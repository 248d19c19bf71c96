"""Pins the CPU oracle (and, on the GPU tier, the sm_100a kernels) against the REFERENCE'S OWN SOURCES.

oracle/_ref/libcerberus_ref.so is built by `make -C oracle ref` from the reference's files (A1Kinematics.cpp, utility.cpp,
pose_local_parameterization.cpp, the three projection factors, imu_leg_integration_base.cpp, imu_leg_factor.cpp,
marginalization_factor.cpp) against the header shims of oracle/shim, because Eigen / Ceres / ROS are not available.
Its outputs for the inputs below are recorded in tests/golden/ref_v1.npz (tests/golden/make_ref_golden.py) and
replayed by ref_golden.GoldenRef, so the comparison runs wherever the repository does.  Every formula statement that
produced them is the reference's; the dense linear-algebra primitives underneath are the shim's.  The solver
(ceres-solver 1.14) is third party and absent, so the trust-region loop itself stays pinned by the oracle restatement only."""
import numpy as np
import pytest
from cerberus_b200 import abi, synth
from oracle_lib import OracleBackend
from ref_golden import reference
from test_oracle_jacobians import proj_inputs, imu_leg_setup
from test_preintegration import make_jobs

ob = OracleBackend()
N_PROJ = 200


@pytest.fixture(scope="module")
def ref():
    return reference()


def test_kinematics_vs_reference(ref):
    rng = np.random.default_rng(0); n = 200
    q = rng.uniform(-1.5, 1.5, (n, 3)); lc = rng.uniform(0.15, 0.25, n)
    fix = np.tile([0.1805, 0.047, 0.0838, 0.21], (n, 1)) * rng.choice([-1.0, 1.0], (n, 4)); fix[:, 3] = 0.21
    for a, b in zip(ob.a1_kinematics(q, lc, fix), ref.a1_kinematics(q, lc, fix)):
        assert np.abs(a - b).max() < 1e-15


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_projection_factors_vs_reference(ref, kind):
    args = proj_inputs(np.random.default_rng(40 + kind), N_PROJ)
    r0, j0 = ref.eval_projection(kind, *args)
    r1, j1 = ob.eval_projection(kind, *args)
    assert np.abs(r0 - r1).max() < 1e-10 * max(1.0, np.abs(r0).max())
    assert np.abs(j0 - j1).max() < 1e-11 * np.abs(j0).max()


def test_imu_leg_factor_vs_reference(ref):
    pre, params = imu_leg_setup(4)
    r0, j0, s0 = ref.eval_imu_leg(pre, params)
    r1, j1, s1 = ob.eval_imu_leg(pre, params)
    assert np.abs(s0 - s1).max() < 1e-9 * np.abs(s0).max()
    assert np.abs(r0 - r1).max() < 1e-9 * np.abs(r0).max()
    assert np.abs(j0 - j1).max() < 1e-9 * np.abs(j0).max()


@pytest.mark.parametrize("contact_type", [0, 2])
def test_preintegration_vs_reference(ref, contact_type):
    jobs, _, _ = make_jobs(4, seed=17, contact_type=contact_type)
    pcfg = abi.default_preint_config(); pcfg.contact_sensor_type = contact_type
    a = ref.preintegrate(pcfg, jobs, 4); b = ob.preintegrate(pcfg, jobs, 4)
    for name in a.dtype.names:
        assert np.abs(a[name] - b[name]).max() <= 1e-12 * max(1e-30, np.abs(a[name]).max()), name


def test_pose_plus_and_prior_vs_reference(ref):
    from oracle_lib import lib as olib
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.normal(0, 1, 3), rng.normal(0, 1, 4)]); x[3:] /= np.linalg.norm(x[3:])
    d = rng.normal(0, 0.1, 6)
    got = ref.pose_plus(x, d)
    # independent statement: p + dp ; q (x) [1, dtheta/2] normalised
    qx, qy, qz, qw = x[3:]; dx, dy, dz, dw = d[3] / 2, d[4] / 2, d[5] / 2, 1.0
    q = np.array([qw * dx + qx * dw + qy * dz - qz * dy, qw * dy + qy * dw + qz * dx - qx * dz, qw * dz + qz * dw + qx * dy - qy * dx, qw * dw - qx * dx - qy * dy - qz * dz])
    assert np.abs(got[:3] - (x[:3] + d[:3])).max() < 1e-15 and np.abs(got[3:] - q / np.linalg.norm(q)).max() < 1e-15
    batch, pr, ncols = prior_probe()
    r0, j0 = ref.eval_prior(pr, batch.states[0], ncols); r1, j1 = ob.eval_prior(pr, batch.states[0], ncols)
    assert np.abs(r0 - r1).max() < 1e-10 * np.abs(r0).max() and np.abs(j0 - j1).max() == 0.0


@pytest.mark.gpu
def test_gpu_kernels_vs_reference_sources(ref):
    """The sm_100a evaluators and the device preintegration directly against the compiled reference sources (the inputs of the
    CPU-tier tests above, whose reference outputs are recorded)."""
    from cerberus_b200 import lib
    cfg = abi.default_config(); cfg.max_batch, cfg.max_features, cfg.max_obs = 8, 32, 32 * 11
    gpu = lib.Backend(cfg)
    for kind in range(3):
        args = proj_inputs(np.random.default_rng(40 + kind), N_PROJ)
        r0, j0 = ref.eval_projection(kind, *args); r1, j1 = gpu.eval_projection(kind, *args)
        assert np.abs(r0 - r1).max() < 1e-9 * max(1.0, np.abs(r0).max()) and np.abs(j0 - j1).max() < 1e-10 * np.abs(j0).max()
    pre, params = imu_leg_setup(4)
    r0, j0, s0 = ref.eval_imu_leg(pre, params); r1, j1, s1 = gpu.eval_imu_leg(pre, params)
    assert np.abs(s0 - s1).max() < 1e-9 * np.abs(s0).max() and np.abs(r0 - r1).max() < 1e-9 * np.abs(r0).max() and np.abs(j0 - j1).max() < 1e-9 * np.abs(j0).max()
    jobs, _, _ = make_jobs(4, seed=17)
    pcfg = abi.default_preint_config()
    a = ref.preintegrate(pcfg, jobs, 4); b = gpu.preintegrate(pcfg, jobs, 4)
    for name in a.dtype.names:
        assert np.abs(a[name] - b[name]).max() <= 1e-11 * max(1e-30, np.abs(a[name]).max()), name


@pytest.mark.parametrize("realistic", [False, True])
def test_marginalization_vs_reference(ref, realistic):
    """MARGIN_OLD with the reference's own MarginalizationInfo::{preMarginalize, marginalize} and ResidualBlockInfo::Evaluate
    (marginalization_factor.cpp:12-333) vs the oracle restatement and vs the product's numpy glue over the kernel evaluators."""
    from helpers import prior_canonical, sim_backend, small_cfg
    cfg = small_cfg()
    mk = lambda: synth.generate_batch(2, 10, ob, realistic=realistic, with_prior=False, window0=31)
    src = mk()
    if realistic:
        src.features[:, :4]["start_frame"] = 0
    a, b, c = mk(), mk(), mk()
    ref.marginalize(cfg, src, a); ob.marginalize(cfg, src, b); sim_backend(cfg).marginalize(cfg, src, c)
    for w in range(2):
        A0, b0, x0 = prior_canonical(a, w)
        for other in (b, c):
            A1, b1, x1 = prior_canonical(other, w)
            assert A0.shape == A1.shape and set(x0) == set(x1)
            assert np.abs(A0 - A1).max() < 1e-5 * np.abs(A0).max() and np.abs(b0 - b1).max() < 1e-4 * np.abs(b0).max()
            assert all(np.abs(x0[k][:7] - x1[k][:7]).max() == 0 for k in x0)


def prior_probe():
    """A window with a prior, its states moved away from the linearization point: (batch, prior, Jacobian columns)."""
    batch = synth.generate_batch(1, 8, ob, prior_features=6)
    st = batch.state_array()
    st["para_Pose"][0, :, :3] += 0.02; st["para_SpeedBias"][0, 0] += 0.01; st["para_LegBias"][0, 0] += 1e-3
    st["para_Pose"][0, :, 3:7] += 0.003; st["para_Pose"][0, :, 3:7] /= np.linalg.norm(st["para_Pose"][0, :, 3:7], axis=-1, keepdims=True)
    st["para_Pose"][0, 2, 3:7] *= -1.0                       # w < 0 branch of the rotation residual (marginalization_factor.cpp:369-375)
    return batch, batch.descs[0].prior, 7 * 12 + 9 + 4 + 1


def imu_setup(n=4, backend=None):
    """IMU-only (USE_LEG == 0) factors of a synthetic window: IntegrationBase results + the 32 parameters."""
    backend = backend or ob
    batch = synth.generate_batch(1, 4, backend, use_leg=False)
    st = batch.state_array()
    pre = batch.imu_preint[0][:n].copy()
    params = np.zeros((n, 32))
    for k in range(n):
        params[k, 0:7] = st["para_Pose"][0, k]; params[k, 7:16] = st["para_SpeedBias"][0, k]
        params[k, 16:23] = st["para_Pose"][0, k + 1]; params[k, 23:32] = st["para_SpeedBias"][0, k + 1]
    params[:, 10:16] += np.random.default_rng(4).normal(0, 1e-3, (n, 6))
    return pre, params


def test_imu_factor_and_preintegration_vs_reference(ref):
    """IMUFactor::Evaluate (imu_factor.h:28-188) and IntegrationBase (integration_base.h:40-198)."""
    jobs, _, _ = make_jobs(5, seed=29)
    pcfg = abi.default_preint_config()
    a = ref.preintegrate_imu(pcfg, jobs, 5); b = ob.preintegrate_imu(pcfg, jobs, 5)
    for name in a.dtype.names:
        assert np.abs(a[name] - b[name]).max() <= 1e-12 * max(1e-30, np.abs(a[name]).max()), name
    pre, params = imu_setup(4)
    r0, j0, s0 = ref.eval_imu(pre, params); r1, j1, s1 = ob.eval_imu(pre, params)
    assert np.abs(s0 - s1).max() < 1e-9 * np.abs(s0).max() and np.abs(r0 - r1).max() < 1e-9 * np.abs(r0).max() and np.abs(j0 - j1).max() < 1e-9 * np.abs(j0).max()


def test_imu_only_kernels_vs_reference_in_simulator(ref):
    from helpers import sim_backend, small_cfg
    sb = sim_backend(small_cfg())
    jobs, _, _ = make_jobs(3, seed=29)
    pcfg = abi.default_preint_config()
    a = ref.preintegrate_imu(pcfg, jobs, 3); b = sb.preintegrate_imu(pcfg, jobs, 3)
    for name in a.dtype.names:
        assert np.abs(a[name] - b[name]).max() <= 1e-11 * max(1e-30, np.abs(a[name]).max()), name
    pre, params = imu_setup(3)
    r0, j0, s0 = ref.eval_imu(pre, params); r1, j1, s1 = sb.eval_imu(pre, params)
    assert np.abs(s0 - s1).max() < 1e-9 * np.abs(s0).max() and np.abs(r0 - r1).max() < 1e-9 * np.abs(r0).max() and np.abs(j0 - j1).max() < 1e-9 * np.abs(j0).max()


@pytest.mark.parametrize("margin_old", [True, False])
def test_marginalization_with_prior_vs_reference(ref, margin_old):
    """Windows that already carry a prior: MARGIN_OLD folds the old MarginalizationFactor in (estimator.cpp:1253-1270),
    MARGIN_SECOND_NEW (estimator.cpp:1377-1455) drops para_Pose[WINDOW_SIZE - 1] from it and keeps the rest; reference classes
    vs oracle restatement vs the product glue (device evaluators + cerb_marginalize_schur in the simulator)."""
    from helpers import prior_canonical, sim_backend, small_cfg
    cfg = small_cfg()
    mk = lambda: synth.generate_batch(2, 10, ob, with_prior=True, window0=47)
    src = mk()
    assert all(src.descs[w].prior.valid for w in range(2))
    a, b, c = mk(), mk(), mk()
    ref.marginalize(cfg, src, a, margin_old); ob.marginalize(cfg, src, b, margin_old); sim_backend(cfg).marginalize(cfg, src, c, margin_old)
    for w in range(2):
        A0, b0, x0 = prior_canonical(a, w)
        assert A0.shape[0] == (86 if margin_old else 80)
        for other in (b, c):
            A1, b1, x1 = prior_canonical(other, w)
            assert A0.shape == A1.shape and set(x0) == set(x1)
            assert np.abs(A0 - A1).max() < 1e-5 * np.abs(A0).max() and np.abs(b0 - b1).max() < 1e-4 * np.abs(b0).max()
            assert all(np.abs(x0[k][:7] - x1[k][:7]).max() == 0 for k in x0)
