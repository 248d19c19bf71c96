"""Parity holes named by the round-1 review, closed (both tiers).

CPU tier (`-m "not gpu"`):
  * cerb_double2vector (the gauge re-anchoring of Estimator::double2vector, estimator.cpp:903-957 -- the function that produces the
    poses the estimator publishes) against the oracle restatement AND against the reference's own Utility::R2ypr / ypr2R
    (utils/utility.cpp compiled into oracle/_ref, outputs recorded in tests/golden/ref_v1.npz), including the singular-pitch
    branch (:925-934);
  * the per-feature steps (triangulate / outlier errors / depth shift) of the oracle and of the kernels (CPU simulator) against
    the reference's own FeatureManager (featureTracker/feature_manager.cpp compiled into oracle/_ref) and the statements of
    Estimator::reprojectionError / outliersRejection executed over it.
GPU tier (`-m gpu`): the sm_100a build of cerb_preintegrate_imu_batch, cerb_eval_imu, cerb_eval_prior, the sum_dt > 10 skipped
factor, MARGIN_SECOND_NEW and marginalization with an old prior, the per-feature steps against the reference sources."""
import ctypes as C
import os
import numpy as np
import pytest
from cerberus_b200 import abi, synth, lib
from oracle_lib import OracleBackend
from ref_golden import reference
from helpers import sim_backend, small_cfg, prior_canonical, state_diffs, SIM_LIB
from test_preintegration import make_jobs

ob = OracleBackend()


# ---------------------------------------------------------------------------------------------------- double2vector
def _Rz(a): return np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1.0]])
def _Ry(a): return np.array([[np.cos(a), 0, np.sin(a)], [0, 1.0, 0], [-np.sin(a), 0, np.cos(a)]])
def _Rx(a): return np.array([[1.0, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])


def _quat(R):
    from cerberus_b200.estimator import R_to_quat
    return R_to_quat(R)


def _d2v_states(rng, pitch_before_deg, pitch_after_deg):
    """(before, after): frame 0 of `before` / `after` have the given pitch; everything else random."""
    before, after = abi.WindowState(), abi.WindowState()
    for st, pitch in ((before, pitch_before_deg), (after, pitch_after_deg)):
        for i in range(abi.NUM_FRAMES):
            y, r = rng.uniform(-np.pi, np.pi), rng.uniform(-0.5, 0.5)
            p = np.deg2rad(pitch) if i == 0 else rng.uniform(-0.6, 0.6)
            q = _quat(_Rz(y) @ _Ry(p) @ _Rx(r)) * (1.0 + (rng.uniform(-1e-9, 1e-9) if st is after else 0.0))   # after: not exactly unit (normalized() matters)
            if rng.uniform() < 0.3: q = -q
            st.para_Pose[i][0:3] = list(rng.normal(0, 3, 3)); st.para_Pose[i][3:7] = list(q)
            st.para_SpeedBias[i][0:9] = list(rng.normal(0, 1, 9))
    return before, after


def _d2v_product(cdll, before, after):
    Ps, Rs, Vs = np.zeros((11, 3)), np.zeros((11, 3, 3)), np.zeros((11, 3))
    cdll.cerb_double2vector.restype = None
    cdll.cerb_double2vector.argtypes = [C.POINTER(abi.WindowState), C.POINTER(abi.WindowState), abi.c_dp, abi.c_dp, abi.c_dp]
    cdll.cerb_double2vector(C.byref(before), C.byref(after), Ps.ctypes.data_as(abi.c_dp), Rs.ctypes.data_as(abi.c_dp), Vs.ctypes.data_as(abi.c_dp))
    return Ps, Rs, Vs


D2V_PITCHES = [(5.0, -7.0), (30.0, 29.0), (-45.0, -44.0), (89.6, 20.0), (10.0, -89.3), (-89.9, -89.9), (88.9, 88.9), (91.0 - 2.0, 40.0)]


def _check_d2v(cdll):
    rng = np.random.default_rng(12)
    ref = reference()
    singular = 0
    for (pb, pa) in D2V_PITCHES * 3:
        before, after = _d2v_states(rng, pb, pa)
        got = _d2v_product(cdll, before, after)
        for arm in (ob, ref):
            want = arm.double2vector(before, after)
            for g, w, name in zip(got, want, ("Ps", "Rs", "Vs")):
                assert np.abs(g - w).max() < 1e-12 * max(1.0, np.abs(w).max()), (name, pb, pa, type(arm).__name__)
        # the property the step exists for: frame 0 keeps its position and its yaw
        assert np.abs(got[0][0] - np.array(before.para_Pose[0][0:3])).max() < 1e-12
        if abs(abs(pb) - 90) < 1.0 or abs(abs(pa) - 90) < 1.0:
            singular += 1
            from cerberus_b200.estimator import quat_to_R
            assert np.abs(got[1][0] - quat_to_R(np.array(before.para_Pose[0][3:7]))).max() < 1e-7      # rot_diff = Rs0 R00^T (R00 from the un-normalised quaternion, as in the reference)
    assert singular >= 9


def test_double2vector_sim_build_vs_oracle_and_reference():
    _check_d2v(C.CDLL(SIM_LIB) if os.path.exists(SIM_LIB) else sim_backend(small_cfg()).lib)


def test_double2vector_product_library_vs_oracle_and_reference():
    """The sm_100a library's host-side cerb_double2vector (no device involved: callable without a GPU)."""
    if not os.path.exists(lib.PRODUCT_LIB):
        pytest.skip("product library not built")
    try:
        cdll = C.CDLL(lib.PRODUCT_LIB)
    except OSError as e:       # libcudart missing on this machine
        pytest.skip(str(e))
    _check_d2v(cdll)


# ---------------------------------------------------------------------------------------------------- n3 against reference source
def _feature_steps_vs_reference(be, ref, realistic):
    """The kernels' outlier errors, depth shift and triangulation against the reference's FeatureManager on fixed inputs: the initial
    states, the states the oracle solves to, and the latter with every second feature not triangulated (estimated_depth = -1)."""
    from test_feature_steps import _batch
    batch = _batch(ob, realistic)
    nf = [batch.descs[w].n_features for w in range(batch.n)]
    for phase in range(3):
        if phase == 1:
            OracleBackend(small_cfg(max_batch=4, max_features=24, iters=3)).solve_batch(batch)
        if phase == 2:
            for w in range(batch.n):
                batch.para_Feature[w, 0:nf[w]:2] = -1.0
        be.upload(batch)
        err, rem = be.outlier_errors(batch.n); e_ref = ref.outlier_errors(batch)
        st_g, dep_g, keep_g = be.shift_depth(batch.n, 7.5); st_r, dep_r, keep_r = ref.shift_depth(batch, 7.5)
        dep = be.triangulate(batch.n); t_ref = ref.triangulate(batch)
        for w in range(batch.n):
            k = nf[w]
            if phase < 2:
                ok = np.isfinite(e_ref[w, :k])       # the reference skips used_num < 4 (estimator.cpp:1750)
                assert ok.sum() >= k - 1 and np.abs(err[w, :k][ok] - e_ref[w, :k][ok]).max() < 1e-12 * max(1.0, np.abs(e_ref[w, :k][ok]).max())
                assert (rem[w, :k][ok] == (e_ref[w, :k][ok] * 460.0 > 3)).all()
            kp = keep_r[w, :k] != 0
            assert (keep_g[w, :k] == keep_r[w, :k]).all() and (st_g[w, :k][kp] == st_r[w, :k][kp]).all()
            assert np.abs(dep_g[w, :k][kp] - dep_r[w, :k][kp]).max() < 1e-12 * np.abs(dep_r[w, :k][kp]).max()
            assert np.abs(dep[w, :k] - t_ref[w, :k]).max() < 1e-8 * np.abs(t_ref[w, :k]).max()


@pytest.mark.parametrize("realistic", [False, True])
def test_feature_steps_oracle_and_sim_vs_reference_feature_manager(realistic):
    """FeatureManager::{triangulate, triangulatePoint, removeBackShiftDepth} (feature_manager.cpp:198-212,302-385,450-488) and the
    statements of Estimator::{reprojectionError, outliersRejection} (estimator.cpp:1729-1798) executed from the reference's source."""
    from test_feature_steps import _batch
    cfg = small_cfg(max_batch=4, max_features=24, iters=3)
    ref = reference()
    # oracle restatement vs reference source
    batch = _batch(ob, realistic)
    nf = [batch.descs[w].n_features for w in range(batch.n)]
    for lamset in (0, 1):
        if lamset:
            for w in range(batch.n):
                batch.para_Feature[w, 0:nf[w]:2] = -1.0
        e0, e1 = ob.outlier_errors(batch), ref.outlier_errors(batch)
        t0, t1 = ob.triangulate(batch), ref.triangulate(batch)
        s0, s1 = ob.shift_depth(batch, 6.5), ref.shift_depth(batch, 6.5)
        for w in range(batch.n):
            k = nf[w]
            if not lamset:
                ok = np.isfinite(e1[w, :k])         # the reference skips used_num < 4 (estimator.cpp:1750)
                assert ok.sum() >= k - 1 and np.abs(e0[w, :k][ok] - e1[w, :k][ok]).max() < 1e-12 * max(1.0, np.abs(e1[w, :k][ok]).max())
            assert np.abs(t0[w, :k] - t1[w, :k]).max() < 1e-8 * np.abs(t1[w, :k]).max()
            keep = s1[2][w, :k] != 0
            assert (s0[0][w, :k][keep] == s1[0][w, :k][keep]).all() and (s0[2][w, :k] == s1[2][w, :k]).all()
            assert np.abs(s0[1][w, :k][keep] - s1[1][w, :k][keep]).max() < 1e-12 * np.abs(s1[1][w, :k][keep]).max()
    # kernels (CPU simulator) vs reference source; the simulator against the oracle through the whole sequence: test_feature_steps.py
    _feature_steps_vs_reference(sim_backend(cfg), ref, realistic)


# ---------------------------------------------------------------------------------------------------- GPU tier
def _gpu(cfg=None):
    return lib.Backend(cfg or small_cfg(max_batch=8, max_features=32))


@pytest.mark.gpu
def test_double2vector_product_library_gpu_box():
    _check_d2v(_gpu().lib)


@pytest.mark.gpu
def test_imu_preintegration_and_imu_factor_gpu():
    """Row a9 / a6 on the sm_100a build: cerb_preintegrate_imu_batch and cerb_eval_imu vs the oracle and the reference's
    integration_base.h / imu_factor.h (oracle/_ref)."""
    from test_reference_pin import imu_setup
    gpu = _gpu()
    arms = [ob, reference()]
    jobs, _, _ = make_jobs(6, seed=29)
    pcfg = abi.default_preint_config()
    got = gpu.preintegrate_imu(pcfg, jobs, 6)
    for arm in arms:
        want = arm.preintegrate_imu(pcfg, jobs, 6)
        for name in want.dtype.names:
            assert np.abs(got[name] - want[name]).max() <= 1e-11 * max(1e-30, np.abs(want[name]).max()), (name, type(arm).__name__)
    pre, params = imu_setup(4)
    r1, j1, s1 = gpu.eval_imu(pre, params)
    for arm in arms:
        r0, j0, s0 = arm.eval_imu(pre, params)
        assert np.abs(s0 - s1).max() < 1e-9 * np.abs(s0).max() and np.abs(r0 - r1).max() < 1e-9 * np.abs(r0).max() and np.abs(j0 - j1).max() < 1e-9 * np.abs(j0).max()
    # the windows a USE_LEG == 0 estimator would solve, fed by the DEVICE preintegration on one arm and the oracle's on the other
    cfg = small_cfg(max_batch=4, max_features=32)
    g2, o2 = lib.Backend(cfg), OracleBackend(cfg)
    bg = synth.generate_batch(2, 24, g2, use_leg=False, window0=310)
    bo = synth.generate_batch(2, 24, o2, use_leg=False, window0=310)
    for name in bo.imu_preint.dtype.names:
        assert np.abs(bg.imu_preint[name] - bo.imu_preint[name]).max() <= 1e-11 * max(1e-30, np.abs(bo.imu_preint[name]).max()), name
    rep_g = g2.solve_batch(bg); rep_o = o2.solve_batch(bo)
    assert (rep_g["iterations"] == rep_o["iterations"]).all()
    assert state_diffs(bg.state_array(), bo.state_array())["para_Pose"] < 1e-6


@pytest.mark.gpu
def test_prior_evaluator_gpu():
    """cerb_eval_prior (MarginalizationFactor::Evaluate, marginalization_factor.cpp:347-395) on the device vs oracle and reference."""
    from test_reference_pin import prior_probe
    gpu = _gpu()
    batch, pr, ncols = prior_probe()
    r1, j1 = gpu.eval_prior(pr, batch.states[0], ncols)
    for arm in (ob, reference()):
        r0, j0 = arm.eval_prior(pr, batch.states[0], ncols)
        assert np.abs(r0 - r1).max() < 1e-10 * np.abs(r0).max() and np.abs(j0 - j1).max() == 0.0


@pytest.mark.gpu
def test_skipped_imu_factor_gpu():
    """estimator.cpp:1119 (sum_dt > 10: factor not added) on the sm_100a build."""
    cfg = small_cfg(max_batch=4, max_features=32, iters=6)
    o, g = OracleBackend(cfg), lib.Backend(cfg)
    batch = synth.generate_batch(3, 24, o, window0=31, prior_features=8)
    batch.preint[0][3]["sum_dt"] = 10.5
    batch.preint[1][0]["sum_dt"] = 12.0; batch.preint[1][9]["sum_dt"] = 11.0
    st = batch.state_array(); saved = batch.copy_states()
    rep_o = o.solve_batch(batch); ref = st.copy(); lam = batch.para_Feature.copy()
    batch.restore_states(saved)
    rep_g = g.solve_batch(batch)
    assert (rep_o["iterations"] == rep_g["iterations"]).all() and (rep_o["num_successful_steps"] == rep_g["num_successful_steps"]).all()
    assert np.abs(rep_o["final_cost"] - rep_g["final_cost"]).max() < 1e-7 * rep_o["final_cost"].max()
    d = state_diffs(batch.state_array(), ref)
    assert d["para_Pose"] < 1e-6 and d["para_SpeedBias"] < 1e-5 and np.abs(batch.para_Feature - lam).max() < 1e-6, d


@pytest.mark.gpu
@pytest.mark.parametrize("margin_old", [True, False])
def test_marginalization_with_prior_gpu(margin_old):
    """MARGIN_OLD with an existing prior and MARGIN_SECOND_NEW on the sm_100a build vs the reference's MarginalizationInfo classes and the oracle."""
    cfg = small_cfg()
    gpu = lib.Backend(cfg)
    mk = lambda: synth.generate_batch(2, 10, ob, with_prior=True, window0=47)
    src = mk()
    arms = [ob, reference()]
    c = mk(); gpu.marginalize(cfg, src, c, margin_old)
    for arm in arms:
        a = mk(); arm.marginalize(cfg, src, a, margin_old)
        for w in range(2):
            A0, b0, x0 = prior_canonical(a, w); A1, b1, x1 = prior_canonical(c, w)
            assert A0.shape[0] == (86 if margin_old else 80) and A0.shape == A1.shape and set(x0) == set(x1)
            assert np.abs(A0 - A1).max() < 1e-5 * np.abs(A0).max() and np.abs(b0 - b1).max() < 1e-4 * np.abs(b0).max()
            assert all(np.abs(x0[k][:7] - x1[k][:7]).max() == 0 for k in x0)


@pytest.mark.gpu
@pytest.mark.parametrize("realistic", [False, True])
def test_feature_steps_gpu_vs_reference_feature_manager(realistic):
    cfg = small_cfg(max_batch=4, max_features=24, iters=4)
    _feature_steps_vs_reference(lib.Backend(cfg), reference(), realistic)


@pytest.mark.gpu
def test_stress_feature_count_gpu():
    """BASELINE.json configs[4]: 10-frame x 2000-feature windows (dense Schur: 32 chunks of tracks, 63 Schur tiles, the inverse-depth scales in the
    global workspace instead of shared memory).  Exceeds the reference's static NUM_OF_F = 1000 (parameters.h:24) on purpose; parity vs the oracle."""
    cfg = abi.default_config()
    cfg.max_batch, cfg.max_features, cfg.max_obs = 2, 2000, 2000 * 11
    big = lib.Backend(cfg)
    o = OracleBackend(cfg)
    batch = synth.generate_batch(2, 2000, big, cfg=cfg, window0=4000, prior_features=16)
    st = batch.state_array(); saved = batch.copy_states()
    rep_o = o.solve_batch(batch, nthreads=2); ref = st.copy(); lam = batch.para_Feature.copy()
    batch.restore_states(saved)
    rep_g = big.solve_batch(batch)
    assert (rep_o["iterations"] == rep_g["iterations"]).all() and (rep_o["num_successful_steps"] == rep_g["num_successful_steps"]).all()
    d = state_diffs(batch.state_array(), ref)
    assert d["para_Pose"] < 1e-6 and d["para_SpeedBias"] < 1e-5 and np.abs(batch.para_Feature - lam).max() < 1e-6, d
    # over the capacity limit of the library
    cfg2 = abi.default_config(); cfg2.max_batch, cfg2.max_features, cfg2.max_obs = 1, 2049, 2049 * 11
    with pytest.raises(lib.CerbError):
        lib.Backend(cfg2)
