"""The C-ABI library loads, exports every symbol include/cerberus_b200.h declares and fails loudly without CUDA."""
import ctypes as C
import os
import re
import subprocess
import pytest
from cerberus_b200 import abi, lib
from helpers import ROOT, SIM_LIB, sim_backend


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "cerberus_b200.h")).read()
    return sorted(set(re.findall(r"\b(cerb_[a-z0-9_]+)\s*\(", hdr)))


def ensure_product_lib():
    if not os.path.exists(lib.PRODUCT_LIB):
        subprocess.check_call(["make", "-s", "-C", ROOT, "lib"])


def test_header_declares_expected_entry_points():
    syms = declared_symbols()
    for s in ("cerb_create", "cerb_destroy", "cerb_solve_window", "cerb_solve_batch", "cerb_batch_upload", "cerb_batch_solve_resident",
              "cerb_batch_download", "cerb_eval_projection", "cerb_eval_imu_leg", "cerb_eval_prior", "cerb_preintegrate_batch",
              "cerb_a1_kinematics", "cerb_double2vector", "cerb_last_error", "cerb_batch_outlier_errors", "cerb_batch_triangulate", "cerb_batch_shift_depth", "cerb_marginalize_schur"):
        assert s in syms


@pytest.mark.parametrize("which", ["product", "sim"])
def test_library_exports_every_declared_symbol(which):
    if which == "product":
        ensure_product_lib()
        path = lib.PRODUCT_LIB
    else:
        sim_backend(None).close()
        path = SIM_LIB
    L = C.CDLL(path)
    for s in declared_symbols():
        assert hasattr(L, s), f"{path} does not export {s}"


def test_struct_sizes_match_the_c_header():
    from oracle_lib import lib as oracle_lib   # compiled against include/cerberus_b200.h; asserts sizes on load
    oracle_lib()


def test_product_sass_is_sm100a_with_fp64_tensor_core_mma():
    ensure_product_lib()
    out = subprocess.run(["cuobjdump", "-lelf", lib.PRODUCT_LIB], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", lib.PRODUCT_LIB], capture_output=True, text=True).stdout
    assert "DMMA" in sass     # mma.sync m8n8k4 f64 of the Gram accumulation


def test_no_cpu_fallback_without_cuda():
    """On a box without a GPU the product library must refuse to create a handle (CERB_ERR_NO_DEVICE)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    ensure_product_lib()
    with pytest.raises(lib.CerbError) as e:
        lib.Backend(abi.default_config())
    assert e.value.code in (abi.ERR_NO_DEVICE, abi.ERR_CUDA)


def test_bad_descriptors_are_rejected():
    from cerberus_b200 import synth
    from oracle_lib import OracleBackend
    from helpers import small_cfg
    cfg = small_cfg()
    sb = sim_backend(cfg)
    batch = synth.generate_batch(1, 6, OracleBackend(cfg), with_prior=False)
    batch.descs[0].n_features = cfg.max_features + 1
    with pytest.raises(lib.CerbError) as e:
        sb.solve_batch(batch)
    assert e.value.code == abi.ERR_BAD_ARGUMENT
    batch.descs[0].n_features = 6
    batch.features[0][2]["n_obs"] = 40
    with pytest.raises(lib.CerbError):
        sb.solve_batch(batch)


def test_integration_stub_compiles_against_the_header_and_reference_headers():
    """tools/integration_stub.cpp (the reference-side binding of INTEGRATION.md) type-checks as C++14 against include/cerberus_b200.h, the
    reference's own headers (where `make -C oracle ref` finds the reference's sources: oracle/Makefile's REF; the repository does not carry
    them) and the Eigen / ROS / OpenCV shims of oracle/shim; the header alone also compiles as plain C."""
    hdr_c = subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-x", "c", os.path.join(ROOT, "include", "cerberus_b200.h")], capture_output=True, text=True)
    assert hdr_c.returncode == 0, hdr_c.stderr
    r = subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "stub-check"], capture_output=True, text=True)
    if "reference sources not present" in r.stdout:
        pytest.skip("the reference's sources are not present (oracle/Makefile REF)")
    assert r.returncode == 0, r.stderr[-3000:]


def test_update_states_and_schur_argument_checks():
    """cerb_batch_update_states needs a resident batch of exactly n windows; cerb_marginalize_schur bounds m by what a window can drop"""
    import numpy as np
    from cerberus_b200 import synth
    from oracle_lib import OracleBackend
    from helpers import small_cfg
    cfg = small_cfg()
    sb = sim_backend(cfg)
    batch = synth.generate_batch(2, 6, OracleBackend(cfg), with_prior=False)
    with pytest.raises(lib.CerbError) as e:
        sb.update_states(batch)                          # nothing resident yet
    assert e.value.code == abi.ERR_BAD_ARGUMENT
    sb.upload(batch)
    one = synth.tile_batch(batch, 1)
    with pytest.raises(lib.CerbError) as e:
        sb.update_states(one)                            # wrong window count
    assert e.value.code == abi.ERR_BAD_ARGUMENT
    sb.update_states(batch)
    A = np.eye(8)[None]; b = np.zeros((1, 8))
    with pytest.raises(lib.CerbError):
        sb.marginalize_schur(np.eye(2100 + 4)[None], np.zeros((1, 2104)), 2100)       # m > 19 + CERB_MAX_FEATURES
    J, r = sb.marginalize_schur(A, b, 3)
    assert J.shape == (1, 5, 5)
