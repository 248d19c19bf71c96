"""Record the reference's outputs for every input the reference-pinning tests feed it: tests/golden/ref_v1.npz.

Needs oracle/_ref/libcerberus_ref.so, which `make -C oracle ref` compiles from the reference's own sources.  Every test that
consults the reference is run once against those compiled sources through a recording ref_golden.GoldenRef; the GPU-tier
ones run on the CPU kernel simulator, which gives them the same reference inputs.  Re-run:  python tests/golden/make_ref_golden.py
"""
import inspect
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from cerberus_b200 import lib                  # noqa: E402
import ref_golden                              # noqa: E402
from helpers import SIM_LIB                    # noqa: E402
from oracle_lib import RefBackend              # noqa: E402

PARITY_TESTS = ("test_double2vector_sim_build_vs_oracle_and_reference", "test_feature_steps_oracle_and_sim_vs_reference_feature_manager",
                "test_imu_preintegration_and_imu_factor_gpu", "test_prior_evaluator_gpu", "test_marginalization_with_prior_gpu",
                "test_feature_steps_gpu_vs_reference_feature_manager")


def run(fn, ref):
    """fn once per parameter set of its (single) parametrize mark, with the `ref` fixture where it takes one."""
    kwargs = {"ref": ref} if "ref" in inspect.signature(fn).parameters else {}
    marks = [m for m in getattr(fn, "pytestmark", []) if m.name == "parametrize"]
    if not marks:
        fn(**kwargs)
    for m in marks:
        for value in m.args[1]:
            fn(**kwargs, **{m.args[0]: value})


def main():
    rec = ref_golden._ACTIVE = ref_golden.GoldenRef(live=RefBackend())
    backend = lib.Backend
    lib.Backend = lambda cfg=None, lib_path=None: backend(cfg, lib_path=SIM_LIB)
    import test_reference_pin
    import test_parity_r2
    names = [n for n in dir(test_reference_pin) if n.startswith("test_")] + list(PARITY_TESTS)
    for name in names:
        mod = test_reference_pin if hasattr(test_reference_pin, name) else test_parity_r2
        run(getattr(mod, name), rec)
        print("recorded", name)
    rec.save()
    print("wrote", ref_golden.GOLDEN, os.path.getsize(ref_golden.GOLDEN), "bytes")


if __name__ == "__main__":
    main()
