"""Recorded outputs of the reference's own sources (oracle/_ref/libcerberus_ref.so) for the inputs the tests feed them.

The compiled reference cannot be rebuilt from this repository, so tests/golden/make_ref_golden.py runs it once on every
input the reference-pinning tests use and stores, per call, a fingerprint of the inputs and the outputs in
tests/golden/ref_v1.npz.  GoldenRef offers the methods of oracle_lib.RefBackend and answers each call with the recorded
outputs of the call whose inputs match; inputs that were never recorded fail the test instead of being guessed.
"""
import ctypes as C
import os
import numpy as np
from cerberus_b200 import abi

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_v1.npz")
FP_RTOL = 1e-11         # of the inputs' absolute sum: inputs rebuilt from the same seeds differ only in the last bits of libm / SIMD results


_ACTIVE = None


def reference():
    """The reference arm of the tests: the recorded outputs (make_ref_golden.py swaps in a recording GoldenRef)."""
    global _ACTIVE
    if _ACTIVE is None:
        _ACTIVE = GoldenRef()
    return _ACTIVE


def _is_ptr(t):
    return issubclass(t, (C._Pointer, C.c_void_p))


def _flat(x):
    """Every numeric input value behind `x` as one float64 vector (pointer fields are followed where they carry data)."""
    parts = [np.zeros(0)]
    if isinstance(x, abi.WindowBatch):
        for w in range(x.n):
            d = x.descs[w]
            pn = d.prior.n if d.prior.valid else 0
            pre = x.preint[w] if x.imu_preint is None else x.imu_preint[w]
            parts += [_flat(v) for v in (d, x.features[w][:d.n_features], x.obs[w][:d.n_obs], pre, x.prior_J[w][:pn * pn],
                                         x.prior_r[w][:pn], x.states[w], x.para_Feature[w][:d.n_features])]
    elif isinstance(x, np.ndarray):
        if x.dtype.names:
            parts += [_flat(x[k]) for k in x.dtype.names]
        else:
            parts.append(x.astype(np.float64).ravel())
    elif isinstance(x, C.Structure):
        parts += [_flat(getattr(x, k)) for k, t in x._fields_ if not _is_ptr(t)]
        if isinstance(x, abi.PreintJob):
            n = x.n_samples * C.sizeof(abi.IMULegSample) // 8
            parts.append(np.ctypeslib.as_array(C.cast(x.samples, C.POINTER(C.c_double)), shape=(n,)).copy())
        elif isinstance(x, abi.Prior) and x.valid:
            parts.append(np.ctypeslib.as_array(x.linearized_jacobians, shape=(x.n * x.n,)).copy())
            parts.append(np.ctypeslib.as_array(x.linearized_residuals, shape=(x.n,)).copy())
    elif isinstance(x, (C.Array, list, tuple)):
        parts += [_flat(e) for e in x]
    else:
        parts.append(np.array([float(x)]))
    return np.concatenate(parts)


def fingerprint(*args):
    f = np.nan_to_num(np.concatenate([_flat(a) for a in args]))
    w = (np.arange(f.size) * 0.6180339887498949) % 1.0
    return np.array([f.size, f.sum(), np.abs(f).sum(), (f * w).sum()])


class GoldenRef:
    """RefBackend's methods answered from tests/golden/ref_v1.npz; with `live` (a RefBackend) the calls run the compiled
    reference and are recorded for save()."""

    def __init__(self, live=None):
        self.live = live
        self.calls = {}
        if live is None:
            g = np.load(GOLDEN, allow_pickle=False)
            for key in g.files:
                method, k, item = key.rsplit(".", 2)
                rec = self.calls.setdefault(method, {}).setdefault(int(k), {})
                rec[item] = g[key]
            self.calls = {m: [(r["fp"], [r[str(i)] for i in range(len(r) - 1)]) for _, r in sorted(recs.items())] for m, recs in self.calls.items()}

    def save(self, path=GOLDEN):
        out = {}
        for method, recs in self.calls.items():
            for k, (fp, outs) in enumerate(recs):
                out[f"{method}.{k}.fp"] = fp
                for i, a in enumerate(outs):
                    out[f"{method}.{k}.{i}"] = a
        np.savez_compressed(path, **out)

    def _find(self, method, fp):
        for rec_fp, outs in self.calls.get(method, []):
            if rec_fp[0] == fp[0] and (np.abs(rec_fp - fp) <= FP_RTOL * max(1.0, rec_fp[2])).all():
                return outs
        return None

    def _call(self, method, inputs, run):
        """`run()` computes the outputs with the live reference (a list of arrays); replay returns the recorded list."""
        fp = fingerprint(*inputs)
        outs = self._find(method, fp)
        if self.live is None:
            assert outs is not None, f"no recorded reference output of {method} for these inputs: regenerate {GOLDEN} with tests/golden/make_ref_golden.py"
            return [a.copy() for a in outs]
        if outs is None:
            outs = [np.array(a) for a in run()]
            self.calls.setdefault(method, []).append((fp, outs))
        return [a.copy() for a in outs]

    # ---- the methods of RefBackend -------------------------------------------------------------------------------
    def a1_kinematics(self, q, rho_opt, rho_fix):
        return tuple(self._call("a1_kinematics", (q, rho_opt, rho_fix), lambda: self.live.a1_kinematics(q, rho_opt, rho_fix)))

    def eval_projection(self, kind, *args):
        return tuple(self._call(f"eval_projection{kind}", args, lambda: self.live.eval_projection(kind, *args)))

    def eval_imu_leg(self, preint, params):
        return tuple(self._call("eval_imu_leg", (preint, params), lambda: self.live.eval_imu_leg(preint, params)))

    def eval_imu(self, preint, params):
        return tuple(self._call("eval_imu", (preint, params), lambda: self.live.eval_imu(preint, params)))

    def preintegrate(self, pcfg, jobs, n):
        return self._call("preintegrate", (pcfg, jobs[:n]), lambda: [self.live.preintegrate(pcfg, jobs, n)])[0]

    def preintegrate_imu(self, pcfg, jobs, n):
        return self._call("preintegrate_imu", (pcfg, jobs[:n]), lambda: [self.live.preintegrate_imu(pcfg, jobs, n)])[0]

    def pose_plus(self, x, delta):
        return self._call("pose_plus", (x, delta), lambda: [self.live.pose_plus(x, delta)])[0]

    def eval_prior(self, prior, state, n_cols):
        return tuple(self._call("eval_prior", (prior, state, n_cols), lambda: self.live.eval_prior(prior, state, n_cols)))

    def double2vector(self, before_state, after_state):
        return tuple(self._call("double2vector", (before_state, after_state), lambda: self.live.double2vector(before_state, after_state)))

    def triangulate(self, batch, init_depth=5.0):
        return self._call("triangulate", (batch, init_depth), lambda: [self.live.triangulate(batch, init_depth)])[0]

    def outlier_errors(self, batch):
        return self._call("outlier_errors", (batch,), lambda: [self.live.outlier_errors(batch)])[0]

    def shift_depth(self, batch, init_depth=5.0):
        return tuple(self._call("shift_depth", (batch, init_depth), lambda: self.live.shift_depth(batch, init_depth)))

    def marginalize(self, cfg, src, dst, margin_old=True):
        """Writes the new prior of every window into dst (descriptor, linearized_jacobians, linearized_residuals)."""
        flags = np.broadcast_to(np.asarray(margin_old, dtype=bool), (src.n,)).astype(np.float64)

        def run():
            self.live.marginalize(cfg, src, dst, margin_old)
            outs = []
            for w in range(src.n):
                pr = dst.descs[w].prior
                # J and r in float32: a prior is compared through J^T J and J^T r at 1e-5 / 1e-4 of their largest entry
                outs += [np.frombuffer(bytes(pr), dtype=np.uint8).copy(), dst.prior_J[w][:pr.n * pr.n].astype(np.float32),
                         dst.prior_r[w][:pr.n].astype(np.float32)]
            return outs
        outs = self._call("marginalize", (src, flags), run)
        for w in range(src.n):
            raw, J, r = outs[3 * w:3 * w + 3]
            pr = dst.descs[w].prior
            C.memmove(C.byref(pr), raw.ctypes.data, C.sizeof(abi.Prior))
            pr.linearized_jacobians = dst.prior_J[w].ctypes.data_as(abi.c_dp)
            pr.linearized_residuals = dst.prior_r[w].ctypes.data_as(abi.c_dp)
            dst.prior_J[w][:J.size] = J
            dst.prior_r[w][:r.size] = r
