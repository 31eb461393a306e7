"""Shared by the NGCF kernel-by-kernel tests (test_ngcf_dense_kernels.py, test_ngcf_step_kernels.py): the float64
reference of one layer's dense transforms, the per-element bounds and checks, the launch grids the bounds depend on, the
per-module summary of error / bound ratios, and the ctypes helpers the GPU tests call the library with. The derivation of
the dense-transform bounds is in test_ngcf_dense_kernels.py's docstring."""
import ctypes as C
import math
from functools import lru_cache

import numpy as np
import torch

U23, U24 = 2.0 ** -23, 2.0 ** -24
SPLIT = 3 * 2.0 ** -20
SLOPES = (0.01, 0.2, 0.0)
FP32_TM = {32: 128, 64: 64, 128: 32}        # rows per tile of the FP32-pipe kernels (csrc/ngcf.cu, DenseCfg<D>::TM)
TC_TM = 128
SENTINEL = np.uint32(0x7FBADBAD)             # a NaN payload no kernel produces: output rows a call must not touch
YR_OK, YR_ERR_BAD_ARG, YR_ERR_BAD_DIM, YR_ERR_WORKSPACE = 0, 1000, 1001, 1003


def tau_fwd(d, tc):
    return SPLIT + 2 * d * (1 + 2.0 ** -8) * U23 + U24 if tc else 2 * d * U24


def tau_rows(d, tc):
    return SPLIT + 3 * d * U23 + 2 * U24 if tc else (d + 2) * U24


def bwd_grid(d, n, tc, sm, reserve=0, cap=None):
    """(grid, row tiles per CTA, rows per tile) of the backward launch (csrc/ngcf_tc_bwd.cu bwd_tc_launch,
    csrc/ngcf.cu dense_bwd_fp32_launch). cap: the row-list launch of the top layer (csrc/ngcf.cu ngcf_layer_bwd_rows)
    sizes its grid for the list's capacity, and the n listed rows are then spread over that grid."""
    tm = TC_TM if tc else FP32_TM[d]
    tiles = -(-n // tm)
    launch = tiles if cap is None else -(-cap // tm)
    grid = min(sm - reserve, launch) if tc else min(sm * (2 if d <= 64 else 1), launch)
    grid = max(grid, 1)
    return grid, -(-tiles // grid), tm


def tau_dw(d, n, tc, sm, reserve=0, cap=None):
    grid, per, tm = bwd_grid(d, n, tc, sm, reserve, cap)
    rows_cta = min(per * tm, n)
    red = math.ceil(grid / 8) + 8
    if tc:
        return SPLIT + 3 * min(rows_cta, 4 * TC_TM) * U23 + (math.ceil(per / 4) + red) * U24
    return (rows_cta + red) * U24


def rms_factor(tau_tc, tau_fp, k):
    return tau_tc / tau_fp * math.sqrt(k)


def ulp(x):
    return np.spacing(np.abs(np.asarray(x, np.float32))).astype(np.float64)


def leaky64(z, slope):
    return np.where(z > 0, z, z * float(np.float32(slope)))


def fwd_ref(E, LE, W1, W2):
    """(z, sum|terms|) in float64, [n x d]"""
    A = np.concatenate([LE + E, E * LE], axis=1).astype(np.float64)          # fp32 S, P, then exact
    W = np.concatenate([W1, W2], axis=1).astype(np.float64)                   # [d x 2d]
    return A @ W.T, np.abs(A) @ np.abs(W).T


def dz_of(Gn, En, slope):
    return np.where(En > 0, Gn, Gn * np.float32(slope)).astype(np.float32)


def rows_ref(dz, E, LE, G0, W1, W2):
    """(T, sum|terms| of T, G, sum|terms| of G) in float64"""
    z = dz.astype(np.float64)
    ds, dp = z @ W1.astype(np.float64), z @ W2.astype(np.float64)
    ms, mp = np.abs(z) @ np.abs(W1).astype(np.float64), np.abs(z) @ np.abs(W2).astype(np.float64)
    E64, LE64, G64 = E.astype(np.float64), LE.astype(np.float64), G0.astype(np.float64)
    return ds + dp * E64, ms + mp * np.abs(E64), G64 + ds + dp * LE64, np.abs(G64) + ms + mp * np.abs(LE64)


def dw_ref(dz, E, LE):
    """(dW1, |dW1| terms, dW2, |dW2| terms) in float64"""
    z = dz.astype(np.float64)
    S, P = (LE + E).astype(np.float64), (E * LE).astype(np.float64)
    return z.T @ S, np.abs(z).T @ np.abs(S), z.T @ P, np.abs(z).T @ np.abs(P)


def bound_ratio(x, ref, mag, tau):
    """per element |x - ref| / (tau * sum|terms| + ulp(x)); NaN / inf count as infinitely far"""
    r = np.abs(x.astype(np.float64) - ref) / (tau * mag + ulp(x))
    return np.where(np.isfinite(r), r, np.inf)


def fwd_ratio(y, z, mag, tau, slope):
    """the bound carried through leaky_relu: y may lie anywhere in leaky([z - b, z + b]) widened by ulp(y)"""
    b = tau * mag
    yc = leaky64(z, slope)
    allow = np.maximum(leaky64(z + b, slope) - yc, yc - leaky64(z - b, slope)) + ulp(y)
    r = np.abs(y.astype(np.float64) - yc) / allow
    return np.where(np.isfinite(r), r, np.inf)


def worst(r, what):
    """assert every ratio <= 1 and name the worst element"""
    i = np.unravel_index(int(np.argmax(r)), r.shape)
    assert r[i] <= 1.0, f"{what}: element {tuple(int(v) for v in i)} is {r[i]:.3g} x its bound"
    return float(r[i])


def rms_rel(x, ref, mag, mask=None):
    ok = mag > 0 if mask is None else (mask & (mag > 0))
    e = (x.astype(np.float64) - ref)[ok] / mag[ok]
    return float(np.sqrt(np.mean(e * e))) if e.size else 0.0


def rms_check(x_tc, x_fp, ref, mag, factor, what, mask=None):
    """RMS of error / sum|terms| of the tensor-core result within `factor` of the FP32 pipe's (needs >= 2048 elements:
    an RMS over fewer is noise)"""
    ok = mag > 0 if mask is None else (mask & (mag > 0))
    if int(ok.sum()) < 2048:
        return None
    a, b = rms_rel(x_tc, ref, mag, ok), rms_rel(x_fp, ref, mag, ok)
    assert a <= factor * b, f"{what}: RMS error {a:.3g} is {a / b:.3g} x the FP32 pipe's {b:.3g} (limit {factor:.3g})"
    return a / b


class Summary:
    """per case family, the largest error / bound ratio and the largest RMS ratio against the FP32 pipe that the GPU tests
    of one module measured; printed once after the module"""

    def __init__(self):
        self.fam = {}

    def note(self, family, ratio, rms=None):
        s = self.fam.setdefault(family, [0.0, 0.0])
        s[0] = max(s[0], ratio)
        if rms is not None:
            s[1] = max(s[1], rms)

    def report(self, request):
        if not self.fam:
            return
        with request.config.pluginmanager.get_plugin("capturemanager").global_and_fixture_disabled():
            print()
            for fam in sorted(self.fam):
                r, rr = self.fam[fam]
                print(f"{fam:24s} max error/bound {r:.3g}" + (f"   max RMS ratio vs FP32 pipe {rr:.3g}" if rr else ""))


# ---- calling the library (GPU) ---------------------------------------------------------------------------------------
class Dev:
    def __init__(self):
        from yelprecommendation_b200 import _cabi
        self.cabi, self.lib = _cabi, _cabi.load()
        c = C.c_int(0)
        _cabi.check(self.lib.yr_device_sm_count(C.byref(c)), "yr_device_sm_count")
        self.sm = c.value

    def st(self):
        return self.cabi.stream_ptr()

    def fwd(self, d, n, E, LE, W1, W2, slope, out, mode):
        return self.lib.yr_ngcf_dense_fwd(d, n, E, LE, W1, W2, slope, out, mode, self.st())

    def bwd(self, d, n, E, LE, En, Gn, W1, W2, slope, G, T, dW1, dW2, ws, ws_bytes, mode):
        return self.lib.yr_ngcf_dense_bwd(d, n, E, LE, En, Gn, W1, W2, slope, G, T, dW1, dW2, ws, ws_bytes, mode,
                                          self.st())


@lru_cache(maxsize=None)
def dev():
    return Dev()


def ptr(t, row=0):
    return t.data_ptr() + row * t.stride(0) * t.element_size()


def ptr1(t, off=0):
    return t.data_ptr() + off * t.element_size()


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def sentinel(rows, d):
    return torch.from_numpy(np.full((rows, d), SENTINEL, np.uint32).view(np.float32)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def fwd_tc(d, mode):
    return mode != 0 and d != 32


def bwd_tc(d, mode):
    return mode == 2 and d != 32


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))
