"""The NGCF dense transforms (yr_ngcf_dense_fwd / yr_ngcf_dense_bwd, all three dense modes) and the dense optimizer step
(yr_dense_opt_step / yr_dense_opt_step_multi), kernel by kernel, against a float64 reference with a per-element bound.

Reference (include/yelprec_b200.h, yr_ngcf_layer_fwd / yr_ngcf_layer_bwd). S = LE + E and P = E * LE are rounded to fp32
first, as every kernel does, and so is dZ = G_next * (E_next > 0 ? 1 : slope); everything after that is float64:
    z = [S | P] . [W1 | W2]^T,   E_next = leaky(z)
    dS = dZ W1,  dP = dZ W2,     T = dS + dP * E,   G = G_old + dS + dP * LE
    dW1 = dZ^T S,  dW2 = dZ^T P

Bound. An element x with float64 value x64 passes when |x - x64| <= tau * sum|terms| + ulp(x). sum|terms| is the same
expression with every operand replaced by its absolute value (the sum of absolute products behind the element), ulp(x)
covers the final rounding to fp32, and tau is the relative error that the kernel's arithmetic can reach:

* FP32 pipe (dense mode 0, every mode at d = 32): one fma chain, round to nearest (u = 2^-24). A chain of K terms errs by
  at most K u sum|terms| (the first-order gamma_K bound). Forward: K = 2d. dS / dP: K = d, plus the epilogue fma and, for
  G, the add: (d + 2) u. dW: each CTA chains over its rows (rows_cta terms), then reduce_partials_kernel adds the CTA
  partials, in 8 strided groups and then the 8 group sums: (rows_cta + ceil(parts / 8) + 8) u.
* Tensor cores, 3xTF32 (tcgen05.mma.kind::tf32, csrc/tc_common.cuh split4): x = hi + lo with hi the top 11 significand
  bits, so |lo| < 2^-10 |x|; the tensor core reads lo as TF32 too (truncated to 11 bits, error < 2^-10 |lo|). The product
  a w is formed as lo_a hi_w + hi_a lo_w + hi_a hi_w: the two truncated lo operands and the dropped lo_a lo_w each err by
  less than 2^-20 |a w|, so the split costs at most 3 * 2^-20 per product. The sums are fp32 in TMEM and truncate
  instead of rounding, so every addend that enters an accumulator can cost up to one ulp of the running sum, 2^-23
  sum|terms|. Forward: 2d addends in the hi.hi accumulator; the lo.hi + hi.lo accumulator holds 4d addends of at most
  2^-9 sum|terms|; the epilogue adds the two (u). GEMM1 of the backward puts all three products, 3d addends, into one
  accumulator, then two rounded epilogue operations. dW: the GEMM2 accumulator takes 3 addends per row for at most 4
  tiles (512 rows, kFlushTiles) before the epilogue drains it into the CTA's partial with a rounded add, then the
  reduction as above.
      tau_fwd_tc  = 3 * 2^-20 + 2d (1 + 2^-8) 2^-23 + 2^-24
      tau_rows_tc = 3 * 2^-20 + 3d 2^-23 + 2 * 2^-24
      tau_dw_tc   = 3 * 2^-20 + 3 min(rows_cta, 512) 2^-23 + (ceil(tiles_cta / 4) + ceil(parts / 8) + 8) 2^-24
  A 1xTF32 product (hi.hi only) errs by up to 2^-9 |a w|, 2^-10 on average, with the sign of a w: over 2d terms of
  random sign its error is about 2^-10 / sqrt(2d) sum|terms|, several times tau_fwd_tc at d = 64 and 128.

Second, self-calibrating check. tau is a worst case; it holds whatever the data. On the same inputs the FP32-pipe mode
runs too, and the RMS over elements of |error| / sum|terms| of the tensor-core result must stay within
    F = (tau_tc / tau_fp32) * sqrt(K)
times that of the FP32 pipe. Round-to-nearest errors are unbiased, so the FP32 pipe's K roundings add up like a random
walk, about sqrt(K) below its worst case, while truncation is biased and can reach its worst case. A tensor-core kernel
that does no worse than its derivation stays inside F; a lost split term (1xTF32) is hundreds of times above it.

The checks have teeth: the CPU tests below show that the C oracle and a numpy emulation of the 3xTF32 split pass them,
and that a 1xTF32 emulation, a dropped or shifted row and a dW without its last partial tile fail them.
"""
import ctypes as C
from functools import lru_cache

import numpy as np
import pytest
import torch

from ngcf_ref import (SENTINEL, SLOPES, TC_TM, YR_ERR_BAD_ARG, YR_ERR_BAD_DIM, YR_ERR_WORKSPACE, YR_OK, Summary, bound_ratio,
                      bwd_tc, cu, dev, dw_ref, dz_of, fwd_ratio, fwd_ref, fwd_tc, host, leaky64, ptr, ptr1, rms_check,
                      rms_factor, rows_ref, same_bits, sentinel, tau_dw, tau_fwd, tau_rows, worst)
from oracle import cport

SUMMARY = Summary()                          # family -> [max error / bound, max RMS ratio against the FP32 pipe]
note = SUMMARY.note


@pytest.fixture(scope="module", autouse=True)
def report_summary(request):
    """after the module: per case family, the largest error / bound ratio and the largest RMS ratio against the FP32
    pipe that the GPU tests measured"""
    yield
    SUMMARY.report(request)


def tf32(x):
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def emulate_3xtf32(E, LE, W1, W2, slope):
    """split4 as csrc/tc_common.cuh does it, lo read as TF32 by the tensor core, exact sums: the split's own error"""
    A = np.concatenate([LE + E, E * LE], axis=1)
    W = np.concatenate([W1, W2], axis=1)
    ah, wh = tf32(A), tf32(W)
    al, wl = tf32(A - ah), tf32(W - wh)
    big = (ah.astype(np.float64) @ wh.astype(np.float64).T).astype(np.float32)
    small = (al.astype(np.float64) @ wh.astype(np.float64).T + ah.astype(np.float64) @ wl.astype(np.float64).T)
    z = big + small.astype(np.float32)
    return np.where(z > 0, z, z * np.float32(slope)).astype(np.float32)


def emulate_1xtf32(E, LE, W1, W2, slope):
    A = np.concatenate([LE + E, E * LE], axis=1)
    W = np.concatenate([W1, W2], axis=1)
    z = (tf32(A).astype(np.float64) @ tf32(W).astype(np.float64).T).astype(np.float32)
    return np.where(z > 0, z, z * np.float32(slope)).astype(np.float32)


def make_inputs(n, d, seed):
    """E, LE with row scales over five decades (a small row must be checked as closely as a large one), W like an
    nn.Linear init, G_next, G_old, and an E_next with exact +0 / -0, negative, tiny and subnormal entries in every row"""
    rng = np.random.default_rng(seed)
    sc = (10.0 ** rng.uniform(-3, 2, (n, 1))).astype(np.float32)
    E = (rng.standard_normal((n, d)) * sc).astype(np.float32)
    LE = (rng.standard_normal((n, d)) * 0.5 * sc).astype(np.float32)
    W1, W2 = ((rng.standard_normal((d, d)) / np.sqrt(d)).astype(np.float32) for _ in range(2))
    Gn = (rng.standard_normal((n, d)) * 10.0 ** rng.uniform(-2, 1, (n, 1))).astype(np.float32)
    G0 = rng.standard_normal((n, d)).astype(np.float32)
    En = rng.standard_normal((n, d)).astype(np.float32)
    special = np.array([0.0, -0.0, 1e-30, -1e-30, 1e-42, -1e-42, -1.0, 3.0], np.float32)
    pick = rng.integers(0, 4, (n, d)) == 0
    En[pick] = special[rng.integers(0, len(special), int(pick.sum()))]
    En[:, :len(special)] = special                            # every row has every kind
    return E, LE, W1, W2, Gn, G0, En


def row_sizes(sm):
    return [1, 127, 128, 129, 255, 257, sm * 128 - 1, sm * 128, sm * 128 + 1, 3 * sm * 128 + 77]


# ---- the checks have teeth: CPU only ---------------------------------------------------------------------------------
def _csr(n, seed, per_row=6):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, per_row + 1, n)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = rng.integers(0, n, int(rowptr[-1])).astype(np.int32)
    val = (rng.standard_normal(int(rowptr[-1])) * 0.3).astype(np.float32)
    return rowptr, col, val


@pytest.mark.parametrize("d", [32, 64, 128])
def test_oracle_forward_within_fp32_bound(d):
    """cport.ngcf_layer_fwd (one fma chain per output, the FP32 pipe's order) on a random L is inside tau_fwd(fp32)"""
    n = 300
    E, *_ = make_inputs(n, d, 1)
    W1, W2 = make_inputs(4, d, 2)[2:4]
    for slope in SLOPES:
        En, LE = cport.ngcf_layer_fwd(_csr(n, 3), E, W1, W2, slope=slope)
        z, mag = fwd_ref(E, LE, W1, W2)
        worst(fwd_ratio(En, z, mag, tau_fwd(d, False), slope), f"oracle fwd d={d} slope={slope}")


@pytest.mark.parametrize("d", [32, 64, 128])
def test_oracle_backward_within_fp32_bound(d):
    """cport.ngcf_layer_bwd with an empty L^T is the dense backward alone: G inside tau_rows, dW inside tau_dw"""
    n = 300
    E, LE, W1, W2, Gn, G0, En = make_inputs(n, d, 4)
    empty = (np.zeros(n + 1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    for slope in SLOPES:
        G, dW1, dW2 = cport.ngcf_layer_bwd(empty, E, LE, En, Gn, W1, W2, G0, slope=slope)
        dz = dz_of(Gn, En, slope)
        _, _, Gr, mG = rows_ref(dz, E, LE, G0, W1, W2)
        worst(bound_ratio(G, Gr, mG, tau_rows(d, False)), f"oracle G d={d}")
        a1, m1, a2, m2 = dw_ref(dz, E, LE)
        for tc in (False, True):                              # dW is float64-accumulated: inside either bound
            worst(bound_ratio(dW1, a1, m1, tau_dw(d, n, tc, 148)), f"oracle dW1 d={d}")
            worst(bound_ratio(dW2, a2, m2, tau_dw(d, n, tc, 148)), f"oracle dW2 d={d}")


@pytest.mark.parametrize("d", [64, 128])
def test_checks_have_teeth(d):
    """3xTF32 emulation passes the bound and the RMS check; 1xTF32, a dropped row, a shifted row and a dW without its
    last partial tile fail"""
    n = 1500
    E, LE, W1, W2, Gn, G0, En = make_inputs(n, d, 5)
    slope = 0.2
    # the FP32 pipe's result: the C oracle's fma chain, with LE = L E through a random L
    LEo = cport.spmm_csr(*_csr(n, 6), E)
    z, mag = fwd_ref(E, LEo, W1, W2)
    y_fp = cport.ngcf_layer_fwd(_csr(n, 6), E, W1, W2, slope=slope)[0]
    tau_tc, tau_fp = tau_fwd(d, True), tau_fwd(d, False)
    F = rms_factor(tau_tc, tau_fp, 2 * d)
    pos = z > tau_tc * mag
    y3 = emulate_3xtf32(E, LEo, W1, W2, slope)
    worst(fwd_ratio(y3, z, mag, tau_tc, slope), "3xTF32 emulation")
    assert rms_check(y3, y_fp, z, mag, F, "3xTF32 emulation", pos) is not None
    y1 = emulate_1xtf32(E, LEo, W1, W2, slope)
    assert fwd_ratio(y1, z, mag, tau_tc, slope).max() > 1.0
    with pytest.raises(AssertionError):
        rms_check(y1, y_fp, z, mag, F, "1xTF32 emulation", pos)
    for k in (0, 128, n - 1):                                   # a row dropped (the rows after it move up) / shifted
        drop = np.concatenate([np.delete(y_fp, k, axis=0), np.zeros((1, d), np.float32)])
        assert fwd_ratio(drop, z, mag, tau_tc, slope)[k:].max() > 1.0, k
    assert fwd_ratio(np.roll(y_fp, 1, axis=0), z, mag, tau_tc, slope).max() > 1.0
    zeroed = y_fp.copy()
    zeroed[700] = 0.0
    assert fwd_ratio(zeroed, z, mag, tau_tc, slope)[700].max() > 1.0
    # dW without the last partial tile (n = 1500 = 11 x 128 + 92)
    dz = dz_of(Gn, En, slope)
    a1, m1, _, _ = dw_ref(dz, E, LE)
    cut = n - n % TC_TM
    b1 = dw_ref(dz[:cut], E[:cut], LE[:cut])[0].astype(np.float32)
    worst(bound_ratio(a1.astype(np.float32), a1, m1, tau_dw(d, n, True, 148, 147)), "full dW")
    assert bound_ratio(b1, a1, m1, tau_dw(d, n, True, 148, 147)).max() > 1.0
    # rows: G / T of another row, and a 1xTF32 GEMM1
    T, mT, G, mG = rows_ref(dz, E, LE, G0, W1, W2)
    assert bound_ratio(np.roll(T, 1, axis=0).astype(np.float32), T, mT, tau_rows(d, True)).max() > 1.0
    T1 = rows_ref(tf32(dz), E, LE, G0, tf32(W1), tf32(W2))[0]
    assert bound_ratio(T1.astype(np.float32), T, mT, tau_rows(d, True)).max() > 1.0


def test_bounds_are_tight_enough_to_see_one_row_of_small_magnitude():
    """rel_err over the whole tensor lets a row 1e-3 times smaller than the others be wrong; the per-element bound does
    not"""
    d, n = 64, 256
    E, LE, W1, W2, *_ = make_inputs(n, d, 8)
    E[5] *= 1e-3
    LE[5] *= 1e-3
    z, mag = fwd_ref(E, LE, W1, W2)
    y = leaky64(z, 0.01).astype(np.float32)
    worst(fwd_ratio(y, z, mag, tau_fwd(d, True), 0.01), "exact")
    y[5] *= np.float32(1 + 1e-4)
    assert np.abs(y - leaky64(z, 0.01)).max() / np.abs(leaky64(z, 0.01)).max() < 2e-6      # invisible norm-wise
    assert fwd_ratio(y, z, mag, tau_fwd(d, True), 0.01)[5].max() > 1.0


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
def modes_for(d):
    return (0, 1, 2)


@lru_cache(maxsize=3)
def case_data(d, nmax):
    E, LE, W1, W2, Gn, G0, En = make_inputs(nmax, d, 100 + d)
    z, mag = fwd_ref(E, LE, W1, W2)
    return dict(E=E, LE=LE, W1=W1, W2=W2, Gn=Gn, G0=G0, En=En, z=z, mag=mag)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 64, 128])
def test_dense_forward_every_element_within_bound(d):
    """Every mode, slopes 0.01 / 0.2 / 0, row counts around one tile, one tile per SM and three per SM plus a ragged
    tile. d = 32 runs on the FP32 pipe in every mode: modes 1 and 2 must be bit-identical to mode 0. n = 0 writes
    nothing."""
    g = dev()
    sizes = row_sizes(g.sm)
    D = case_data(d, sizes[-1])
    E, LE, W1, W2 = (cu(D[k]) for k in ("E", "LE", "W1", "W2"))
    out = sentinel(sizes[-1], d)
    assert g.fwd(d, 0, ptr(E), ptr(LE), ptr(W1), ptr(W2), 0.01, ptr(out), 2) == YR_OK
    assert np.array_equal(host(out).view(np.uint32), np.full((sizes[-1], d), SENTINEL, np.uint32))
    for n in sizes:
        z, mag = D["z"][:n], D["mag"][:n]
        for slope in SLOPES:
            res = {}
            for mode in modes_for(d):
                out = sentinel(n, d)
                assert g.fwd(d, n, ptr(E), ptr(LE), ptr(W1), ptr(W2), slope, ptr(out), mode) == YR_OK
                y = res[mode] = host(out)
                tc = fwd_tc(d, mode)
                r = worst(fwd_ratio(y, z, mag, tau_fwd(d, tc), slope), f"fwd d={d} mode={mode} n={n} slope={slope}")
                rr = None
                if tc:
                    rr = rms_check(y, res[0], z, mag, rms_factor(tau_fwd(d, True), tau_fwd(d, False), 2 * d),
                                   f"fwd d={d} mode={mode} n={n} slope={slope}", z > tau_fwd(d, True) * mag)
                note(f"fwd d={d} {'tc' if tc else 'fp32'}", r, rr)
            if d == 32:
                for mode in (1, 2):
                    assert np.array_equal(res[mode].view(np.uint32), res[0].view(np.uint32)), (mode, n, slope)


def _bwd_ws(g, d):
    nb = g.lib.yr_ngcf_layer_bwd_ws_bytes(d)
    return torch.empty(nb, dtype=torch.uint8, device="cuda"), nb


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 64, 128])
def test_dense_backward_every_element_within_bound(d):
    """G accumulates, T is overwritten, dW1 / dW2 are overwritten: per element within tau_rows / tau_dw for every mode,
    slope and row count. E_next carries exact +0 / -0, negative, tiny and subnormal values, so both leaky branches and
    the zero boundary are taken. For a fixed grid a second identical call gives the same bits. Mode 1 runs the FP32-pipe
    backward: bit-identical to mode 0, as is every mode at d = 32."""
    g = dev()
    sizes = row_sizes(g.sm)
    D = case_data(d, sizes[-1])
    E, LE, W1, W2, Gn, En = (cu(D[k]) for k in ("E", "LE", "W1", "W2", "Gn", "En"))
    ws, nb = _bwd_ws(g, d)
    for slope in SLOPES:
        dz = dz_of(D["Gn"], D["En"], slope)
        Tr, mT, Gr, mG = rows_ref(dz, D["E"], D["LE"], D["G0"], D["W1"], D["W2"])
        for n in sizes:
            a1, m1, a2, m2 = dw_ref(dz[:n], D["E"][:n], D["LE"][:n])
            res = {}
            for mode in modes_for(d):
                tc = bwd_tc(d, mode)
                runs = []
                for _ in range(2):
                    G, T = cu(D["G0"][:n]), sentinel(n, d)
                    dW1, dW2 = sentinel(d, d), sentinel(d, d)
                    assert g.bwd(d, n, ptr(E), ptr(LE), ptr(En), ptr(Gn), ptr(W1), ptr(W2), slope, ptr(G), ptr(T),
                                 ptr(dW1), ptr(dW2), ptr(ws), nb, mode) == YR_OK
                    runs.append([host(x) for x in (G, T, dW1, dW2)])
                    if mode == 1:
                        break
                for a, b in zip(runs[0], runs[-1]):
                    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"bwd d={d} mode={mode} n={n}: not deterministic"
                Gk, Tk, dW1k, dW2k = res[mode] = runs[0]
                what = f"bwd d={d} mode={mode} n={n} slope={slope}"
                r = max(worst(bound_ratio(Gk, Gr[:n], mG[:n], tau_rows(d, tc)), what + " G"),
                        worst(bound_ratio(Tk, Tr[:n], mT[:n], tau_rows(d, tc)), what + " T"))
                rw = max(worst(bound_ratio(dW1k, a1, m1, tau_dw(d, n, tc, g.sm)), what + " dW1"),
                         worst(bound_ratio(dW2k, a2, m2, tau_dw(d, n, tc, g.sm)), what + " dW2"))
                rr = None
                if tc:
                    F = rms_factor(tau_rows(d, True), tau_rows(d, False), d)
                    r1 = rms_check(Gk, res[0][0], Gr[:n], mG[:n], F, what + " G")
                    r2 = rms_check(Tk, res[0][1], Tr[:n], mT[:n], F, what + " T")
                    rr = max(x for x in (r1, r2, 0.0) if x is not None)
                kind = "tc" if tc else "fp32"
                note(f"bwd d={d} {kind} G,T", r, rr)
                note(f"bwd d={d} {kind} dW", rw)
            for a, b in zip(res[1], res[0]):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"bwd d={d} n={n}: mode 1 != mode 0"
            if d == 32:
                for a, b in zip(res[2], res[0]):
                    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"bwd d=32 n={n}: mode 2 != mode 0"


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 64, 128])
def test_row_windows_touch_only_their_rows(d):
    """Both passes on rows [r0, r0 + n) of larger buffers, as the row-sharded trainer calls them: input rows outside the
    window hold NaN, output rows outside it (E_next, G, T) hold a sentinel and must keep it; inside, every element is
    within its bound and dW is finite and within its bound."""
    g = dev()
    sizes = row_sizes(g.sm)
    D = case_data(d, sizes[-1])
    slope = 0.01
    dz = dz_of(D["Gn"], D["En"], slope)
    Tr, mT, Gr, mG = rows_ref(dz, D["E"], D["LE"], D["G0"], D["W1"], D["W2"])
    W1, W2 = cu(D["W1"]), cu(D["W2"])
    ws, nb = _bwd_ws(g, d)
    r0, after = 37, 53
    for n in sizes:
        rows = r0 + n + after
        win = slice(r0, r0 + n)

        def framed(a):
            x = np.full((rows, d), np.nan, np.float32)
            x[win] = a[:n]
            return cu(x)

        E, LE, En, Gn = (framed(D[k]) for k in ("E", "LE", "En", "Gn"))
        a1, m1, a2, m2 = dw_ref(dz[:n], D["E"][:n], D["LE"][:n])
        for mode in (0, 2):
            what = f"window d={d} mode={mode} n={n}"
            out = sentinel(rows, d)
            assert g.fwd(d, n, ptr(E, r0), ptr(LE, r0), ptr(W1), ptr(W2), slope, ptr(out, r0), mode) == YR_OK
            y = host(out)
            for part in (y[:r0], y[r0 + n:]):
                assert np.all(part.view(np.uint32) == SENTINEL), what + ": E_next written outside the window"
            worst(fwd_ratio(y[win], D["z"][:n], D["mag"][:n], tau_fwd(d, fwd_tc(d, mode)), slope), what + " E_next")
            G, T = sentinel(rows, d), sentinel(rows, d)
            G[win] = cu(D["G0"][:n])
            dW1, dW2 = sentinel(d, d), sentinel(d, d)
            assert g.bwd(d, n, ptr(E, r0), ptr(LE, r0), ptr(En, r0), ptr(Gn, r0), ptr(W1), ptr(W2), slope, ptr(G, r0),
                         ptr(T, r0), ptr(dW1), ptr(dW2), ptr(ws), nb, mode) == YR_OK
            Gh, Th, w1, w2 = (host(x) for x in (G, T, dW1, dW2))
            for X, name in ((Gh, "G"), (Th, "T")):
                for part in (X[:r0], X[r0 + n:]):
                    assert np.all(part.view(np.uint32) == SENTINEL), f"{what}: {name} written outside the window"
            tc = bwd_tc(d, mode)
            worst(bound_ratio(Gh[win], Gr[:n], mG[:n], tau_rows(d, tc)), what + " G")
            worst(bound_ratio(Th[win], Tr[:n], mT[:n], tau_rows(d, tc)), what + " T")
            assert np.all(np.isfinite(w1)) and np.all(np.isfinite(w2)), what + ": dW not finite"
            worst(bound_ratio(w1, a1, m1, tau_dw(d, n, tc, g.sm)), what + " dW1")
            worst(bound_ratio(w2, a2, m2, tau_dw(d, n, tc, g.sm)), what + " dW2")


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 128])
def test_sm_reservation_same_rows_dw_within_bound(d):
    """YR_DENSE_RESERVE(mode, r): the tensor-core kernels run on SM count - r CTAs (one CTA at r = 255, which walks every
    tile). Forward output, G and T are row-local: bit-identical to r = 0. dW is not: its per-CTA partials follow the
    grid (n_parts), so it is checked against tau_dw for that grid."""
    g = dev()
    sizes = row_sizes(g.sm)
    D = case_data(d, sizes[-1])
    E, LE, W1, W2, Gn, En = (cu(D[k]) for k in ("E", "LE", "W1", "W2", "Gn", "En"))
    ws, nb = _bwd_ws(g, d)
    slope = 0.2
    dz = dz_of(D["Gn"], D["En"], slope)
    for n in (sizes[-1], g.sm * 128 + 1, 257):
        a1, m1, a2, m2 = dw_ref(dz[:n], D["E"][:n], D["LE"][:n])
        base = None
        for r in (0, 1, 7, g.sm - 1, 255):
            mode = 2 | ((r & 0xFF) << 8)
            what = f"reserve d={d} n={n} r={r}"
            out = sentinel(n, d)
            assert g.fwd(d, n, ptr(E), ptr(LE), ptr(W1), ptr(W2), slope, ptr(out), mode) == YR_OK
            G, T = cu(D["G0"][:n]), sentinel(n, d)
            dW1, dW2 = sentinel(d, d), sentinel(d, d)
            assert g.bwd(d, n, ptr(E), ptr(LE), ptr(En), ptr(Gn), ptr(W1), ptr(W2), slope, ptr(G), ptr(T), ptr(dW1),
                         ptr(dW2), ptr(ws), nb, mode) == YR_OK
            got = [host(x) for x in (out, G, T)]
            if base is None:
                base = got
            for a, b, name in zip(got, base, ("E_next", "G", "T")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"{what}: {name} differs from r = 0"
            rw = max(worst(bound_ratio(host(dW1), a1, m1, tau_dw(d, n, True, g.sm, r)), what + " dW1"),
                     worst(bound_ratio(host(dW2), a2, m2, tau_dw(d, n, True, g.sm, r)), what + " dW2"))
            note(f"reserve d={d} dW", rw)


@pytest.mark.gpu
def test_spmm_sm_reservation_bit_exact():
    """yr_csr.reserve_sms = r runs the SpMM as SM count - r persistent CTAs: bit-identical to r = 0 and to the oracle, on
    a graph with split rows and hub rows (more than YR_SPMM_BIG_CHUNKS chunks), plain and accumulating."""
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.data.graph import CSRMatrix
    g = dev()
    rng = np.random.default_rng(7)
    n = 90_000
    lens = rng.integers(0, 60, n)
    lens[5], lens[77], lens[4000], lens[n - 1] = 70_001, 33_000, 20_000, 40_321
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = rng.integers(0, n, int(rowptr[-1])).astype(np.int32)
    val = (rng.standard_normal(int(rowptr[-1])) * 0.05).astype(np.float32)
    A = CSRMatrix(rowptr, col, val, "cuda")
    assert A.n_big_rows == 3 and A.n_split_rows >= 4
    for d in (64, 128):
        X = rng.standard_normal((n, d)).astype(np.float32)
        Y0 = rng.standard_normal((n, d)).astype(np.float32)
        want = cport.spmm_csr(rowptr, col, val, X).view(np.uint32)
        want_acc = cport.spmm_csr(rowptr, col, val, X, Y0).view(np.uint32)
        Xd = cu(X)
        for r in (0, 1, 7, g.sm - 1, 255):
            A.reserve_sms = r
            y = ops.spmm_csr(A, Xd)
            assert np.array_equal(host(y).view(np.uint32), want), (d, r)
            ya = cu(Y0)
            ops.spmm_csr(A, Xd, out=ya, accumulate=True)
            assert np.array_equal(host(ya).view(np.uint32), want_acc), (d, r)
    A.reserve_sms = 0


@pytest.mark.gpu
def test_dense_input_checks():
    """d not in {32, 64, 128}: YR_ERR_BAD_DIM; mode bits >= 1 << 16: YR_ERR_BAD_ARG; a backward workspace below
    yr_ngcf_layer_bwd_ws_bytes(d): YR_ERR_WORKSPACE. Nothing is written."""
    g = dev()
    d, n = 64, 300
    buf = [sentinel(n, 128) for _ in range(6)]
    W = [sentinel(128, 128) for _ in range(4)]
    ws, nb = _bwd_ws(g, 128)
    P = [ptr(b) for b in buf]
    fwd = lambda dd, mode: g.fwd(dd, n, P[0], P[1], ptr(W[0]), ptr(W[1]), 0.01, P[2], mode)
    bwd = lambda dd, mode, nbytes: g.bwd(dd, n, P[0], P[1], P[3], P[4], ptr(W[0]), ptr(W[1]), 0.01, P[5], P[2],
                                         ptr(W[2]), ptr(W[3]), ptr(ws), nbytes, mode)
    for dd in (0, 16, 48, 96, 256):
        for mode in (0, 1, 2):
            assert fwd(dd, mode) == YR_ERR_BAD_DIM, (dd, mode)
            assert bwd(dd, mode, nb) == YR_ERR_BAD_DIM, (dd, mode)
    for mode in (1 << 16, 2 | (1 << 16), 1 << 20, -1, 3, 0xFF):
        assert fwd(d, mode) == YR_ERR_BAD_ARG, mode
        assert bwd(d, mode, nb) == YR_ERR_BAD_ARG, mode
    for dd in (32, 64, 128):
        need = g.lib.yr_ngcf_layer_bwd_ws_bytes(dd)
        for mode in (0, 1, 2):
            assert bwd(dd, mode, need - 1) == YR_ERR_WORKSPACE, (dd, mode)
            assert bwd(dd, mode, 0) == YR_ERR_WORKSPACE, (dd, mode)
    for b in buf + W:
        assert np.all(host(b).view(np.uint32) == SENTINEL)


# ---- optimizer step --------------------------------------------------------------------------------------------------
OPTS = {"sgd": ("sgd", 0.05, 0.0), "sgd_wd": ("sgd", 0.05, 1e-2), "adam": ("adam", 1e-3, 0.0),
        "adam_wd": ("adam", 1e-3, 1e-2), "adamw": ("adamw", 1e-3, 1e-2)}


def opt_state(n, seed):
    rng = np.random.default_rng(seed)
    p = rng.standard_normal(n).astype(np.float32)
    gr = (rng.standard_normal(n) * 10.0 ** rng.uniform(-6, 1, n)).astype(np.float32)
    gr[::7] = 0.0
    m = (rng.standard_normal(n) * 0.1).astype(np.float32)
    v = (np.abs(rng.standard_normal(n)) * 10.0 ** rng.uniform(-8, -1, n)).astype(np.float32)
    return p, gr, m, v


def opt_oracle(kind, lr, wd, step, p, gr, m, v):
    p, m, v = p.copy(), m.copy(), v.copy()
    cport.dense_opt_step(p, gr, m, v, cport.make_opt(kind, lr, wd, step))
    return p, m, v



@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 4, 5, 1023, (1 << 20) + 3])
def test_dense_opt_step_bit_exact_vs_oracle(n):
    """yr_dense_opt_step against orc_dense_opt_step bit for bit: the float4 body and the scalar tail (n % 4 != 0), SGD
    with and without weight decay, Adam with and without, AdamW, at steps 1, 2 and 1000 (bias correction)"""
    g = dev()
    for name, (kind, lr, wd) in OPTS.items():
        for step in (1, 2, 1000):
            p, gr, m, v = opt_state(n, step + n)
            pd, gd, md, vd = (cu(x) for x in (p, gr, m, v))
            adam = kind != "sgd"
            opt = g.cabi.make_opt(kind, lr, wd, step)
            assert g.lib.yr_dense_opt_step(ptr1(pd), ptr1(gd), ptr1(md) if adam else None, ptr1(vd) if adam else None,
                                           n, C.byref(opt), g.st()) == YR_OK
            want = opt_oracle(kind, lr, wd, step, p, gr, m, v)
            assert same_bits(host(pd), want[0]), (name, step)
            assert same_bits(host(gd), gr), (name, step)
            if adam:
                assert same_bits(host(md), want[1]) and same_bits(host(vd), want[2]), (name, step)


@pytest.mark.gpu
def test_dense_opt_step_unaligned_views_bit_exact():
    """Views that start inside a tensor (pointers 4, 8 or 12 bytes past a 16-byte boundary) take the scalar path: same
    bits as the oracle, nothing outside the view touched"""
    g = dev()
    for n in (5, 1023, 4096):
        for off in ((1, 0, 0, 0), (0, 2, 0, 0), (0, 0, 3, 0), (0, 0, 0, 1), (3, 3, 3, 3)):
            p, gr, m, v = opt_state(n, n + sum(off))
            bufs = []
            for x, o in zip((p, gr, m, v), off):
                b = np.full(n + 8, 7.0, np.float32)
                b[o:o + n] = x
                bufs.append(cu(b))
            opt = g.cabi.make_opt("adam", 1e-3, 1e-2, 3)
            assert g.lib.yr_dense_opt_step(*(ptr1(b, o) for b, o in zip(bufs, off)), n, C.byref(opt), g.st()) == YR_OK
            want = opt_oracle("adam", 1e-3, 1e-2, 3, p, gr, m, v)
            got = [host(b) for b in bufs]
            for x, o, w in zip(got, off, (want[0], gr, want[1], want[2])):
                assert same_bits(x[o:o + n], w), (n, off)
                assert np.all(x[:o] == 7.0) and np.all(x[o + n:] == 7.0), (n, off)


def _carve(sizes, fill, seed):
    """one device buffer per role with every tensor at a 16-byte-aligned offset and 8 guard floats after it"""
    offs, o = [], 0
    for s in sizes:
        offs.append(o)
        o += s + 8
    host_bufs = [np.full(o, fill, np.float32) for _ in range(4)]
    parts = []
    for t, s in enumerate(sizes):
        st = opt_state(s, seed + t) if s else tuple(np.zeros(0, np.float32) for _ in range(4))
        for hb, x in zip(host_bufs, st):
            hb[offs[t]:offs[t] + s] = x
        parts.append(st)
    return offs, host_bufs, parts


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [[1028], [12, 0, 4100], [4, 0, 64, 4096, 8, 0, 65540, 20]])
def test_dense_opt_step_multi_bit_exact_and_zero_grad(sizes):
    """yr_dense_opt_step_multi over 1, 3 and 8 tensors of mixed sizes with empty ones among them: every tensor bit-exact
    against its own oracle call; zero_grad = 1 clears exactly the gradients it consumed (the guards between them keep
    their values), zero_grad = 0 leaves them alone"""
    g = dev()
    k = len(sizes)
    for name, (kind, lr, wd) in OPTS.items():
        adam = kind != "sgd"
        for step, zero_grad in ((1, 1), (1000, 0)):
            offs, hb, parts = _carve(sizes, 7.0, step + k)
            P, Gd, M, V = (cu(b) for b in hb)
            ptrs = lambda b: (C.c_void_p * k)(*[ptr1(b, o) for o in offs])
            opt = g.cabi.make_opt(kind, lr, wd, step)
            rc = g.lib.yr_dense_opt_step_multi(k, ptrs(P), ptrs(Gd), ptrs(M) if adam else None, ptrs(V) if adam else None,
                                               (C.c_int64 * k)(*sizes), C.byref(opt), zero_grad, g.st())
            assert rc == YR_OK
            got = [host(b) for b in (P, Gd, M, V)]
            for t, (s, o) in enumerate(zip(sizes, offs)):
                p, gr, m, v = parts[t]
                want = opt_oracle(kind, lr, wd, step, p, gr, m, v) if s else (p, m, v)
                assert same_bits(got[0][o:o + s], want[0]), (name, step, t)
                assert same_bits(got[1][o:o + s], np.zeros(s, np.float32) if zero_grad else gr), (name, step, t)
                if adam:
                    assert same_bits(got[2][o:o + s], want[1]) and same_bits(got[3][o:o + s], want[2]), (name, step, t)
                for b in got if adam else got[:2]:
                    assert np.all(b[o + s:o + s + 8] == 7.0), (name, step, t, "guard")


@pytest.mark.gpu
def test_dense_opt_step_multi_rejects_ragged_or_unaligned():
    """a size that is not a multiple of 4, or any pointer that is not 16-byte aligned: YR_ERR_BAD_ARG, nothing written"""
    g = dev()
    sizes = [8, 16, 4]
    offs, hb, _ = _carve(sizes, 7.0, 1)
    bufs = [cu(b) for b in hb]
    before = [b.copy() for b in hb]
    opt = g.cabi.make_opt("adam", 1e-3, 0.0, 1)

    def call(sz, shift=None):
        arrs = []
        for r, b in enumerate(bufs):
            arrs.append((C.c_void_p * 3)(*[ptr1(b, o + (1 if shift == (r, t) else 0)) for t, o in enumerate(offs)]))
        return g.lib.yr_dense_opt_step_multi(3, *arrs, (C.c_int64 * 3)(*sz), C.byref(opt), 1, g.st())

    for bad in ([8, 6, 4], [1, 16, 4], [8, 16, 3], [8, 16, -4]):
        assert call(bad) == YR_ERR_BAD_ARG, bad
    for r in range(4):
        for t in range(3):
            assert call([8, 12, 4], (r, t)) == YR_ERR_BAD_ARG, (r, t)
    for b, w in zip(bufs, before):
        assert same_bits(host(b), w)
