"""The rest of the NGCF train step (yr_ngcf_train_step_ex) kernel by kernel: the BPR tail (yr_ngcf_tail), the SpMM plan
edges and launch variants (yr_spmm_csr), and the row-sparse top layer stage by stage, each against a float64 reference
with a per-element bound (the dense transforms and the optimizer step are test_ngcf_dense_kernels.py's; this file reuses
their reference and bounds from ngcf_ref.py). u = 2^-24 throughout; ulp(x) covers the final rounding to fp32.

BPR tail. The float64 reference reads the fp32 layer tables E_0..E_L and rounds nothing:
    x_b = sum_l (u . p - u . n),  loss = mean_b -log sigmoid(x_b),  g_b = -sigmoid(-x_b) / B
    G_l[u] += g_b (p - n),  G_l[nU + p] += g_b u,  G_l[nU + n] -= g_b u
* Scores (pos_out / neg_out): a warp per triple, every lane one fma chain of K = (L + 1) d / 32 terms, then a 5-level
  shuffle tree: tau_s = (K + 5) u against sum|u p|.
* x = fl(dp - dn) errs by bx = tau_s (sum|u p| + sum|u n|) + ulp(dp) + ulp(dn) + ulp(x).
* Loss: |d(-log sigmoid)/dx| <= 1 carries bx; exp_cr / log1p_cr are correctly rounded and log1p(exp(-|x|)) - min(x, 0) has
  at most 4 roundings of relative size u on a sum of like-signed terms: 4 u loss_b, plus 2^-148 for the subnormal
  exp(-|x|) of a saturated triple. The double-precision sum is exact to far below that; the mean is rounded to fp32 once.
* g: |dsigma| <= 1/4 carries bx / (4B); the division z / (1 + z), the 1 - q, 1/B and the product add 8 u |g|.
* G: gu = fl(fl(g p) - fl(g n)) and gp = fl(g u) cost 2 u sum|terms|; m atomic addends into a zeroed row, in any order,
  at most (m - 1) u sum|terms|: tau_G = (m + 3) u. The error of g enters as sum_b |dg_b| |operand|. fp32 atomics
  flush subnormals to zero, so every addend may also lose up to 2^-126.

Row-sparse top layer (d = 64, cfg.ngcf_top_rows_mode = 1). Each stage is checked from the GPU's own inputs to it:
* LE_l (yr_spmm_csr and the row-subset yr_spmm_csr_rows) bit-exact against cport.spmm_csr, E_{l+1} within tau_fwd.
* G_L = the tail alone: within the tail bound, exactly 0 on every row the batch does not touch.
* G_l after its layer's backward, from G_{l+1}, E_{l+1} (dZ rounded to fp32 first), E_l and LE_l. The dense row part
  is tau_rows(d, tc) as in the dense-kernel test, on the touched rows of the top layer and on every row below it. Then
  G_l += L^T T: the SpMM accumulates a row's nnz products and its chunk partials onto G, the scatter form of the top
  layer adds one float4 RED per (touched row, stored entry); both are m = nnz + chunks addends on the existing value,
  so (m + 2) u sum|terms|. T itself carries tau_rows mT + ulp(T) into every product: |L|^T (tau_rows mT + ulp(T)).
  The error that G_l's input carried (the tail's allowance) adds on.
* dW1 / dW2: tau_dw of the dense-kernel test with the grid of the launch that ran. The row-list launch sizes its grid for
  the list's capacity cap = 3 max(batch_size, 4096) and spreads the listed rows over it: FP32 pipe min(ceil(cap / 64),
  2 SM) CTAs, tensor cores (dense mode 2, cap >= 16,384) min(SM, ceil(cap / 128)).
* The SGD step is bit-exact: fl(p - lr g) from the GPU's G_0 / dW through the C oracle.

The checks have teeth: the CPU tests show that the C oracle passes them and that a tail gradient without its 1/B, a
dropped triple, a scatter without one 128-non-zero chunk of a split row, a touched row listed twice or left out and a
top-layer dW without one touched row fail them.
"""
import ctypes as C
from functools import lru_cache

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from ngcf_ref import (SENTINEL, U24, YR_ERR_BAD_ARG, YR_ERR_BAD_DIM, YR_OK, Summary, bwd_tc, cu, dev, dw_ref, dz_of,
                      fwd_ratio, fwd_ref, fwd_tc, host, ptr1, rows_ref, same_bits, sentinel, tau_dw, tau_fwd, tau_rows,
                      ulp, worst)
from oracle import cport
from util import cfg

SUMMARY = Summary()
note = SUMMARY.note
SLOPE = 0.01                         # models/ngcf.py _LEAKY_SLOPE
TINY = 2.0 ** -148                   # a subnormal exp(-|x|) of a saturated triple
FTZ = 2.0 ** -126                    # fp32 atomic adds flush subnormal operands and results to zero: per addend


@pytest.fixture(scope="module", autouse=True)
def report_summary(request):
    """after the module: per case family, the largest error / bound ratio the GPU tests measured"""
    yield
    SUMMARY.report(request)


# ----------------------------------------------------------------------------------------------------------------------
# float64 references and bounds (CPU)
# ----------------------------------------------------------------------------------------------------------------------
def ratio(x, ref, allow):
    """per element |x - ref| / (allow + ulp(x)); NaN / inf count as infinitely far"""
    r = np.abs(np.asarray(x, np.float64) - ref) / (allow + ulp(x))
    return np.where(np.isfinite(r), r, np.inf)


def tau_score(d, n_layers):
    return ((n_layers + 1) * d // 32 + 5) * U24


def tail_ref(E_layers, nU, uid, pos, neg):
    """float64 tail over the valid triples, divided by the full B. Returns the scores with their sum|terms|, the loss and
    its allowance, and per layer G (float64) with its allowance (everything but the final ulp)."""
    uid, pos, neg = (np.asarray(a, np.int64) for a in (uid, pos, neg))
    B = len(uid)
    n, d = E_layers[0].shape
    nI, L = n - nU, len(E_layers) - 1
    ok = (uid >= 0) & (uid < nU) & (pos >= 0) & (pos < nI) & (neg >= 0) & (neg < nI)
    u, p, q = uid[ok], nU + pos[ok], nU + neg[ok]
    b = len(u)
    dp, dn, mp, mn = (np.zeros(b) for _ in range(4))
    for E in E_layers:
        E = E.astype(np.float64)
        up, un = E[u] * E[p], E[u] * E[q]
        dp += up.sum(1)
        dn += un.sum(1)
        mp += np.abs(up).sum(1)
        mn += np.abs(un).sum(1)
    x = dp - dn
    ts = tau_score(d, L)
    bx = ts * (mp + mn) + ulp(dp) + ulp(dn) + ulp(x)
    lossb = np.logaddexp(0.0, -x)
    loss = lossb.sum() / B
    loss_allow = (bx + 4 * U24 * lossb + TINY).sum() / B
    g = -0.5 * (1.0 - np.tanh(0.5 * x)) / B                   # -sigmoid(-x) / B without overflow
    ag = bx / (4 * B) + 8 * U24 * np.abs(g) + TINY
    cols = np.arange(b)
    S = lambda rows, w: sp.csr_matrix((w, (rows, cols)), shape=(n, b))
    Su, Sp, Sn = S(u, g), S(p, g), S(q, g)
    Au, Ap, An = S(u, np.abs(g)), S(p, np.abs(g)), S(q, np.abs(g))
    Du, Dp, Dn = S(u, ag), S(p, ag), S(q, ag)
    cnt = (np.bincount(u, minlength=n) + np.bincount(p, minlength=n) + np.bincount(q, minlength=n)).astype(np.float64)
    G, allow = [], []
    for E in E_layers:
        E = E.astype(np.float64)
        Eu, Ep, Eq = E[u], E[p], E[q]
        G.append(Su @ (Ep - Eq) + Sp @ Eu - Sn @ Eu)
        mag = Au @ (np.abs(Ep) + np.abs(Eq)) + (Ap + An) @ np.abs(Eu)
        dg = Du @ (np.abs(Ep) + np.abs(Eq)) + (Dp + Dn) @ np.abs(Eu)
        allow.append((cnt[:, None] + 3) * U24 * mag + dg + cnt[:, None] * FTZ)
    return dict(ok=ok, dp=dp, dn=dn, mp=mp, mn=mn, ts=ts, loss=loss, loss_allow=loss_allow, G=G, allow=allow, x=x)


def csr_parts(rowptr, col, val, n):
    A = sp.csr_matrix((np.asarray(val, np.float64), np.asarray(col), np.asarray(rowptr)), shape=(n, n))
    At = A.T.tocsr()
    nnz = np.diff(At.indptr).astype(np.float64)
    return dict(At=At, absAt=abs(At), cnt=nnz + np.ceil(nnz / 128.0))


def layer_g_ref(Gpre, pre_allow, dz, E, LE, W1, W2, Ap, tc):
    """G_l after one layer's backward from G_pre (float64, with the allowance it carries): dense row part + L^T T"""
    d = E.shape[1]
    T, mT, Gr, mG = rows_ref(dz, E, LE, Gpre, W1, W2)
    tr = tau_rows(d, tc)
    At, absAt = Ap["At"], Ap["absAt"]
    ref = Gr + At @ T
    allow = (pre_allow + tr * mG + absAt @ (tr * mT + ulp(T))
             + (Ap["cnt"][:, None] + 2) * (U24 * (np.abs(Gr) + absAt @ np.abs(T)) + FTZ))
    return ref, allow


# ---- the checks have teeth: CPU only ---------------------------------------------------------------------------------
def _tables(n, d, L, seed):
    """layer tables with row scales over four decades, exact +0 / -0 and subnormal entries in a tenth of the rows"""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(L + 1):
        E = (rng.standard_normal((n, d)) * 10.0 ** rng.uniform(-2, 0.5, (n, 1))).astype(np.float32)
        rows = rng.choice(n, n // 10, replace=False)
        E[rows, :6] = np.array([0.0, -0.0, 1e-42, -1e-42, 1e-39, -3e-39], np.float32)
        out.append(E)
    return out


def _triples(B, nU, nI, seed, hub=True):
    """random triples plus: a hub user in a third of them (>= 1,000 once B > 3,000), an item that is pos in some and neg
    in others, a triple with pos == neg, and two saturated triples (x = +-100, rows nU - 1 / items nI - 1, nI - 2)"""
    rng = np.random.default_rng(seed)
    uid, pos, neg = rng.integers(0, nU - 1, B), rng.integers(0, nI - 2, B), rng.integers(0, nI - 2, B)
    if hub and B > 3000:
        uid[: B // 3] = 0
    pos[1::7], neg[4::7] = 7, 7
    if B >= 3:
        pos[2] = neg[2]
    if B >= 5:
        uid[3:5] = nU - 1
        pos[3], neg[3], pos[4], neg[4] = nI - 1, nI - 2, nI - 2, nI - 1
    return uid, pos, neg


def _saturate(E_layers, nU, x=100.0):
    d, L = E_layers[0].shape[1], len(E_layers) - 1
    s = np.float32(x / (2 * d * (L + 1)))
    for E in E_layers:
        E[nU - 1], E[-1], E[-2] = 1.0, s, -s


def tail_ratios(ref, nU, pos_out, neg_out, loss, G_layers):
    ok = ref["ok"]
    r = {"scores": max(worst(ratio(pos_out[ok], ref["dp"], ref["ts"] * ref["mp"]), "pos_out"),
                       worst(ratio(neg_out[ok], ref["dn"], ref["ts"] * ref["mn"]), "neg_out")),
         "loss": worst(ratio(np.float32(loss), ref["loss"], ref["loss_allow"]), "loss")}
    if G_layers is not None:
        r["G"] = max(worst(ratio(G, Gr, a), f"G_{l}") for l, (G, Gr, a) in enumerate(zip(G_layers, ref["G"], ref["allow"])))
    return r


@pytest.mark.parametrize("d,L", [(32, 0), (64, 3), (128, 1), (256, 7)])
def test_oracle_tail_within_bounds(d, L):
    """cport.ngcf_tail (one fma chain per score, sequential accumulation) passes the tail bounds, saturated triples
    included"""
    nU, nI = 300, 400
    E = _tables(nU + nI, d, L, d + L)
    _saturate(E, nU)
    uid, pos, neg = _triples(4000, nU, nI, 3)
    loss, po, no, G = cport.ngcf_tail(E, nU, uid, pos, neg)
    ref = tail_ref(E, nU, uid, pos, neg)
    assert ref["x"][3] == pytest.approx(100.0, rel=1e-4) and ref["x"][4] == pytest.approx(-100.0, rel=1e-4)
    tail_ratios(ref, nU, po, no, loss, G)


def test_tail_mutations_fail():
    """a tail gradient without its 1/B and a dropped triple are outside the G bound; a triple whose loss is counted
    twice is outside the loss bound"""
    nU, nI, d, L = 300, 400, 64, 1
    E = _tables(nU + nI, d, L, 9)
    uid, pos, neg = _triples(257, nU, nI, 4, hub=False)
    ref = tail_ref(E, nU, uid, pos, neg)
    loss, po, no, G = cport.ngcf_tail(E, nU, uid, pos, neg)
    tail_ratios(ref, nU, po, no, loss, G)
    assert ratio(G[1] * np.float32(len(uid)), ref["G"][1], ref["allow"][1]).max() > 1.0        # no 1/B
    for k in (0, 100, 256):                                                                   # one triple dropped
        keep = np.arange(len(uid)) != k
        Gd = cport.ngcf_tail(E, nU, uid[keep], pos[keep], neg[keep])[3]
        Gd = [x * np.float32((len(uid) - 1) / len(uid)) for x in Gd]                          # same 1/B as the full batch
        assert max(ratio(a, r, al).max() for a, r, al in zip(Gd, ref["G"], ref["allow"])) > 1.0, k
    twice = loss + float(np.logaddexp(0.0, -ref["x"][5])) / len(uid)
    assert ratio(np.float32(twice), ref["loss"], ref["loss_allow"]).max() > 1.0


def _split_graph(n=700, seed=2):
    """a symmetric-pattern CSR with one 300-non-zero row (three chunks) and short rows"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 8, n)
    lens[11] = 300
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = np.concatenate([rng.choice(n, k, replace=False) for k in lens]).astype(np.int32)
    val = (rng.uniform(0.01, 0.2, int(rowptr[-1]))).astype(np.float32)
    return rowptr, col, val


def _top_layer_case(n=700, d=64, seed=3):
    """inputs of the top layer's backward as the train step sees them: G_L non-zero on the touched rows only"""
    rowptr, col, val = _split_graph(n)
    rng = np.random.default_rng(seed)
    E, LE, En = (rng.standard_normal((n, d)).astype(np.float32) for _ in range(3))
    W1, W2 = ((rng.standard_normal((d, d)) / np.sqrt(d)).astype(np.float32) for _ in range(2))
    touched = np.zeros(n, bool)
    touched[rng.choice(n, n // 5, replace=False)] = True
    touched[11] = True                                         # the split row is touched
    Gn = np.where(touched[:, None], rng.standard_normal((n, d)), 0.0).astype(np.float32)
    Gpre = (rng.standard_normal((n, d)) * 0.1).astype(np.float32)   # what the tail left in G_{L-1}
    return rowptr, col, val, E, LE, En, Gn, W1, W2, touched, Gpre


def test_oracle_layer_backward_within_g_bound_and_scatter_mutations_fail():
    """cport.ngcf_layer_bwd on the touched rows (dZ = 0 elsewhere) passes the G_{L-1} bound; a scatter without one
    128-non-zero chunk of the split row, a touched row listed twice, a touched row missing from the list and a top-layer
    dW without one touched row fail"""
    n, d = 700, 64
    rowptr, col, val, E, LE, En, Gn, W1, W2, touched, Gpre = _top_layer_case(n, d)
    Ap = csr_parts(rowptr, col, val, n)
    At = Ap["At"]
    csrT = (At.indptr.astype(np.int32), At.indices.astype(np.int32), At.data.astype(np.float32))
    G, dW1, dW2 = cport.ngcf_layer_bwd(csrT, E, LE, En, Gn, W1, W2, Gpre, slope=SLOPE)
    dz = dz_of(Gn, En, SLOPE)
    ref, allow = layer_g_ref(Gpre.astype(np.float64), 0.0, dz, E, LE, W1, W2, Ap, False)
    worst(ratio(G, ref, allow), "oracle G_{L-1}")
    T = rows_ref(dz, E, LE, Gpre, W1, W2)[0]
    A = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(n, n))

    def scatter_from(rows_w):                                  # G with the row part as computed and L^T T over rows_w
        return (ref - At @ T + A.T @ (rows_w[:, None] * T)).astype(np.float32)

    one = touched.astype(np.float64)
    worst(ratio(scatter_from(one), ref, allow), "exact scatter")
    twice = one.copy()
    twice[np.flatnonzero(touched)[3]] = 2.0
    assert ratio(scatter_from(twice), ref, allow).max() > 1.0, "row listed twice"
    missing = one.copy()
    missing[np.flatnonzero(touched)[3]] = 0.0
    assert ratio(scatter_from(missing), ref, allow).max() > 1.0, "row missing from the list"
    chunk = A.copy().tolil()
    cols11 = col[rowptr[11] + 128: rowptr[11] + 256]
    for c in cols11:
        chunk[11, c] = 0.0
    Gc = (ref - At @ T + chunk.tocsr().T @ (one[:, None] * T)).astype(np.float32)
    assert ratio(Gc, ref, allow).max() > 1.0, "scatter without one chunk"
    rows = np.flatnonzero(touched)
    for tc, cap in ((False, 3 * 2048), (True, 3 * 8192)):
        a1, m1, a2, m2 = dw_ref(dz[rows], E[rows], LE[rows])
        tau = tau_dw(d, len(rows), tc, 148, cap=cap)
        worst(ratio(dW1, a1, tau * m1), "oracle dW1")
        worst(ratio(dW2, a2, tau * m2), "oracle dW2")
        for k in (0, len(rows) // 2, len(rows) - 1):
            keep = np.delete(rows, k)
            b1 = dw_ref(dz[keep], E[keep], LE[keep])[0].astype(np.float32)
            assert ratio(b1, a1, tau * m1).max() > 1.0, ("dW without a touched row", tc, k)


# ----------------------------------------------------------------------------------------------------------------------
# GPU: BPR tail
# ----------------------------------------------------------------------------------------------------------------------
def _tail(g, E_dev, G_dev, L, nU, nI, d, uid, pos, neg, B, po, no, loss, sl, err):
    return g.lib.yr_ngcf_tail(E_dev, G_dev, L, nU, nI, d, uid, pos, neg, B, po, no, loss, sl, err, g.st())


def _dptrs(ts):
    from yelprecommendation_b200 import ops
    return ops.device_ptr_array(ts)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [32, 64, 128, 256])
@pytest.mark.parametrize("L", [0, 1, 3, 7])
def test_tail_every_element_within_bound(d, L):
    """Batch sizes 1, 31, 32 and around SM * 64 (one triple per warp of the capped grid) up to 3 SM * 64 + 5, where warps
    loop. Scores, loss and every G_l element within their bounds; the scores are bit-identical across calls; loss_sum[0]
    accumulates the step means and loss_sum[1] is 0 after every call; G_layers = NULL and NULL pos_out / neg_out /
    step_loss write nothing."""
    g = dev()
    nU, nI = 600, 800
    E = _tables(nU + nI, d, L, 7 * d + L)
    _saturate(E, nU)
    Ed = [cu(x) for x in E]
    E_dev = _dptrs(Ed)
    sizes = (1, 31, 32, g.sm * 64 - 1, g.sm * 64, g.sm * 64 + 1, 3 * g.sm * 64 + 5)
    for B in sizes if L in (0, 3) or d == 64 else sizes[:3] + sizes[5:6]:
        uid, pos, neg = _triples(B, nU, nI, B)
        ref = tail_ref(E, nU, uid, pos, neg)
        ud, pd, nd = (cu(a.astype(np.int64)) for a in (uid, pos, neg))
        G = [torch.zeros_like(x) for x in Ed]
        G_dev = _dptrs(G)
        po, no, po2, no2 = (sentinel(B, 1) for _ in range(4))
        loss = torch.zeros(2, dtype=torch.float64, device="cuda")
        sl, sl2 = sentinel(1, 1), sentinel(1, 1)
        err = torch.zeros(1, dtype=torch.int32, device="cuda")
        what = f"tail d={d} L={L} B={B}"
        assert _tail(g, ptr1(E_dev), ptr1(G_dev), L, nU, nI, d, ptr1(ud), ptr1(pd), ptr1(nd), B, ptr1(po), ptr1(no),
                     ptr1(loss), ptr1(sl), ptr1(err)) == YR_OK
        Gh = [host(x) for x in G]
        r = tail_ratios(ref, nU, host(po)[:, 0], host(no)[:, 0], host(sl)[0, 0], Gh)
        lh = host(loss)
        assert lh[0] == np.float64(host(sl)[0, 0]) and lh[1] == 0.0, what
        assert _tail(g, ptr1(E_dev), None, L, nU, nI, d, ptr1(ud), ptr1(pd), ptr1(nd), B, ptr1(po2), ptr1(no2),
                     ptr1(loss), ptr1(sl2), ptr1(err)) == YR_OK
        assert same_bits(host(po2), host(po)) and same_bits(host(no2), host(no)), what + ": scores not reproducible"
        assert all(same_bits(host(x), y) for x, y in zip(G, Gh)), what + ": G_layers = NULL wrote G"
        lh2 = host(loss)
        assert lh2[0] == lh[0] + np.float64(host(sl2)[0, 0]) and lh2[1] == 0.0, what
        worst(ratio(host(sl2)[0, 0], ref["loss"], ref["loss_allow"]), what + " second loss")
        assert _tail(g, ptr1(E_dev), None, L, nU, nI, d, ptr1(ud), ptr1(pd), ptr1(nd), B, None, None, ptr1(loss), None,
                     ptr1(err)) == YR_OK
        assert all(same_bits(host(x), y) for x, y in zip(G, Gh)), what + ": G_layers = NULL wrote G"
        assert host(loss)[0] > lh2[0] or ref["loss"] == 0.0, what + ": loss_sum[0] did not accumulate"
        assert host(loss)[1] == 0.0 and host(err)[0] == 0, what
        for k, v in r.items():
            note(f"tail {k}", v)


@pytest.mark.gpu
def test_tail_bad_ids_flag_and_contribute_nothing():
    """uid -1 / nU, pos nI, neg -1: err = 1, those triples add nothing to G or to the loss, and the loss and g of the
    others are still divided by the full B (current behaviour, pinned)"""
    g = dev()
    nU, nI, d, L = 600, 800, 64, 2
    E = _tables(nU + nI, d, L, 5)
    Ed = [cu(x) for x in E]
    B = 200
    uid, pos, neg = _triples(B, nU, nI, 8, hub=False)
    uid[10], uid[20], pos[30], neg[40] = -1, nU, nI, -1
    ref = tail_ref(E, nU, uid, pos, neg)
    assert int(ref["ok"].sum()) == B - 4
    G = [torch.zeros_like(x) for x in Ed]
    po, no = sentinel(B, 1), sentinel(B, 1)
    loss = torch.zeros(2, dtype=torch.float64, device="cuda")
    sl, err = sentinel(1, 1), torch.zeros(1, dtype=torch.int32, device="cuda")
    ud, pd, nd = (cu(a.astype(np.int64)) for a in (uid, pos, neg))
    assert _tail(g, ptr1(_dptrs(Ed)), ptr1(_dptrs(G)), L, nU, nI, d, ptr1(ud), ptr1(pd), ptr1(nd), B, ptr1(po), ptr1(no),
                 ptr1(loss), ptr1(sl), ptr1(err)) == YR_OK
    assert host(err)[0] == 1
    r = tail_ratios(ref, nU, host(po)[:, 0], host(no)[:, 0], host(sl)[0, 0], [host(x) for x in G])
    for k, v in r.items():
        note(f"tail bad ids {k}", v)


@pytest.mark.gpu
def test_tail_argument_errors_write_nothing():
    """d = 48 / 512: YR_ERR_BAD_DIM; n_layers 8 or -1, B = 0, NULL E_layers / uid / pos / neg / loss_sum: YR_ERR_BAD_ARG.
    Neither writes G, the scores, the loss, step_loss or err."""
    g = dev()
    nU, nI, d = 60, 80, 64
    E = [cu(x) for x in _tables(nU + nI, 512, 7, 1)]
    Ep = ptr1(_dptrs(E))
    G = [sentinel(nU + nI, 512) for _ in range(8)]
    Gp = ptr1(_dptrs(G))
    ids = cu(np.arange(16, dtype=np.int64))
    po, no, sl = sentinel(16, 1), sentinel(16, 1), sentinel(1, 1)
    loss = torch.full((2,), 3.0, dtype=torch.float64, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    base = dict(E=Ep, G=Gp, L=1, d=d, u=ptr1(ids), p=ptr1(ids), n=ptr1(ids), B=16, loss=ptr1(loss))

    def call(**kw):
        a = dict(base, **kw)
        return _tail(g, a["E"], a["G"], a["L"], nU, nI, a["d"], a["u"], a["p"], a["n"], a["B"], ptr1(po), ptr1(no),
                     a["loss"], ptr1(sl), ptr1(err))

    for dd in (48, 512):
        assert call(d=dd) == YR_ERR_BAD_DIM, dd
    for kw in (dict(L=8), dict(L=-1), dict(B=0), dict(E=None), dict(u=None), dict(p=None), dict(n=None), dict(loss=None)):
        assert call(**kw) == YR_ERR_BAD_ARG, kw
    for t in G + [po, no, sl]:
        assert np.all(host(t).view(np.uint32) == SENTINEL)
    assert np.array_equal(host(loss), [3.0, 3.0]) and host(err)[0] == 0


# ----------------------------------------------------------------------------------------------------------------------
# GPU: SpMM plan edges and launch variants
# ----------------------------------------------------------------------------------------------------------------------
EDGE_LENS = (0, 1, 127, 128, 129, 255, 256, 257, 32768, 32769)


@lru_cache(maxsize=1)
def edge_matrix():
    """rows of every plan edge (one chunk / two chunks / the last non-hub row of 256 chunks / the first hub row of 257)
    among short random rows; every 97th row of X is referenced by no column"""
    rng = np.random.default_rng(21)
    n = 40_000
    lens = rng.integers(0, 9, n)
    at = np.linspace(5, n - 5, len(EDGE_LENS)).astype(int)
    lens[at] = EDGE_LENS
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    live = np.setdiff1d(np.arange(n), np.arange(0, n, 97))
    col = rng.choice(live, int(rowptr[-1])).astype(np.int32)
    val = (rng.standard_normal(int(rowptr[-1])) * 0.05).astype(np.float32)
    return rowptr, col, val


@lru_cache(maxsize=4)
def edge_oracle(d):
    rowptr, col, val = edge_matrix()
    n = len(rowptr) - 1
    rng = np.random.default_rng(d)
    X = rng.standard_normal((n, d)).astype(np.float32)
    X[::97] = np.nan
    Y0 = rng.standard_normal((n, d)).astype(np.float32)
    return X, Y0, cport.spmm_csr(rowptr, col, val, X), cport.spmm_csr(rowptr, col, val, X, Y0)


def _spmm_sweep(g, A, what):
    for d in (32, 64, 128, 256):
        X, Y0, want, want_acc = edge_oracle(d)
        assert np.all(np.isfinite(want)) and np.all(np.isfinite(want_acc))
        Xd = cu(X)
        st = A.struct(d)
        for _ in range(2):                                    # back to back: the arrival counters re-arm
            Y = sentinel(A.n_rows, d)
            assert g.lib.yr_spmm_csr(C.byref(st), d, ptr1(Xd), ptr1(Y), 0, g.st()) == YR_OK
            assert same_bits(host(Y), want), f"{what} d={d}"
            assert not np.any(host(A.split_count)), f"{what} d={d}: split_count not re-armed"
            Ya = cu(Y0)
            assert g.lib.yr_spmm_csr(C.byref(st), d, ptr1(Xd), ptr1(Ya), 1, g.st()) == YR_OK
            assert same_bits(host(Ya), want_acc), f"{what} d={d} accumulate"
            assert not np.any(host(A.split_count)), f"{what} d={d}: split_count not re-armed"


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["default", "0", "1", "2", "3", "4", "unsorted", "reserve1", "reserve_all_but_1"])
def test_spmm_plan_edges_bit_exact_every_variant(variant, monkeypatch):
    """Row lengths 0 / 1 / 127 / 128 / 129 / 255 / 256 / 257, 256 chunks (last split row) and 257 chunks (first hub row),
    d = 32 .. 256, plain and accumulating: bit-exact against the oracle in every YR_SPMM_VARIANT launch shape, with the
    row-order plan and with reserved SMs. Every row of Y is written, the NaN rows of X no column references stay out."""
    from yelprecommendation_b200.data.graph import CSRMatrix
    g = dev()
    rowptr, col, val = edge_matrix()
    if variant == "unsorted":
        monkeypatch.setenv("YR_SPMM_PLAN_SORT", "0")
    A = CSRMatrix(rowptr, col, val, "cuda")
    monkeypatch.delenv("YR_SPMM_PLAN_SORT", raising=False)
    assert A.n_big_rows == 1 and A.n_split_rows == 6
    if variant in "01234":
        monkeypatch.setenv("YR_SPMM_VARIANT", variant)
    if variant.startswith("reserve"):
        A.reserve_sms = 1 if variant == "reserve1" else g.sm - 1
    _spmm_sweep(g, A, f"variant {variant}")


@pytest.mark.gpu
def test_spmm_all_rows_empty():
    """a matrix without a single non-zero: Y = 0 in every row, Y += 0 leaves Y as it was"""
    from yelprecommendation_b200.data.graph import CSRMatrix
    g = dev()
    n = 1000
    A = CSRMatrix(np.zeros(n + 1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32), "cuda")
    dummy = torch.zeros(4, device="cuda")
    for d in (32, 64, 128, 256):
        st = A.struct(d)
        st.col = st.val = dummy.data_ptr()                   # nnz = 0: the pointers are never read
        X = cu(np.full((n, d), np.nan, np.float32))
        Y = sentinel(n, d)
        assert g.lib.yr_spmm_csr(C.byref(st), d, ptr1(X), ptr1(Y), 0, g.st()) == YR_OK
        assert same_bits(host(Y), np.zeros((n, d), np.float32)), d
        Y0 = np.random.default_rng(d).standard_normal((n, d)).astype(np.float32)
        Ya = cu(Y0)
        assert g.lib.yr_spmm_csr(C.byref(st), d, ptr1(X), ptr1(Ya), 1, g.st()) == YR_OK
        assert same_bits(host(Ya), Y0), d


# ----------------------------------------------------------------------------------------------------------------------
# GPU: the row-sparse top layer, stage by stage, through NGCFTrainer.train_step_on_device
# ----------------------------------------------------------------------------------------------------------------------
LR = 0.05


@lru_cache(maxsize=2)
def graph(kind):
    """'skewed': the 2,500 x 3,500 degree-skewed synthetic graph; 'hub': 34,000 users x 300 items with item 0 in 33,000
    interactions (a row of 258 chunks: the scatter and the row-subset SpMM walk a hub row)"""
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.data.graph import build_laplacian
    if kind == "skewed":
        inter = syn.make_interactions(num_users=2500, num_items=3500, nnz=90_000, seed=8, n_clusters=8)
        nU, nI, user, item, rating = inter.num_users, inter.num_items, inter.user, inter.item, inter.rating
    else:
        rng = np.random.default_rng(4)
        nU, nI = 34_000, 300
        user = np.concatenate([np.arange(33_000), np.arange(nU)])
        item = np.concatenate([np.zeros(33_000, np.int64), rng.integers(1, nI, nU)])
        rating = rng.integers(1, 6, len(user)).astype(np.float32)
    Lap = build_laplacian(user, item, rating, nU, nI)
    Lc = Lap.coalesce()
    idx, val = Lc.indices().numpy(), Lc.values().numpy()
    from yelprecommendation_b200.data.graph import coo_to_csr
    rowptr, col, v = coo_to_csr(idx[0], idx[1], val, nU + nI)
    return nU, nI, Lap, (rowptr, col, v), csr_parts(rowptr, col, v, nU + nI)


def batch(kind, B, seed):
    nU, nI = graph(kind)[:2]
    rng = np.random.default_rng(seed)
    uid, pos, neg = rng.integers(0, nU, B), rng.integers(0, nI, B), rng.integers(0, nI, B)
    if kind == "hub":
        pos[::2] = 0
    return uid, pos, neg


def trainer(kind, n_layers, bs, mode, top_rows=1):
    from yelprecommendation_b200.trainers import NGCFTrainer
    nU, nI, Lap = graph(kind)[:3]
    torch.manual_seed(11)
    return NGCFTrainer(cfg(optimizer="sgd", lr=LR, num_orders=n_layers, batch_size=bs, ngcf_dense_mode=mode,
                           ngcf_top_rows_mode=top_rows), nI, nU, Lap)


def params(tr):
    m = tr.model
    return dict(E0=host(m.embedding.weight.data).copy(), W1=[host(w.weight.data).copy() for w in m.W1],
                W2=[host(w.weight.data).copy() for w in m.W2])


def step(tr, uid, pos, neg):
    """one step; returns the pre-step parameters and the step loss"""
    pre = params(tr)
    sl = torch.zeros(1, device="cuda")
    tr.train_step_on_device(*(cu(np.asarray(a, np.int64)) for a in (uid, pos, neg)), step_loss=sl)
    return pre, float(host(sl)[0])


def check_step(tr, kind, pre, uid, pos, neg, loss, what):
    """every stage of the step just taken, from the GPU's own inputs to that stage (module docstring)"""
    g = dev()
    st, b = tr._state()
    nU, nI, _, (rowptr, col, val), Ap = graph(kind)
    n, d, L, mode = nU + nI, int(st.d), int(st.n_layers), int(st.dense_mode)
    B = len(uid)
    rows_path = int(st.top_rows_mode) != 0 and 3 * B <= int(st.row_list_cap)
    cap = int(st.row_list_cap)
    # 1. the row scratch is re-armed
    assert not np.any(host(b["row_flag"])) and host(b["row_count"])[0] == 0, what + ": row scratch not re-armed"
    E = [pre["E0"]] + [host(x) for x in b["E"]]
    LE = [host(x) for x in b["LE"]]
    G = [host(x) for x in b["G"]]
    dW1, dW2 = [host(x) for x in b["dW1"]], [host(x) for x in b["dW2"]]
    uid, pos, neg = (np.asarray(a, np.int64) for a in (uid, pos, neg))
    touched = np.zeros(n, bool)
    touched[uid[(uid >= 0) & (uid < nU)]] = True
    touched[nU + pos[(pos >= 0) & (pos < nI)]] = True
    touched[nU + neg[(neg >= 0) & (neg < nI)]] = True
    rows = np.flatnonzero(touched)
    # 2. / 3. forward: LE bit-exact (on the touched rows only for the top layer), E_{l+1} within tau_fwd
    for l in range(L):
        want = cport.spmm_csr(rowptr, col, val, E[l])
        sel = rows if l == L - 1 else slice(None)
        assert same_bits(LE[l][sel], want[sel]), f"{what}: LE_{l} differs from the oracle SpMM"
        z, mag = fwd_ref(E[l][sel], LE[l][sel], pre["W1"][l], pre["W2"][l])
        note(f"step fwd {'tc' if fwd_tc(d, mode) else 'fp32'}",
             worst(fwd_ratio(E[l + 1][sel], z, mag, tau_fwd(d, fwd_tc(d, mode)), SLOPE), f"{what}: E_{l + 1}"))
    # 4. the tail: G_L, and the step loss
    ref = tail_ref(E, nU, uid, pos, neg)
    note("step tail G_L", worst(ratio(G[L], ref["G"][L], ref["allow"][L]), f"{what}: G_{L}"))
    assert not np.any(G[L][~touched]), f"{what}: G_{L} written outside the batch rows"
    note("step loss", worst(ratio(np.float32(loss), ref["loss"], ref["loss_allow"]), f"{what}: step loss"))
    # 5. - 7. backward, top layer first
    for l in range(L - 1, -1, -1):
        top = l == L - 1
        dz = dz_of(G[l + 1], E[l + 1], SLOPE)
        if top:
            dz[~touched] = 0.0                  # E_L is stale off the batch rows; G_L is exactly 0 there
        tc = bwd_tc(d, mode) and (cap >= 16384 if top and rows_path else True)
        Gr, allow = layer_g_ref(ref["G"][l], ref["allow"][l], dz, E[l], LE[l], pre["W1"][l], pre["W2"][l], Ap, tc)
        fam = f"{'top' if top else 'lower'} {'rows' if top and rows_path else 'dense'} {'tc' if tc else 'fp32'}"
        note(f"step G {fam}", worst(ratio(G[l], Gr, allow), f"{what}: G_{l}"))
        sel = rows if top else slice(None)
        a1, m1, a2, m2 = dw_ref(dz[sel], E[l][sel], LE[l][sel])
        tau = (tau_dw(d, len(rows), tc, g.sm, cap=cap) if top and rows_path else tau_dw(d, n, tc, g.sm))
        note(f"step dW {fam}", max(worst(ratio(dW1[l], a1, tau * m1), f"{what}: dW1_{l}"),
                                   worst(ratio(dW2[l], a2, tau * m2), f"{what}: dW2_{l}")))
    # 8. SGD, bit for bit from the GPU's gradients
    m = tr.model
    zero = lambda a: np.zeros_like(a)

    def sgd(p, gr):
        p = p.copy()
        cport.dense_opt_step(p, gr, zero(p), zero(p), cport.make_opt("sgd", LR, 0.0, 1))
        return p

    assert same_bits(host(m.embedding.weight.data), sgd(pre["E0"], G[0])), f"{what}: embedding update"
    for l in range(L):
        assert same_bits(host(m.W1[l].weight.data), sgd(pre["W1"][l], dW1[l])), f"{what}: W1_{l} update"
        assert same_bits(host(m.W2[l].weight.data), sgd(pre["W2"][l], dW2[l])), f"{what}: W2_{l} update"
    return rows_path


@pytest.mark.gpu
@pytest.mark.parametrize("n_layers", [1, 3])
@pytest.mark.parametrize("bs", [2048, 8192])
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("B", ["1", "37", "bs"])
def test_row_sparse_top_layer_stage_by_stage(n_layers, bs, mode, B):
    """cfg.batch_size 2,048 lists up to 12,288 rows (FP32-pipe row backward), 8,192 up to 24,576 (tensor-core row
    backward in dense mode 2); the actual batch is 1 (three listed rows: most CTAs write zero partials), 37 or the full
    batch. Every stage within its bound."""
    Bn = bs if B == "bs" else int(B)
    tr = trainer("skewed", n_layers, bs, mode)
    uid, pos, neg = batch("skewed", Bn, Bn + mode)
    pre, loss = step(tr, uid, pos, neg)
    assert check_step(tr, "skewed", pre, uid, pos, neg, loss, f"L={n_layers} bs={bs} mode={mode} B={Bn}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("n_layers", [1, 3])
def test_dense_top_layer_passes_the_same_stage_checks(mode, n_layers):
    """cfg.ngcf_top_rows_mode = 0 (the top layer on every row) on the same inputs: the same stage checks hold"""
    for B in (37, 2048):
        tr = trainer("skewed", n_layers, 2048, mode, top_rows=0)
        uid, pos, neg = batch("skewed", B, B + mode)
        pre, loss = step(tr, uid, pos, neg)
        assert not check_step(tr, "skewed", pre, uid, pos, neg, loss, f"dense top L={n_layers} mode={mode} B={B}")


@pytest.mark.gpu
@pytest.mark.parametrize("bs,kernel,absent", [(2048, "ngcf_dense_bwd_kernel", "ngcf_dense_bwd_tc_kernel"),
                                              (8192, "ngcf_dense_bwd_tc_kernel", "ngcf_dense_bwd_kernel")])
def test_row_backward_branch_is_the_one_that_ran(bs, kernel, absent):
    """One layer in dense mode 2, so the top layer's row backward is the only backward of the step: the profiler sees the
    FP32-pipe row kernel at batch size 2,048 and the tensor-core one at 8,192, each with the scatter of L^T T"""
    from torch.profiler import ProfilerActivity, profile
    tr = trainer("skewed", 1, bs, 2)
    uid, pos, neg = batch("skewed", bs, 3)
    tr._state()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pre, loss = step(tr, uid, pos, neg)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert any(kernel in k for k in names), sorted(names)
    assert not any(absent in k for k in names), sorted(names)
    assert any("spmm_scatter_rows_kernel" in k for k in names), sorted(names)
    assert check_step(tr, "skewed", pre, uid, pos, neg, loss, f"profiled bs={bs}")


@pytest.mark.gpu
@pytest.mark.parametrize("bs", [2048, 8192])
def test_consecutive_steps_on_overlapping_batches(bs):
    """the second step lists the rows the first one listed too: a stale flag would silently drop them from the list"""
    tr = trainer("skewed", 3, bs, 2)
    u1, p1, n1 = batch("skewed", bs, 5)
    u2, p2, n2 = batch("skewed", bs, 6)
    h = bs // 2
    u2[:h], p2[:h], n2[:h] = u1[h:], p1[h:], n1[h:]
    for k, (u, p, q) in enumerate(((u1, p1, n1), (u2, p2, n2))):
        pre, loss = step(tr, u, p, q)
        assert check_step(tr, "skewed", pre, u, p, q, loss, f"consecutive bs={bs} step {k}")


@pytest.mark.gpu
def test_error_exit_rearms_row_scratch_and_leaves_parameters():
    """yr_ngcf_train_step_ex on a copy of the state with dW1[L-1] = NULL fails in the backward, after the row list was
    built: YR_ERR_BAD_ARG, the row scratch re-armed, no parameter changed; the next normal step passes every check"""
    from yelprecommendation_b200 import _cabi
    tr = trainer("skewed", 3, 2048, 2)
    st, b = tr._state()
    uid, pos, neg = batch("skewed", 2048, 9)
    bad = _cabi.YrNgcfState.from_buffer_copy(st)
    bad.dW1[2] = None
    before = params(tr)
    opt = tr.optimizer.opt_struct(tr.optimizer.step_count + 1)
    ud, pd, nd = (cu(a.astype(np.int64)) for a in (uid, pos, neg))
    rc = _cabi.load().yr_ngcf_train_step_ex(C.byref(bad), C.byref(opt), SLOPE, ptr1(ud), ptr1(pd), ptr1(nd), 2048, None, 0,
                                            _cabi.stream_ptr())
    assert rc == YR_ERR_BAD_ARG
    assert not np.any(host(b["row_flag"])) and host(b["row_count"])[0] == 0
    after = params(tr)
    assert same_bits(after["E0"], before["E0"]) and all(same_bits(a, c) for a, c in zip(after["W1"] + after["W2"],
                                                                                      before["W1"] + before["W2"]))
    b["loss"].zero_()
    pre, loss = step(tr, uid, pos, neg)
    assert check_step(tr, "skewed", pre, uid, pos, neg, loss, "after the error exit")


@pytest.mark.gpu
def test_out_of_range_id_flags_rearms_and_drops_only_that_triple():
    """one out-of-range item id: err = 1 (the trainer raises IndexError), the scratch is re-armed, and G matches the
    reference without that triple (the others still divided by the full B)"""
    tr = trainer("skewed", 3, 2048, 2)
    nI = graph("skewed")[1]
    uid, pos, neg = batch("skewed", 2048, 10)
    pos[100] = nI
    pre, loss = step(tr, uid, pos, neg)
    assert host(tr._bufs["err"])[0] == 1
    with pytest.raises(IndexError):
        tr.loss_sum()
    assert check_step(tr, "skewed", pre, uid, pos, neg, loss, "bad id")


@pytest.mark.gpu
def test_prefix_done_gives_the_same_stages():
    """the batch-independent layers pre-propagated behind the previous step (prefix_done = L - 1): same bounds"""
    tr = trainer("skewed", 3, 2048, 2)
    uid, pos, neg = batch("skewed", 2048, 12)
    st, _ = tr._state()
    tr._prepropagate(st)
    assert tr._prefix_tag is not None and tr._prefix_tag[1] == 2
    pre, loss = step(tr, uid, pos, neg)
    assert check_step(tr, "skewed", pre, uid, pos, neg, loss, "prefix_done = L - 1")


@pytest.mark.gpu
@pytest.mark.parametrize("n_layers", [1, 3])
def test_hub_row_scatter_and_row_subset_spmm(n_layers):
    """an item row of 33,000 non-zeros in the batch: the row-subset SpMM finishes a hub row and the scatter walks its
    258 chunks"""
    tr = trainer("hub", n_layers, 2048, 2)
    uid, pos, neg = batch("hub", 2048, 13)
    pre, loss = step(tr, uid, pos, neg)
    assert check_step(tr, "hub", pre, uid, pos, neg, loss, f"hub L={n_layers}")
