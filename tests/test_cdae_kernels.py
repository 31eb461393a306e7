"""The CDAE train step (yr_cdae_step_ex, yr_cdae_step_idx) kernel by kernel, and the dense drop-ins yr_cdae_output /
yr_nsbce_loss, each against a float64 reference with a per-element bound |x - ref| <= allowance + ulp(x). u = 2^-24;
ulp(x) covers the final rounding to fp32. Shared helpers come from ngcf_ref.py.

Reading the gradients. Every step entry point runs the optimizer and then clears the gradients. The GPU tests step with
Adam at beta1 = 0, step 1, zeroed moments: the first moment is fmaf(1, g - 0, 0) = g bit for bit (common.cuh opt_update),
so m is the gradient. The second moment and the updated parameters are then checked bit for bit against the C oracle's
dense step fed with that gradient, which also checks that every tensor was stepped with its own size; the gradient
buffers must be all zero on return.

Hidden layer (cdae_compact_kernel + phase 1 of cdae_row_kernel; the index-list path stages its lists instead).
    pre = bh + Vu[u] + sum_j xv_j Wh[:, j],  xv = fl(x keep),  z = act(pre)
* G = 256 / h fma chains (G = 1 from h = 256) of ceil(nx / G) terms over the nx compacted (or listed) inputs, G - 1 adds
  combining them, one add for bh + Vu and one for the sum: tau_pre = (ceil(nx / G) + G + 1) u on
  |bh| + |Vu| + sum |xv Wh|.
* identity: z = pre within that. sigmoid: sigmoidf_ = 1 / (1 + expf(-x)) with expf within 2 ulp (4 u) and the add and
  the divide rounded to nearest, all monotone: for an input within pre +- b the kernel returns an fp32 value between the
  two ends sig_range() computes, and the allowance is the larger distance of an end from sigmoid(pre). The padding
  columns of z_out are exactly 1 (column h) and 0.
* Downstream, the kernel's z may be off by az = that allowance + ulp(z).

Logits, loss and dl (warp per loss position).
* logit = sum over lanes of a VPL-term fma chain (VPL = h / 32), a 5-level shuffle tree, + bo: (VPL + 6) u on
  sum |z Wo| + |bo|, plus sum |Wo| az for z's error.
* p = sigmoidf_(logit) lies in sig_range(logit, that). The reference p is the same three steps each rounded to nearest:
  at logit >= 16.64, 1 + expf(-logit) rounds to 1 and p is exactly 1 (torch's CPU sigmoid has the same form). Every test
  logit is kept at least 1 away from 16.64 and from -27.63, where (1 - p) p = 1e-12, so both ends of the range are on
  the reference's side of either threshold.
* Loss term per position -(t max(log p, -100) + (1 - t) max(log1p(-p), -100)) in float64 on the fp32 p; the kernel's
  term lies between its values at the two ends of p's range, plus 2 roundings of logf / log1pf (4 u). The terms are
  summed in double (M 2^-53 relative at most) and the mean is rounded to fp32 once.
* dl = torch's autograd chain: binary_cross_entropy's (p - t) / max((1 - p) p, 1e-12) / m, then sigmoid's (1 - p) p, in
  float64 on the fp32 p (m = loss positions of the batch). It equals (p - t) / m unless (1 - p) p < 1e-12. The kernel's
  dl = (p - t) inv_m min(1, (1 - p) p 1e12f) lies between the chain's values at the ends of p's range, plus 6 roundings
  and those of inv_m and 1e12f (12 u).

Gradients. fp32 atomics from a zeroed buffer: c addends in any order cost (c - 1) u on sum |addends|, and each addend
may lose 2^-126 to flush-to-zero. The error of an addend's factors enters as sum |factor| x allowance of the other.
* dbo[i] = sum_rows dl: (c + 1) u.   dWo[i, :] = sum_rows dl z (one product each): (c + 1) u.
* dz[r, k] = sum_positions dl Wo[i, k]: each warp one fma chain over its positions (at most ceil(nt / (8 UN)) UN of
  them, UN = 4 / 2 / 1 positions per round for VPL <= 2 / <= 8 / above), then the 8 warp partials in order:
  (n_w + 8) u on sum |dl Wo|.
* dpre = dz z (1 - z) for sigmoid (3 roundings, and z's error through d(z(1 - z))/dz = 1 - 2z) or dz for identity.
* dbh = sum_rows dpre, dVu[u] = sum over the rows of user u of dpre (duplicate user ids accumulate): (c + 1) u.
* dWh[:, j] = sum_rows dpre xv_j: (c + 1) u. An input dropped by keep is not an addend, so its element is exactly 0
  when no other row has it.

yr_cdae_output: one fma chain of h terms plus bo, (h + 1) u, then sig_range. yr_nsbce_loss: the same loss terms on the
given p, summed in double in any order, mean rounded once.

The checks have teeth: the CPU tests show that a straightforward fp32 step passes them, that torch's autograd through
oracle/torch_port.CDAEPort passes them at saturated logits, and that a gradient without its 1/m, a compaction that drops
the last column of a warp segment, dWh without keep, one batch row missing from dVu and dl = (p - t) / m at a saturated
position fail them.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from ngcf_ref import SENTINEL, U24, YR_ERR_BAD_ARG, YR_OK, Summary, cu, dev, host, ptr1, same_bits, ulp, worst
from oracle import cport

SUMMARY = Summary()
note = SUMMARY.note
KEYS = ("Wh", "bh", "Vu", "Wo", "bo")
FTZ = 2.0 ** -126                    # fp32 atomics flush subnormal operands and results to zero: per addend
SAT_HI, SAT_LO = 16.64, -27.63       # logit where p rounds to 1.0f / where (1 - p) p drops below 1e-12
ACT = {"sigmoid": 0, "identity": 1}
LR = 1e-3
NW = 32                              # warps of cdae_compact_kernel


@pytest.fixture(scope="module", autouse=True)
def report_summary(request):
    """after the module: per family, the largest error / bound ratio the GPU tests measured"""
    yield
    SUMMARY.report(request)


# ----------------------------------------------------------------------------------------------------------------------
# float64 reference and bounds (CPU)
# ----------------------------------------------------------------------------------------------------------------------
def ratio(x, ref, allow):
    """per element |x - ref| / (allow + ulp(x)); NaN / inf count as infinitely far"""
    with np.errstate(invalid="ignore"):
        r = np.abs(np.asarray(x, np.float64) - ref) / (allow + ulp(x))
    return np.where(np.isfinite(r), r, np.inf)


def _rn32(x):
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float64)


def sig32(x):
    """sigmoidf_ with expf, the add and the divide each rounded to nearest: the fp32 p of the reference"""
    with np.errstate(over="ignore"):
        return _rn32(1.0 / _rn32(1.0 + _rn32(np.exp(-x))))


def sig_range(x, a):
    """the ends of the fp32 values sigmoidf_ can return for an input within x +- a (expf within 2 ulp)"""
    with np.errstate(over="ignore"):
        e_lo, e_hi = np.exp(-(x + a)) * (1 - 4 * U24), np.exp(-(x - a)) * (1 + 4 * U24)
        return _rn32(1.0 / _rn32(1.0 + e_hi)), _rn32(1.0 / _rn32(1.0 + e_lo))


def bce(p, t):
    """the loss term with torch's -100 clamps, float64 on the fp32 p"""
    with np.errstate(divide="ignore"):
        return -(t * np.maximum(np.log(p), -100.0) + (1 - t) * np.maximum(np.log1p(-p), -100.0))


def dlogit(p, t):
    """torch's autograd chain d bce / d logit: (p - t) / max((1 - p) p, 1e-12) * (1 - p) p"""
    q = (1 - p) * p
    return (p - t) / np.maximum(q, 1e-12) * q


def _spread(f, p, lo, hi, t):
    v, a, b = f(p, t), f(lo, t), f(hi, t)
    return v, np.maximum(np.abs(a - v), np.abs(b - v)), np.maximum(np.abs(a), np.abs(b))


def shape_of(h):
    """(G, VPL, UN) of cdae_row_kernel at hidden size h"""
    vpl = h // 32
    return max(1, 256 // h), vpl, (4 if vpl <= 2 else (2 if vpl <= 8 else 1))


def cdae_ref(P, uid, xv, tgt, pos, act, listed=None, rule=dlogit):
    """Forward, loss and dl of one step in float64 with their allowances (module docstring). xv: the fp32 inputs after
    keep; tgt: the targets; pos: the loss positions; listed: the inputs the hidden chains walk (default xv != 0, the
    compaction; the index-list path walks every listed input, zeros included)."""
    Wh, bh, Vu, Wo, bo = (P[k].astype(np.float64) for k in KEYS)
    h = Wh.shape[0]
    uid = np.asarray(uid, np.int64)
    G, vpl, un = shape_of(h)
    x = xv.astype(np.float64)
    nx = (xv != 0 if listed is None else listed).sum(1)
    pre = bh + Vu[uid] + x @ Wh.T
    b_pre = ((np.ceil(nx / G) + G + 1) * U24)[:, None] * (np.abs(bh) + np.abs(Vu[uid]) + np.abs(x) @ np.abs(Wh).T)
    if act == "sigmoid":
        z = 1.0 / (1.0 + np.exp(-pre))
        lo, hi = sig_range(pre, b_pre)
        a_z = np.maximum(hi - z, z - lo)
    else:
        z, a_z = pre, b_pre
    az = a_z + ulp(z)
    aWo = np.abs(Wo)
    logit = z @ Wo.T + bo
    a_logit = (vpl + 6) * U24 * (np.abs(z) @ aWo.T + np.abs(bo)) + az @ aWo.T
    lp = logit[pos]
    assert np.all((np.abs(lp - SAT_HI) >= 1) & (np.abs(lp - SAT_LO) >= 1)), "a test logit is near a threshold"
    t = tgt.astype(np.float64)
    p = sig32(logit)
    p_lo, p_hi = sig_range(logit, a_logit)
    ell, d_ell, m_ell = _spread(bce, p, p_lo, p_hi, t)
    M = int(pos.sum())
    f, d_f, m_f = _spread(rule, p, p_lo, p_hi, t)
    inv = 1.0 / M if M else np.nan
    D = np.where(pos, f * inv, 0.0)
    A = np.where(pos, (d_f + 12 * U24 * m_f) * inv, 0.0)
    loss = ell[pos].sum() * inv
    a_loss = (d_ell + 4 * U24 * m_ell)[pos].sum() * inv + M * 2.0 ** -53 * abs(loss)
    nt = pos.sum(1)
    n_w = np.ceil(nt / (8 * un)) * un
    dz = D @ Wo
    a_dz = A @ aWo + ((n_w + 8) * U24)[:, None] * (np.abs(D) @ aWo)
    if act == "sigmoid":
        s = z * (1 - z)
        dpre = dz * s
        a_dpre = a_dz * s + np.abs(dz) * np.abs(1 - 2 * z) * az + 3 * U24 * np.abs(dpre)
    else:
        dpre, a_dpre = dz, a_dz
    return dict(pre=pre, z=z, a_z=a_z, az=az, logit=logit, loss=loss, a_loss=a_loss, D=D, A=A, dpre=dpre,
                a_dpre=a_dpre, uid=uid, x=x, pos=pos, nU=P["Vu"].shape[0], M=M)


def grad_refs(r):
    """(name, float64 gradient, allowance) per parameter, one at a time (the h = 1,024 Yelp-shape tensors are large)"""
    D, A, z, az, dpre, a_dpre, x, uid = (r[k] for k in ("D", "A", "z", "az", "dpre", "a_dpre", "x", "uid"))
    B = len(uid)
    aD, az_, adp, ax = np.abs(D), np.abs(z), np.abs(dpre), np.abs(x)
    c = r["pos"].sum(0).astype(np.float64)
    yield "bo", D.sum(0), A.sum(0) + (c + 1) * U24 * aD.sum(0) + c * FTZ
    c = c[:, None]
    yield "Wo", D.T @ z, A.T @ az_ + aD.T @ az + (c + 1) * U24 * (aD.T @ az_) + c * FTZ
    yield "bh", dpre.sum(0), a_dpre.sum(0) + (B + 1) * U24 * adp.sum(0) + B * FTZ
    U = np.zeros((r["nU"], B))
    U[uid, np.arange(B)] = 1.0
    c = U.sum(1)[:, None]
    yield "Vu", U @ dpre, U @ a_dpre + (c + 1) * U24 * (U @ adp) + c * FTZ
    c = (x != 0).sum(0)[None, :].astype(np.float64)
    yield "Wh", dpre.T @ x, a_dpre.T @ ax + (c + 1) * U24 * (adp.T @ ax) + c * FTZ


def z_ratio(z, r):
    return ratio(z, r["z"], r["a_z"])


def check_step(r, z, loss, grads, what, fam=None):
    """z (if given), the step loss and every gradient element within bound; notes the ratios under `fam`"""
    out = {}
    if z is not None:
        out["hidden z"] = worst(z_ratio(z, r), f"{what}: z")
    if loss is None:
        pass
    elif r["M"] == 0:
        assert np.isnan(loss), f"{what}: the mean over no loss positions is NaN"
    else:
        out["loss"] = worst(ratio(np.float32(loss), r["loss"], r["a_loss"]), f"{what}: loss")
    if grads is not None:
        for k, ref, allow in grad_refs(r):
            out[f"d{k}"] = worst(ratio(grads[k], ref, allow), f"{what}: d{k}")
    if fam is not None:
        for k, v in out.items():
            note(f"{fam} {k}", v)
    return out


# ---- cases ------------------------------------------------------------------------------------------------------------
def make_params(nI, h, nU, rng):
    f = np.float32
    a = np.sqrt(6.0 / (h + nI))
    return {"Wh": rng.uniform(-a, a, (h, nI)).astype(f), "bh": rng.uniform(-0.5, 0.5, h).astype(f),
            "Vu": (rng.standard_normal((nU, h)) * 0.3).astype(f),
            "Wo": (rng.standard_normal((nI, h)) * 0.5 / np.sqrt(h)).astype(f), "bo": rng.uniform(-1, 1, nI).astype(f)}


def seg_ends(nI):
    """the last column of every non-empty warp segment of cdae_compact_kernel"""
    per_warp = -(-nI // NW)
    seg = -(-per_warp // 32) * 32
    return np.unique(np.minimum(np.arange(1, NW + 1) * seg, nI) - 1)


def edge_case(nI, h=64, seed=0, nU=40):
    """B = 8 rows: 0 no inputs (negatives only), 1 every column an input and a target (non-binary x), 2 inputs but no
    loss position, 3 keep zeroes every input, 4 / 5 hold the last column of every warp segment, 4 has a position that is
    both a target and a sampled negative, 5 / 6 share a user; non-binary x and dropout keep (0 or 2.5) elsewhere"""
    rng = np.random.default_rng(1000 * seed + nI)
    P = make_params(nI, h, nU, rng)
    B = 8
    uid = rng.choice(nU, B, replace=False)
    uid[6] = uid[5]
    dens = min(0.5, 24.0 / nI)
    x = (rng.random((B, nI)) < dens).astype(np.float32)
    x[0] = 0.0
    x[1] = rng.uniform(0.5, 3.0, nI)
    x[4:6, seg_ends(nI)] = 1.0
    x[5] *= rng.integers(1, 6, nI)                                   # ratings 1..5
    keep = np.where(rng.random((B, nI)) < 0.6, 0.0, 2.5).astype(np.float32)
    keep[1] = 1.0
    keep[4:6, seg_ends(nI)] = 2.5
    keep[3] = 0.0
    tgt = (x != 0).astype(np.float32)
    tgt[2] = 0.0
    neg = np.zeros_like(x)
    for b in (0, 3, 4, 5, 6, 7):
        free = np.flatnonzero(tgt[b] == 0)
        neg[b, rng.choice(free, min(len(free), 5 * max(1, int(tgt[b].sum())) if b else 3), replace=False)] = 1.0
    on = np.flatnonzero(tgt[4])
    neg[4, on[len(on) // 2]] = 1.0                                   # target and negative: one loss position
    return P, uid, x, keep, tgt, neg


def positions(tgt, neg):
    return (tgt + neg) != 0


def yelp_rows(nI, B, seed):
    """Yelp-like train lists (a heavy-tailed length, popularity-skewed items, one user with 2,500) and 5x sampled
    negatives drawn the way bench.py's CDAE block draws them"""
    rng = np.random.default_rng(seed)
    pop = 1.0 / (np.arange(nI) + 10.0) ** 0.8
    pop = pop[rng.permutation(nI)]
    pop /= pop.sum()
    lens = np.clip(rng.lognormal(3.0, 1.0, B), 1, 1500).astype(int)
    lens[0] = 2500
    x = np.zeros((B, nI), np.float32)
    neg = np.zeros_like(x)
    for r in range(B):
        items = rng.choice(nI, lens[r], replace=False, p=pop)
        x[r, items] = 1.0
        cand = rng.integers(0, nI, size=5 * len(items) + 8)
        cand = cand[x[r, cand] == 0][: 5 * len(items)]
        neg[r, cand] = 1.0
    keep = np.where(rng.random((B, nI)) < 0.6, 0.0, 2.5).astype(np.float32)
    return x, keep, neg


def saturation_case(h=64, nI=300, nU=20, seed=5):
    """items 0..7 have Wo = 0, so their logit is exactly bo: 18 and 19 as sampled negatives and targets, 18.5 as a
    negative only, -30 and -40 as targets, unsaturated controls 15 (negative and target) and -25 (target)"""
    rng = np.random.default_rng(seed)
    P = make_params(nI, h, nU, rng)
    P["Wo"][:8] = 0.0
    P["bo"][:8] = [18.0, 19.0, 18.5, -30.0, -40.0, 15.0, -25.0, 15.0]
    B = 4
    uid = np.array([3, 7, 3, 11])
    x = (rng.random((B, nI)) < 0.08).astype(np.float32)
    x[:, :8] = 0.0
    tgt = x.copy()
    neg = np.zeros_like(x)
    for b in range(B):
        free = np.flatnonzero((tgt[b] == 0) & (np.arange(nI) >= 8))
        neg[b, rng.choice(free, 20, replace=False)] = 1.0
    neg[:3, 0] = neg[:2, 2] = neg[2:, 1] = neg[0, 5] = 1.0           # saturated negatives, a control negative
    tgt[:2, 1] = tgt[3, 0] = tgt[:, 3] = tgt[1:3, 4] = tgt[2:, 6] = tgt[1, 7] = 1.0
    keep = np.where(rng.random((B, nI)) < 0.6, 0.0, 2.5).astype(np.float32)
    return P, uid, x, keep, tgt, neg


# ---- a straightforward fp32 step and its mutants (CPU) ----------------------------------------------------------------
def step_fp32(P, uid, xv, tgt, pos, act, simple_dl=False):
    """(z, loss, gradients) of one step in plain numpy fp32: BLAS sums, sigmoid as 1 / (1 + exp(-x))"""
    f = np.float32
    sig = lambda v: (f(1) / (f(1) + np.exp(-v))).astype(f)
    pre = P["bh"] + P["Vu"][uid] + xv @ P["Wh"].T
    z = sig(pre) if act == "sigmoid" else pre
    p = sig(z @ P["Wo"].T + P["bo"])
    M = int(pos.sum())
    loss = f(bce(p.astype(np.float64), tgt)[pos].sum() / M)
    inv = f(1.0 / M)
    if simple_dl:
        dl = (p - tgt) * inv
    else:
        dl = (p - tgt) / np.maximum((f(1) - p) * p, f(1e-12)) * inv * (f(1) - p) * p
    D = np.where(pos, dl, f(0)).astype(f)
    dz = D @ P["Wo"]
    dpre = (dz * z * (f(1) - z)).astype(f) if act == "sigmoid" else dz
    dVu = np.zeros_like(P["Vu"])
    np.add.at(dVu, uid, dpre)
    return z, loss, {"bo": D.sum(0), "Wo": D.T @ z, "bh": dpre.sum(0), "Vu": dVu, "Wh": dpre.T @ xv}, dpre


@pytest.mark.parametrize("h,act", [(32, "sigmoid"), (64, "sigmoid"), (256, "identity"), (1024, "sigmoid")])
@pytest.mark.parametrize("nI", [33, 1025])
def test_fp32_step_within_bounds(h, act, nI):
    P, uid, x, keep, tgt, neg = edge_case(nI, h, seed=1)
    xv, pos = x * keep, positions(tgt, neg)
    r = cdae_ref(P, uid, xv, tgt, pos, act)
    z, loss, grads, _ = step_fp32(P, uid, xv, tgt, pos, act)
    check_step(r, z, loss, grads, f"fp32 step h={h} {act} nI={nI}")


def test_mutants_fail():
    """a gradient without its 1/m, a compaction that drops the last column of a warp segment, dWh without keep and one
    batch row missing from dVu are each outside the bound they target"""
    nI, h, act = 8193, 64, "sigmoid"
    P, uid, x, keep, tgt, neg = edge_case(nI, h, seed=2)
    xv, pos = x * keep, positions(tgt, neg)
    r = cdae_ref(P, uid, xv, tgt, pos, act)
    z, loss, grads, dpre = step_fp32(P, uid, xv, tgt, pos, act)
    check_step(r, z, loss, grads, "exact fp32 step")
    refs = {k: (ref, allow) for k, ref, allow in grad_refs(r)}
    over = lambda k, g: ratio(g, *refs[k]).max() > 1.0
    for k in KEYS:
        assert over(k, grads[k] * np.float32(r["M"])), f"d{k} without 1/m"
    ends = seg_ends(nI)
    assert len(ends) == 29 and ends[-2] == 28 * 288 - 1                # 288-column segments, warps 29 .. 31 empty
    for c in ends[[0, 13, -2]]:                                      # a full segment's last column
        dropped = xv.copy()
        dropped[4, c] = 0.0
        zd = step_fp32(P, uid, dropped, tgt, pos, act)[0]
        assert z_ratio(zd, r)[4].max() > 1.0, f"compaction without column {c}"
    assert not np.array_equal(x, xv)
    assert over("Wh", dpre.T @ x), "dWh without keep"
    dVu = grads["Vu"].copy()
    dVu[uid[6]] -= dpre[6]
    assert uid[6] == uid[5] and over("Vu", dVu), "dVu without row 6"


def test_saturated_positions_take_torchs_gradient_cpu():
    """CDAEPort's autograd (torch's sigmoid and binary_cross_entropy backward) and the torch-chain fp32 step pass the
    bounds on the saturation batch; dl = (p - t) / m at a saturated position fails the dbo bound"""
    from oracle import torch_port as tp
    act = "sigmoid"
    P, uid, x, keep, tgt, neg = saturation_case()
    xv, pos = x * keep, positions(tgt, neg)
    r = cdae_ref(P, uid, xv, tgt, pos, act)
    L = r["logit"]
    assert np.all(L[:, :8][pos[:, :8]] == np.repeat(P["bo"][None, :8], 4, 0)[pos[:, :8]])
    dbo = dict((k, (a, b)) for k, a, b in grad_refs(r))["bo"]
    assert np.all(dbo[0][[0, 1, 2]] == 0.0) and np.all(dbo[0][[3, 4]] != 0.0)
    z, loss, grads, _ = step_fp32(P, uid, xv, tgt, pos, act)
    check_step(r, z, None, grads, "fp32 step, saturated")
    names = {"Wh": "hidden_layer.weight", "bh": "hidden_layer.bias", "Vu": "user_nodes.weight",
             "Wo": "output_layer.weight", "bo": "output_layer.bias"}
    port = tp.CDAEPort({names[k]: torch.from_numpy(P[k].copy()) for k in KEYS})
    t = lambda a: torch.from_numpy(a.copy())
    pl = tp.nsbce_loss(port.forward(t(uid), t(x), t(keep)), t(tgt), t(neg))
    pl.backward()
    pg = {k: getattr(port, k).grad.numpy() for k in KEYS}
    check_step(r, None, pl.item(), pg, "CDAEPort autograd, saturated")
    simple = step_fp32(P, uid, xv, tgt, pos, act, simple_dl=True)[2]["bo"]
    rb = ratio(simple, *dbo)
    assert rb[[0, 1, 2, 3, 4]].min() > 1.0 and rb[5:].max() <= 1.0, rb[:8]


def test_sig_range_and_thresholds():
    """the reference's p: exactly 1 from 16.64 up, (1 - p) p = 1e-12 at -27.63; sig_range brackets the float32
    evaluation of sigmoidf_ at every input within the allowance"""
    f = np.float32
    assert sig32(np.float64(SAT_HI + 0.01)) == 1.0 and sig32(np.float64(SAT_HI - 0.01)) < 1.0
    q = lambda v: (1 - sig32(v)) * sig32(v)
    assert q(SAT_LO + 0.01) > 1e-12 > q(SAT_LO - 0.01)
    xs = np.random.default_rng(0).uniform(-40, 40, 100_000)
    a = np.abs(xs) * 4 * U24
    lo, hi = sig_range(xs, a)
    for d in (-0.5, 0.0, 0.5):                                        # fp32 rounding of x + d a stays within a
        xk = (xs + d * a).astype(f)
        pk = (f(1) / (f(1) + np.exp(-xk))).astype(np.float64)
        assert np.all((lo <= pk) & (pk <= hi))


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
def _opt():
    from yelprecommendation_b200 import _cabi
    return _cabi.YrOpt(_cabi.YR_OPT_ADAM, 1, LR, 0.0, 0.0, 0.999, 1e-8)


def _pack(d):
    from yelprecommendation_b200 import _cabi
    return _cabi.YrCdaeTensors(*[ptr1(d[k]) for k in KEYS])


def _sets(P, layout):
    """device parameters, gradients, m and v: separate allocations, or views of one flat buffer. "offset": every view
    starts 4 bytes past a 16-byte boundary except P.Wo and g.Wo, which the row kernel reads as float4 (all five tensors
    take the optimizer's single-tensor path: m.Wo and v.Wo are off); "wo_off": P.Wo too, "gwo_off": g.Wo too."""
    names = [(s, k) for s in ("P", "g", "m", "v") for k in KEYS]
    if layout == "separate":
        out = {(s, k): (cu(P[k]) if s == "P" else torch.zeros(P[k].shape, device="cuda")) for s, k in names}
    else:
        vec = {("P", "Wo"), ("g", "Wo")} - {{"wo_off": ("P", "Wo"), "gwo_off": ("g", "Wo")}.get(layout)}
        offs, o = [], 0
        for s, k in names:
            o += (-o) % 4 if (s, k) in vec else (1 - o) % 4
            offs.append(o)
            o += P[k].size
        flat = torch.zeros(o + 4, device="cuda")
        out = {}
        for (s, k), o in zip(names, offs):
            out[(s, k)] = flat[o: o + P[k].size].view(P[k].shape)
            assert (out[(s, k)].data_ptr() % 16) == (0 if (s, k) in vec else 4)
            if s == "P":
                out[(s, k)].copy_(cu(P[k]))
    return {s: {k: out[(s, k)] for k in KEYS} for s in ("P", "g", "m", "v")}


def lists(x, keep, tgt, neg):
    """index-list batch (data/cdae_sparse.py's layout): inputs x != 0 with their value after keep, loss positions
    (target + negative != 0) with the target"""
    def csr(mask):
        r, c = np.nonzero(mask)
        return np.concatenate([[0], np.cumsum(mask.sum(1))]).astype(np.int32), c.astype(np.int32), r
    in_ptr, in_idx, ir = csr(x != 0)
    lp, li, lr = csr(positions(tgt, neg))
    in_val = None if keep is None else (x * keep)[ir, in_idx].astype(np.float32)
    return in_ptr, in_idx, in_val, lp, li, tgt[lr, li].astype(np.float32)


def ws_z(ws, B, nI, h):
    """the step's hidden activations, [B x h], in its workspace (csrc/cdae.cu cdae_ws_layout: two [B] counts, the
    total, four [B x nI] lists, then z; every piece 256-byte aligned)"""
    r = lambda b: -(-b // 256) * 256
    o = 2 * r(4 * B) + r(16) + 4 * r(4 * B * nI)
    return host(ws[o: o + 4 * B * h].view(torch.float32)).reshape(B, h).copy()


def run_step(P, uid, x, keep, tgt, neg, act, entry="dense", layout="separate", train=True, lst=None, rc_want=YR_OK):
    """one yr_cdae_step_ex (dense) or yr_cdae_step_idx (lists) call. With train: the gradients read out through Adam at
    beta1 = 0 (module docstring), v and the parameters checked bit for bit against the C oracle's step, the gradient
    buffers all zero. Without: parameters, gradients and moments (pre-filled) untouched bit for bit."""
    g = dev()
    nU, h = P["Vu"].shape
    nI, B = P["bo"].size, len(uid)
    S = _sets(P, layout)
    if not train or rc_want != YR_OK:
        for s in ("g", "m", "v"):
            for k in KEYS:
                S[s][k].copy_(cu(np.full(P[k].shape, SENTINEL, np.uint32).view(np.float32)))
    before = {s: {k: host(t).copy() for k, t in S[s].items()} for s in (S if not train or rc_want else ("P",))}
    Pt, Gt, Mt, Vt = (_pack(S[s]) for s in ("P", "g", "m", "v"))
    ws = torch.empty(g.lib.yr_cdae_ws_bytes(B, nI), dtype=torch.uint8, device="cuda")
    loss = torch.zeros(2, dtype=torch.float64, device="cuda")
    sl = torch.full((1,), 7.0, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    ud = cu(np.asarray(uid, np.int64))
    opt = _opt()
    head = (C.byref(Pt), C.byref(Gt), C.byref(Mt), C.byref(Vt), C.byref(opt) if train else None, nU, nI, h, ACT[act],
            ptr1(ud))
    tail = (B, ptr1(loss), ptr1(sl), ptr1(ws), ws.numel(), ptr1(err), g.st())
    if entry == "dense":
        xd, td, nd = cu(x), cu(tgt), cu(neg)
        kd = cu(keep) if keep is not None else None
        rc = g.lib.yr_cdae_step_ex(*head, ptr1(xd), ptr1(kd) if kd is not None else None, ptr1(td), ptr1(nd), *tail)
    else:
        ip, ii, iv, lp, li, lv = lst if lst is not None else lists(x, keep, tgt, neg)
        pad = lambda a: np.concatenate([a, np.zeros(1, a.dtype)])   # an empty list still has a buffer
        dl = [cu(ip), cu(pad(ii)), cu(lp), cu(pad(li)), cu(pad(lv))] + [cu(pad(iv)) if iv is not None else None]
        rc = g.lib.yr_cdae_step_idx(*head, ptr1(dl[0]), ptr1(dl[1]), ptr1(dl[5]) if iv is not None else None,
                                    ptr1(dl[2]), ptr1(dl[3]), ptr1(dl[4]), *tail)
    assert rc == rc_want
    if rc != YR_OK:
        assert host(sl)[0] == 7.0 and not np.any(host(loss)) and host(err)[0] == 0
        for s in S:
            for k in KEYS:
                assert same_bits(host(S[s][k]), before[s][k]), f"rejected call changed {s}.{k}"
        return None
    out = {"loss": float(host(sl)[0]), "loss_sum": host(loss).copy(), "z": ws_z(ws, B, nI, h)}
    assert host(err)[0] == 0
    assert out["loss_sum"][1] == 0.0 and (out["loss_sum"][0] == out["loss"] or np.isnan(out["loss"]))
    after = {s: {k: host(t).copy() for k, t in S[s].items()} for s in S}
    if not train:
        for s in before:
            for k in KEYS:
                assert same_bits(after[s][k], before[s][k]), f"loss-only pass changed {s}.{k}"
        return out
    copt = cport.make_opt("adam", LR, 0.0, 1, (0.0, 0.999), 1e-8)
    grads = {}
    for k in KEYS:
        gk = after["m"][k]
        p, m, v = before["P"][k].copy(), np.zeros_like(gk), np.zeros_like(gk)
        cport.dense_opt_step(p, gk, m, v, copt)
        assert same_bits(m, gk) and same_bits(after["v"][k], v) and same_bits(after["P"][k], p), f"Adam step of {k}"
        assert not np.any(after["g"][k]), f"gradient {k} not cleared"
        grads[k] = gk
    out["grads"], out["v"], out["P"] = grads, {k: after["v"][k] for k in KEYS}, {k: after["P"][k] for k in KEYS}
    return out


def run_hidden(P, uid, x, keep, act, extra=32):
    """yr_cdae_hidden_ex into z_out [B x (h + extra)] filled with the sentinel"""
    g = dev()
    nU, h = P["Vu"].shape
    nI, B = P["bo"].size, len(uid)
    Pd = {k: cu(P[k]) for k in KEYS}
    Pt = _pack(Pd)
    ldz = h + extra
    zo = cu(np.full((B, ldz), SENTINEL, np.uint32).view(np.float32))
    ws = torch.empty(g.lib.yr_cdae_ws_bytes(B, nI), dtype=torch.uint8, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    ud, xd = cu(np.asarray(uid, np.int64)), cu(x)
    kd = cu(keep) if keep is not None else None
    assert g.lib.yr_cdae_hidden_ex(C.byref(Pt), nU, nI, h, ACT[act], ptr1(ud), ptr1(xd), ptr1(kd) if kd is not None
                                   else None, B, ptr1(zo), ldz, ptr1(ws), ws.numel(), ptr1(err), g.st()) == YR_OK
    z = host(zo)
    pad = np.zeros((B, extra), np.float32)
    pad[:, 0] = 1.0
    assert same_bits(z[:, h:], pad), "padding columns of z_out"
    assert host(err)[0] == 0
    return z[:, :h]


def check_both_entries(P, uid, x, keep, tgt, neg, act, what, fam):
    """the dense and the index-list step against the same reference (the lists keep dropped inputs as zeros in their
    chains: their own chain lengths), the hidden layer alone, and the loss-only pass of both"""
    xv, pos = x * keep, positions(tgt, neg)
    r = cdae_ref(P, uid, xv, tgt, pos, act)
    rl = cdae_ref(P, uid, xv, tgt, pos, act, listed=x != 0)
    note(f"{fam} hidden z", worst(z_ratio(run_hidden(P, uid, x, keep, act), r), f"{what}: yr_cdae_hidden_ex z"))
    for entry, ref in (("dense", r), ("lists", rl)):
        o = run_step(P, uid, x, keep, tgt, neg, act, entry)
        check_step(ref, o["z"], o["loss"], o["grads"], f"{what} {entry}", fam)
        o = run_step(P, uid, x, keep, tgt, neg, act, entry, train=False)
        check_step(ref, None, o["loss"], None, f"{what} {entry} loss only", fam)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("nI", [1, 31, 32, 33, 255, 257, 1025, 7937, 8193])
def test_compaction_edges_every_element_within_bound(nI):
    """one or several 256-column rounds per warp segment and empty trailing warps; rows without inputs, with every
    column an input, without loss positions, with every input dropped by keep, a position that is both a target and a
    negative (counted once), non-binary x and a duplicate user (module docstring, edge_case)"""
    P, uid, x, keep, tgt, neg = edge_case(nI)
    r = check_both_entries(P, uid, x, keep, tgt, neg, "sigmoid", f"edges nI={nI}", "edges")
    assert r["M"] == int(positions(tgt, neg).sum()) and (nI == 1 or positions(tgt, neg)[4].sum() < (tgt[4] + neg[4]).sum())


@pytest.mark.gpu
def test_batch_without_loss_positions():
    """no loss position at all: the step loss is NaN (torch's mean of nothing), the gradients are 0 and Adam leaves
    every parameter as it was"""
    P, uid, x, keep, tgt, neg = edge_case(257)
    tgt[:], neg[:] = 0.0, 0.0
    for entry in ("dense", "lists"):
        o = run_step(P, uid, x, keep, tgt, neg, "sigmoid", entry)
        assert np.isnan(o["loss"]) and np.isnan(o["loss_sum"][0]), entry
        for k in KEYS:
            assert not np.any(o["grads"][k]) and same_bits(o["P"][k], P[k]), (entry, k)


@pytest.mark.gpu
@pytest.mark.parametrize("act", ["sigmoid", "identity"])
@pytest.mark.parametrize("h", [32, 64, 128, 256, 512, 1024])
def test_every_width_every_element_within_bound(h, act):
    """G = 8, 4, 2, 1 partial sums per hidden unit and VPL = 1 .. 32 floats per lane"""
    P, uid, x, keep, tgt, neg = edge_case(1025, h, seed=h)
    check_both_entries(P, uid, x, keep, tgt, neg, act, f"h={h} {act}", "widths")


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 1024])
def test_yelp_shape_every_element_within_bound(h):
    """the bench's CDAE configuration: 38,048 items, B = 32, Adam, Yelp-like rows with 5x negatives and dropout. At
    h = 64 also the index-list step, its lists built by data/cdae_sparse.sparse_cdae_batch."""
    from yelprecommendation_b200.data.cdae_sparse import sparse_cdae_batch
    nI, B, nU = 38_048, 32, 1000
    x, keep, neg = yelp_rows(nI, B, 11)
    P = make_params(nI, h, nU, np.random.default_rng(h))
    uid = np.random.default_rng(3).choice(nU, B, replace=False)
    xv, pos = x * keep, positions(x, neg)
    r = cdae_ref(P, uid, xv, x, pos, "sigmoid")
    o = run_step(P, uid, x, keep, x, neg, "sigmoid")
    check_step(r, o["z"], o["loss"], o["grads"], f"Yelp shape h={h}", "yelp")
    if h == 64:
        t = torch.from_numpy
        sb = sparse_cdae_batch({"user_id": t(uid), "input_mask": t(x), "negative_mask": t(neg)})
        ip, ii = sb["input_ptr"].numpy(), sb["input_idx"].numpy()
        iv = keep[np.repeat(np.arange(B), np.diff(ip)), ii]
        lst = (ip, ii, iv, sb["loss_ptr"].numpy(), sb["loss_idx"].numpy(), sb["loss_val"].numpy())
        assert all(np.array_equal(a, b) for a, b in zip(lst, lists(x, keep, x, neg)) if a is not None)
        rl = cdae_ref(P, uid, xv, x, pos, "sigmoid", listed=x != 0)
        o = run_step(P, uid, x, keep, x, neg, "sigmoid", "lists", lst=lst)
        check_step(rl, o["z"], o["loss"], o["grads"], "Yelp shape lists", "yelp")


def single_addend_case(nI, h, seed):
    """B = 1: every gradient element has at most one addend, so the step is deterministic"""
    rng = np.random.default_rng(seed)
    P = make_params(nI, h, 30, rng)
    x = (rng.random((1, nI)) < min(0.5, 60.0 / nI)).astype(np.float32)
    x[0, seg_ends(nI)] = 1.0
    neg = np.zeros_like(x)
    neg[0, rng.choice(np.flatnonzero(x[0] == 0), min(int(x.sum()) * 5, int((x == 0).sum())), replace=False)] = 1.0
    return P, np.array([17]), x, neg


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 1024])
@pytest.mark.parametrize("vals", ["null", "nonzero", "dropout"])
def test_entry_points_agree_bit_for_bit_without_zero_inputs(h, vals):
    """On a single-addend batch the dense and the index-list step give the same z, step loss, gradients, v and parameters
    bit for bit when in_val is NULL (keep NULL) or has no zero. With dropout zeros in in_val both stay within the
    reference's bound (the lists keep the zeros in their chains, so the bits may differ)."""
    nI = 2000
    P, uid, x, neg = single_addend_case(nI, h, h)
    rng = np.random.default_rng(7)
    keep = {"null": None, "nonzero": rng.uniform(0.5, 3.0, x.shape).astype(np.float32),
            "dropout": np.where(rng.random(x.shape) < 0.6, 0.0, 2.5).astype(np.float32)}[vals]
    a = run_step(P, uid, x, keep, x, neg, "sigmoid", "dense")
    b = run_step(P, uid, x, keep, x, neg, "sigmoid", "lists")
    if vals != "dropout":
        assert same_bits(a["z"], b["z"]) and a["loss"] == b["loss"]
        for k in KEYS:
            assert same_bits(a["grads"][k], b["grads"][k]) and same_bits(a["v"][k], b["v"][k]), k
            assert same_bits(a["P"][k], b["P"][k]), k
    xv = x if keep is None else x * keep
    for o, listed in ((a, None), (b, x != 0)):
        r = cdae_ref(P, uid, xv, x, positions(x, neg), "sigmoid", listed=listed)
        check_step(r, o["z"], o["loss"], o["grads"], f"single addend h={h} {vals}", "entries")


@pytest.mark.gpu
@pytest.mark.parametrize("nI", [38_047, 113])
def test_optimizer_routing_unaligned_tensors(nI):
    """bo of a catalog size that is not a multiple of 4 takes the single-tensor optimizer path (then a memset of its
    gradient); with every tensor carved out of one flat buffer at 4-byte-but-not-16-byte offsets, all five do. On a
    single-addend batch the parameters, m and v are bit-identical to the separately allocated layout, every gradient is
    zero on return and within bound."""
    h = 64
    P, uid, x, neg = single_addend_case(nI, h, nI)
    keep = np.where(np.random.default_rng(1).random(x.shape) < 0.6, 0.0, 2.5).astype(np.float32)
    a = run_step(P, uid, x, keep, x, neg, "sigmoid", layout="separate")
    b = run_step(P, uid, x, keep, x, neg, "sigmoid", layout="offset")
    for k in KEYS:
        assert same_bits(a["P"][k], b["P"][k]) and same_bits(a["grads"][k], b["grads"][k]), k
        assert same_bits(a["v"][k], b["v"][k]), k
    r = cdae_ref(P, uid, x * keep, x, positions(x, neg), "sigmoid")
    check_step(r, b["z"], b["loss"], b["grads"], f"offset layout nI={nI}", "routing")


@pytest.mark.gpu
@pytest.mark.parametrize("h", [32, 64, 128])
def test_misaligned_output_layer_is_rejected(h):
    """P.Wo or g.Wo 4 bytes past a 16-byte boundary: h = 32 reads its rows as floats and runs; from h = 64 (float2 /
    float4 rows) both entry points return YR_ERR_BAD_ARG and write nothing"""
    P, uid, x, neg = single_addend_case(113, h, 3)
    for layout in ("wo_off", "gwo_off"):
        for entry in ("dense", "lists"):
            o = run_step(P, uid, x, None, x, neg, "sigmoid", entry, layout, rc_want=YR_OK if h == 32 else YR_ERR_BAD_ARG)
            if h == 32:
                r = cdae_ref(P, uid, x, x, positions(x, neg), "sigmoid", listed=None if entry == "dense" else x != 0)
                check_step(r, o["z"], o["loss"], o["grads"], f"{layout} {entry} h=32", "routing")


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["dense", "lists"])
def test_saturated_logits_take_torchs_gradient(entry):
    """logits >= 18 as sampled negatives and as targets, targets at -30 and -40, controls at 15 and -25: every element
    within the bound of torch's autograd chain, and dbo of the saturated items equal to CDAEPort's autograd dbo within
    the same bound (a negative at p = 1 gets 0, not 1/m)"""
    from oracle import torch_port as tp
    act = "sigmoid"
    P, uid, x, keep, tgt, neg = saturation_case()
    xv, pos = x * keep, positions(tgt, neg)
    r = cdae_ref(P, uid, xv, tgt, pos, act, listed=None if entry == "dense" else x != 0)
    o = run_step(P, uid, x, keep, tgt, neg, act, entry)
    check_step(r, o["z"], o["loss"], o["grads"], f"saturation {entry}", "saturation")
    names = {"Wh": "hidden_layer.weight", "bh": "hidden_layer.bias", "Vu": "user_nodes.weight",
             "Wo": "output_layer.weight", "bo": "output_layer.bias"}
    port = tp.CDAEPort({names[k]: torch.from_numpy(P[k].copy()) for k in KEYS})
    t = lambda a: torch.from_numpy(a.copy())
    tp.nsbce_loss(port.forward(t(uid), t(x), t(keep)), t(tgt), t(neg)).backward()
    pbo = port.bo.grad.numpy()
    _, ref, allow = next(grad_refs(r))
    assert np.all(o["grads"]["bo"][:3] == 0.0) and np.all(pbo[:3] == 0.0)
    note("saturation dbo vs port", worst(np.abs(o["grads"]["bo"][:8] - pbo[:8]) / (2 * allow[:8] + ulp(pbo[:8])),
                                         f"saturation {entry}: dbo vs CDAEPort"))


@pytest.mark.gpu
def test_output_and_nsbce_loss_within_bound():
    """yr_cdae_output (z with ldz > h) and yr_nsbce_loss with n past sm * 8 * 256, so the grid-stride loop turns more
    than once; p exactly 0 and 1 where the -100 clamp applies; an all-masked input gives NaN"""
    g = dev()
    rng = np.random.default_rng(8)
    nI, h, ldz, B = 1000, 64, 96, 3
    P = make_params(nI, h, 4, rng)
    z = rng.uniform(-1, 1, (B, ldz)).astype(np.float32)
    Pd = {k: cu(P[k]) for k in KEYS}
    Pt = _pack(Pd)
    pred = cu(np.full((B, nI), SENTINEL, np.uint32).view(np.float32))
    zd = cu(z)
    assert g.lib.yr_cdae_output(C.byref(Pt), nI, h, ptr1(zd), ldz, B, ptr1(pred), g.st()) == YR_OK
    Wo, bo, z64 = P["Wo"].astype(np.float64), P["bo"].astype(np.float64), z[:, :h].astype(np.float64)
    logit = z64 @ Wo.T + bo
    a = (h + 1) * U24 * (np.abs(z64) @ np.abs(Wo).T + np.abs(bo))
    lo, hi = sig_range(logit, a)
    pe = 1.0 / (1.0 + np.exp(-logit))
    note("output pred", worst(ratio(host(pred), pe, np.maximum(hi - pe, pe - lo)), "yr_cdae_output"))

    n = 2 * g.sm * 8 * 256 + 77
    p = rng.random(n).astype(np.float32)
    p[:4] = [0.0, 0.0, 1.0, 1.0]
    t = (rng.random(n) < 0.3).astype(np.float32)
    t[:4] = [1.0, 0.0, 0.0, 1.0]
    m = (rng.random(n) < 0.5).astype(np.float32)
    m[:4] = 1.0
    sel = (t + m) != 0
    ell = bce(p.astype(np.float64), t)[sel]
    assert ell[0] == 100.0 and ell[2] == 100.0 and ell[1] == 0.0 and ell[3] == 0.0
    c = ell.size
    ref = ell.sum() / c
    ws = torch.empty(64, dtype=torch.uint8, device="cuda")
    out = torch.full((1,), 7.0, device="cuda")
    pd, td, md = cu(p), cu(t), cu(m)
    assert g.lib.yr_nsbce_loss(ptr1(pd), ptr1(td), ptr1(md), n, ptr1(out), ptr1(ws), ws.numel(), g.st()) == YR_OK
    note("nsbce loss", worst(ratio(host(out)[0], ref, (4 * U24 + c * 2.0 ** -53) * np.abs(ell).sum() / c), "yr_nsbce_loss"))
    zero = cu(np.zeros(n, np.float32))
    assert g.lib.yr_nsbce_loss(ptr1(pd), ptr1(zero), ptr1(zero), n, ptr1(out), ptr1(ws), ws.numel(), g.st()) == YR_OK
    assert np.isnan(host(out)[0])
