// CDAE kernels (sm_100a) — BASELINE config 4: the reference's denoising auto-encoder
//   models/cdae.py:46-52     out = sigmoid(Wo . act(Wh . dropout(x) + bh + Vu[u]) + bo),  act = sigmoid | identity
//   loss.py:7-16             NSBCELoss: BCE (mean) over the positions where target + negative_mask != 0
//   trainers/cdae_trainer.py:36-54 (train step), :56-70 (validate loss)
// The reference pushes dense [B x nI] tensors through two nn.Linear layers and materialises the dense output.
// Here: the multi-hot input and the loss positions are compacted once per batch (ordered, deterministic), the first
// layer is a gather-sum over the ~|x| active columns, logits are evaluated ONLY at the loss positions, and the
// backward pass touches only those positions and the active columns — the dense [B x nI] output never exists during
// training. The optimizer keeps torch's dense semantics (every element of every tensor is stepped).
#include "common.cuh"

namespace yr {

constexpr int kCdaeThreads = 256;
constexpr int kCdaeMaxH = 1024;
constexpr int kCompactThreads = 1024;   // 32 warps per row: the compaction is a latency chain, parallelism is what it needs

struct CdaeWs {
  int32_t* xin_cnt;   // [B]
  int32_t* tgt_cnt;   // [B]
  int32_t* total;     // [1] number of loss positions in the batch
  int32_t* xin_idx;   // [B x nI]
  float* xin_val;     // [B x nI]
  int32_t* tgt_idx;   // [B x nI]
  float* tgt_val;     // [B x nI]
  float* z;           // [B x h]
};

static size_t cdae_ws_layout(int64_t B, int64_t nI, void* base, CdaeWs* w) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_xc = take((size_t)B * 4), o_tc = take((size_t)B * 4), o_tot = take(16);
  const size_t o_xi = take((size_t)B * nI * 4), o_xv = take((size_t)B * nI * 4);
  const size_t o_ti = take((size_t)B * nI * 4), o_tv = take((size_t)B * nI * 4);
  const size_t o_z = take((size_t)B * kCdaeMaxH * 4);
  if (w && base) {
    unsigned char* p = (unsigned char*)base;
    w->xin_cnt = (int32_t*)(p + o_xc); w->tgt_cnt = (int32_t*)(p + o_tc); w->total = (int32_t*)(p + o_tot);
    w->xin_idx = (int32_t*)(p + o_xi); w->xin_val = (float*)(p + o_xv);
    w->tgt_idx = (int32_t*)(p + o_ti); w->tgt_val = (float*)(p + o_tv); w->z = (float*)(p + o_z);
  }
  return off;
}

// Block per batch row: ordered compaction of (a) the active inputs x*keep != 0 and (b) the loss positions
// target + negative != 0 (value kept = target). Each warp owns a contiguous segment of the row; two passes.
__global__ void __launch_bounds__(kCompactThreads)
cdae_compact_kernel(const float* __restrict__ x, const float* __restrict__ keep, const float* __restrict__ target,
                    const float* __restrict__ neg, int64_t nI, CdaeWs w) {
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = kCompactThreads / 32;
  const int64_t seg = ((nI + NW - 1) / NW + 31) / 32 * 32;
  const int64_t s0 = warp * seg, s1 = min(nI, s0 + seg);
  const float* xr = x + (int64_t)b * nI;
  const float* kr = keep ? keep + (int64_t)b * nI : nullptr;
  const float* tr = target ? target + (int64_t)b * nI : nullptr;
  const float* nr = neg ? neg + (int64_t)b * nI : nullptr;
  __shared__ int cx[NW], ct[NW];
  int nx = 0, nt = 0;
  constexpr int UN = 8;                                   // 8 x 32 columns per round: all loads of a round are in flight
  // pass 1: counts
  for (int64_t i0 = s0; i0 < s1; i0 += 32 * UN) {
    float xv_[UN], kv_[UN], tv_[UN], nv_[UN];
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      const int64_t i = i0 + q * 32 + lane;
      const bool in = i < s1;
      xv_[q] = in ? xr[i] : 0.f;
      kv_[q] = (in && kr) ? kr[i] : 1.f;
      tv_[q] = (in && tr) ? tr[i] : 0.f;
      nv_[q] = (in && nr) ? nr[i] : 0.f;
    }
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      const float v = kr ? xv_[q] * kv_[q] : xv_[q];
      const bool px = v != 0.f;
      const bool pt = tr ? ((tv_[q] + nv_[q]) != 0.f) : false;
      nx += __popc(__ballot_sync(kFull, px));
      nt += __popc(__ballot_sync(kFull, pt));
    }
  }
  if (lane == 0) { cx[warp] = nx; ct[warp] = nt; }
  __syncthreads();
  int bx = 0, bt = 0, totx = 0, tott = 0;
  for (int q = 0; q < NW; ++q) {
    if (q < warp) { bx += cx[q]; bt += ct[q]; }
    totx += cx[q]; tott += ct[q];
  }
  if (threadIdx.x == 0) {
    w.xin_cnt[b] = totx;
    w.tgt_cnt[b] = tott;
    if (tott) atomicAdd(w.total, tott);
  }
  int32_t* xi = w.xin_idx + (int64_t)b * nI;
  float* xv = w.xin_val + (int64_t)b * nI;
  int32_t* ti = w.tgt_idx + (int64_t)b * nI;
  float* tv = w.tgt_val + (int64_t)b * nI;
  // pass 2: ordered writes (the second read of the row comes from L2)
  for (int64_t i0 = s0; i0 < s1; i0 += 32 * UN) {
    float xv_[UN], kv_[UN], tv_[UN], nv_[UN];
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      const int64_t i = i0 + q * 32 + lane;
      const bool in = i < s1;
      xv_[q] = in ? xr[i] : 0.f;
      kv_[q] = (in && kr) ? kr[i] : 1.f;
      tv_[q] = (in && tr) ? tr[i] : 0.f;
      nv_[q] = (in && nr) ? nr[i] : 0.f;
    }
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      const int64_t i = i0 + q * 32 + lane;
      const float v = kr ? xv_[q] * kv_[q] : xv_[q];
      const bool px = v != 0.f;
      const bool pt = tr ? ((tv_[q] + nv_[q]) != 0.f) : false;
      const unsigned mx = __ballot_sync(kFull, px), mt = __ballot_sync(kFull, pt);
      const unsigned lower = (1u << lane) - 1u;
      if (px) { const int p = bx + __popc(mx & lower); xi[p] = (int32_t)i; xv[p] = v; }
      if (pt) { const int p = bt + __popc(mt & lower); ti[p] = (int32_t)i; tv[p] = tv_[q]; }
      bx += __popc(mx);
      bt += __popc(mt);
    }
  }
}

// Index-list form of a batch (no dense [B x nI] tensors anywhere): block per row copies its lists into the layout the row
// kernel reads. in_val == NULL: every listed input is 1 (evaluation / no dropout); otherwise the value after dropout
// (0 or 1/(1-p); zeros are harmless). Loss positions: tgt_idx ascending per row with tgt_val = the target (1 / 0).
__global__ void __launch_bounds__(256)
cdae_lists_kernel(const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_idx, const float* __restrict__ in_val,
                  const int32_t* __restrict__ tgt_ptr, const int32_t* __restrict__ tgt_idx, const float* __restrict__ tgt_val,
                  int64_t nI, CdaeWs w, int32_t* err) {
  const int b = blockIdx.x;
  const int i0 = in_ptr[b], ni = in_ptr[b + 1] - i0;
  int32_t* xi = w.xin_idx + (int64_t)b * nI;
  float* xv = w.xin_val + (int64_t)b * nI;
  bool bad = ni < 0 || ni > nI;
  for (int j = threadIdx.x; j < ni && !bad; j += blockDim.x) {
    const int it = in_idx[i0 + j];
    if (it < 0 || it >= nI) { if (err) atomicExch(err, 1); xi[j] = 0; xv[j] = 0.f; continue; }
    xi[j] = it;
    xv[j] = in_val ? in_val[i0 + j] : 1.f;
  }
  int nt = 0;
  if (tgt_ptr) {
    const int t0 = tgt_ptr[b];
    nt = tgt_ptr[b + 1] - t0;
    bad = bad || nt < 0 || nt > nI;
    int32_t* ti = w.tgt_idx + (int64_t)b * nI;
    float* tv = w.tgt_val + (int64_t)b * nI;
    for (int j = threadIdx.x; j < nt && !bad; j += blockDim.x) {
      const int it = tgt_idx[t0 + j];
      if (it < 0 || it >= nI) { if (err) atomicExch(err, 1); ti[j] = 0; tv[j] = 0.f; continue; }
      ti[j] = it;
      tv[j] = tgt_val[t0 + j];
    }
  }
  if (threadIdx.x == 0) {
    if (bad && err) atomicExch(err, 1);
    w.xin_cnt[b] = bad ? 0 : ni;
    w.tgt_cnt[b] = bad ? 0 : nt;
    if (!bad && nt) atomicAdd(w.total, nt);
  }
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// Hidden layer, phase 1: part[g][k] = sum over j = g, g + G, ... < nx of xv[j] * Wh[k, xi[j]], one fma chain each
// (G partial sums per unit, KS units per pass of the CTA). xv: the input values, or CdaeOnes for a multi-hot list.
template <int H, int G, int KS, typename XV>
__device__ __forceinline__ void cdae_hidden_part(int tid, const float* Wh, int64_t nI, const int32_t* xi, XV xv, int nx,
                                                 float (*part)[H]) {
  const int g = tid / KS;
  for (int k = tid % KS; k < H; k += KS) {
    float acc = 0.f;
    for (int j = g; j < nx; j += G) acc = fmaf(xv[j], __ldg(Wh + (int64_t)k * nI + xi[j]), acc);
    part[g][k] = acc;
  }
}

// Hidden layer, phase 2 for unit k: act(pre + the G partial sums), pre = bh[k] + Vu[u, k].
template <int H, int G>
__device__ __forceinline__ float cdae_hidden_unit(const float (*part)[H], int k, float pre, int act) {
  if constexpr (G == 4) {
    pre += (part[0][k] + part[1][k]) + (part[2][k] + part[3][k]);
  } else {
    float t = part[0][k];
#pragma unroll
    for (int g = 1; g < G; ++g) t += part[g][k];
    pre += t;
  }
  return act ? pre : sigmoidf_(pre);
}

struct CdaeOnes {
  __device__ __forceinline__ float operator[](int) const { return 1.f; }
};

// Block per batch row. H = 32 * VPL = hidden size (32 ... 1,024: the values of the reference's cdae_sweep_config.yaml).
// Phase 1: hidden activation (act: 0 sigmoid, 1 identity — models/base_model.py:10-14) from the compacted inputs.
// Phase 2 (targets given): logits at the loss positions, BCE terms, and — if GRAD — every gradient.
template <int VPL, bool GRAD>
__global__ void __launch_bounds__(kCdaeThreads)
cdae_row_kernel(yr_cdae_tensors P, yr_cdae_tensors Gr, int64_t nU, int64_t nI, const int64_t* __restrict__ uid,
                CdaeWs w, bool with_loss, float* __restrict__ z_out, int64_t ldz, double* loss_acc, int32_t* err, int act) {
  constexpr int H = VPL * 32;
  constexpr int NW = kCdaeThreads / 32;
  constexpr int G = H >= kCdaeThreads ? 1 : kCdaeThreads / H;      // partial sums per hidden unit (4 at H = 64)
  constexpr int KS = H >= kCdaeThreads ? kCdaeThreads : H;         // hidden units covered per pass of the CTA
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ float part[G][H];
  __shared__ __align__(16) float z_s[H];
  __shared__ __align__(16) float dz_s[NW][H];
  __shared__ double loss_s[NW];
  int64_t u = uid[b];
  if (u < 0 || u >= nU) { if (tid == 0 && err) atomicExch(err, 1); u = 0; }
  const int nx = w.xin_cnt[b];
  const int32_t* xi = w.xin_idx + (int64_t)b * nI;
  const float* xv = w.xin_val + (int64_t)b * nI;

  // ---- hidden: z = act(bh + Vu[u] + sum_j xv_j * Wh[:, xi_j]) ; thread = (group g of G, unit k)
  cdae_hidden_part<H, G, KS>(tid, P.Wh, nI, xi, xv, nx, part);
  __syncthreads();
  for (int k = tid; k < H; k += kCdaeThreads) {
    const float z = cdae_hidden_unit<H, G>(part, k, P.bh[k] + P.Vu[u * H + k], act);
    z_s[k] = z;
    w.z[(int64_t)b * H + k] = z;
    if (z_out) z_out[(int64_t)b * ldz + k] = z;
  }
  if (z_out)
    for (int k = H + tid; k < ldz; k += kCdaeThreads) z_out[(int64_t)b * ldz + k] = (k == H) ? 1.f : 0.f;
  __syncthreads();
  if (!with_loss) return;

  // ---- loss positions: warp per position, lanes hold VPL hidden units each (Row<VPL> slices) ----
  const int nt = w.tgt_cnt[b];
  const int32_t* ti = w.tgt_idx + (int64_t)b * nI;
  const float* tv = w.tgt_val + (int64_t)b * nI;
  const float inv_m = 1.f / (float)(*w.total);
  const Row<VPL> zz = ld_row<VPL>(z_s, lane);
  Row<VPL> dz;
#pragma unroll
  for (int i = 0; i < VPL; ++i) dz.x[i] = 0.f;
  double lsum = 0.0;
  constexpr int UN = VPL <= 2 ? 4 : (VPL <= 8 ? 2 : 1);   // positions per warp round: their ids, then their Wo rows, are in flight together
  for (int j0 = warp * UN; j0 < nt; j0 += NW * UN) {
    int item[UN];
    float t[UN], bo[UN];
    Row<VPL> wo[UN];
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      const bool in = j0 + q < nt;
      item[q] = in ? ti[j0 + q] : -1;
      t[q] = in ? tv[j0 + q] : 0.f;
    }
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      const int it = item[q] < 0 ? 0 : item[q];
      wo[q] = ld_row<VPL>(P.Wo + (int64_t)it * H, lane);
      bo[q] = __ldg(P.bo + it);
    }
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      if (item[q] < 0) continue;                                 // warp-uniform
      const float logit = warp_sum(dot_partial<VPL>(zz, wo[q])) + bo[q];
      const float p = sigmoidf_(logit);
      // torch.nn.functional.binary_cross_entropy clamps both logs at -100
      const float lp = fmaxf(logf(p), -100.f), lq = fmaxf(log1pf(-p), -100.f);
      lsum += (double)(-(t[q] * lp + (1.f - t[q]) * lq));
      if (GRAD) {
        const float dl = (p - t[q]) * inv_m;                     // d loss / d logit (mean over all loss positions)
        Row<VPL> gw;
#pragma unroll
        for (int i = 0; i < VPL; ++i) { dz.x[i] = fmaf(dl, wo[q].x[i], dz.x[i]); gw.x[i] = dl * zz.x[i]; }
        red_row<VPL>(Gr.Wo + (int64_t)item[q] * H, lane, gw);
        if (lane == 0) atomicAdd(Gr.bo + item[q], dl);
      }
    }
  }
  if (lane == 0) loss_s[warp] = lsum;
  if (GRAD) st_row<VPL>(dz_s[warp], lane, dz);
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int q = 0; q < NW; ++q) t += loss_s[q];
    if (t != 0.0) atomicAdd(loss_acc, t);
  }
  if (!GRAD) return;
  for (int k = tid; k < H; k += kCdaeThreads) {
    float d = 0.f;
#pragma unroll
    for (int q = 0; q < NW; ++q) d += dz_s[q][k];
    const float z = z_s[k];
    const float dpre = act ? d : d * z * (1.f - z);
    z_s[k] = dpre;                                              // reuse: z_s now holds d loss / d pre-activation
    atomicAdd(Gr.bh + k, dpre);
    atomicAdd(Gr.Vu + u * H + k, dpre);
  }
  __syncthreads();
  {
    const int g = tid / KS;
    for (int k = tid % KS; k < H; k += KS) {
      const float dpre = z_s[k];
      for (int j = g; j < nx; j += G) atomicAdd(Gr.Wh + (int64_t)k * nI + xi[j], dpre * xv[j]);
    }
  }
}

// Block per batch row: the hidden activations from the row's interaction list (a CSR indexed by user id), with the
// arithmetic of cdae_row_kernel's phase 1 on the dense multi-hot of the same list.
template <int VPL>
__global__ void __launch_bounds__(kCdaeThreads)
cdae_encode_kernel(yr_cdae_tensors P, int64_t nU, int64_t nI, const int64_t* __restrict__ uid,
                   const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_idx, float* __restrict__ z,
                   int64_t ldz, int32_t* err, int act) {
  constexpr int H = VPL * 32;
  constexpr int G = H >= kCdaeThreads ? 1 : kCdaeThreads / H;
  constexpr int KS = H >= kCdaeThreads ? kCdaeThreads : H;
  __shared__ float part[G][H];
  const int b = blockIdx.x, tid = threadIdx.x;
  int64_t u = uid[b];
  if (u < 0 || u >= nU) { if (tid == 0 && err) atomicOr(err, 1); u = 0; }
  const int64_t i0 = in_ptr[u], i1 = in_ptr[u + 1];
  bool bad = i0 < 0 || i1 < i0 || i1 > in_ptr[nU];
  const int32_t* xi = in_idx + (bad ? 0 : i0);
  int nx = bad ? 0 : (int)(i1 - i0);
  int out = 0;                                                  // every id checked before any is used as a column
  for (int j = tid; j < nx; j += kCdaeThreads) out |= (xi[j] < 0) | (xi[j] >= nI);
  bad = __syncthreads_or(out) || bad;
  if (bad) {
    nx = 0;
    if (tid == 0 && err) atomicOr(err, 2);
  }
  cdae_hidden_part<H, G, KS>(tid, P.Wh, nI, xi, CdaeOnes{}, nx, part);
  __syncthreads();
  for (int k = tid; k < H; k += kCdaeThreads)
    z[(int64_t)b * ldz + k] = cdae_hidden_unit<H, G>(part, k, P.bh[k] + P.Vu[u * H + k], act);
}

template <bool GRAD>
static int launch_cdae_row(int h, int64_t B, cudaStream_t s, const yr_cdae_tensors& P, const yr_cdae_tensors& Gr, int64_t nU,
                           int64_t nI, const int64_t* uid, const CdaeWs& w, bool with_loss, float* z_out, int64_t ldz,
                           double* loss_acc, int32_t* err, int act) {
#define YR_CDAE_ROW(V) cdae_row_kernel<V, GRAD><<<(unsigned)B, kCdaeThreads, 0, s>>>(P, Gr, nU, nI, uid, w, with_loss, z_out, ldz, loss_acc, err, act)
  switch (dim_vpl(h)) {
    case 1: YR_CDAE_ROW(1); break;
    case 2: YR_CDAE_ROW(2); break;
    case 4: YR_CDAE_ROW(4); break;
    case 8: YR_CDAE_ROW(8); break;
    case 16: YR_CDAE_ROW(16); break;
    case 32: YR_CDAE_ROW(32); break;
    default: return YR_ERR_BAD_DIM;
  }
#undef YR_CDAE_ROW
  YR_CHECK_LAUNCH();
  return YR_OK;
}

__global__ void cdae_finish_kernel(double* loss, const int32_t* total, float* step_loss) {
  const float mean = (*total > 0) ? (float)(loss[1] / (double)(*total)) : nanf("");
  if (step_loss) *step_loss = mean;
  loss[0] += (double)mean;
  loss[1] = 0.0;
}

// pred[b, i] = sigmoid(z[b,:] . Wo[i,:] + bo[i])
__global__ void __launch_bounds__(256)
cdae_output_kernel(const float* __restrict__ Wo, const float* __restrict__ bo, int64_t nI, int h,
                   const float* __restrict__ z, int64_t ldz, float* __restrict__ pred) {
  extern __shared__ float zs[];
  const int b = blockIdx.y;
  for (int k = threadIdx.x; k < h; k += blockDim.x) zs[k] = z[(int64_t)b * ldz + k];
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nI) return;
  const float* wr = Wo + i * h;
  float acc = 0.f;
  for (int k = 0; k < h; ++k) acc = fmaf(zs[k], __ldg(wr + k), acc);
  pred[(int64_t)b * nI + i] = sigmoidf_(acc + bo[i]);
}

__global__ void __launch_bounds__(256)
nsbce_kernel(const float* __restrict__ pred, const float* __restrict__ target, const float* __restrict__ neg,
             int64_t n, double* acc /* [0] sum, [1] count */) {
  double s = 0.0, c = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float t = target[i];
    if (t + neg[i] != 0.f) {
      const float p = pred[i];
      s += (double)(-(t * fmaxf(logf(p), -100.f) + (1.f - t) * fmaxf(log1pf(-p), -100.f)));
      c += 1.0;
    }
  }
  s = warp_sum_d(s); c = warp_sum_d(c);
  if ((threadIdx.x & 31) == 0) { atomicAdd(acc, s); atomicAdd(acc + 1, c); }
}
__global__ void nsbce_finish_kernel(const double* acc, float* loss) { *loss = (float)(acc[0] / acc[1]); }

}  // namespace yr

using namespace yr;

extern "C" size_t yr_cdae_ws_bytes(int64_t B, int64_t nI) { return cdae_ws_layout(B, nI, nullptr, nullptr) + 256; }

static int cdae_tensors_ok(const yr_cdae_tensors* t) {
  return (t && t->Wh && t->bh && t->Vu && t->Wo && t->bo) ? YR_OK : YR_ERR_BAD_ARG;
}

extern "C" int yr_cdae_hidden(const yr_cdae_tensors* P, int64_t nU, int64_t nI, int h, const int64_t* uid,
                              const float* x, const float* keep, int64_t B, float* z_out, int64_t ldz, void* ws,
                              size_t ws_bytes, int32_t* err, yr_stream stream) {
  return yr_cdae_hidden_ex(P, nU, nI, h, YR_ACT_SIGMOID, uid, x, keep, B, z_out, ldz, ws, ws_bytes, err, stream);
}

extern "C" int yr_cdae_hidden_ex(const yr_cdae_tensors* P, int64_t nU, int64_t nI, int h, int hidden_act,
                                 const int64_t* uid, const float* x, const float* keep, int64_t B, float* z_out,
                                 int64_t ldz, void* ws, size_t ws_bytes, int32_t* err, yr_stream stream) {
  if (cdae_tensors_ok(P) || !uid || !x || !z_out || !ws || B <= 0 || nI <= 0 || ldz < h) return YR_ERR_BAD_ARG;
  if (hidden_act != YR_ACT_SIGMOID && hidden_act != YR_ACT_IDENTITY) return YR_ERR_BAD_ARG;
  if (!dim_vpl(h)) return YR_ERR_BAD_DIM;
  if (ws_bytes < yr_cdae_ws_bytes(B, nI)) return YR_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  CdaeWs w;
  cdae_ws_layout(B, nI, ws, &w);
  YR_CUDA(cudaMemsetAsync(w.total, 0, 16, s));
  cdae_compact_kernel<<<(unsigned)B, kCompactThreads, 0, s>>>(x, keep, nullptr, nullptr, nI, w);
  YR_CHECK_LAUNCH();
  yr_cdae_tensors none = {};
  return launch_cdae_row<false>(h, B, s, *P, none, nU, nI, uid, w, false, z_out, ldz, nullptr, err, hidden_act);
}

extern "C" int yr_cdae_encode(const yr_cdae_tensors* P, int64_t nU, int64_t nI, int h, int hidden_act,
                              const int64_t* user_ids, int64_t B, const int32_t* in_ptr, const int32_t* in_idx, float* z,
                              int64_t ldz, int32_t* err, yr_stream stream) {
  if (cdae_tensors_ok(P) || !user_ids || !in_ptr || !in_idx || !z || B < 0 || nU <= 0 || nI <= 0 || ldz < h)
    return YR_ERR_BAD_ARG;
  if (hidden_act != YR_ACT_SIGMOID && hidden_act != YR_ACT_IDENTITY) return YR_ERR_BAD_ARG;
  if (!dim_vpl(h)) return YR_ERR_BAD_DIM;
  if (B == 0) return YR_OK;
  cudaStream_t s = (cudaStream_t)stream;
#define YR_CDAE_ENCODE(V) \
  cdae_encode_kernel<V><<<(unsigned)B, kCdaeThreads, 0, s>>>(*P, nU, nI, user_ids, in_ptr, in_idx, z, ldz, err, hidden_act)
  switch (dim_vpl(h)) {
    case 1: YR_CDAE_ENCODE(1); break;
    case 2: YR_CDAE_ENCODE(2); break;
    case 4: YR_CDAE_ENCODE(4); break;
    case 8: YR_CDAE_ENCODE(8); break;
    case 16: YR_CDAE_ENCODE(16); break;
    case 32: YR_CDAE_ENCODE(32); break;
    default: return YR_ERR_BAD_DIM;
  }
#undef YR_CDAE_ENCODE
  YR_CHECK_LAUNCH();
  return YR_OK;
}

extern "C" int yr_cdae_output(const yr_cdae_tensors* P, int64_t nI, int h, const float* z, int64_t ldz, int64_t B,
                              float* pred, yr_stream stream) {
  if (cdae_tensors_ok(P) || !z || !pred || B <= 0 || nI <= 0 || h <= 0 || ldz < h) return YR_ERR_BAD_ARG;
  dim3 grid((unsigned)((nI + 255) / 256), (unsigned)B);
  cdae_output_kernel<<<grid, 256, h * sizeof(float), (cudaStream_t)stream>>>(P->Wo, P->bo, nI, h, z, ldz, pred);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

static int cdae_step_tail(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                          const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h, int hidden_act,
                          const int64_t* uid, int64_t B, double* loss, float* step_loss, const CdaeWs& w, int32_t* err,
                          yr_stream stream);

static int cdae_step_args_ok(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                             const yr_cdae_tensors* v, const yr_opt* opt, int h, int hidden_act) {
  if (cdae_tensors_ok(P)) return YR_ERR_BAD_ARG;
  if (hidden_act != YR_ACT_SIGMOID && hidden_act != YR_ACT_IDENTITY) return YR_ERR_BAD_ARG;
  if (!dim_vpl(h)) return YR_ERR_BAD_DIM;
  if (opt) {
    if (cdae_tensors_ok(grads)) return YR_ERR_BAD_ARG;
    if (opt->kind < YR_OPT_SGD || opt->kind > YR_OPT_ADAMW) return YR_ERR_BAD_OPT;
    if (opt->kind != YR_OPT_SGD && (cdae_tensors_ok(m) || cdae_tensors_ok(v))) return YR_ERR_BAD_ARG;
  }
  return YR_OK;
}

extern "C" int yr_cdae_step_idx(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                                const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h, int hidden_act,
                                const int64_t* uid, const int32_t* in_ptr, const int32_t* in_idx, const float* in_val,
                                const int32_t* tgt_ptr, const int32_t* tgt_idx, const float* tgt_val, int64_t B,
                                double* loss, float* step_loss, void* ws, size_t ws_bytes, int32_t* err, yr_stream stream) {
  if (!uid || !in_ptr || !in_idx || !tgt_ptr || !tgt_idx || !tgt_val || !loss || !ws || B <= 0 || nI <= 0) return YR_ERR_BAD_ARG;
  int rc = cdae_step_args_ok(P, grads, m, v, opt, h, hidden_act);
  if (rc) return rc;
  if (ws_bytes < yr_cdae_ws_bytes(B, nI)) return YR_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  CdaeWs w;
  cdae_ws_layout(B, nI, ws, &w);
  YR_CUDA(cudaMemsetAsync(w.total, 0, 16, s));
  cdae_lists_kernel<<<(unsigned)B, 256, 0, s>>>(in_ptr, in_idx, in_val, tgt_ptr, tgt_idx, tgt_val, nI, w, err);
  YR_CHECK_LAUNCH();
  return cdae_step_tail(P, grads, m, v, opt, nU, nI, h, hidden_act, uid, B, loss, step_loss, w, err, stream);
}

extern "C" int yr_cdae_step(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                            const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h,
                            const int64_t* uid, const float* x, const float* keep, const float* target,
                            const float* negative_mask, int64_t B, double* loss, float* step_loss, void* ws,
                            size_t ws_bytes, int32_t* err, yr_stream stream) {
  return yr_cdae_step_ex(P, grads, m, v, opt, nU, nI, h, YR_ACT_SIGMOID, uid, x, keep, target, negative_mask, B, loss,
                         step_loss, ws, ws_bytes, err, stream);
}

extern "C" int yr_cdae_step_ex(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                               const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h, int hidden_act,
                               const int64_t* uid, const float* x, const float* keep, const float* target,
                               const float* negative_mask, int64_t B, double* loss, float* step_loss, void* ws,
                               size_t ws_bytes, int32_t* err, yr_stream stream) {
  if (cdae_tensors_ok(P) || !uid || !x || !target || !loss || !ws || B <= 0 || nI <= 0) return YR_ERR_BAD_ARG;
  if (hidden_act != YR_ACT_SIGMOID && hidden_act != YR_ACT_IDENTITY) return YR_ERR_BAD_ARG;
  if (!dim_vpl(h)) return YR_ERR_BAD_DIM;
  if (ws_bytes < yr_cdae_ws_bytes(B, nI)) return YR_ERR_WORKSPACE;
  const bool train = opt != nullptr;
  if (train) {
    if (cdae_tensors_ok(grads)) return YR_ERR_BAD_ARG;
    if (opt->kind < YR_OPT_SGD || opt->kind > YR_OPT_ADAMW) return YR_ERR_BAD_OPT;
    if (opt->kind != YR_OPT_SGD && (cdae_tensors_ok(m) || cdae_tensors_ok(v))) return YR_ERR_BAD_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  CdaeWs w;
  cdae_ws_layout(B, nI, ws, &w);
  YR_CUDA(cudaMemsetAsync(w.total, 0, 16, s));
  cdae_compact_kernel<<<(unsigned)B, kCompactThreads, 0, s>>>(x, keep, target, negative_mask, nI, w);
  YR_CHECK_LAUNCH();
  return cdae_step_tail(P, grads, m, v, opt, nU, nI, h, hidden_act, uid, B, loss, step_loss, w, err, stream);
}

// everything of a step behind the compaction / list staging: row kernel (forward, loss, backward), loss finish, optimizer
static int cdae_step_tail(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                          const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h, int hidden_act,
                          const int64_t* uid, int64_t B, double* loss, float* step_loss, const CdaeWs& w, int32_t* err,
                          yr_stream stream) {
  cudaStream_t s = (cudaStream_t)stream;
  const bool train = opt != nullptr;
  yr_cdae_tensors none = {};
  int rrc = train ? launch_cdae_row<true>(h, B, s, *P, *grads, nU, nI, uid, w, true, nullptr, 0, loss + 1, err, hidden_act)
                  : launch_cdae_row<false>(h, B, s, *P, none, nU, nI, uid, w, true, nullptr, 0, loss + 1, err, hidden_act);
  if (rrc) return rrc;
  cdae_finish_kernel<<<1, 1, 0, s>>>(loss, w.total, step_loss);
  YR_CHECK_LAUNCH();
  if (!train) return YR_OK;
  const bool adam = opt->kind != YR_OPT_SGD;
  struct { float* p; float* g; float* m; float* v; int64_t n; } ts[5] = {
      {P->Wh, grads->Wh, adam ? m->Wh : nullptr, adam ? v->Wh : nullptr, (int64_t)h * nI},
      {P->bh, grads->bh, adam ? m->bh : nullptr, adam ? v->bh : nullptr, (int64_t)h},
      {P->Vu, grads->Vu, adam ? m->Vu : nullptr, adam ? v->Vu : nullptr, nU * h},
      {P->Wo, grads->Wo, adam ? m->Wo : nullptr, adam ? v->Wo : nullptr, nI * h},
      {P->bo, grads->bo, adam ? m->bo : nullptr, adam ? v->bo : nullptr, nI}};
  // one launch for the tensors whose size is a multiple of 4 (all of them at h = 64 and a catalog size % 4 == 0),
  // gradients cleared in the same pass; anything else takes the single-tensor path
  float *pp[5], *gg[5], *mm[5], *vv[5];
  int64_t nn[5];
  int cnt = 0;
  for (auto& t : ts) {
    const bool aligned = ((t.n & 3) == 0) &&
        ((((uintptr_t)t.p | (uintptr_t)t.g | (adam ? ((uintptr_t)t.m | (uintptr_t)t.v) : 0)) & 15) == 0);
    if (aligned) {
      pp[cnt] = t.p; gg[cnt] = t.g; mm[cnt] = t.m; vv[cnt] = t.v; nn[cnt++] = t.n;
    } else {
      int rc = yr_dense_opt_step(t.p, t.g, t.m, t.v, t.n, opt, stream);
      if (rc) return rc;
      YR_CUDA(cudaMemsetAsync(t.g, 0, sizeof(float) * (size_t)t.n, s));
    }
  }
  if (cnt) {
    int rc = yr_dense_opt_step_multi(cnt, pp, gg, mm, vv, nn, opt, 1, stream);
    if (rc) return rc;
  }
  return YR_OK;
}

extern "C" int yr_nsbce_loss(const float* pred, const float* target, const float* negative_mask, int64_t n,
                             float* loss, void* ws, size_t ws_bytes, yr_stream stream) {
  if (!pred || !target || !negative_mask || !loss || !ws || ws_bytes < 16 || n <= 0) return YR_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  YR_CUDA(cudaMemsetAsync(ws, 0, 16, s));
  int64_t blocks = (n + 255) / 256;
  if (blocks > yr_sm_count() * 8) blocks = yr_sm_count() * 8;
  nsbce_kernel<<<(unsigned)blocks, 256, 0, s>>>(pred, target, negative_mask, n, (double*)ws);
  YR_CHECK_LAUNCH();
  nsbce_finish_kernel<<<1, 1, 0, s>>>((const double*)ws, loss);
  YR_CHECK_LAUNCH();
  return YR_OK;
}
