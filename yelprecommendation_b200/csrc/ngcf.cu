// NGCF propagation kernels (sm_100a).
//   (the CSR SpMM lives in spmm.cu)
//   yr_ngcf_layer_fwd    — NGCF.embedding_propagation (reference models/ngcf.py:60-72)
//   yr_ngcf_layer_bwd    — its gradient (autograd through the two SpMMs / two Linear layers)
//   yr_ngcf_tail         — gather/concat/dot tail of bpr_forward + BPRLoss and its scatter backward
//                          (reference models/ngcf.py:37-45, loss.py:25-27)
//   yr_dense_opt_step    — torch.optim Adam/AdamW/SGD single-tensor step (trainers/base_trainer.py:34-40)
#include <stdlib.h>
#include "common.cuh"

namespace yr {

// ---------------------------------------------------------------------------------------------
// Dense part of one layer, forward: out = leaky( [LE+E | E*LE] . [W1^T ; W2^T] ).
// 256 threads, tile = TM rows x D cols, thread = 4 rows x 4 cols, k runs 0..2D-1 as one fma chain
// (first the W1 term, then the W2 term — the order the oracle restates).
// ---------------------------------------------------------------------------------------------
// Packed FP32 FMA (FFMA2, sm_100): two IEEE fmas per lane per instruction — each component is exactly fmaf(), so results
// are bit-identical to the scalar chain while the FMA pipe does twice the work per issue slot (a 3-register FFMA issues
// every other cycle per scheduler on Blackwell).
__device__ __forceinline__ void fma2(float2& acc, float a, const float2 b) { acc = __ffma2_rn(make_float2(a, a), b, acc); }

template <int D>
struct DenseCfg {
  static constexpr int kThreads = 256;
  static constexpr int kColGroups = D / 4;
  static constexpr int kRowGroups = kThreads / kColGroups;
  static constexpr int TM = 4 * kRowGroups;                       // 64 for D=64
  static constexpr int RO = D / kRowGroups;                       // dW rows (o) per thread: 1 / 4 / 16 for D = 32 / 64 / 128
  static constexpr size_t kSmemFwd = (size_t)(2 * D * TM + 2 * D * D) * sizeof(float);
  static constexpr size_t kSmemBwd = (size_t)(3 * TM * D + 2 * D * D) * sizeof(float);
  static_assert(D == 32 || D == 64 || D == 128, "dense transforms: D in {32, 64, 128}");
};

template <int D>
__global__ void __launch_bounds__(256)
ngcf_dense_fwd_kernel(const float* __restrict__ E, const float* __restrict__ LE,
                      const float* __restrict__ W1, const float* __restrict__ W2, float slope,
                      int64_t n, float* __restrict__ Eout) {
  using C = DenseCfg<D>;
  constexpr int TM = C::TM;
  extern __shared__ __align__(16) float smem[];
  float* As = smem;                 // [2D][TM]   k-major: S then P
  float* Ws = smem + 2 * D * TM;    // [2D][D]    Ws[k][o] = Wcat[o][k]
  const int tid = threadIdx.x;
  const int tx = tid % C::kColGroups, ty = tid / C::kColGroups;

  for (int idx = tid; idx < D * D; idx += C::kThreads) {
    const int o = idx / D, k = idx % D;
    Ws[k * D + o] = W1[idx];
    Ws[(D + k) * D + o] = W2[idx];
  }
  const int64_t n_tiles = (n + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * TM;
    __syncthreads();   // previous tile's readers are done with As (and Ws is written on the first pass)
    for (int idx = tid; idx < TM * (D / 4); idx += C::kThreads) {
      const int r = idx % TM, c4 = idx / TM;
      float4 e = make_float4(0.f, 0.f, 0.f, 0.f), le = e;
      if (r0 + r < n) {
        e = __ldg(reinterpret_cast<const float4*>(E + (r0 + r) * D) + c4);
        le = __ldg(reinterpret_cast<const float4*>(LE + (r0 + r) * D) + c4);
      }
      const int k = c4 * 4;
      As[(k + 0) * TM + r] = le.x + e.x; As[(k + 1) * TM + r] = le.y + e.y;
      As[(k + 2) * TM + r] = le.z + e.z; As[(k + 3) * TM + r] = le.w + e.w;
      As[(D + k + 0) * TM + r] = e.x * le.x; As[(D + k + 1) * TM + r] = e.y * le.y;
      As[(D + k + 2) * TM + r] = e.z * le.z; As[(D + k + 3) * TM + r] = e.w * le.w;
    }
    __syncthreads();
    float2 acc[4][2];                    // [row][column pair]
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) acc[i][j] = make_float2(0.f, 0.f);
#pragma unroll 8
    for (int k = 0; k < 2 * D; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(As + k * TM + ty * 4);
      const float4 w = *reinterpret_cast<const float4*>(Ws + k * D + tx * 4);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float2 wv[2] = {make_float2(w.x, w.y), make_float2(w.z, w.w)};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) fma2(acc[i][j], av[i], wv[j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t r = r0 + ty * 4 + i;
      if (r < n) {
        float4 o;
        o.x = acc[i][0].x > 0.f ? acc[i][0].x : acc[i][0].x * slope;
        o.y = acc[i][0].y > 0.f ? acc[i][0].y : acc[i][0].y * slope;
        o.z = acc[i][1].x > 0.f ? acc[i][1].x : acc[i][1].x * slope;
        o.w = acc[i][1].y > 0.f ? acc[i][1].y : acc[i][1].y * slope;
        reinterpret_cast<float4*>(Eout + r * D)[tx] = o;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Dense part of one layer, backward. Per tile of TM rows:
//   dZ = G_next * (E_next > 0 ? 1 : slope)
//   dS = dZ W1, dP = dZ W2          -> T = dS + dP*E (SpMM operand), G += dS + dP*LE
//   dW1 += dZ^T (LE+E), dW2 += dZ^T (E*LE)   (register accumulators across the CTA's tiles,
//                                             per-CTA partials to ws, fixed-order reduce afterwards)
// ---------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256)
ngcf_dense_bwd_kernel(const float* __restrict__ E, const float* __restrict__ LE,
                      const float* __restrict__ Enext, const float* __restrict__ Gnext,
                      const float* __restrict__ W1, const float* __restrict__ W2, float slope,
                      int64_t n, float* __restrict__ G, float* __restrict__ T,
                      float* __restrict__ ws, const int32_t* __restrict__ row_list,
                      const int32_t* __restrict__ row_count) {
  // row_list != NULL: only the listed rows carry a gradient (top layer of a BPR step: the 3B batch rows); tile row q
  // is graph row row_list[q], everything else is unchanged.
  using C = DenseCfg<D>;
  constexpr int TM = C::TM;
  constexpr int RO = C::RO;
  if (row_list) n = *row_count;
  extern __shared__ __align__(16) float smem[];
  float* dZs = smem;                    // [TM][D]
  float* Ss = dZs + TM * D;             // [TM][D]  LE + E
  float* Ps = Ss + TM * D;              // [TM][D]  E * LE
  float* W1s = Ps + TM * D;             // [D][D]  (o, i) as stored
  float* W2s = W1s + D * D;
  const int tid = threadIdx.x;
  const int tx = tid % C::kColGroups, ty = tid / C::kColGroups;

  for (int idx = tid; idx < D * D / 4; idx += C::kThreads) {
    reinterpret_cast<float4*>(W1s)[idx] = __ldg(reinterpret_cast<const float4*>(W1) + idx);
    reinterpret_cast<float4*>(W2s)[idx] = __ldg(reinterpret_cast<const float4*>(W2) + idx);
  }
  float2 dw1[RO][2], dw2[RO][2];         // [o][column pair]
#pragma unroll
  for (int i = 0; i < RO; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) { dw1[i][j] = make_float2(0.f, 0.f); dw2[i][j] = make_float2(0.f, 0.f); }

  const int64_t n_tiles = (n + TM - 1) / TM;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * TM;
    __syncthreads();
    // all global loads of the tile first (16 independent float4 per thread in flight), then the transforms
    constexpr int kLd = TM * (D / 4) / C::kThreads;
    float4 e4[kLd], le4[kLd], en4[kLd], g4[kLd];
#pragma unroll
    for (int q = 0; q < kLd; ++q) {
      const int idx = tid + q * C::kThreads;
      const int r = idx / (D / 4), c4 = idx % (D / 4);
      const bool ok = r0 + r < n;
      const int64_t rr = ok ? r0 + r : r0;                                   // r0 < n: a valid row to read instead
      const int64_t off = (row_list ? (int64_t)__ldg(row_list + rr) : rr) * D;
      e4[q] = __ldg(reinterpret_cast<const float4*>(E + off) + c4);
      le4[q] = __ldg(reinterpret_cast<const float4*>(LE + off) + c4);
      en4[q] = __ldg(reinterpret_cast<const float4*>(Enext + off) + c4);
      g4[q] = __ldg(reinterpret_cast<const float4*>(Gnext + off) + c4);
    }
#pragma unroll
    for (int q = 0; q < kLd; ++q) {
      const int idx = tid + q * C::kThreads;
      const int r = idx / (D / 4);
      float4 sv = make_float4(0.f, 0.f, 0.f, 0.f), pv = sv, dz = sv;
      if (r0 + r < n) {
        const float4 e = e4[q], le = le4[q], en = en4[q], g = g4[q];
        dz.x = en.x > 0.f ? g.x : g.x * slope; dz.y = en.y > 0.f ? g.y : g.y * slope;
        dz.z = en.z > 0.f ? g.z : g.z * slope; dz.w = en.w > 0.f ? g.w : g.w * slope;
        sv = make_float4(le.x + e.x, le.y + e.y, le.z + e.z, le.w + e.w);
        pv = make_float4(e.x * le.x, e.y * le.y, e.z * le.z, e.w * le.w);
      }
      reinterpret_cast<float4*>(Ss)[idx] = sv;
      reinterpret_cast<float4*>(Ps)[idx] = pv;
      reinterpret_cast<float4*>(dZs)[idx] = dz;
    }
    __syncthreads();

    // ---- dS, dP: rows ty*4.., cols tx*4.. ; k = o, four k per shared-memory round ----
    float2 ds[4][2], dp[4][2];          // [row][column pair]
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) { ds[i][j] = make_float2(0.f, 0.f); dp[i][j] = make_float2(0.f, 0.f); }
#pragma unroll 2
    for (int o = 0; o < D; o += 4) {
      float av[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 a4 = *reinterpret_cast<const float4*>(dZs + (ty * 4 + i) * D + o);
        av[i][0] = a4.x; av[i][1] = a4.y; av[i][2] = a4.z; av[i][3] = a4.w;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 w1 = *reinterpret_cast<const float4*>(W1s + (o + k) * D + tx * 4);
        const float4 w2 = *reinterpret_cast<const float4*>(W2s + (o + k) * D + tx * 4);
        const float2 w1v[2] = {make_float2(w1.x, w1.y), make_float2(w1.z, w1.w)};
        const float2 w2v[2] = {make_float2(w2.x, w2.y), make_float2(w2.z, w2.w)};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            fma2(ds[i][j], av[i][k], w1v[j]);
            fma2(dp[i][j], av[i][k], w2v[j]);
          }
      }
    }
    // epilogue two rows at a time: their E / LE / G loads (L1 / L2 hits: this CTA has just read the tile) are issued
    // together, then T is stored and G updated — shared memory holds S and P instead of E and LE
#pragma unroll
    for (int i0 = 0; i0 < 4; i0 += 2) {
      float4 e[2], le[2], g[2];
      int64_t rg[2];
      bool ok[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int64_t r = r0 + ty * 4 + i0 + h;
        ok[h] = r < n;
        const int64_t rr = ok[h] ? r : r0;
        rg[h] = row_list ? (int64_t)__ldg(row_list + rr) : rr;
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        e[h] = __ldg(reinterpret_cast<const float4*>(E + rg[h] * D) + tx);
        le[h] = __ldg(reinterpret_cast<const float4*>(LE + rg[h] * D) + tx);
        g[h] = *(reinterpret_cast<const float4*>(G + rg[h] * D) + tx);
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (!ok[h]) continue;
        const int i = i0 + h;
        float4 t, dd;
        t.x = fmaf(dp[i][0].x, e[h].x, ds[i][0].x); t.y = fmaf(dp[i][0].y, e[h].y, ds[i][0].y);
        t.z = fmaf(dp[i][1].x, e[h].z, ds[i][1].x); t.w = fmaf(dp[i][1].y, e[h].w, ds[i][1].y);
        dd.x = fmaf(dp[i][0].x, le[h].x, ds[i][0].x); dd.y = fmaf(dp[i][0].y, le[h].y, ds[i][0].y);
        dd.z = fmaf(dp[i][1].x, le[h].z, ds[i][1].x); dd.w = fmaf(dp[i][1].y, le[h].w, ds[i][1].y);
        reinterpret_cast<float4*>(T + rg[h] * D)[tx] = t;
        float4 gn = g[h];
        gn.x += dd.x; gn.y += dd.y; gn.z += dd.z; gn.w += dd.w;
        reinterpret_cast<float4*>(G + rg[h] * D)[tx] = gn;
      }
    }

    // ---- dW1[o,i], dW2[o,i]: o = ty*RO.., i = tx*4.. ; k = row (rows past n hold dZ = 0) ----
#pragma unroll 4
    for (int r = 0; r < TM; ++r) {
      float dzv[RO];
      if constexpr (RO >= 4) {
#pragma unroll
        for (int i = 0; i < RO; i += 4) {
          const float4 dz = *reinterpret_cast<const float4*>(dZs + r * D + ty * RO + i);
          dzv[i] = dz.x; dzv[i + 1] = dz.y; dzv[i + 2] = dz.z; dzv[i + 3] = dz.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < RO; ++i) dzv[i] = dZs[r * D + ty * RO + i];
      }
      const float4 s4 = *reinterpret_cast<const float4*>(Ss + r * D + tx * 4);
      const float4 p4 = *reinterpret_cast<const float4*>(Ps + r * D + tx * 4);
      const float2 sv[2] = {make_float2(s4.x, s4.y), make_float2(s4.z, s4.w)};
      const float2 pv[2] = {make_float2(p4.x, p4.y), make_float2(p4.z, p4.w)};
#pragma unroll
      for (int i = 0; i < RO; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          fma2(dw1[i][j], dzv[i], sv[j]);
          fma2(dw2[i][j], dzv[i], pv[j]);
        }
    }
  }
  float* my = ws + (size_t)blockIdx.x * 2 * D * D;
#pragma unroll
  for (int i = 0; i < RO; ++i) {
    const int o = ty * RO + i;
    reinterpret_cast<float4*>(my + o * D)[tx] = make_float4(dw1[i][0].x, dw1[i][0].y, dw1[i][1].x, dw1[i][1].y);
    reinterpret_cast<float4*>(my + D * D + o * D)[tx] = make_float4(dw2[i][0].x, dw2[i][0].y, dw2[i][1].x, dw2[i][1].y);
  }
}

// Several parameter tensors in ONE launch (a step of a model with many small tensors is launch-bound otherwise).
// Tensor t covers float4 units [start4[t], start4[t+1]) of a virtual concatenation; sizes must be multiples of 4.
struct MultiOptArgs {
  float* p[YR_OPT_MAX_TENSORS]; float* g[YR_OPT_MAX_TENSORS]; float* m[YR_OPT_MAX_TENSORS]; float* v[YR_OPT_MAX_TENSORS];
  int64_t start4[YR_OPT_MAX_TENSORS + 1];
  int count, zero_grad;
};

__global__ void __launch_bounds__(256)
dense_opt_multi_kernel(MultiOptArgs a, yr_opt opt) {
  OptScalars os;
  opt_scalars_for_step(os, opt, opt.step);
  const bool adam = opt.kind != YR_OPT_SGD;
  const int64_t total4 = a.start4[a.count];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += stride) {
    int t = 0;
#pragma unroll
    for (int q = 1; q < YR_OPT_MAX_TENSORS; ++q) t += (q < a.count && i >= a.start4[q]) ? 1 : 0;
    const int64_t k = i - a.start4[t];
    float4* pp = reinterpret_cast<float4*>(a.p[t]) + k;
    float4* gp = reinterpret_cast<float4*>(a.g[t]) + k;
    float4 pv = *pp;
    const float4 gv = *gp;
    float4 mv = make_float4(0.f, 0.f, 0.f, 0.f), vv = mv;
    if (adam) { mv = reinterpret_cast<float4*>(a.m[t])[k]; vv = reinterpret_cast<float4*>(a.v[t])[k]; }
    opt_update(os, pv.x, gv.x, mv.x, vv.x);
    opt_update(os, pv.y, gv.y, mv.y, vv.y);
    opt_update(os, pv.z, gv.z, mv.z, vv.z);
    opt_update(os, pv.w, gv.w, mv.w, vv.w);
    *pp = pv;
    if (adam) { reinterpret_cast<float4*>(a.m[t])[k] = mv; reinterpret_cast<float4*>(a.v[t])[k] = vv; }
    if (a.zero_grad) *gp = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

// dW[idx] = sum over CTA partials in CTA order (deterministic).
// Block = 32 outputs x 8 partial-groups: group g sums partials g, g+8, ... (8 loads in flight), then the 8 group
// sums are added in group order.
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const float* __restrict__ ws, int n_parts, int len,
                       float* __restrict__ out1, float* __restrict__ out2, int half) {
  __shared__ float sh[8][33];
  const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5;
  const int idx = blockIdx.x * 32 + lane;
  float acc = 0.f;
  if (idx < len) {
    int p = grp;
    for (; p + 56 < n_parts; p += 64) {
      float x[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) x[q] = ws[(size_t)(p + 8 * q) * len + idx];
#pragma unroll
      for (int q = 0; q < 8; ++q) acc += x[q];
    }
    for (; p < n_parts; p += 8) acc += ws[(size_t)p * len + idx];
  }
  sh[grp][lane] = acc;
  __syncthreads();
  if (grp == 0 && idx < len) {
    float t = sh[0][lane];
#pragma unroll
    for (int g = 1; g < 8; ++g) t += sh[g][lane];
    if (idx < half) out1[idx] = t; else out2[idx - half] = t;
  }
}

// ---------------------------------------------------------------------------------------------
// Tail: warp per triple, all layers.
// ---------------------------------------------------------------------------------------------
template <int VPL>
__global__ void __launch_bounds__(256)
ngcf_tail_kernel(const float* const* __restrict__ E_layers, float* const* __restrict__ G_layers,
                 int n_layers, int64_t nU, int64_t nI, const int64_t* __restrict__ uid,
                 const int64_t* __restrict__ pos, const int64_t* __restrict__ neg, int64_t B,
                 float* __restrict__ pos_out, float* __restrict__ neg_out, double* loss_acc,
                 int32_t* err) {
  constexpr int D = VPL * 32;
  constexpr int kMaxL = 8;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  __shared__ double s_part[8];
  double wl = 0.0;
  const float inv_b = 1.f / (float)B;
  for (int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; b < B; b += nwarps) {
    const int64_t u = uid[b], p = pos[b], n = neg[b];
    if (u < 0 || u >= nU || p < 0 || p >= nI || n < 0 || n >= nI) {
      if (lane == 0 && err) atomicExch(err, 1);
      continue;
    }
    float dp = 0.f, dn = 0.f;
    for (int l = 0; l <= n_layers && l < kMaxL; ++l) {
      const float* El = E_layers[l];
      const Row<VPL> ur = ld_row<VPL>(El + u * D, lane);
      const Row<VPL> pr = ld_row<VPL>(El + (nU + p) * D, lane);
      const Row<VPL> nr = ld_row<VPL>(El + (nU + n) * D, lane);
#pragma unroll
      for (int j = 0; j < VPL; ++j) { dp = fmaf(ur.x[j], pr.x[j], dp); dn = fmaf(ur.x[j], nr.x[j], dn); }
    }
    dp = warp_sum(dp);
    dn = warp_sum(dn);
    const float x = dp - dn;
    if (lane == 0) {
      if (pos_out) pos_out[b] = dp;
      if (neg_out) neg_out[b] = dn;
    }
    wl += (double)neg_logsigmoid(x);
    if (G_layers) {
      const float g = neg_logsigmoid_grad(x) * inv_b;
      for (int l = 0; l <= n_layers && l < kMaxL; ++l) {
        const float* El = E_layers[l];
        float* Gl = G_layers[l];
        const Row<VPL> ur = ld_row<VPL>(El + u * D, lane);
        const Row<VPL> pr = ld_row<VPL>(El + (nU + p) * D, lane);
        const Row<VPL> nr = ld_row<VPL>(El + (nU + n) * D, lane);
        Row<VPL> gu, gp, gn;
#pragma unroll
        for (int j = 0; j < VPL; ++j) {
          gu.x[j] = __fsub_rn(__fmul_rn(g, pr.x[j]), __fmul_rn(g, nr.x[j]));   // two rounded products, like autograd
          gp.x[j] = g * ur.x[j];
          gn.x[j] = -gp.x[j];
        }
        red_row<VPL>(Gl + u * D, lane, gu);
        red_row<VPL>(Gl + (nU + p) * D, lane, gp);
        red_row<VPL>(Gl + (nU + n) * D, lane, gn);
      }
    }
  }
  if (lane == 0) s_part[wib] = wl;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += s_part[i];
    if (t != 0.0) atomicAdd(loss_acc, t);
  }
}

__global__ void tail_finish_kernel(double* loss_acc, int64_t B, double* loss_sum, float* step_loss) {
  const float mean = (float)(*loss_acc / (double)B);
  if (step_loss) *step_loss = mean;
  if (loss_sum) *loss_sum += (double)mean;
  *loss_acc = 0.0;
}

// ---------------------------------------------------------------------------------------------
// Dense optimizer step, float4 vectorised with scalar tail. vec == 0 (a pointer that is not 16-byte aligned, e.g. a view
// that starts inside a tensor): every element takes the scalar loop — same per-element arithmetic, same bits.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
dense_opt_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                 float* __restrict__ v, int64_t n, yr_opt opt, int vec) {
  OptScalars os;
  opt_scalars_for_step(os, opt, opt.step);
  const bool adam = opt.kind != YR_OPT_SGD;
  const int64_t n4 = vec ? n >> 2 : 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pv = reinterpret_cast<float4*>(p)[i];
    const float4 gv = __ldg(reinterpret_cast<const float4*>(g) + i);
    float4 mv = make_float4(0.f, 0.f, 0.f, 0.f), vv = mv;
    if (adam) { mv = reinterpret_cast<float4*>(m)[i]; vv = reinterpret_cast<float4*>(v)[i]; }
    opt_update(os, pv.x, gv.x, mv.x, vv.x);
    opt_update(os, pv.y, gv.y, mv.y, vv.y);
    opt_update(os, pv.z, gv.z, mv.z, vv.z);
    opt_update(os, pv.w, gv.w, mv.w, vv.w);
    reinterpret_cast<float4*>(p)[i] = pv;
    if (adam) { reinterpret_cast<float4*>(m)[i] = mv; reinterpret_cast<float4*>(v)[i] = vv; }
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float mv = 0.f, vv = 0.f, pv = p[i];
    if (adam) { mv = m[i]; vv = v[i]; }
    opt_update(os, pv, g[i], mv, vv);
    p[i] = pv;
    if (adam) { m[i] = mv; v[i] = vv; }
  }
}

constexpr int kBwdCtasPerSm = 2;

}  // namespace yr

using namespace yr;

// yr_dense_mode (include/yelprec_b200.h) travels per call / per trainer state; nothing here is process-wide.
// bits 0..7: yr_dense_mode; bits 8..15: SMs the tensor-core kernels leave empty (YR_DENSE_RESERVE)
static inline int mode_of(int m) { return m & 0xff; }
static inline int reserve_of(int m) { return (m >> 8) & 0xff; }
static inline bool mode_ok(int m) {
  return m >= 0 && (m >> 16) == 0 && (mode_of(m) == YR_DENSE_FP32 || mode_of(m) == YR_DENSE_TC_FWD || mode_of(m) == YR_DENSE_TC);
}
static inline bool fwd_tc(int m) { return mode_of(m) != YR_DENSE_FP32; }
static inline bool bwd_tc(int m) { return mode_of(m) == YR_DENSE_TC; }

template <int D>
static int dense_fwd_fp32_launch(int64_t n, const float* E, const float* LE, const float* W1, const float* W2, float slope,
                                 float* E_next, cudaStream_t s) {
  using C = DenseCfg<D>;
  static AttrOnce attr;
  { int rc_ = attr.set(ngcf_dense_fwd_kernel<D>, (int)C::kSmemFwd); if (rc_) return rc_; }
  const int64_t n_tiles = (n + C::TM - 1) / C::TM;
  int64_t grid = (int64_t)yr_sm_count() * (D <= 64 ? 3 : 1);
  if (grid > n_tiles) grid = n_tiles;
  ngcf_dense_fwd_kernel<D><<<(unsigned)grid, C::kThreads, C::kSmemFwd, s>>>(E, LE, W1, W2, slope, n, E_next);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

template <int D>
static int dense_bwd_fp32_launch(int64_t n, const float* E, const float* LE, const float* E_next, const float* G_next,
                                 const float* W1, const float* W2, float slope, float* G, float* T, float* ws,
                                 cudaStream_t s, int* n_parts) {
  using C = DenseCfg<D>;
  static AttrOnce attr;
  { int rc_ = attr.set(ngcf_dense_bwd_kernel<D>, (int)C::kSmemBwd); if (rc_) return rc_; }
  const int64_t n_tiles = (n + C::TM - 1) / C::TM;
  int64_t grid = (int64_t)yr_sm_count() * (D <= 64 ? kBwdCtasPerSm : 1);       // D = 128: 176 KB of shared memory per CTA
  if (grid > n_tiles) grid = n_tiles;
  ngcf_dense_bwd_kernel<D><<<(unsigned)grid, C::kThreads, C::kSmemBwd, s>>>(E, LE, E_next, G_next, W1, W2, slope, n, G, T, ws,
                                                                          nullptr, nullptr);
  YR_CHECK_LAUNCH();
  *n_parts = (int)grid;
  return YR_OK;
}

extern "C" int yr_ngcf_dense_fwd(int d, int64_t n, const float* E, const float* LE, const float* W1, const float* W2,
                                 float slope, float* E_next, int dense_mode, yr_stream stream) {
  if (!E || !LE || !W1 || !W2 || !E_next || n < 0 || !mode_ok(dense_mode)) return YR_ERR_BAD_ARG;
  if (d != 32 && d != 64 && d != 128) return YR_ERR_BAD_DIM;
  if (n == 0) return YR_OK;
  if (fwd_tc(dense_mode) && (d == 64 || d == 128))      // tcgen05 3xTF32 (ngcf_tc.cu); d = 32 runs on the FP32 pipe
    return yr_ngcf_dense_fwd_tc_launch_d(d, E, LE, W1, W2, slope, n, E_next, (cudaStream_t)stream, nullptr, nullptr, 0,
                                         reserve_of(dense_mode));
  switch (d) {
    case 32: return dense_fwd_fp32_launch<32>(n, E, LE, W1, W2, slope, E_next, (cudaStream_t)stream);
    case 64: return dense_fwd_fp32_launch<64>(n, E, LE, W1, W2, slope, E_next, (cudaStream_t)stream);
    default: return dense_fwd_fp32_launch<128>(n, E, LE, W1, W2, slope, E_next, (cudaStream_t)stream);
  }
}

extern "C" int yr_ngcf_layer_fwd(const yr_csr* L, int d, const float* E, const float* W1, const float* W2,
                                 float slope, float* E_next, float* LE_save, int dense_mode, yr_stream stream) {
  if (!L || !E || !W1 || !W2 || !E_next || !LE_save || L->n_rows <= 0 || !mode_ok(dense_mode)) return YR_ERR_BAD_ARG;
  if (d != 32 && d != 64 && d != 128) return YR_ERR_BAD_DIM;
  int rc = yr_spmm_csr(L, d, E, LE_save, 0, stream);
  if (rc) return rc;
  return yr_ngcf_dense_fwd(d, L->n_rows, E, LE_save, W1, W2, slope, E_next, dense_mode, stream);
}

extern "C" size_t yr_ngcf_layer_bwd_ws_bytes(int d) {
  return (size_t)yr_sm_count() * kBwdCtasPerSm * 2 * (size_t)d * d * sizeof(float);
}

// the dense backward kernel WITHOUT the reduction of its per-CTA dW partials (n_parts of them are left in ws)
static int dense_bwd_launch(int d, int64_t n, const float* E, const float* LE, const float* E_next, const float* G_next,
                            const float* W1, const float* W2, float slope, float* G, float* T, void* ws, size_t ws_bytes,
                            int dense_mode, cudaStream_t s, int* n_parts) {
  if (!E || !LE || !E_next || !G_next || !W1 || !W2 || !G || !T || !ws || n <= 0 || !mode_ok(dense_mode)) return YR_ERR_BAD_ARG;
  if (d != 32 && d != 64 && d != 128) return YR_ERR_BAD_DIM;
  if (ws_bytes < yr_ngcf_layer_bwd_ws_bytes(d)) return YR_ERR_WORKSPACE;
  if (bwd_tc(dense_mode) && (d == 64 || d == 128))          // tcgen05 3xTF32 (ngcf_tc_bwd.cu); d = 32 runs on the FP32 pipe
    return yr_ngcf_dense_bwd_tc_launch(d, E, LE, E_next, G_next, W1, W2, slope, n, G, T, (float*)ws, n_parts, s, nullptr, nullptr,
                                       0, reserve_of(dense_mode));
  switch (d) {
    case 32: return dense_bwd_fp32_launch<32>(n, E, LE, E_next, G_next, W1, W2, slope, G, T, (float*)ws, s, n_parts);
    case 64: return dense_bwd_fp32_launch<64>(n, E, LE, E_next, G_next, W1, W2, slope, G, T, (float*)ws, s, n_parts);
    default: return dense_bwd_fp32_launch<128>(n, E, LE, E_next, G_next, W1, W2, slope, G, T, (float*)ws, s, n_parts);
  }
}

static int dense_bwd_reduce(int d, const void* ws, int n_parts, float* dW1, float* dW2, cudaStream_t s) {
  const int len = 2 * d * d;
  reduce_partials_kernel<<<(len + 31) / 32, 256, 0, s>>>((const float*)ws, n_parts, len, dW1, dW2, d * d);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

extern "C" int yr_ngcf_dense_bwd(int d, int64_t n, const float* E, const float* LE, const float* E_next,
                                 const float* G_next, const float* W1, const float* W2, float slope,
                                 float* G, float* T, float* dW1, float* dW2, void* ws, size_t ws_bytes,
                                 int dense_mode, yr_stream stream) {
  if (!dW1 || !dW2) return YR_ERR_BAD_ARG;
  int parts = 0;
  int rc = dense_bwd_launch(d, n, E, LE, E_next, G_next, W1, W2, slope, G, T, ws, ws_bytes, dense_mode, (cudaStream_t)stream,
                            &parts);
  if (rc) return rc;
  return dense_bwd_reduce(d, ws, parts, dW1, dW2, (cudaStream_t)stream);
}

// ---- top layer of a BPR step: only the <= 3B batch rows carry a gradient -------------------------------------
namespace yr {
__global__ void __launch_bounds__(256)
touched_rows_kernel(const int64_t* __restrict__ uid, const int64_t* __restrict__ pos, const int64_t* __restrict__ neg,
                    int64_t B, int64_t nU, int64_t nI, int32_t* flag, int32_t* list, int32_t* count) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < 3 * B; i += (int64_t)gridDim.x * blockDim.x) {
    const int which = (int)(i / B);
    const int64_t b = i - which * B;
    const int64_t id = which == 0 ? uid[b] : (which == 1 ? pos[b] : neg[b]);
    if (id < 0 || id >= (which == 0 ? nU : nI)) continue;          // the tail kernel has flagged the error
    const int64_t row = which == 0 ? id : nU + id;
    if (atomicExch(flag + row, 1) == 0) list[atomicAdd(count, 1)] = (int32_t)row;
  }
}

__global__ void __launch_bounds__(256)
untouch_rows_kernel(int32_t* flag, const int32_t* __restrict__ list, const int32_t* __restrict__ count) {
  const int n = *count;                 // the counter itself is cleared by a memset node after this kernel
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) flag[list[i]] = 0;
}

// G += A^T T restricted to the flagged rows j of T: every stored A[j, i] scatters a(j,i) * T[j] into G[i] with one
// vector RED per lane. Walks the SpMM plan of A (chunks of <= 128 non-zeros), so hub rows are spread over many groups.
template <int D>
__global__ void __launch_bounds__(256)
spmm_scatter_rows_kernel(yr_csr A, const int32_t* __restrict__ flag, const float* __restrict__ T, float* __restrict__ G) {
  constexpr int kVec = D / 4, LPR = kVec >= 32 ? 32 : kVec, VPT = kVec / LPR, CPW = 32 / LPR;
  const int lane = threadIdx.x & 31, sub = lane / LPR, sl = lane % LPR;
  const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int4* __restrict__ desc = reinterpret_cast<const int4*>(A.chunk_desc);
  for (int cb = gwarp * CPW; cb < A.n_chunks; cb += nwarps * CPW) {
    const int c = cb + sub;
    int4 dsc = make_int4(0, 0, 0, -1);
    if (c < A.n_chunks) dsc = __ldg(desc + c);
    const int row = dsc.x, s0 = dsc.y;
    int len = dsc.z & 0xff;
    if (c >= A.n_chunks || !__ldg(flag + row)) len = 0;
    int maxlen = len;
#pragma unroll
    for (int o = LPR; o < 32; o <<= 1) maxlen = max(maxlen, __shfl_xor_sync(kFull, maxlen, o));
    if (maxlen == 0) continue;
    float4 t[VPT];
#pragma unroll
    for (int v = 0; v < VPT; ++v)
      t[v] = len ? reinterpret_cast<const float4*>(T + (int64_t)row * D)[sl * VPT + v] : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j0 = 0; j0 < maxlen; j0 += LPR) {
      const int j = j0 + sl;
      const int cc = (j < len) ? __ldg(A.col + s0 + j) : -1;
      const float aa = (j < len) ? __ldg(A.val + s0 + j) : 0.f;
      for (int q = 0; q < LPR && j0 + q < maxlen; ++q) {
        const int cq = __shfl_sync(kFull, cc, q, LPR);
        const float a = __shfl_sync(kFull, aa, q, LPR);
        if (cq >= 0) {
#pragma unroll
          for (int v = 0; v < VPT; ++v)
            atomicAdd(reinterpret_cast<float4*>(G + (int64_t)cq * D) + sl * VPT + v,
                      make_float4(a * t[v].x, a * t[v].y, a * t[v].z, a * t[v].w));
        }
      }
    }
  }
}
}  // namespace yr

// dense backward of one layer on the listed rows + scatter form of G += L^T T (ngcf_train_step, top layer)
// One helper stream + two events per device, created on first use (the only resources the library ever creates):
// independent memsets of a step run on it, ordered against the caller's stream with events. YR_NGCF_SIDE_STREAM=0
// keeps everything on the caller's stream.
struct SideStream { cudaStream_t stream; cudaEvent_t fork, join; };
static SideStream* side_stream() {
  static SideStream pool[64];
  static int state[64];                 // 0 = not tried, 1 = ready, -1 = unavailable
  const char* e = getenv("YR_NGCF_SIDE_STREAM");
  if (e && e[0] == '0') return nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (state[dev] == 0) {
    SideStream& x = pool[dev];
    const bool ok = cudaStreamCreateWithFlags(&x.stream, cudaStreamNonBlocking) == cudaSuccess &&
                    cudaEventCreateWithFlags(&x.fork, cudaEventDisableTiming) == cudaSuccess &&
                    cudaEventCreateWithFlags(&x.join, cudaEventDisableTiming) == cudaSuccess;
    state[dev] = ok ? 1 : -1;
  }
  return state[dev] == 1 ? &pool[dev] : nullptr;
}

static int rows_reduce(const yr_ngcf_state* st, int l, int parts, cudaStream_t s, SideStream* side);

static int ngcf_layer_bwd_rows(const yr_ngcf_state* st, int l, float slope, cudaStream_t s, SideStream* side) {
  const int d = st->d;
  using C = DenseCfg<64>;
  if (d != 64) return YR_ERR_BAD_DIM;
  // The tensor-core kernel has fixed costs (weight split launch, TMEM, ring fill: 22.7 us for the 48 tiles of a B = 2,048
  // step against 15.4 us for the FP32-pipe kernel, profiles/r02_launches_ngcf_step.csv; 42 vs 67 us on all 69,716 rows): it
  // takes over from ~16 k listed rows.
  if (bwd_tc(st->dense_mode) && st->row_list_cap >= 16384) {
    int parts = 0;
    int rc = yr_ngcf_dense_bwd_tc_launch(d, st->E[l], st->LE[l], st->E[l + 1], st->G[l + 1], st->W1[l], st->W2[l], slope,
                                         st->nU + st->nI, st->G[l], st->T, (float*)st->ws, &parts, s, st->row_list,
                                         st->row_count, st->row_list_cap);
    if (rc) return rc;
    rc = rows_reduce(st, l, parts, s, side);
    if (rc) return rc;
    const int64_t blocks_tc = ((int64_t)st->L.n_chunks + 15) / 16;
    spmm_scatter_rows_kernel<64><<<(unsigned)blocks_tc, 256, 0, s>>>(st->L, st->row_flag, st->T, st->G[l]);
    YR_CHECK_LAUNCH();
    return YR_OK;
  }
  int64_t grid = (st->row_list_cap + C::TM - 1) / C::TM;
  const int64_t cap = (int64_t)yr_sm_count() * kBwdCtasPerSm;
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  static AttrOnce attr;
  { int rc_ = attr.set(ngcf_dense_bwd_kernel<64>, (int)C::kSmemBwd); if (rc_) return rc_; }
  ngcf_dense_bwd_kernel<64><<<(unsigned)grid, C::kThreads, C::kSmemBwd, s>>>(
      st->E[l], st->LE[l], st->E[l + 1], st->G[l + 1], st->W1[l], st->W2[l], slope, st->nU + st->nI, st->G[l], st->T,
      (float*)st->ws, st->row_list, st->row_count);
  YR_CHECK_LAUNCH();
  int rc = rows_reduce(st, l, (int)grid, s, side);
  if (rc) return rc;
  const int wpb = 8, cpw = 2;
  int64_t blocks = ((int64_t)st->L.n_chunks + wpb * cpw - 1) / (wpb * cpw);
  spmm_scatter_rows_kernel<64><<<(unsigned)blocks, 256, 0, s>>>(st->L, st->row_flag, st->T, st->G[l]);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

// reduction of the rows-layer dW partials: on the side stream (joined by the caller) when there is one
static int rows_reduce(const yr_ngcf_state* st, int l, int parts, cudaStream_t s, SideStream* side) {
  const int len = 2 * st->d * st->d;
  cudaStream_t rs = s;
  if (side) {
    YR_CUDA(cudaEventRecord(side->fork, s));
    YR_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    rs = side->stream;
  }
  reduce_partials_kernel<<<(len + 31) / 32, 256, 0, rs>>>((const float*)st->ws, parts, len, st->dW1[l], st->dW2[l],
                                                         st->d * st->d);
  YR_CHECK_LAUNCH();
  if (side) YR_CUDA(cudaEventRecord(side->join, side->stream));
  return YR_OK;
}

extern "C" int yr_ngcf_layer_bwd(const yr_csr* LT, int d, const float* E, const float* LE, const float* E_next,
                                 const float* G_next, const float* W1, const float* W2, float slope,
                                 float* G, float* T, float* dW1, float* dW2, void* ws, size_t ws_bytes,
                                 int dense_mode, yr_stream stream) {
  if (!LT || LT->n_rows <= 0) return YR_ERR_BAD_ARG;
  int rc = yr_ngcf_dense_bwd(d, LT->n_rows, E, LE, E_next, G_next, W1, W2, slope, G, T, dW1, dW2, ws, ws_bytes, dense_mode,
                             stream);
  if (rc) return rc;
  return yr_spmm_csr(LT, d, T, G, 1, stream);
}

extern "C" int yr_ngcf_tail(const float* const* E_layers, float* const* G_layers, int n_layers,
                            int64_t nU, int64_t nI, int d, const int64_t* uid, const int64_t* pos,
                            const int64_t* neg, int64_t B, float* pos_out, float* neg_out,
                            double* loss_sum, float* step_loss, int32_t* err, yr_stream stream) {
  // loss_sum doubles as [0] running sum (+= batch mean) and needs a private accumulator: callers pass a
  // 2-double block: loss_sum[0] = running sum, loss_sum[1] = scratch accumulator (zero between calls).
  if (!E_layers || !uid || !pos || !neg || !loss_sum || B <= 0 || n_layers < 0 || n_layers > 7)
    return YR_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 256;
  int64_t blocks = (B * 32 + threads - 1) / threads;
  const int64_t cap = (int64_t)yr_sm_count() * 8;
  if (blocks > cap) blocks = cap;
  const unsigned g = (unsigned)blocks;
  double* acc = loss_sum + 1;
  switch (dim_vpl(d)) {
    case 1: ngcf_tail_kernel<1><<<g, threads, 0, s>>>(E_layers, G_layers, n_layers, nU, nI, uid, pos, neg, B, pos_out, neg_out, acc, err); break;
    case 2: ngcf_tail_kernel<2><<<g, threads, 0, s>>>(E_layers, G_layers, n_layers, nU, nI, uid, pos, neg, B, pos_out, neg_out, acc, err); break;
    case 4: ngcf_tail_kernel<4><<<g, threads, 0, s>>>(E_layers, G_layers, n_layers, nU, nI, uid, pos, neg, B, pos_out, neg_out, acc, err); break;
    case 8: ngcf_tail_kernel<8><<<g, threads, 0, s>>>(E_layers, G_layers, n_layers, nU, nI, uid, pos, neg, B, pos_out, neg_out, acc, err); break;
    default: return YR_ERR_BAD_DIM;
  }
  YR_CHECK_LAUNCH();
  tail_finish_kernel<<<1, 1, 0, s>>>(acc, B, loss_sum, step_loss);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

extern "C" int yr_dense_opt_step(float* p, const float* g, float* m, float* v, int64_t n,
                                 const yr_opt* opt, yr_stream stream) {
  if (!p || !g || !opt || n < 0) return YR_ERR_BAD_ARG;
  if (opt->kind < YR_OPT_SGD || opt->kind > YR_OPT_ADAMW) return YR_ERR_BAD_OPT;
  if (opt->kind != YR_OPT_SGD && (!m || !v)) return YR_ERR_BAD_ARG;
  if (n == 0) return YR_OK;
  const int threads = 256;
  int64_t blocks = ((n >> 2) + threads - 1) / threads;
  if (blocks < 1) blocks = 1;
  const int64_t cap = (int64_t)yr_sm_count() * 8;
  if (blocks > cap) blocks = cap;
  const bool adam = opt->kind != YR_OPT_SGD;
  const int vec = (((uintptr_t)p | (uintptr_t)g | (adam ? ((uintptr_t)m | (uintptr_t)v) : 0)) & 15) == 0;
  dense_opt_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(p, g, m, v, n, *opt, vec);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

extern "C" int yr_dense_opt_step_multi(int count, float* const* p, float* const* g, float* const* m, float* const* v,
                                       const int64_t* n, const yr_opt* opt, int zero_grad, yr_stream stream) {
  if (count < 0 || count > YR_OPT_MAX_TENSORS || !p || !g || !n || !opt) return YR_ERR_BAD_ARG;
  if (opt->kind < YR_OPT_SGD || opt->kind > YR_OPT_ADAMW) return YR_ERR_BAD_OPT;
  const bool adam = opt->kind != YR_OPT_SGD;
  if (adam && (!m || !v)) return YR_ERR_BAD_ARG;
  MultiOptArgs a;
  a.count = 0; a.zero_grad = zero_grad ? 1 : 0; a.start4[0] = 0;
  for (int t = 0; t < count; ++t) {
    if (n[t] < 0 || (n[t] & 3) || !p[t] || !g[t] || (adam && (!m[t] || !v[t]))) return YR_ERR_BAD_ARG;
    if (((uintptr_t)p[t] | (uintptr_t)g[t] | (adam ? ((uintptr_t)m[t] | (uintptr_t)v[t]) : 0)) & 15) return YR_ERR_BAD_ARG;
    if (n[t] == 0) continue;
    const int c = a.count++;
    a.p[c] = p[t]; a.g[c] = g[t]; a.m[c] = adam ? m[t] : nullptr; a.v[c] = adam ? v[t] : nullptr;
    a.start4[c + 1] = a.start4[c] + (n[t] >> 2);
  }
  if (a.count == 0) return YR_OK;
  const int threads = 256;
  int64_t blocks = (a.start4[a.count] + threads - 1) / threads;
  const int64_t cap = (int64_t)yr_sm_count() * 8;
  if (blocks > cap) blocks = cap;
  dense_opt_multi_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(a, *opt);
  YR_CHECK_LAUNCH();
  return YR_OK;
}

// ---------------------------------------------------------------------------------------------
// Composite entry points: a whole propagate / train step per host call.
// ---------------------------------------------------------------------------------------------
namespace yr {
__global__ void concat_layers_kernel(const float* const* __restrict__ E_layers, int n_layers, int64_t n,
                                     int d, float* __restrict__ out) {
  const int width = (n_layers + 1) * d;
  const int64_t total4 = n * (width / 4);
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total4;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = idx / (width / 4);
    const int c = (int)(idx % (width / 4)) * 4;
    const int l = c / d, k = c % d;
    reinterpret_cast<float4*>(out)[idx] = __ldg(reinterpret_cast<const float4*>(E_layers[l] + r * d + k));
  }
}
}  // namespace yr

static int ngcf_state_ok(const yr_ngcf_state* st) {
  if (!st || st->n_layers < 1 || st->n_layers > YR_NGCF_MAX_LAYERS || st->nU <= 0 || st->nI <= 0)
    return YR_ERR_BAD_ARG;
  if (yr_csr_ok(&st->L) || !st->E[0] || !mode_ok(st->dense_mode)) return YR_ERR_BAD_ARG;
  for (int l = 0; l < st->n_layers; ++l)
    if (!st->E[l + 1] || !st->LE[l] || !st->W1[l] || !st->W2[l]) return YR_ERR_BAD_ARG;
  return YR_OK;
}

extern "C" int yr_ngcf_propagate_prefix(const yr_ngcf_state* st, float slope, int n_prefix, yr_stream stream) {
  int rc = ngcf_state_ok(st);
  if (rc) return rc;
  if (n_prefix < 0 || n_prefix > st->n_layers) return YR_ERR_BAD_ARG;
  for (int l = 0; l < n_prefix; ++l) {
    rc = yr_ngcf_layer_fwd(&st->L, st->d, st->E[l], st->W1[l], st->W2[l], slope, st->E[l + 1], st->LE[l], st->dense_mode,
                           stream);
    if (rc) return rc;
  }
  return YR_OK;
}

extern "C" int yr_ngcf_propagate(const yr_ngcf_state* st, float slope, yr_stream stream) {
  int rc = ngcf_state_ok(st);
  if (rc) return rc;
  for (int l = 0; l < st->n_layers; ++l) {
    rc = yr_ngcf_layer_fwd(&st->L, st->d, st->E[l], st->W1[l], st->W2[l], slope,
                           st->E[l + 1], st->LE[l], st->dense_mode, stream);
    if (rc) return rc;
  }
  return YR_OK;
}

extern "C" int yr_ngcf_train_step_ex(const yr_ngcf_state* st, const yr_opt* opt, float slope,
                                     const int64_t* uid, const int64_t* pos, const int64_t* neg, int64_t B,
                                     float* step_loss, int prefix_done, yr_stream stream);

extern "C" int yr_ngcf_train_step(const yr_ngcf_state* st, const yr_opt* opt, float slope,
                                  const int64_t* uid, const int64_t* pos, const int64_t* neg, int64_t B,
                                  float* step_loss, yr_stream stream) {
  return yr_ngcf_train_step_ex(st, opt, slope, uid, pos, neg, B, step_loss, 0, stream);
}

// *rows_armed is true while row_flag / row_list / row_count hold the current batch (set after touched_rows_kernel,
// cleared once the re-arming kernels are enqueued): the wrapper below re-arms them on every early error return.
static int train_step_body(const yr_ngcf_state* st, const yr_opt* opt, float slope,
                           const int64_t* uid, const int64_t* pos, const int64_t* neg, int64_t B,
                           float* step_loss, int prefix_done, yr_stream stream, bool* rows_armed) {
  int rc = ngcf_state_ok(st);
  if (rc) return rc;
  if (prefix_done < 0 || prefix_done > st->n_layers) return YR_ERR_BAD_ARG;
  if (!opt || !uid || !pos || !neg || B <= 0 || yr_csr_ok(&st->LT) || !st->T ||
      !st->E_dev || !st->G_dev || !st->ws || !st->loss)
    return YR_ERR_BAD_ARG;
  if (opt->kind < YR_OPT_SGD || opt->kind > YR_OPT_ADAMW) return YR_ERR_BAD_OPT;
  const int L = st->n_layers, d = st->d;
  const int64_t n = st->nU + st->nI;
  cudaStream_t s = (cudaStream_t)stream;
  // The gradient buffers are first written by the tail, after the whole forward: clear them on a side stream
  // underneath the forward SpMMs (HBM writes next to an L2-bound kernel) and join before the tail.
  SideStream* side = side_stream();
  for (int l = 0; l <= L; ++l)
    if (!st->G[l]) return YR_ERR_BAD_ARG;
  cudaStream_t ms = side ? side->stream : s;
  if (side) {
    YR_CUDA(cudaEventRecord(side->fork, s));                 // everything enqueued so far (the previous optimizer step reads G[0])
    YR_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
  }
  for (int l = 0; l <= L; ++l) YR_CUDA(cudaMemsetAsync(st->G[l], 0, sizeof(float) * (size_t)n * d, ms));
  // Top layer: E_L is READ only at the <= 3B rows the batch touches (the tail) and dLoss/dE_L is non-zero only there.
  // So the last layer's forward (SpMM + transform) and backward run on those rows, and G_{L-1} += L^T T becomes a
  // scatter from them (same sums, different fp32 order). Needs the row scratch; E_L / LE_{L-1} keep stale values in
  // the other rows (yr_ngcf_propagate recomputes everything for validate / evaluate).
  const bool rows_path = st->row_flag && st->row_list && st->row_count && st->row_list_cap >= 3 * B && d == 64 &&
                         st->top_rows_mode != 0;
  if (rows_path) {                                            // list of the batch rows: also off the critical path
    touched_rows_kernel<<<(unsigned)((3 * B + 255) / 256), 256, 0, ms>>>(uid, pos, neg, B, st->nU, st->nI, st->row_flag,
                                                                        st->row_list, st->row_count);
    YR_CHECK_LAUNCH();
    *rows_armed = true;
  }
  if (side) YR_CUDA(cudaEventRecord(side->join, side->stream));
  if (rows_path && fwd_tc(st->dense_mode)) {
    for (int l = (prefix_done < L - 1 ? prefix_done : L - 1); l + 1 < L; ++l) {
      rc = yr_ngcf_layer_fwd(&st->L, d, st->E[l], st->W1[l], st->W2[l], slope, st->E[l + 1], st->LE[l], st->dense_mode,
                           stream);
      if (rc) return rc;
    }
    if (side) YR_CUDA(cudaStreamWaitEvent(s, side->join, 0));       // row list (and the cleared gradients) ready
    rc = yr_spmm_csr_rows(&st->L, d, st->E[L - 1], st->LE[L - 1], st->row_flag, s);
    if (rc) return rc;
    rc = yr_ngcf_dense_fwd_tc_launch_d(d, st->E[L - 1], st->LE[L - 1], st->W1[L - 1], st->W2[L - 1], slope, n, st->E[L], s,
                                       st->row_list, st->row_count, 3 * B);
    if (rc) return rc;
  } else {
    for (int l = prefix_done; l < L; ++l) {
      rc = yr_ngcf_layer_fwd(&st->L, d, st->E[l], st->W1[l], st->W2[l], slope, st->E[l + 1], st->LE[l], st->dense_mode,
                           stream);
      if (rc) return rc;
    }
  }
  if (side) YR_CUDA(cudaStreamWaitEvent(s, side->join, 0));
  rc = yr_ngcf_tail(st->E_dev, st->G_dev, L, st->nU, st->nI, d, uid, pos, neg, B, nullptr, nullptr, st->loss,
                    step_loss, st->err, stream);
  if (rc) return rc;
  bool reduce_pending = false;
  for (int l = L - 1; l >= 0; --l) {
    if (!st->dW1[l] || !st->dW2[l]) return YR_ERR_BAD_ARG;
    if (rows_path && l == L - 1) {
      rc = ngcf_layer_bwd_rows(st, l, slope, s, side);
      if (rc) return rc;
      reduce_pending = side != nullptr;
      // re-arm the row scratch for the next step: behind the scatter, next to the following layers
      cudaStream_t us = s;
      if (side) {
        YR_CUDA(cudaStreamWaitEvent(s, side->join, 0));          // the reduce has read ws; also lets `fork` be reused
        reduce_pending = false;
        YR_CUDA(cudaEventRecord(side->fork, s));                  // scatter (reads row_flag) enqueued before this point
        YR_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
        us = side->stream;
      }
      untouch_rows_kernel<<<(unsigned)((3 * B + 255) / 256), 256, 0, us>>>(st->row_flag, st->row_list, st->row_count);
      YR_CHECK_LAUNCH();
      YR_CUDA(cudaMemsetAsync(st->row_count, 0, sizeof(int32_t), us));
      *rows_armed = false;
      continue;
    }
    // dense backward, then the reduction of its dW partials on the side stream underneath the transposed SpMM
    if (side && reduce_pending) { YR_CUDA(cudaStreamWaitEvent(s, side->join, 0)); reduce_pending = false; }   // ws is free again
    int parts = 0;
    rc = dense_bwd_launch(d, n, st->E[l], st->LE[l], st->E[l + 1], st->G[l + 1], st->W1[l], st->W2[l], slope, st->G[l],
                          st->T, st->ws, st->ws_bytes, st->dense_mode, s, &parts);
    if (rc) return rc;
    if (side) {
      YR_CUDA(cudaEventRecord(side->fork, s));
      YR_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
      rc = dense_bwd_reduce(d, st->ws, parts, st->dW1[l], st->dW2[l], side->stream);
      if (rc) return rc;
      YR_CUDA(cudaEventRecord(side->join, side->stream));
      reduce_pending = true;
    } else {
      rc = dense_bwd_reduce(d, st->ws, parts, st->dW1[l], st->dW2[l], s);
      if (rc) return rc;
    }
    rc = yr_spmm_csr(&st->LT, d, st->T, st->G[l], 1, stream);
    if (rc) return rc;
  }
  if (side && reduce_pending) YR_CUDA(cudaStreamWaitEvent(s, side->join, 0));
  // embedding.weight and the 2L weights: parameter order of nn.Module.parameters() does not matter for a per-tensor
  // optimizer; two launches (1 + 2L <= 15 tensors, 8 per launch)
  float *pp[2 * YR_NGCF_MAX_LAYERS + 1], *gg[2 * YR_NGCF_MAX_LAYERS + 1], *mm[2 * YR_NGCF_MAX_LAYERS + 1],
      *vv[2 * YR_NGCF_MAX_LAYERS + 1];
  int64_t nn[2 * YR_NGCF_MAX_LAYERS + 1];
  int cnt = 0;
  pp[cnt] = st->E[0]; gg[cnt] = st->G[0]; mm[cnt] = st->mE; vv[cnt] = st->vE; nn[cnt++] = n * d;
  for (int l = 0; l < L; ++l) {
    pp[cnt] = st->W1[l]; gg[cnt] = st->dW1[l]; mm[cnt] = st->mW1[l]; vv[cnt] = st->vW1[l]; nn[cnt++] = (int64_t)d * d;
    pp[cnt] = st->W2[l]; gg[cnt] = st->dW2[l]; mm[cnt] = st->mW2[l]; vv[cnt] = st->vW2[l]; nn[cnt++] = (int64_t)d * d;
  }
  for (int c0 = 0; c0 < cnt; c0 += YR_OPT_MAX_TENSORS) {
    const int c = (cnt - c0 < YR_OPT_MAX_TENSORS) ? cnt - c0 : YR_OPT_MAX_TENSORS;
    rc = yr_dense_opt_step_multi(c, pp + c0, gg + c0, mm + c0, vv + c0, nn + c0, opt, 0, stream);
    if (rc) return rc;
  }
  return YR_OK;
}

extern "C" int yr_ngcf_train_step_ex(const yr_ngcf_state* st, const yr_opt* opt, float slope,
                                     const int64_t* uid, const int64_t* pos, const int64_t* neg, int64_t B,
                                     float* step_loss, int prefix_done, yr_stream stream) {
  bool rows_armed = false;
  const int rc = train_step_body(st, opt, slope, uid, pos, neg, B, step_loss, prefix_done, stream, &rows_armed);
  if (rc == YR_OK) return rc;
  // Error exit in the middle of a step: join the helper stream and re-arm the row scratch, so that a later step does
  // not find rows still flagged (atomicExch would return 1 and those rows would silently drop out of row_list).
  cudaStream_t s = (cudaStream_t)stream;
  if (SideStream* side = side_stream()) {
    if (cudaEventRecord(side->join, side->stream) == cudaSuccess) cudaStreamWaitEvent(s, side->join, 0);
  }
  if (rows_armed && st && st->row_flag && st->row_list && st->row_count) {
    untouch_rows_kernel<<<(unsigned)((3 * B + 255) / 256), 256, 0, s>>>(st->row_flag, st->row_list, st->row_count);
    cudaMemsetAsync(st->row_count, 0, sizeof(int32_t), s);
  }
  return rc;
}

extern "C" int yr_ngcf_concat(const float* const* E_layers, int n_layers, int64_t n, int d, float* out,
                              yr_stream stream) {
  if (!E_layers || !out || n <= 0 || d <= 0 || (d & 3) || n_layers < 0 || n_layers > YR_NGCF_MAX_LAYERS)
    return YR_ERR_BAD_ARG;
  const int64_t total4 = n * ((n_layers + 1) * d / 4);
  int64_t blocks = (total4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  yr::concat_layers_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(E_layers, n_layers, n, d, out);
  YR_CHECK_LAUNCH();
  return YR_OK;
}
