// CUDA-core kernels of the LCN hot path: weight preparation (clip_by_norm + mask + pack), the edge
// layers (17*in_F -> 17*F and 17*F -> 51), BatchNorm statistics / apply, the elementwise half of the backward
// pass, the fused masked TF1-Adam step, and the orchestration of the forward / backward passes of both arithmetic
// paths.  The tensor-core (tcgen05) mid-layer GEMMs of both paths live in lcn_gemm_tc.cu, the data-parallel exchange
// and the gradient pack / unpack in lcn_dp.cu.
//
// Reference semantics implemented here (paths relative to the reference root):
//   network/models_att.py:534-586 (mask, mask_weights), :588-612 (BN), :630-775 (layers, head),
//   :352-421 (loss, Adam); SURVEY.md section 9 lists the TF behaviours relied on.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <type_traits>

#include "lcn_internal.cuh"

// Activation types of the two arithmetic paths (include/lcn_b200.h): __nv_bfloat16 = LCN_PATH_BF16 (every GEMM on the
// tensor cores, fused BatchNorm statistics, tensor-core edge layers), lcn_sp16 = LCN_PATH_FP32 (split-bf16 storage,
// three tensor-core products per block: fp32 parity; the K = 17*in_F first layer and the N = 51 head stay on CUDA cores,
// < 1.3 % of the FLOPs).  There is no CUDA-core GEMM for the mid layers any more.
template <typename T>
struct PathTraits {
  static constexpr bool bf16 = std::is_same<T, __nv_bfloat16>::value;
  static constexpr bool x3 = std::is_same<T, lcn_sp16>::value;
};

struct ConstMask {
  float v[LCN_J * LCN_J];
};

__device__ __forceinline__ double block_reduce_sum_d(double v, double* sh /* >= 32 */) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[w] = v;
  __syncthreads();
  v = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.0;
  if (w == 0)
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;  // valid in thread 0
}

// ------------------------------------------------------------------------------------------------
// weight preparation
// ------------------------------------------------------------------------------------------------
__global__ void k_zero_norm2(LayerScalars* sc, int n) {
  lcn_pdl_prologue();
  if (threadIdx.x < n) sc[threadIdx.x].norm2 = 0.0;
}

// ||W_l||_F^2 of the full, unmasked matrix (tf.clip_by_norm, models_att.py:659)
__global__ void k_sumsq(const float* __restrict__ params, LinTable lt, LayerScalars* sc) {
  lcn_pdl_prologue();
  __shared__ double sh[32];
  int l = blockIdx.y;
  int64_t n4 = (int64_t)lt.Fi[l] * lt.Fo[l] * LCN_J * LCN_J / 4;
  const float4* w = reinterpret_cast<const float4*>(params + lt.w_off[l]);
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 v = w[i];
    s += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
  }
  s = block_reduce_sum_d(s, sh);
  if (threadIdx.x == 0) atomicAdd(&sc[l].norm2, s);
}

// mask = softmax(var, axis=0) * support (models_att.py:569-571) or the constant; per-layer clip scale.
// The weight-pack kernels evaluate these two helpers themselves (one thread per block), so that storing the mask values
// and scalars is not a launch of its own in front of them on the tail of every train step: block (0, 0, 0) of
// k_pack_edges stores them (lcn_write_mask_scalars) for the kernels that follow the weight preparation.
__device__ __forceinline__ float lcn_mask_value(const float* __restrict__ params, int64_t mask_off, const ConstMask& cmask,
                                                const SupportBits& sup, int i, int j) {
  if (!((sup.row[i] >> j) & 1u)) return 0.f;
  if (mask_off < 0) return cmask.v[i * LCN_J + j];
  const float* var = params + mask_off;
  float mx = -INFINITY;
  for (int k = 0; k < LCN_J; ++k) mx = fmaxf(mx, var[k * LCN_J + j]);
  float den = 0.f;
  for (int k = 0; k < LCN_J; ++k) den += expf(var[k * LCN_J + j] - mx);
  return expf(var[i * LCN_J + j] - mx) / den;
}
__device__ __forceinline__ float lcn_inv_norm(const LayerScalars* sc, int l, int max_norm, bool* clipped) {
  const double nrm = sqrt(sc[l].norm2);
  const bool clip = max_norm && nrm > 1.0;
  if (clipped) *clipped = clip;
  return clip ? (float)(1.0 / nrm) : 1.0f;
}
__device__ __forceinline__ void lcn_write_mask_scalars(const float* __restrict__ params, int64_t mask_off,
                                                       const ConstMask& cmask, const SupportBits& sup, int n_lin,
                                                       int max_norm, LayerScalars* sc, float* mask_out, int t) {
  if (t < LCN_J * LCN_J) mask_out[t] = lcn_mask_value(params, mask_off, cmask, sup, t / LCN_J, t % LCN_J);
  if (t < n_lin) {
    bool clip;
    const float inv = lcn_inv_norm(sc, t, max_norm, &clip);
    sc[t].inv_norm = inv;
    sc[t].clipped = clip ? 1.f : 0.f;
  }
}
// packed 64x64 sub-blocks of the mid layers.  grid (nnz*FC*FC, n_mid), 256 threads.  Every block derives its own
// scale from ||W||^2 and the mask variable (see lcn_mask_value).
//   wp32 : [mid][pair][hi][ho][fi][fo] fp32, when given (the mid-layer weight tap of the fp32-parity path)
//   wp16f: bf16, UMMA K-major SWIZZLE_128B image of B[n=fo][k=fi], input-chunk-major order
//   wp16b: bf16, same for the transposed operand B[n=fi][k=fo], output-chunk-major order
__global__ void __launch_bounds__(256) k_pack_mid(const float* __restrict__ params, LinTable lt, PairTable pt,
                                                  SupportBits sup, const LayerScalars* sc, int F, int FC, int nnz,
                                                  float* __restrict__ wp32, __nv_bfloat16* __restrict__ wp16f,
                                                  __nv_bfloat16* __restrict__ wp16b, __nv_bfloat16* __restrict__ wp16f_lo,
                                                  __nv_bfloat16* __restrict__ wp16b_lo, int64_t mask_off, ConstMask cmask,
                                                  int max_norm) {
  lcn_pdl_prologue();
  __shared__ float tile[64][65];     // tile[fi][fo], scaled
  __shared__ float s_scale;
  int mid = blockIdx.y, l = mid + 1;
  int sb = blockIdx.x;
  int p = sb / (FC * FC), hi = (sb / FC) % FC, ho = sb % FC;
  int i = pt.pi[p], j = pt.pj[p];
  int P = LCN_J * F;
  if (threadIdx.x == 0)
    s_scale = lcn_inv_norm(sc, l, max_norm, nullptr) * lcn_mask_value(params, mask_off, cmask, sup, i, j);
  __syncthreads();
  const float scale = s_scale;
  const float* w = params + lt.w_off[l] + (size_t)(i * F + hi * 64) * P + j * F + ho * 64;
  size_t mid_sb = (size_t)nnz * FC * FC;
  float* d32 = wp32 ? wp32 + ((size_t)mid * mid_sb + sb) * 4096 : nullptr;
  for (int f4 = threadIdx.x; f4 < 1024; f4 += 256) {     // coalesced 16-byte loads of the 64x64 block
    int fi = f4 >> 4, c4 = (f4 & 15) * 4;
    float4 v = *reinterpret_cast<const float4*>(w + (size_t)fi * P + c4);
    v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
    tile[fi][c4] = v.x; tile[fi][c4 + 1] = v.y; tile[fi][c4 + 2] = v.z; tile[fi][c4 + 3] = v.w;
    if (d32 != nullptr) *reinterpret_cast<float4*>(d32 + fi * 64 + c4) = v;
  }
  __syncthreads();
  // destination sub-block slots
  int base_i = 0, base_j = 0;
  for (int q = 0; q < i; ++q) base_i += __popc(sup.row[q]);
  for (int q = 0; q < j; ++q) base_j += __popc(sup.col[q]);
  int rank_out = __popc(sup.row[i] & ((1u << j) - 1u));   // rank of j among outputs of i
  int rank_in = __popc(sup.col[j] & ((1u << i) - 1u));    // rank of i among inputs of j
  int cnt_out = __popc(sup.row[i]), cnt_in = __popc(sup.col[j]);
  size_t slot_f = (size_t)FC * FC * base_i + (size_t)hi * (cnt_out * FC) + rank_out * FC + ho;
  size_t slot_b = (size_t)FC * FC * base_j + (size_t)ho * (cnt_in * FC) + rank_in * FC + hi;
  uint4* df = reinterpret_cast<uint4*>(wp16f + ((size_t)mid * mid_sb + slot_f) * 4096);
  uint4* db = reinterpret_cast<uint4*>(wp16b + ((size_t)mid * mid_sb + slot_b) * 4096);
  // split-bf16 path: the lo parts w - bf16(w) of the same blocks, same layout, separate arrays
  uint4* dfl = wp16f_lo ? reinterpret_cast<uint4*>(wp16f_lo + ((size_t)mid * mid_sb + slot_f) * 4096) : nullptr;
  uint4* dbl = wp16b_lo ? reinterpret_cast<uint4*>(wp16b_lo + ((size_t)mid * mid_sb + slot_b) * 4096) : nullptr;
  for (int e = threadIdx.x; e < 512; e += 256) {          // one 16-byte chunk (8 bf16) per store
    int n = e >> 3, kc = e & 7;
    __nv_bfloat162 hf[4], hb[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      hf[q] = __floats2bfloat162_rn(tile[kc * 8 + 2 * q][n], tile[kc * 8 + 2 * q + 1][n]);   // row n=fo, k=fi
      hb[q] = __floats2bfloat162_rn(tile[n][kc * 8 + 2 * q], tile[n][kc * 8 + 2 * q + 1]);   // row n=fi, k=fo
    }
    df[n * 8 + (kc ^ (n & 7))] = *reinterpret_cast<uint4*>(hf);
    db[n * 8 + (kc ^ (n & 7))] = *reinterpret_cast<uint4*>(hb);
    if (dfl != nullptr) {
      __nv_bfloat162 lf[4], lb[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 f = __bfloat1622float2(hf[q]), b = __bfloat1622float2(hb[q]);
        lf[q] = __floats2bfloat162_rn(tile[kc * 8 + 2 * q][n] - f.x, tile[kc * 8 + 2 * q + 1][n] - f.y);
        lb[q] = __floats2bfloat162_rn(tile[n][kc * 8 + 2 * q] - b.x, tile[n][kc * 8 + 2 * q + 1] - b.y);
      }
      dfl[n * 8 + (kc ^ (n & 7))] = *reinterpret_cast<uint4*>(lf);
      dbl[n * 8 + (kc ^ (n & 7))] = *reinterpret_cast<uint4*>(lb);
    }
  }
}

// Both edge layers in one launch (17*in_F <= 64): the dense masked weights Wm = W * inv_norm * mask[i,j] in fp32
// (CUDA-core first layer / head of the fp32-parity path, parity taps) and, when the bf16 pointers are given, their
// tensor-core tiles: wf16 one 64x64 block per output chunk of the first layer, B[n = output column][k = input feature,
// zero padded to 64]; wl16f / wl16b one block per channel chunk of the last layer, B[n = output column (51 padded to 64)]
// [k = channel] for the forward pass and B[n = channel][k = output column] for dgrad.  grid (17*FC, 4, 2): z = 0 first
// layer (x = output chunk), z = 1 last layer (x = channel chunk); y = 16 of the 64 rows of the tile.  Scales from ||W||^2
// and the mask variable directly (see lcn_mask_value); block (0, 0, 0) also stores the 289 mask values and the
// per-layer scalars.
__global__ void __launch_bounds__(256) k_pack_edges(const float* __restrict__ params, int64_t w_first, int64_t w_last,
                                                    int in_F, int F, int P, int n_lin, LayerScalars* sc,
                                                    int64_t mask_off, ConstMask cmask, SupportBits sup, int max_norm,
                                                    float* __restrict__ mask_out,
                                                    float* __restrict__ wm_first, float* __restrict__ wm_last,
                                                    __nv_bfloat16* __restrict__ wf16, __nv_bfloat16* __restrict__ wl16f,
                                                    __nv_bfloat16* __restrict__ wl16b) {
  lcn_pdl_prologue();
  __shared__ float s_m[LCN_J];       // mask column / row of this tile, times inv_norm
  const int x = blockIdx.x, last = n_lin - 1;
  if (blockIdx.z == 0) {
    // first layer: rows k = input feature (joint i = k / in_F), columns of output chunk x (joint j = x*64 / F)
    const int Kin = LCN_J * in_F, j = (x * 64) / F;
    if ((int)threadIdx.x < LCN_J)
      s_m[threadIdx.x] = lcn_inv_norm(sc, 0, max_norm, nullptr) * lcn_mask_value(params, mask_off, cmask, sup, threadIdx.x, j);
    __syncthreads();
    const float* w = params + w_first;
    for (int e = blockIdx.y * 1024 + threadIdx.x; e < (int)(blockIdx.y + 1) * 1024; e += blockDim.x) {
      const int k = e >> 6, n = e & 63;
      float v = 0.f;
      if (k < Kin) {
        const size_t o = (size_t)k * P + x * 64 + n;
        v = w[o] * s_m[k / in_F];
        wm_first[o] = v;
      }
      if (wf16 != nullptr) wf16[(size_t)x * 4096 + n * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7))] = __float2bfloat16_rn(v);
    }
  } else {
    // last layer: rows = channels of chunk x (joint i = x*64 / F), columns n = 3*j + c < 51
    const int i = (x * 64) / F;
    if ((int)threadIdx.x < LCN_J)
      s_m[threadIdx.x] = lcn_inv_norm(sc, last, max_norm, nullptr) * lcn_mask_value(params, mask_off, cmask, sup, i, threadIdx.x);
    __syncthreads();
    const float* w = params + w_last;
    for (int e = blockIdx.y * 1024 + threadIdx.x; e < (int)(blockIdx.y + 1) * 1024; e += blockDim.x) {
      const int k = e >> 6, n = e & 63;
      float v = 0.f;
      if (n < 51) {
        const size_t o = (size_t)(x * 64 + k) * 51 + n;
        v = w[o] * s_m[n / 3];
        wm_last[o] = v;
      }
      if (wl16f != nullptr) {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        wl16f[(size_t)x * 4096 + n * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7))] = h;
        wl16b[(size_t)x * 4096 + k * 64 + ((((n >> 3) ^ (k & 7)) << 3) | (n & 7))] = h;
      }
    }
  }
  // after the tiles and not unrolled: the kernel stays at 32 registers
  if (x == 0 && blockIdx.y == 0 && blockIdx.z == 0)
#pragma unroll 1
    for (int t = threadIdx.x; t < LCN_J * LCN_J; t += blockDim.x)
      lcn_write_mask_scalars(params, mask_off, cmask, sup, n_lin, max_norm, sc, mask_out, t);
}

// side stream + events of the model (LcnAux), created on first use under aux.mu (held by the caller).  A creation that
// fails releases what was created and returns LCN_ECUDA; the next call tries again.
void lcn_aux_release(LcnAux& a) {
  for (cudaStream_t* s : {&a.st, &a.xst}) {
    if (*s != nullptr) cudaStreamDestroy(*s);
    *s = nullptr;
  }
  for (cudaEvent_t* e : {&a.ev_go, &a.ev_done, &a.ev_dz[0], &a.ev_dz[1], &a.ev_wg[0], &a.ev_wg[1], &a.ev_ms, &a.ev_loss,
                         &a.ev_xdone}) {
    if (*e != nullptr) cudaEventDestroy(*e);
    *e = nullptr;
  }
  a.ready = false;
}

static int lcn_aux_get(const lcn_model* m, LcnAux** out) {
  LcnAux& a = m->aux;
  if (!a.ready) {
    const char* call = "cudaStreamCreateWithFlags";
    cudaError_t e = cudaSuccess;
    for (cudaStream_t* s : {&a.st, &a.xst})
      if (e == cudaSuccess) e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
      call = "cudaEventCreateWithFlags";
      for (cudaEvent_t* ev : {&a.ev_go, &a.ev_done, &a.ev_dz[0], &a.ev_dz[1], &a.ev_wg[0], &a.ev_wg[1], &a.ev_ms,
                              &a.ev_loss, &a.ev_xdone})
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      lcn_aux_release(a);
      lcn_set_error("side streams of the model: %s -> %s", call, cudaGetErrorString(e));
      return LCN_ECUDA;
    }
    a.ready = true;
  }
  *out = &a;
  return LCN_OK;
}

int lcn_launch_prepare(const lcn_model* m, const float* params, char* ws, const WsLayout& lay,
                       bool recompute_norm, cudaStream_t st) {
  LayerScalars* sc = reinterpret_cast<LayerScalars*>(ws + lay.off_scalars);
  float* mask = reinterpret_cast<float*>(ws + lay.off_mask);
  LinTable lt = make_lin(m);
  if (recompute_norm) {
    lcn_launch(k_zero_norm2, dim3(1), dim3(32), 0, st, sc, m->n_lin);
    lcn_launch(k_sumsq, dim3(dim3(64, m->n_lin)), dim3(256), 0, st, params, lt, sc);
    LCN_CHECK_LAUNCH();
  }
  ConstMask cmask;
  memcpy(cmask.v, m->d.const_mask, sizeof(cmask.v));
  int last = m->n_lin - 1;
  int n_mid = m->n_lin - 2;
  const bool x3 = m->d.path == LCN_PATH_FP32;
  const bool bf = m->d.path == LCN_PATH_BF16;
  // The weight preparation is k_pack_edges on the model's side stream (it also stores the mask values and the per-layer
  // scalars for the kernels that follow) beside k_pack_mid on the caller's stream, for models with mid layers.
  std::lock_guard<std::mutex> aux_lock(m->aux.mu);
  LcnAux* ax;
  int rc = lcn_aux_get(m, &ax);
  if (rc) return rc;
  LCN_CHECK_CUDA(cudaEventRecord(ax->ev_go, st));
  LCN_CHECK_CUDA(cudaStreamWaitEvent(ax->st, ax->ev_go, 0));
  lcn_launch(k_pack_edges, dim3(LCN_J * m->FC, 4, 2), dim3(256), 0, ax->st, params, m->L[0].w_off, m->L[last].w_off, m->d.in_F,
             m->d.F, m->P, m->n_lin, sc, m->mask_off, cmask, m->sup, m->d.max_norm, mask,
             reinterpret_cast<float*>(ws + lay.off_wm_first), reinterpret_cast<float*>(ws + lay.off_wm_last),
             bf ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wf16) : nullptr,
             bf ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wl16f) : nullptr,
             bf ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wl16b) : nullptr);
  LCN_CHECK_CUDA(cudaEventRecord(ax->ev_done, ax->st));
  if (n_mid > 0)
    lcn_launch(k_pack_mid, dim3(dim3(m->nnz * m->FC * m->FC, n_mid)), dim3(256), 0, st,
        params, lt, make_pairs(m), m->sup, sc, m->d.F, m->FC, m->nnz,
        x3 ? reinterpret_cast<float*>(ws + lay.off_wp32) : nullptr /* the parity tap (lcn_model_read_tensor kind 2) */,
        reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wp16f), reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wp16b),
        x3 ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wp16f_lo) : nullptr,
        x3 ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_wp16b_lo) : nullptr,
        m->mask_off, cmask, m->d.max_norm);
  LCN_CHECK_LAUNCH();
  LCN_CHECK_CUDA(cudaStreamWaitEvent(st, ax->ev_done, 0));
  return LCN_OK;
}

// ------------------------------------------------------------------------------------------------
// row geometry helpers
// ------------------------------------------------------------------------------------------------
struct RowGeom {
  int64_t n_rows;   // real poses
  int bn_group;     // rows per BN group (logical)
  int gstride;      // physical rows per group (multiple of 128)
};
// physical row -> (valid for BN statistics, source row or -1 when zero padded)
__device__ __forceinline__ bool row_valid(const RowGeom& g, int64_t pr, int64_t* src) {
  int64_t grp = pr / g.gstride;
  int rin = (int)(pr - grp * g.gstride);
  int64_t s = grp * g.bn_group + rin;
  *src = (rin < g.bn_group && s < g.n_rows) ? s : -1;
  return rin < g.bn_group;
}

// ------------------------------------------------------------------------------------------------
// first layer: Z0 = X * Wm1 + b1  (models_att.py:729), K = 17*in_F, plus BN partials.  CUDA cores on purpose: K is
// too small for an MMA tile and the fp32 input stays exact.
// grid (tiles, P/64), 256 threads: a CTA owns a 128-row x 64-column tile, a thread 4 rows x 8 columns (the K loop
// reads 3 x 16 B of shared memory per 32 FMAs; rows leave as 16-byte vectors of the tiled layout).  BN partials
// (mean, M2 per column over the tile's valid rows) use sums shifted by the bias, reduced by shuffles across the 4
// row groups of a warp and through shared memory across the 8 warps.
// ------------------------------------------------------------------------------------------------
template <typename T, int IN_F>
__global__ void __launch_bounds__(256) k_first_layer(const float* __restrict__ x, RowGeom g,
                                                     const float* __restrict__ wm, const float* __restrict__ bias,
                                                     T* __restrict__ Z, float* __restrict__ part, int P,
                                                     __nv_bfloat16* __restrict__ x16, double* __restrict__ gacc, int F,
                                                     SupportBits sup) {
  lcn_pdl_prologue();
  constexpr int KIN = LCN_J * IN_F;
  __shared__ __align__(16) float xs[KIN][LCN_TILE];
  __shared__ __align__(16) float wsm[KIN][64];
  __shared__ __align__(16) float red[8][64][2];
  __shared__ unsigned char valid_s[LCN_TILE];
  const int tile = blockIdx.x, col0 = blockIdx.y * 64;
  {
    // thread = (row, k parity): conflict-free shared-memory stores; the strided global reads of a row hit L1
    const int r = threadIdx.x & (LCN_TILE - 1);
    int64_t src;
    const bool v = row_valid(g, (int64_t)tile * LCN_TILE + r, &src);
    if (threadIdx.x < LCN_TILE) valid_s[r] = v;
    for (int k = threadIdx.x >> 7; k < KIN; k += 2) xs[k][r] = (src >= 0) ? x[src * KIN + k] : 0.f;
  }
  for (int e = threadIdx.x; e < KIN * 16; e += 256) {
    int k = e >> 4, c4 = (e & 15) * 4;
    *reinterpret_cast<float4*>(&wsm[k][c4]) = *reinterpret_cast<const float4*>(wm + (size_t)k * P + col0 + c4);
  }
  __syncthreads();
  if (x16 != nullptr && blockIdx.y == 0) {   // bf16 tile of the (zero padded) input: operand of the tensor-core wgrad
    for (int e = threadIdx.x; e < LCN_TILE * 64; e += 256) {
      int r = e >> 6, cc = e & 63;
      x16[lcn_off<__nv_bfloat16>((int64_t)tile * LCN_TILE + r, cc, 64)] = __float2bfloat16_rn(cc < KIN ? xs[cc][r] : 0.f);
    }
  }
  const int cg = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c0 = cg * 8, r0 = rg * 4;
  float b[8];
  {
    const float4 b0 = *reinterpret_cast<const float4*>(bias + col0 + c0), b1 = *reinterpret_cast<const float4*>(bias + col0 + c0 + 4);
    b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w; b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
  }
  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[i][q] = b[q];
  // only the input joints with a block into this output joint contribute (the masked weights of the others are zero):
  // 20 of 34 rows of the reduction on average for knn=3
  const uint32_t in_bits = sup.col[(col0 / 64) / (F / 64)];
#pragma unroll 2
  for (int k = 0; k < KIN; ++k) {
    if (!((in_bits >> (k / IN_F)) & 1u)) continue;
    const float4 xv = *reinterpret_cast<const float4*>(&xs[k][r0]);
    const float4 w0 = *reinterpret_cast<const float4*>(&wsm[k][c0]), w1 = *reinterpret_cast<const float4*>(&wsm[k][c0 + 4]);
    const float xr[4] = {xv.x, xv.y, xv.z, xv.w};
    const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[i][q] = fmaf(xr[i], wv[q], acc[i][q]);
  }
  float s1[8], s2[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) s1[q] = s2[q] = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool v = valid_s[r0 + i];
    float y[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      y[q] = v ? acc[i][q] : 0.f;
      const float d = v ? acc[i][q] - b[q] : 0.f;
      s1[q] += d;
      s2[q] = fmaf(d, d, s2[q]);
    }
    lcn_st8(Z, lcn_off<T>((int64_t)tile * LCN_TILE + r0 + i, col0 + c0, P), y);
  }
  // reduce over the 32 row groups: lanes {cg, cg+8, cg+16, cg+24} of a warp, then the 8 warps
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    s1[q] += __shfl_xor_sync(0xffffffffu, s1[q], 8);
    s2[q] += __shfl_xor_sync(0xffffffffu, s2[q], 8);
    s1[q] += __shfl_xor_sync(0xffffffffu, s1[q], 16);
    s2[q] += __shfl_xor_sync(0xffffffffu, s2[q], 16);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane < 8) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      red[warp][c0 + q][0] = s1[q];
      red[warp][c0 + q][1] = s2[q];
    }
  }
  __syncthreads();
  if (threadIdx.x < 64) {
    const int tig = tile % (int)(g.gstride / LCN_TILE);
    const int n = min(LCN_TILE, (int)g.bn_group - tig * LCN_TILE);   // valid rows of this tile (row_valid: rin < bn_group)
    float t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      t1 += red[w][threadIdx.x][0];
      t2 += red[w][threadIdx.x][1];
    }
    const float nf = (float)max(n, 1);
    const int c = col0 + threadIdx.x;
    if (gacc != nullptr) {
      // per-channel fp64 accumulators instead of partials + k_bn_finalize (TcFuse, lcn_internal.cuh): the sums are
      // shifted by the bias, sum x = n b + t1, sum x^2 = t2 + 2 b t1 + n b^2
      const double nd = (double)n, bd = (double)bias[c], d1 = (double)t1;
      double* dst = gacc + ((size_t)(tile & (LCN_GACC_REP - 1)) * F + c % F) * 2;
      atomicAdd(dst, nd * bd + d1);
      atomicAdd(dst + 1, (double)t2 + 2.0 * bd * d1 + nd * bd * bd);
    } else {
      *reinterpret_cast<float2*>(part + ((size_t)tile * P + c) * 2) =
          make_float2(bias[c] + t1 / nf, fmaxf(t2 - t1 * t1 / nf, 0.f));
    }
  }
}

// shared-memory pitches of k_last_layer (activation rows / weight rows)
#define GS_APAD 65
#define GS_BPAD 68

// ------------------------------------------------------------------------------------------------
// BatchNorm statistics: merge per-tile (mean, M2) partials over the tiles of a group and the 17
// joints (Keras BN axis=-1 on [B,17,F]: per channel over batch x joints, biased variance).
// grid (n_groups, F/2), 256 threads = 2 channels x 128 slices.  Two-pass merge in fp64:
//   mean = sum n_b mean_b / N ;  M2 = sum [ M2_b + n_b (mean_b - mean)^2 ]   (exact, no per-item division)
// mom != nullptr (synchronised BatchNorm, one group): the fp64 moments (N, mean, M2) go to mom[F][3] for k_bn_sync
// instead of (mean, rstd) to stat.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bn_finalize(const float* __restrict__ part, float* __restrict__ stat, int P,
                                                     int F, int tiles_per_group, int bn_group, double* __restrict__ mom) {
  lcn_pdl_prologue();
  __shared__ double sa[256];
  __shared__ double smean[2];
  int g = blockIdx.x, tid = threadIdx.x;
  int c = tid & 1, slice = tid >> 1;
  int f = blockIdx.y * 2 + c;
  int items = tiles_per_group * LCN_J;
  double ntot = (double)bn_group * LCN_J;
  double acc = 0;
  for (int it = slice; it < items; it += 128) {
    int t = it / LCN_J, j = it - t * LCN_J;
    double nb = (double)min(LCN_TILE, bn_group - t * LCN_TILE);
    acc += nb * (double)part[((size_t)(g * tiles_per_group + t) * P + j * F + f) * 2];
  }
  sa[tid] = acc;
  for (int off = 64; off > 0; off >>= 1) {
    __syncthreads();
    if (slice < off) sa[tid] += sa[tid + off * 2];
  }
  __syncthreads();
  if (slice == 0) smean[c] = sa[tid] / ntot;
  __syncthreads();
  double mean = smean[c];
  acc = 0;
  for (int it = slice; it < items; it += 128) {
    int t = it / LCN_J, j = it - t * LCN_J;
    double nb = (double)min(LCN_TILE, bn_group - t * LCN_TILE);
    size_t o = ((size_t)(g * tiles_per_group + t) * P + j * F + f) * 2;
    double d = (double)part[o] - mean;
    acc += (double)part[o + 1] + nb * d * d;
  }
  __syncthreads();
  sa[tid] = acc;
  for (int off = 64; off > 0; off >>= 1) {
    __syncthreads();
    if (slice < off) sa[tid] += sa[tid + off * 2];
  }
  if (slice == 0 && mom != nullptr) {
    mom[f * 3] = ntot;
    mom[f * 3 + 1] = mean;
    mom[f * 3 + 2] = sa[tid];
  } else if (slice == 0) {
    double var = sa[tid] / ntot;
    stat[((size_t)g * F + f) * 2 + 0] = (float)mean;
    stat[((size_t)g * F + f) * 2 + 1] = (float)(1.0 / sqrt(var + (double)LCN_BN_EPS));
  }
}

// ------------------------------------------------------------------------------------------------
// BN apply + LeakyReLU(0.2) + dropout + residual (models_att.py:664-673,704).  HBM/L2-bound elementwise pass.
// Persistent: grid = 2 x SMs blocks of (P/8, Y) threads, each block owns a contiguous range of rows; a thread
// owns 8 consecutive columns (16 B of bf16) and walks the rows with a register double buffer (the loads of
// row r+Y are in flight while row r is processed).  Per-channel scale/shift live in shared memory and are
// reloaded when the row range crosses into the next BatchNorm group.  In training, per (row, 8 columns) the keep
// decisions (low byte: backward does not redraw Philox) and the signs ybn > 0 of the LeakyReLU (high byte: backward
// takes the branch the forward took without forming ybn again) are written as one uint16.
// ------------------------------------------------------------------------------------------------
#define EW_MAXT 288   // (P/8) x Y threads: (136,2) for F=64, (272,1) for F=128
template <typename T>
__global__ void __launch_bounds__(EW_MAXT, 2) k_bn_act(const T* __restrict__ Z, const float* __restrict__ stat,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       const T* __restrict__ res, T* __restrict__ Aout,
                                                       uint16_t* __restrict__ keepbits, int P, int F, int rows_pad,
                                                       int bn_group, int gstride, float rate, uint64_t seed,
                                                       uint64_t step, int layer, const lcn_step_scalars* __restrict__ dyn) {
  lcn_pdl_prologue();
  __shared__ __align__(16) float s_sc[256], s_sh[256];
  if (dyn != nullptr) step = dyn->step;        // CUDA-graph replay: the step counter lives in device memory
  const int Y = blockDim.y, c8 = threadIdx.x * 8, f0 = c8 % F;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  // contiguous row range of this block (multiple of Y rows)
  int per = ((rows_pad / Y + gridDim.x - 1) / gridDim.x) * Y;
  int r_begin = blockIdx.x * per, r_end = min(r_begin + per, rows_pad);
  if (r_begin >= r_end) return;
  float inv_keep = rate > 0.f ? 1.f / (1.f - rate) : 1.f;
  const uint32_t thr16 = lcn_keep_thr16(rate);
  float sc[8], sh[8];
  int cur_g = -1;
  float zc[8], rc[8], zn[8], rn[8];
  int r = r_begin + threadIdx.y;
  bool vc = false, vn = false;
  size_t oc = 0, on = 0;
  if (r < r_end) {
    oc = lcn_off<T>(r, c8, P);
    vc = (r % gstride) < bn_group;
    if (vc) {
      lcn_ld8(Z, oc, zc);
      if (res != nullptr) lcn_ld8(res, oc, rc);
    }
  }
  // r_end - r_begin is a multiple of Y, so every thread of the block runs the same number of iterations
  for (; r < r_end; r += Y) {
    int g = (r - (int)threadIdx.y) / gstride;     // block-uniform (Y divides gstride)
    if (g != cur_g) {
      __syncthreads();
      if (tid < F) {
        float mean = stat[((size_t)g * F + tid) * 2], rstd = stat[((size_t)g * F + tid) * 2 + 1];
        float a = gamma[tid] * rstd;
        s_sc[tid] = a;
        s_sh[tid] = beta[tid] - mean * a;
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        sc[q] = s_sc[f0 + q];
        sh[q] = s_sh[f0 + q];
      }
      cur_g = g;
    }
    int rn_row = r + Y;
    vn = false;
    if (rn_row < r_end) {                          // prefetch the next row of this thread
      on = lcn_off<T>(rn_row, c8, P);
      vn = (rn_row % gstride) < bn_group;
      if (vn) {
        lcn_ld8(Z, on, zn);
        if (res != nullptr) lcn_ld8(res, on, rn);
      }
    }
    if (r < r_end) {
      float y[8];
      uint32_t kb = 0xffu;
      if (!vc) {
#pragma unroll
        for (int q = 0; q < 8; ++q) y[q] = 0.f;
      } else {
        if (rate > 0.f) {
          kb = lcn_keep8(seed, step, (uint32_t)layer, ((uint64_t)r * P + c8) >> 3, thr16);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float v = fmaf(zc[q], sc[q], sh[q]);
          if (v > 0.f) kb |= 0x100u << q;
          v = v > 0.f ? v : LCN_LRELU * v;
          v = ((kb >> q) & 1u) ? v * inv_keep : 0.f;
          if (res != nullptr) v += rc[q];
          y[q] = v;
        }
      }
      lcn_st8(Aout, oc, y);
      if (keepbits != nullptr) keepbits[(size_t)r * (P >> 3) + threadIdx.x] = (uint16_t)kb;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      zc[q] = zn[q];
      rc[q] = rn[q];
    }
    vc = vn;
    oc = on;
  }
}

// Same arithmetic for ONE BatchNorm group in bf16 with <= BA_R rows per thread (training at batch <= ~4.7 k): every
// load of the thread's rows (Z, residual) is issued before the first use, so the L2 latency is paid once per
// block instead of once per row (the register double buffer of k_bn_act exposes it BA_R-1 times); the Philox
// draws of the dropout mask overlap the loads.
#define BA_R 8
__global__ void __launch_bounds__(EW_MAXT, 2) k_bn_act_pre(const __nv_bfloat16* __restrict__ Z,
                                                           const float* __restrict__ stat,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ beta,
                                                           const __nv_bfloat16* __restrict__ res,
                                                           __nv_bfloat16* __restrict__ Aout,
                                                           uint16_t* __restrict__ keepbits, int P, int F, int rows_pad,
                                                           int bn_group, float rate, uint64_t seed, uint64_t step,
                                                           int layer, const lcn_step_scalars* __restrict__ dyn,
                                                           const double* __restrict__ gacc, float* __restrict__ stat_out,
                                                           double inv_n) {
  lcn_pdl_prologue();
  __shared__ __align__(16) float s_sc[256], s_sh[256];
  if (dyn != nullptr) step = dyn->step;
  const int Y = blockDim.y, c8 = threadIdx.x * 8, f0 = c8 % F;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int per = ((rows_pad / Y + gridDim.x - 1) / gridDim.x) * Y;      // contiguous rows of this block (<= BA_R * Y)
  const int r_begin = blockIdx.x * per, r_end = min(r_begin + per, rows_pad);
  if (r_begin >= r_end) return;
  uint4 zr[BA_R], rr[BA_R];
#pragma unroll
  for (int i = 0; i < BA_R; ++i) {
    const int r = r_begin + threadIdx.y + i * Y;
    zr[i] = make_uint4(0u, 0u, 0u, 0u);
    rr[i] = make_uint4(0u, 0u, 0u, 0u);
    if (r < r_end && r < bn_group) {
      const size_t o = lcn_off<__nv_bfloat16>(r, c8, P);
      zr[i] = *reinterpret_cast<const uint4*>(Z + o);
      if (res != nullptr) rr[i] = *reinterpret_cast<const uint4*>(res + o);
    }
  }
  if (tid < F) {
    float mean, rstd;
    if (gacc != nullptr) {
      // statistics straight from the GEMM's per-channel fp64 accumulators (sum x, sum x^2 over batch x joints,
      // LCN_GACC_REP replicas): what k_bn_finalize would have produced, without the launch
      double S1 = 0.0, S2 = 0.0;
#pragma unroll
      for (int rep = 0; rep < LCN_GACC_REP; ++rep) {
        S1 += gacc[((size_t)rep * F + tid) * 2];
        S2 += gacc[((size_t)rep * F + tid) * 2 + 1];
      }
      // (fp64 only where the cancellation is; no fp64 division or square root on every block's critical path)
      const double md = S1 * inv_n;
      const double var = fmax(S2 * inv_n - md * md, 0.0);
      mean = (float)md;
      rstd = rsqrtf((float)var + LCN_BN_EPS);
      rstd = rstd * (1.5f - 0.5f * ((float)var + LCN_BN_EPS) * rstd * rstd);    // one Newton step: full fp32 accuracy
      if (blockIdx.x == 0) {            // for the backward pass
        stat_out[tid * 2] = mean;
        stat_out[tid * 2 + 1] = rstd;
      }
    } else {
      mean = stat[tid * 2];
      rstd = stat[tid * 2 + 1];
    }
    const float a = gamma[tid] * rstd;
    s_sc[tid] = a;
    s_sh[tid] = beta[tid] - mean * a;
  }
  __syncthreads();
  float sc[8], sh[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    sc[q] = s_sc[f0 + q];
    sh[q] = s_sh[f0 + q];
  }
  const float inv_keep = rate > 0.f ? 1.f / (1.f - rate) : 1.f;
  const uint32_t thr16 = lcn_keep_thr16(rate);
#pragma unroll
  for (int i = 0; i < BA_R; ++i) {
    const int r = r_begin + threadIdx.y + i * Y;
    if (r >= r_end) continue;
    float y[8];
    uint32_t kb = 0xffu;
    if (r >= bn_group) {
#pragma unroll
      for (int q = 0; q < 8; ++q) y[q] = 0.f;
    } else {
      if (rate > 0.f) {
        kb = lcn_keep8(seed, step, (uint32_t)layer, ((uint64_t)r * P + c8) >> 3, thr16);
      }
      const __nv_bfloat162* hz = reinterpret_cast<const __nv_bfloat162*>(&zr[i]);
      const __nv_bfloat162* hr = reinterpret_cast<const __nv_bfloat162*>(&rr[i]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 z2 = __bfloat1622float2(hz[e]), r2 = __bfloat1622float2(hr[e]);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int q = 2 * e + h;
          float v = fmaf(h ? z2.y : z2.x, sc[q], sh[q]);
          if (v > 0.f) kb |= 0x100u << q;
          v = v > 0.f ? v : LCN_LRELU * v;
          v = ((kb >> q) & 1u) ? v * inv_keep : 0.f;
          if (res != nullptr) v += h ? r2.y : r2.x;
          y[q] = v;
        }
      }
    }
    lcn_st8(Aout, lcn_off<__nv_bfloat16>(r, c8, P), y);
    if (keepbits != nullptr) keepbits[(size_t)r * (P >> 3) + threadIdx.x] = (uint16_t)kb;
  }
}

// ------------------------------------------------------------------------------------------------
// last layer + output head: out = A * Wm4 + b4, xy residual from the 2D input (models_att.py:750-773)
// grid tiles, 128 threads (thread = row), input chunks streamed through shared memory.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) k_last_layer(const T* __restrict__ A, const float* __restrict__ wm,
                                                    const float* __restrict__ bias, const float* __restrict__ x,
                                                    int in_F, RowGeom g, float* __restrict__ out_user,
                                                    float* __restrict__ out_ws, SupportBits sup, int P, int FC) {
  lcn_pdl_prologue();
  extern __shared__ __align__(16) float smem[];
  float* As = smem;                         // [128][65]
  float* Ws = smem + LCN_TILE * GS_APAD;    // [64][17][4]
  int tile = blockIdx.x, tid = threadIdx.x;
  size_t row0 = (size_t)tile * LCN_TILE;
  float acc[LCN_J][3];
#pragma unroll
  for (int j = 0; j < LCN_J; ++j) acc[j][0] = acc[j][1] = acc[j][2] = 0.f;
  for (int ic = 0; ic < LCN_J * FC; ++ic) {
    int i = ic / FC;
    __syncthreads();
    for (int f = tid; f < LCN_TILE * 16; f += 128) {
      int r = f >> 4, kq = f & 15;
      float4 v = lcn_ld4(A, lcn_off<T>(row0 + r, ic * 64 + kq * 4, P));
      float* dst = As + r * GS_APAD + kq * 4;
      dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    }
    for (int e = tid; e < 64 * LCN_J * 3; e += 128) {
      int k = e / (LCN_J * 3), jc = e - k * (LCN_J * 3);
      Ws[(k * LCN_J + jc / 3) * 4 + jc % 3] = wm[(size_t)(ic * 64 + k) * (LCN_J * 3) + jc];
    }
    __syncthreads();
    uint32_t outs = sup.row[i];
    for (int k = 0; k < 64; ++k) {
      float av = As[tid * GS_APAD + k];
#pragma unroll
      for (int j = 0; j < LCN_J; ++j) {
        if ((outs >> j) & 1u) {
          float4 wv = *reinterpret_cast<const float4*>(Ws + (k * LCN_J + j) * 4);
          acc[j][0] = fmaf(av, wv.x, acc[j][0]);
          acc[j][1] = fmaf(av, wv.y, acc[j][1]);
          acc[j][2] = fmaf(av, wv.z, acc[j][2]);
        }
      }
    }
  }
  int64_t pr = (int64_t)row0 + tid, src;
  bool valid = row_valid(g, pr, &src);
  int kin = LCN_J * in_F;
#pragma unroll
  for (int j = 0; j < LCN_J; ++j) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float v = acc[j][c] + bias[j * 3 + c];
      if (c < 2 && src >= 0) v += x[src * kin + j * in_F + c];
      if (out_ws != nullptr) out_ws[(size_t)pr * 51 + j * 3 + c] = valid ? v : 0.f;
      if (src >= 0) out_user[src * 51 + j * 3 + c] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// loss and its gradient: mean((out-labels)^2) over B*51 (models_att.py:356); dOut = 2 (out-y)/(B*51)
// ------------------------------------------------------------------------------------------------
// grid rows_pad/64, 256 threads: thread = (column c = tid%64, row slice tid/64)
__global__ void __launch_bounds__(256) k_loss_dout(const float* __restrict__ out_ws, const float* __restrict__ labels,
                                                   int64_t n_rows, float* __restrict__ dout,
                                                   __nv_bfloat16* __restrict__ dout16, float* __restrict__ db,
                                                   double* loss_acc, float* __restrict__ loss_out) {
  lcn_pdl_prologue();
  __shared__ double sh[32];
  __shared__ float csum[4][64];
  int c = threadIdx.x & 63, rs = threadIdx.x >> 6;
  float inv = 2.0f / ((float)n_rows * 51.f);
  double s = 0.0;
  float cs = 0.f;
  int64_t pr0 = (int64_t)blockIdx.x * 16;              // 16 rows per block (rows_pad is a multiple of 128)
  for (int r = rs; r < 16; r += 4) {
    int64_t pr = pr0 + r;
    float gsc = 0.f;
    if (c < 51) {
      float d = 0.f;
      if (pr < n_rows) {
        d = out_ws[pr * 51 + c] - labels[pr * 51 + c];
        s += (double)d * d;
      }
      gsc = d * inv;
      dout[pr * 51 + c] = gsc;
      cs += gsc;
    }
    if (dout16 != nullptr) dout16[lcn_off<__nv_bfloat16>(pr, c, 64)] = __float2bfloat16_rn(gsc);
  }
  csum[rs][c] = cs;
  s = block_reduce_sum_d(s, sh);
  __syncthreads();
  if (db != nullptr && threadIdx.x < 51)
    atomicAdd(&db[threadIdx.x], csum[0][threadIdx.x] + csum[1][threadIdx.x] + csum[2][threadIdx.x] + csum[3][threadIdx.x]);
  // loss = mean((out - y)^2) (models_att.py:356): the block that arrives last divides the fp64 sum
  if (threadIdx.x == 0) {
    atomicAdd(loss_acc, s);
    __threadfence();
    unsigned ticket = atomicAdd(reinterpret_cast<unsigned*>(loss_acc + 1), 1u);
    if (ticket == gridDim.x - 1) {
      __threadfence();
      double tot = *reinterpret_cast<volatile double*>(loss_acc);
      loss_out[0] = (float)(tot / ((double)n_rows * 51.0));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// last layer backward: dA = dOut * Wm4^T, dWm4 = A^T dOut, db4 = sum_rows dOut
// grid (rows_pad/rows_per_block, ceil(P/256)), 256 threads; thread = one input column
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_last_layer_bwd(const T* __restrict__ A, const float* __restrict__ dout,
                                                        const float* __restrict__ wm, T* __restrict__ dA,
                                                        float* __restrict__ dwm, float* __restrict__ db, int P,
                                                        int rows_per_block) {
  lcn_pdl_prologue();
  __shared__ float ds[32][52];
  int c = blockIdx.y * 256 + threadIdx.x;
  bool act = c < P;
  float w[51], gw[51];
#pragma unroll
  for (int q = 0; q < 51; ++q) {
    w[q] = act ? wm[(size_t)c * 51 + q] : 0.f;
    gw[q] = 0.f;
  }
  float sdb = 0.f;
  size_t row0 = (size_t)blockIdx.x * rows_per_block;
  for (int rc = 0; rc < rows_per_block; rc += 32) {
    __syncthreads();
    for (int e = threadIdx.x; e < 32 * 51; e += 256) ds[e / 51][e % 51] = dout[(row0 + rc) * 51 + e];
    __syncthreads();
    if (blockIdx.y == 0 && threadIdx.x < 51)
      for (int r = 0; r < 32; ++r) sdb += ds[r][threadIdx.x];
    if (act) {
      for (int r = 0; r < 32; ++r) {
        size_t o = lcn_off<T>(row0 + rc + r, c, P);
        float av = lcn_ld(A, o), da = 0.f;
#pragma unroll
        for (int q = 0; q < 51; ++q) {
          float d = ds[r][q];
          da = fmaf(w[q], d, da);
          gw[q] = fmaf(av, d, gw[q]);
        }
        lcn_st(dA, o, da);
      }
    }
  }
  if (act) {
#pragma unroll
    for (int q = 0; q < 51; ++q) atomicAdd(&dwm[(size_t)c * 51 + q], gw[q]);
  }
  if (blockIdx.y == 0 && threadIdx.x < 51) atomicAdd(&db[threadIdx.x], sdb);
}

// ------------------------------------------------------------------------------------------------
// BN / LeakyReLU / dropout backward (training = one group).
//   dy   = dOut * keep/(1-rate) * (ybn > 0 ? 1 : 0.2),  keep and ybn > 0 as stored by k_bn_act(_pre)
//   sums = (sum dy, rstd * sum dy*(z - mean)) = (sum dy, sum dy*xhat) per channel   [k_bn_bwd_reduce]
//   dZ   = sc*(dy - s1/n - xhat*s2/n) = sc*dy + alpha + beta*z                     [k_bn_bwd_apply], db = sum_rows dZ
// Persistent like k_bn_act: grid = 2 x SMs blocks of (P/8, Y) threads, strided rows, a register double buffer of the
// rows as loaded (Raw8); keep decisions and LeakyReLU branches come from the bits written by k_bn_act(_pre), so neither
// kernel forms ybn; one block-level reduction, then one atomic per channel (reduce) / one partial row (apply) per block.
//
// Both kernels run while the weight-gradient GEMM of the layer before (k_tc_wgrad, one 224-thread CTA with ~195 KB of
// shared memory and 72 registers per thread on 124 of the SMs) is still running on the side stream.  Their grid
// assumes two blocks per SM, so two blocks must fit BESIDE that CTA (else 124 of 296 run as a second wave): at most
// 72 registers per thread (register files are per SM sub-partition: 16 K registers, 2 wgrad warps + 5 of these warps
// in each), the per-channel constants in shared memory rather than registers, <= 15 KB of shared memory per block,
// and the maximum shared-memory carveout (backward_impl).  lcn_debug_bn_bwd_fit reports the fit for the device.
// ------------------------------------------------------------------------------------------------
#define LCN_BN_BWD_MAXREG 72

// one thread's 8 consecutive elements of a row, as loaded: 16 B per bf16 plane (4 registers for bf16, 8 for split
// bf16 instead of 8 floats); at(q) is what lcn_ld8 would have produced for element q
template <typename T>
struct Raw8;
__device__ __forceinline__ float bf16_word_at(const uint4& u, int q) {
  const uint32_t w = q < 2 ? u.x : q < 4 ? u.y : q < 6 ? u.z : u.w;
  return __uint_as_float((q & 1) ? (w & 0xffff0000u) : (w << 16));
}
template <>
struct Raw8<__nv_bfloat16> {
  uint4 h;
  __device__ __forceinline__ void load(const __nv_bfloat16* p, size_t i) { h = *reinterpret_cast<const uint4*>(p + i); }
  __device__ __forceinline__ float at(int q) const { return bf16_word_at(h, q); }
};
template <>
struct Raw8<lcn_sp16> {
  uint4 h, l;
  __device__ __forceinline__ void load(const lcn_sp16* p, size_t i) {
    const __nv_bfloat16* q = reinterpret_cast<const __nv_bfloat16*>(p);
    h = *reinterpret_cast<const uint4*>(q + i);
    l = *reinterpret_cast<const uint4*>(q + i + LCN_SP_LO);
  }
  __device__ __forceinline__ float at(int q) const { return bf16_word_at(h, q) + bf16_word_at(l, q); }
};

// Per-channel constants of the backward kernels: s_k[k][f] in shared memory.  lds<W>(s_f0, k, h, v) reads constants k
// of the thread's channels f0 + h .. f0 + h + W - 1, s_f0 being the shared address of s_k[0][f0].  volatile: read again
// for every row, where they are used, instead of hoisted out of the row loop into live registers.
#define BN_BWD_KSTRIDE 256
template <int W>
__device__ __forceinline__ void lds(uint32_t s_f0, int k, int h, float v[W]) {
  static_assert(W == 2 || W == 4, "2 or 4 channels");
  const uint32_t a = s_f0 + (uint32_t)(k * BN_BWD_KSTRIDE + h) * 4u;
  if constexpr (W == 4)
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a));
  else
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "r"(a));
}

// dy of element q: its dropout keep bit (bit q) and the LeakyReLU branch the forward pass took (bit 8 + q), both as
// k_bn_act(_pre) wrote them
__device__ __forceinline__ float bn_bwd_dy(float d, uint32_t kb, int q, float inv_keep) {
  const float v = ((kb >> q) & 1u) ? d * inv_keep : 0.f;
  return ((kb >> (8 + q)) & 1u) ? v : LCN_LRELU * v;
}

template <typename T>
__global__ void __maxnreg__(LCN_BN_BWD_MAXREG) k_bn_bwd_reduce(const T* __restrict__ dOut, const T* __restrict__ Z,
                                                               const uint16_t* __restrict__ keepbits,
                                                               const float* __restrict__ stat, float* __restrict__ sums,
                                                               int P, int F, int bn_group, float rate) {
  lcn_pdl_prologue();
  __shared__ __align__(16) float s_k[1][BN_BWD_KSTRIDE];    // mean
  extern __shared__ float red[];                 // [warps][16 values][F/8 octets]: warp sums of (dy, dy*(z - mean))
  const int Y = blockDim.y, c8 = threadIdx.x * 8, f0 = c8 % F;
  const int nt = blockDim.x * Y, tid = threadIdx.y * blockDim.x + threadIdx.x;
  if (tid < F) s_k[0][tid] = stat[tid * 2];
  __syncthreads();
  const uint32_t s_f0 = (uint32_t)__cvta_generic_to_shared(&s_k[0][f0]);
  const float inv_keep = rate > 0.f ? 1.f / (1.f - rate) : 1.f;
  float s1[8], s2[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) s1[q] = s2[q] = 0.f;
  const int stride = gridDim.x * Y;
  int r = blockIdx.x * Y + threadIdx.y;
  Raw8<T> zc, dc, zn, dn;
  uint32_t kc = 0u, kn = 0u;
  if (r < bn_group) {
    const size_t o = lcn_off<T>(r, c8, P);
    zc.load(Z, o);
    dc.load(dOut, o);
    kc = keepbits[(size_t)r * (P >> 3) + threadIdx.x];
  }
  for (; r < bn_group; r += stride) {
    const int rn = r + stride;
    if (rn < bn_group) {
      const size_t o = lcn_off<T>(rn, c8, P);
      zn.load(Z, o);
      dn.load(dOut, o);
      kn = keepbits[(size_t)rn * (P >> 3) + threadIdx.x];
    }
#pragma unroll
    for (int h = 0; h < 8; h += 4) {             // the means of 4 channels are live at a time
      float mu[4];
      lds<4>(s_f0, 0, h, mu);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int q = h + e;
        const float dy = bn_bwd_dy(dc.at(q), kc, q, inv_keep);
        s1[q] += dy;
        s2[q] = fmaf(dy, zc.at(q) - mu[e], s2[q]);
      }
    }
    zc = zn;
    dc = dn;
    kc = kn;
  }
  // Threads tid, tid ^ F/8, ... of a warp hold the same channel octet (tid % (F/8); F/8 divides 32 and the row length
  // P/8): butterfly over them (the partial last warp has 16 lanes), then lanes 0 .. F/8-1 store the warp's sums and
  // 2F threads add up the warps (plain stores: shared-memory float atomics are compare-and-swap loops that the 9 warps
  // of a block, arriving together, serialise on)
  const int lane = tid & 31, per = F / 8, nv = min(32, nt - (tid & ~31));
  const unsigned mask = nv == 32 ? 0xffffffffu : (1u << nv) - 1u;
  for (int off = per; off < nv; off <<= 1) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      s1[q] += __shfl_xor_sync(mask, s1[q], off);
      s2[q] += __shfl_xor_sync(mask, s2[q], off);
    }
  }
  if (lane < per) {
    float* mine = red + (tid >> 5) * 2 * F + lane;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      mine[q * per] = s1[q];
      mine[(8 + q) * per] = s2[q];
    }
  }
  __syncthreads();
  const int nw = (nt + 31) >> 5;
  for (int i = tid; i < 2 * F; i += nt) {
    float a = 0.f;
    for (int w = 0; w < nw; ++w) a += red[w * 2 * F + i];
    const int v = i / per, f = (i % per) * 8 + (v & 7);
    atomicAdd(&sums[f * 2 + (v >> 3)], v < 8 ? a : a * stat[f * 2 + 1]);
  }
}

template <typename T, bool kSync>
__global__ void __maxnreg__(LCN_BN_BWD_MAXREG) k_bn_bwd_apply(const T* __restrict__ dOut, const T* __restrict__ Z,
                                                              const uint16_t* __restrict__ keepbits,
                                                              const float* __restrict__ stat,
                                                              const float* __restrict__ gamma,
                                                              const float* __restrict__ sums, T* __restrict__ dZ,
                                                              float* __restrict__ dbpart, float* __restrict__ dgamma,
                                                              float* __restrict__ dbeta, int P, int F, int rows_pad,
                                                              int bn_group, float rate, const float* __restrict__ gmean) {
  lcn_pdl_prologue();
  extern __shared__ __align__(16) float red[];   // [Y-1][P] column sums of the other row-threads
  __shared__ __align__(16) float s_k[3][BN_BWD_KSTRIDE];    // sc, alpha, beta
  const int Y = blockDim.y, c8 = threadIdx.x * 8, f0 = c8 % F;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if (tid < F) {
    const float mean = stat[tid * 2], rstd = stat[tid * 2 + 1];
    const float sc = gamma[tid] * rstd;
    float m1, m2;
    if constexpr (kSync) {       // synchronised BatchNorm: (S1, S2) / N over all ranks' rows, from k_bn_sync
      m1 = gmean[tid * 2];
      m2 = gmean[tid * 2 + 1];
    } else {
      const float inv_n = 1.f / ((float)bn_group * (float)LCN_J);
      m1 = sums[tid * 2] * inv_n;
      m2 = sums[tid * 2 + 1] * inv_n;
    }
    s_k[0][tid] = sc;
    // sc*(dy - m1 - xhat*m2) with xhat = z*rstd - mean*rstd
    s_k[1][tid] = sc * (m2 * (mean * rstd) - m1);
    s_k[2][tid] = -(sc * m2) * rstd;
    if (blockIdx.x == 0) {
      dbeta[tid] = sums[tid * 2];
      dgamma[tid] = sums[tid * 2 + 1];
    }
  }
  __syncthreads();
  const uint32_t s_f0 = (uint32_t)__cvta_generic_to_shared(&s_k[0][f0]);
  const float inv_keep = rate > 0.f ? 1.f / (1.f - rate) : 1.f;
  float bsum[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) bsum[q] = 0.f;
  const int stride = gridDim.x * Y;
  int r = blockIdx.x * Y + threadIdx.y;
  Raw8<T> zc, dc, zn, dn;
  uint32_t kc = 0u, kn = 0u;
  if (r < bn_group) {
    const size_t o = lcn_off<T>(r, c8, P);
    zc.load(Z, o);
    dc.load(dOut, o);
    kc = keepbits[(size_t)r * (P >> 3) + threadIdx.x];
  }
  for (; r < rows_pad; r += stride) {
    const int rn = r + stride;
    if (rn < bn_group) {
      const size_t o = lcn_off<T>(rn, c8, P);
      zn.load(Z, o);
      dn.load(dOut, o);
      kn = keepbits[(size_t)rn * (P >> 3) + threadIdx.x];
    }
    float dz[8];
    if (r >= bn_group) {                          // tile padding rows: dZ must be zero (wgrad reduces over rows)
#pragma unroll
      for (int q = 0; q < 8; ++q) dz[q] = 0.f;
    } else {
#pragma unroll
      for (int h = 0; h < 8; h += 4) {           // the constants of 4 channels are live at a time
        float sc[4], al[4], be[4];
        lds<4>(s_f0, 0, h, sc);
        lds<4>(s_f0, 1, h, al);
        lds<4>(s_f0, 2, h, be);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int q = h + e;
          const float dy = bn_bwd_dy(dc.at(q), kc, q, inv_keep);
          dz[q] = fmaf(sc[e], dy, fmaf(be[e], zc.at(q), al[e]));
          bsum[q] += dz[q];
        }
      }
    }
    lcn_st8(dZ, lcn_off<T>(r, c8, P), dz);
    zc = zn;
    dc = dn;
    kc = kn;
  }
  // db: combine the row-threads of a column octet in shared memory; one partial row per block (no atomics:
  // 2*SMs blocks adding into the same 17F addresses serialise in L2 -- measured 19 us per layer)
  if (threadIdx.y > 0) {
#pragma unroll
    for (int q = 0; q < 8; ++q) red[(size_t)(threadIdx.y - 1) * P + c8 + q] = bsum[q];
  }
  __syncthreads();
  if (threadIdx.y == 0) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float a = bsum[q];
      for (int y = 1; y < Y; ++y) a += red[(size_t)(y - 1) * P + c8 + q];
      dbpart[(size_t)blockIdx.x * P + c8 + q] = a;
    }
  }
}

// db[l][col] = sum over the per-block partial rows written by k_bn_bwd_apply.  grid (ceil(P/64), n_bn), 256 threads
__global__ void __launch_bounds__(256) k_db_reduce(const float* __restrict__ dbpart, int nblocks, int P,
                                                   float* __restrict__ graw, LinTable lt_b /* w_off holds b_off */) {
  // grid (P/64, n_bn): 16 row lanes x 16 column quads; a thread adds every 16th partial row of its 4 columns with four
  // independent accumulators (all of its <= 19 loads in flight), then the lanes are combined in a fixed order
  lcn_pdl_prologue();
  __shared__ float4 sh[16][16];
  const int l = blockIdx.y, q = threadIdx.x & 15, lane = threadIdx.x >> 4;
  const int c = blockIdx.x * 64 + q * 4;
  float4 a[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) a[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < P) {
    const float* src = dbpart + (size_t)l * nblocks * P + c;
    int b = lane;
    for (; b + 48 < nblocks; b += 64) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float4 v = *reinterpret_cast<const float4*>(src + (size_t)(b + 16 * k) * P);
        a[k].x += v.x; a[k].y += v.y; a[k].z += v.z; a[k].w += v.w;
      }
    }
    for (int k = 0; b < nblocks; b += 16, ++k) {
      const float4 v = *reinterpret_cast<const float4*>(src + (size_t)b * P);
      a[k & 3].x += v.x; a[k & 3].y += v.y; a[k & 3].z += v.z; a[k & 3].w += v.w;
    }
  }
  sh[lane][q] = make_float4((a[0].x + a[1].x) + (a[2].x + a[3].x), (a[0].y + a[1].y) + (a[2].y + a[3].y),
                            (a[0].z + a[1].z) + (a[2].z + a[3].z), (a[0].w + a[1].w) + (a[2].w + a[3].w));
  __syncthreads();
  if (lane == 0 && c < P) {
    float4 r = sh[0][q];
#pragma unroll
    for (int k = 1; k < 16; ++k) { r.x += sh[k][q].x; r.y += sh[k][q].y; r.z += sh[k][q].z; r.w += sh[k][q].w; }
    *reinterpret_cast<float4*>(graw + lt_b.w_off[l] + c) = r;
  }
}

// first layer weight gradient: dWm1[k][c] = sum_rows X[row][k] dZ0[row][c]  (dense 17*in_F x P)
template <typename T, int IN_F>
__global__ void __launch_bounds__(256) k_first_wgrad(const float* __restrict__ x, int64_t n_rows,
                                                     const T* __restrict__ dZ, float* __restrict__ dW, int P,
                                                     int rows_per_block) {
  lcn_pdl_prologue();
  constexpr int KIN = LCN_J * IN_F;
  __shared__ float xs[32][KIN];
  int c = blockIdx.y * 256 + threadIdx.x;
  bool act = c < P;
  float acc[KIN];
#pragma unroll
  for (int k = 0; k < KIN; ++k) acc[k] = 0.f;
  int64_t row0 = (int64_t)blockIdx.x * rows_per_block;
  for (int rc = 0; rc < rows_per_block; rc += 32) {
    __syncthreads();
    for (int e = threadIdx.x; e < 32 * KIN; e += 256) {
      int64_t pr = row0 + rc + e / KIN;
      xs[e / KIN][e % KIN] = pr < n_rows ? x[pr * KIN + e % KIN] : 0.f;
    }
    __syncthreads();
    if (act) {
      for (int r = 0; r < 32; ++r) {
        float dz = lcn_ld(dZ, lcn_off<T>(row0 + rc + r, c, P));
#pragma unroll
        for (int k = 0; k < KIN; ++k) acc[k] = fmaf(xs[r][k], dz, acc[k]);
      }
    }
  }
  if (act) {
#pragma unroll
    for (int k = 0; k < KIN; ++k) atomicAdd(&dW[(size_t)k * P + c], acc[k]);
  }
}

// ------------------------------------------------------------------------------------------------
// chain rule through mask_weights / clip_by_norm / mask softmax, and the fused masked Adam
// ------------------------------------------------------------------------------------------------
// pairdot[l][p] = <dWm_l(block p), W_l(block p)>      grid (nnz, n_lin), 256 threads
__global__ void __launch_bounds__(256) k_pairdot(const float* __restrict__ params, const float* __restrict__ graw, LinTable lt,
                                                 PairTable pt, float* __restrict__ pairdot) {
  lcn_pdl_prologue();
  __shared__ double sh[32];
  int p = blockIdx.x, l = blockIdx.y;
  int Fi = lt.Fi[l], Fo = lt.Fo[l], Kout = LCN_J * Fo;
  int i = pt.pi[p], j = pt.pj[p];
  const size_t base = (size_t)lt.w_off[l] + (size_t)(i * Fi) * Kout + j * Fo;
  const float* w = params + base;
  const float* g = graw + base;
  double s = 0.0;
  if ((Fo & 3) == 0 && (base & 3) == 0) {
    // 16-byte loads, four rows of the block in flight per thread
    const int q = Fo >> 2, n4 = Fi * q;
    for (int t0 = threadIdx.x; t0 < n4; t0 += 4 * 256) {
      float4 wv[4], gv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int t = t0 + k * 256;
        wv[k] = gv[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < n4) {
          const int fi = t / q, c4 = (t - fi * q) * 4;
          const size_t o = (size_t)fi * Kout + c4;
          wv[k] = *reinterpret_cast<const float4*>(w + o);
          gv[k] = *reinterpret_cast<const float4*>(g + o);
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k)
        s += (double)gv[k].x * (double)wv[k].x + (double)gv[k].y * (double)wv[k].y + (double)gv[k].z * (double)wv[k].z +
             (double)gv[k].w * (double)wv[k].w;
    }
  } else {
    for (int e = threadIdx.x; e < Fi * Fo; e += blockDim.x) {
      int fi = e / Fo, fo = e - fi * Fo;
      size_t o = (size_t)fi * Kout + fo;
      s += (double)g[o] * (double)w[o];
    }
  }
  s = block_reduce_sum_d(s, sh);
  if (threadIdx.x == 0) pairdot[l * LCN_J * LCN_J + p] = (float)s;
}

// per-layer <dWc,W> -> clip coefficient; mask gradient through the column softmax (SURVEY 9-Q5/Q6)
__global__ void k_maskgrad(const float* __restrict__ params, int64_t mask_off, SupportBits sup, PairTable pt,
                           int nnz, int n_lin, const float* __restrict__ pairdot, const float* __restrict__ mask,
                           LayerScalars* sc, float* __restrict__ maskgrad /*[289]*/, int zero_norm2) {
  lcn_pdl_prologue();
  __shared__ float dM[LCN_J * LCN_J];
  if (zero_norm2 && threadIdx.x < n_lin) sc[threadIdx.x].norm2 = 0.0;   // the Adam kernel that follows accumulates ||W_new||^2
  __shared__ float soft[LCN_J * LCN_J];
  int t = threadIdx.x;
  for (int l = t >> 5; l < n_lin; l += (int)(blockDim.x >> 5)) {      // one warp per layer, lanes over the pairs
    double s = 0.0;
    for (int p = t & 31; p < nnz; p += 32)
      s += (double)mask[pt.pi[p] * LCN_J + pt.pj[p]] * (double)pairdot[l * LCN_J * LCN_J + p];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((t & 31) == 0) {
      sc[l].sdot = s;
      double inv = sc[l].inv_norm;
      sc[l].coef = sc[l].clipped > 0.f ? (float)(s * inv * inv * inv) : 0.f;
    }
  }
  if (t < LCN_J * LCN_J) {
    int i = t / LCN_J, j = t % LCN_J;
    float d = 0.f;
    int p = sup.pair[i][j];
    if (p >= 0)
      for (int l = 0; l < n_lin; ++l) d += pairdot[l * LCN_J * LCN_J + p] * sc[l].inv_norm;
    dM[t] = d;
    if (mask_off >= 0) {
      const float* var = params + mask_off;
      float mx = -INFINITY;
      for (int k = 0; k < LCN_J; ++k) mx = fmaxf(mx, var[k * LCN_J + j]);
      float den = 0.f;
      for (int k = 0; k < LCN_J; ++k) den += expf(var[k * LCN_J + j] - mx);
      soft[t] = expf(var[t] - mx) / den;
    }
  }
  __syncthreads();
  if (t < LCN_J * LCN_J && mask_off >= 0) {
    int j = t % LCN_J;
    float dot = 0.f;
    for (int k = 0; k < LCN_J; ++k) dot += soft[k * LCN_J + j] * dM[k * LCN_J + j];
    maskgrad[t] = soft[t] * (dM[t] - dot);
  }
}

// Fused: true gradient from the raw one, TF1 Adam update, ||W_new||^2 accumulation.
// WRITE_G: only materialise the true gradients (tests / inspection).
template <bool WRITE_G>
__global__ void __launch_bounds__(256) k_adam(float* __restrict__ params, float* __restrict__ mm,
                                              float* __restrict__ vv, const float* __restrict__ graw,
                                              float* __restrict__ gout, SegTable segs, LinTable lt, SupportBits sup,
                                              const float* __restrict__ mask, const float* __restrict__ maskgrad,
                                              LayerScalars* sc, float lr_t, float b1, float b2, float eps, float reg,
                                              const lcn_step_scalars* __restrict__ dyn) {
  lcn_pdl_prologue();
  __shared__ double sh[32];
  if (dyn != nullptr) lr_t = dyn->lr_t;        // CUDA-graph replay: the step size lives in device memory
  // Persistent: gridDim.x blocks (8 per SM) walk the parameter vector in quarter chunks of 1024 elements with a grid
  // stride, so the last wave is 1/6 of the work instead of half of it and the per-block prologue / norm reduction is
  // paid once per block and layer, not once per 4096 elements.
  constexpr int SUB = LCN_ADAM_CHUNK / 1024;
  const int nsub = segs.total_chunks * SUB;
  const float omb1 = 1.f - b1, omb2 = 1.f - b2;
  double nrm = 0.0;
  int nrm_layer = -1;
  int s = 0;
  for (int sub = blockIdx.x; sub < nsub; sub += gridDim.x) {
    const int chunk = sub / SUB, part = sub - chunk * SUB;
    while (s + 1 < segs.n && segs.s[s + 1].chunk_start <= chunk) ++s;
    const SegInfo sg = segs.s[s];
    const int64_t e0 = (int64_t)(chunk - sg.chunk_start) * LCN_ADAM_CHUNK + part * 1024;
    const int64_t e1 = min(e0 + (int64_t)1024, sg.size);
    const int l = sg.layer;
    int Fi = 1, Fo = 1, Kout = 1;
    float inv = 1.f, coef = 0.f;
    if (sg.kind == SEG_W) {
      if (!WRITE_G && l != nrm_layer) {          // block-uniform: flush the previous layer's ||W_new||^2
        if (nrm_layer >= 0) {
          nrm = block_reduce_sum_d(nrm, sh);
          if (threadIdx.x == 0) atomicAdd(&sc[nrm_layer].norm2, nrm);
          __syncthreads();
        }
        nrm = 0.0;
        nrm_layer = l;
      }
      Fi = lt.Fi[l]; Fo = lt.Fo[l]; Kout = LCN_J * Fo;
      inv = sc[l].inv_norm; coef = sc[l].coef;
    }
    if (sg.kind == SEG_W && (Fo & 3) == 0) {
      // fast path: 4 consecutive elements share the row and the joint pair; 28 B/parameter of HBM traffic
      const int64_t e = e0 + 4 * threadIdx.x;
      if (e < e1) {
        int64_t o = sg.off + e;
        uint32_t r = (uint32_t)e / (uint32_t)Kout, c = (uint32_t)e - r * (uint32_t)Kout;
        uint32_t i = r / (uint32_t)Fi, j = c / (uint32_t)Fo;
        float4 w4 = *reinterpret_cast<const float4*>(params + o);
        float w[4] = {w4.x, w4.y, w4.z, w4.w}, g[4];
        bool on = (sup.row[i] >> j) & 1u;
        float ms = on ? mask[i * LCN_J + j] * inv : 0.f;
        float4 gr = on ? *reinterpret_cast<const float4*>(graw + o) : make_float4(0.f, 0.f, 0.f, 0.f);
        float grr[4] = {gr.x, gr.y, gr.z, gr.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) g[q] = fmaf(reg, w[q], fmaf(grr[q], ms, -coef * w[q]));
        if (WRITE_G) {
          *reinterpret_cast<float4*>(gout + o) = make_float4(g[0], g[1], g[2], g[3]);
        } else {
          float4 m4 = *reinterpret_cast<const float4*>(mm + o), v4 = *reinterpret_cast<const float4*>(vv + o);
          float m[4] = {m4.x, m4.y, m4.z, m4.w}, v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            m[q] = b1 * m[q] + omb1 * g[q];
            v[q] = b2 * v[q] + omb2 * g[q] * g[q];
            w[q] -= lr_t * m[q] / (sqrtf(v[q]) + eps);
            nrm += (double)w[q] * w[q];
          }
          *reinterpret_cast<float4*>(mm + o) = make_float4(m[0], m[1], m[2], m[3]);
          *reinterpret_cast<float4*>(vv + o) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(params + o) = make_float4(w[0], w[1], w[2], w[3]);
        }
      }
    } else {
      for (int64_t e = e0 + threadIdx.x; e < e1; e += 256) {
        int64_t o = sg.off + e;
        float w = params[o];
        float g;
        if (sg.kind == SEG_W) {
          int r = (int)(e / Kout), c = (int)(e - (int64_t)r * Kout);
          int i = r / Fi, j = c / Fo;
          g = -coef * w;
          if ((sup.row[i] >> j) & 1u) g = fmaf(graw[o], mask[i * LCN_J + j] * inv, g);
          g = fmaf(reg, w, g);
        } else if (sg.kind == SEG_B) {
          g = fmaf(reg, w, graw[o]);
        } else if (sg.kind == SEG_MASK) {
          g = maskgrad[e];
        } else {
          g = graw[o];
        }
        if (WRITE_G) {
          gout[o] = g;
        } else {
          float m = b1 * mm[o] + omb1 * g;
          float v = b2 * vv[o] + omb2 * g * g;
          mm[o] = m;
          vv[o] = v;
          w -= lr_t * m / (sqrtf(v) + eps);
          params[o] = w;
          if (sg.kind == SEG_W) nrm += (double)w * w;
        }
      }
    }
  }
  if (!WRITE_G && nrm_layer >= 0) {
    nrm = block_reduce_sum_d(nrm, sh);
    if (threadIdx.x == 0) atomicAdd(&sc[nrm_layer].norm2, nrm);
  }
}

static int launch_grad_chain(const lcn_model* m, const float* params, char* ws, const WsLayout& lay,
                             const float* graw, cudaStream_t st, int zero_norm2) {
  LayerScalars* sc = reinterpret_cast<LayerScalars*>(ws + lay.off_scalars);
  float* mask = reinterpret_cast<float*>(ws + lay.off_mask);
  float* pairdot = reinterpret_cast<float*>(ws + lay.off_pairdot);
  float* maskgrad = mask + 2 * LCN_J * LCN_J;
  lcn_launch(k_pairdot, dim3(dim3(m->nnz, m->n_lin)), dim3(256), 0, st, params, graw, make_lin(m), make_pairs(m), pairdot);
  lcn_launch(k_maskgrad, dim3(1), dim3(320), 0, st, params, m->mask_off, m->sup, make_pairs(m), m->nnz, m->n_lin, pairdot, mask, sc,
                                maskgrad, zero_norm2);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

int lcn_launch_grad_finalize(const lcn_model* m, const float* params, char* ws, const WsLayout& lay,
                             const float* grads_raw, float* grads_out, cudaStream_t st) {
  int rc = launch_grad_chain(m, params, ws, lay, grads_raw, st, /*zero_norm2=*/0);
  if (rc) return rc;
  LayerScalars* sc = reinterpret_cast<LayerScalars*>(ws + lay.off_scalars);
  float* mask = reinterpret_cast<float*>(ws + lay.off_mask);
  lcn_launch(k_adam<true>, dim3(std::min(m->segs.total_chunks * (LCN_ADAM_CHUNK / 1024), 8 * m->sm_count)), dim3(256), 0, st, const_cast<float*>(params), nullptr, nullptr, grads_raw,
                                                     grads_out, m->segs, make_lin(m), m->sup, mask,
                                                     mask + 2 * LCN_J * LCN_J, sc, 0.f, 0.f, 0.f, 0.f, 0.f, nullptr);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

int lcn_launch_adam(const lcn_model* m, float* params, float* mm, float* vv, char* ws, const WsLayout& lay,
                    const float* grads_raw, float lr_t, float b1, float b2, float eps, float reg,
                    const lcn_step_scalars* dyn, cudaStream_t st) {
  int rc = launch_grad_chain(m, params, ws, lay, grads_raw, st, /*zero_norm2=*/1);
  if (rc) return rc;
  LayerScalars* sc = reinterpret_cast<LayerScalars*>(ws + lay.off_scalars);
  float* mask = reinterpret_cast<float*>(ws + lay.off_mask);
  lcn_launch(k_adam<false>, dim3(std::min(m->segs.total_chunks * (LCN_ADAM_CHUNK / 1024), 8 * m->sm_count)), dim3(256), 0, st, params, mm, vv, grads_raw, nullptr, m->segs, make_lin(m),
                                                      m->sup, mask, mask + 2 * LCN_J * LCN_J, sc, lr_t, b1, b2, eps,
                                                      reg, dyn);
  LCN_CHECK_LAUNCH();
  return lcn_launch_prepare(m, params, ws, lay, /*recompute_norm=*/false, st);
}

// ------------------------------------------------------------------------------------------------
// forward / backward orchestration
// ------------------------------------------------------------------------------------------------
static inline char* z_buf(char* ws, const WsLayout& lay, int l) {
  return ws + lay.off_z + (size_t)(lay.training ? l : 0) * lay.z_stride;
}
static inline char* a_buf(char* ws, const WsLayout& lay, int l) {
  return ws + lay.off_a + (size_t)(lay.training ? l : l % 3) * lay.a_stride;
}
static inline float* bn_stat(char* ws, const WsLayout& lay, const lcn_model* m, int l) {
  return reinterpret_cast<float*>(ws + lay.off_bnstat) + (size_t)l * lay.n_groups * m->d.F * 2;
}
// launch geometry of the elementwise BatchNorm kernels (k_bn_act*, k_bn_bwd_*): blocks of (P/8, ewy) threads over
// grid-stride row ranges of rows_thr rows per thread
struct EwGeom {
  int ewy, grid, rows_thr;
};
static inline int ew_rows_per_block(int P) { return (P / 8) * 2 <= EW_MAXT ? 2 : 1; }
static inline EwGeom ew_geom(const lcn_model* m, const WsLayout& lay) {
  const int ewy = ew_rows_per_block(m->P);
  const int grid = (int)std::min<int64_t>(2 * m->sm_count, lay.rows_pad / ewy);
  return {ewy, grid, (int)((lay.rows_pad / ewy + grid - 1) / grid)};
}
// dynamic shared memory of k_bn_bwd_reduce: 2F warp sums per warp; of k_bn_bwd_apply: the column sums of the
// row-threads 1 .. ewy-1
static inline size_t bn_bwd_reduce_smem(int P, int ewy) {
  return (size_t)((P / 8 * ewy + 31) / 32) * 2 * (P / LCN_J) * sizeof(float);
}
static inline size_t bn_bwd_apply_smem(int P, int ewy) { return (size_t)(ewy - 1) * P * sizeof(float); }
// packed bf16 blocks of mid layer l: forward (Y = A*Wm) or transposed (dA = dZ*Wm^T); lo: their lo parts on the
// split-bf16 path, nullptr on the bf16 path
struct MidWeights {
  const char *hi, *lo;
};
static inline MidWeights mid_weights(const lcn_model* m, const char* ws, const WsLayout& lay, int l, int transposed) {
  const size_t ofs = (size_t)(l - 1) * m->nnz * m->FC * m->FC * 4096 * 2;
  const bool x3 = m->d.path == LCN_PATH_FP32;
  return {ws + (transposed ? lay.off_wp16b : lay.off_wp16f) + ofs,
          x3 ? ws + (transposed ? lay.off_wp16b_lo : lay.off_wp16f_lo) + ofs : nullptr};
}

template <typename T>
static int forward_impl(const FwdArgs& a) {
  const lcn_model* m = a.m;
  const WsLayout& lay = a.lay;
  char* ws = a.ws;
  cudaStream_t st = a.st;
  const int P = m->P, F = m->d.F, FC = m->FC;
  RowGeom g{lay.n_rows, lay.bn_group, lay.gstride};
  float* part = reinterpret_cast<float*>(ws + lay.off_part);
  constexpr bool kBf = PathTraits<T>::bf16;
  size_t gemm_smem = (LCN_TILE * GS_APAD + 64 * GS_BPAD) * sizeof(float);
  static std::once_flag attr_once;                 // one per instantiation; thread safe (header: re-entrancy)
  static cudaError_t attr_rc = cudaSuccess;
  std::call_once(attr_once, [&] {
    attr_rc = cudaFuncSetAttribute(k_last_layer<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem);
  });
  LCN_CHECK_CUDA(attr_rc);
  int n_bn = m->n_bn;
  const EwGeom ew = ew_geom(m, lay);
  // k_bn_act_pre takes every layer on the bf16 path at one BatchNorm group and <= BA_R rows per thread (all loads up
  // front).  In training the mid-layer GEMMs then accumulate the BatchNorm statistics themselves (TcFuse,
  // lcn_gemm_tc.cu) and k_bn_act_pre finalises them; the accumulators are cleared here, once per pass
  const bool pre = kBf && lay.n_groups == 1 && ew.rows_thr <= BA_R;
  const bool try_fuse = pre && lay.training;
  const bool bn_sync = lay.training && lcn_bn_sync_on(m);      // lcn_model_forward admits it only at one group
  if (bn_sync && lay.n_groups != 1) {
    lcn_set_error("synchronised BatchNorm: a training forward pass must be one BatchNorm group (bn_group = n_rows)");
    return LCN_EINVAL;
  }
  if (try_fuse) LCN_CHECK_CUDA(cudaMemsetAsync(ws + lay.off_gacc, 0, lay.gacc_stride * (size_t)n_bn, st));
  const int lb = a.layer_begin, le = a.layer_end < 0 ? m->n_lin : a.layer_end;   // linear layers [lb, le)
  for (int l = lb; l < n_bn && l < le; ++l) {
    const LayerInfo& L = m->L[l];
    T* Z = reinterpret_cast<T*>(z_buf(ws, lay, l));
    T* Aout = reinterpret_cast<T*>(a_buf(ws, lay, l));
    int fused_bn = 0;
    if (l == 0) {
      dim3 grid(lay.tiles, P / 64);
      const float* wm = reinterpret_cast<const float*>(ws + lay.off_wm_first);
      __nv_bfloat16* x16 = (kBf && lay.training) ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_x16) : nullptr;
      double* gacc0 = try_fuse ? reinterpret_cast<double*>(ws + lay.off_gacc) : nullptr;
      fused_bn = gacc0 != nullptr;
      switch (m->d.in_F) {
        case 2: lcn_launch(k_first_layer<T, 2>, dim3(grid), dim3(256), 0, st, a.x, g, wm, a.params + L.b_off, Z, part, P, x16, gacc0, F, m->sup); break;
        case 3: lcn_launch(k_first_layer<T, 3>, dim3(grid), dim3(256), 0, st, a.x, g, wm, a.params + L.b_off, Z, part, P, x16, gacc0, F, m->sup); break;
        default: lcn_set_error("in_F=%d not supported (2 or 3)", m->d.in_F); return LCN_EINVAL;
      }
    } else {
      const T* Ain = reinterpret_cast<const T*>(a_buf(ws, lay, l - 1));
      const MidWeights w = mid_weights(m, ws, lay, l, 0);
      TcFuse fu;
      memset(&fu, 0, sizeof(fu));
      if (try_fuse) {
        fu.gacc = reinterpret_cast<double*>(ws + lay.off_gacc + (size_t)l * lay.gacc_stride);
        fu.F = F;
      }
      int rc = lcn_tc_gemm(m, lay, l - 1, 0, reinterpret_cast<const __nv_bfloat16*>(Ain), w.hi, a.params + L.b_off,
                           nullptr, reinterpret_cast<__nv_bfloat16*>(Z), part, st, try_fuse ? &fu : nullptr, &fused_bn,
                           w.lo);
      if (rc) return rc;
    }
    LCN_CHECK_LAUNCH();
    float* stat = bn_stat(ws, lay, m, l);
    const double* gacc = fused_bn ? reinterpret_cast<const double*>(ws + lay.off_gacc + (size_t)l * lay.gacc_stride) : nullptr;
    // synchronised BatchNorm: k_bn_finalize leaves fp64 moments in the (otherwise unused) accumulator area of the layer,
    // k_bn_sync merges them -- or the GEMM's sums -- with the other ranks' and writes the global (mean, rstd) to stat
    double* mom = bn_sync ? reinterpret_cast<double*>(ws + lay.off_gacc + (size_t)l * lay.gacc_stride) : nullptr;
    if (fused_bn == 0)
    lcn_launch(k_bn_finalize, dim3(dim3(lay.n_groups, F / 2)), dim3(256), 0, st, part, stat, P, F, lay.tiles_per_group, lay.bn_group, mom);
    if (bn_sync) {
      LCN_CHECK_LAUNCH();
      int rc = lcn_bn_sync(m, l, fused_bn ? LCN_BN_SYNC_GACC : LCN_BN_SYNC_MOMENTS, fused_bn ? (const void*)gacc : mom, stat,
                           lay.n_rows, st);
      if (rc) return rc;
      gacc = nullptr;                  // k_bn_act_pre reads the global statistics from stat
    }
    const T* res = L.res_from >= 0 ? reinterpret_cast<const T*>(a_buf(ws, lay, L.res_from)) : nullptr;
    uint16_t* keepbits = lay.training ? reinterpret_cast<uint16_t*>(ws + lay.off_keep) + (size_t)l * lay.rows_pad * (P / 8)
                                      : nullptr;
    if (pre)
      lcn_launch(k_bn_act_pre, dim3(ew.grid), dim3(P / 8, ew.ewy), 0, st, reinterpret_cast<const __nv_bfloat16*>(Z), stat,
                 a.params + L.gamma_off, a.params + L.beta_off, reinterpret_cast<const __nv_bfloat16*>(res),
                 reinterpret_cast<__nv_bfloat16*>(Aout), keepbits, P, F, (int)lay.rows_pad, lay.bn_group, a.dropout_rate,
                 a.seed, a.step, l, a.dyn, gacc, stat, 1.0 / ((double)lay.bn_group * LCN_J));
    else
      lcn_launch(k_bn_act<T>, dim3(ew.grid), dim3(dim3(P / 8, ew.ewy)), 0, st, Z, stat, a.params + L.gamma_off, a.params + L.beta_off, res, Aout,
                                                      keepbits, P, F, (int)lay.rows_pad, lay.bn_group, lay.gstride,
                                                      a.dropout_rate, a.seed, a.step, l, a.dyn);
    LCN_CHECK_LAUNCH();
  }
  int last = m->n_lin - 1;
  if (le <= last) return LCN_OK;
  const T* Ain = reinterpret_cast<const T*>(a_buf(ws, lay, n_bn - 1));
  float* out_ws = lay.training ? reinterpret_cast<float*>(ws + lay.off_out) : nullptr;
  if constexpr (kBf) {
    int rc = lcn_tc_head(m, lay, reinterpret_cast<const __nv_bfloat16*>(Ain), ws + lay.off_wl16f,
                         a.params + m->L[last].b_off, a.x, a.out, out_ws, st);
    if (rc) return rc;
  } else {
    lcn_launch(k_last_layer<T>, dim3(lay.tiles), dim3(128), gemm_smem, st, Ain, reinterpret_cast<const float*>(ws + lay.off_wm_last),
                                                       a.params + m->L[last].b_off, a.x, m->d.in_F, g, a.out, out_ws,
                                                       m->sup, P, FC);
  }
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

int lcn_launch_forward(const FwdArgs& a) {
  if (a.lay.fused) return lcn_stack_forward(a.m, a.lay, a.params, a.ws, a.x, a.out, nullptr, a.st);
  return a.m->d.path == LCN_PATH_BF16 ? forward_impl<__nv_bfloat16>(a) : forward_impl<lcn_sp16>(a);
}

template <typename T>
static int backward_impl(const lcn_model* m, const float* params, char* ws, const WsLayout& lay, const float* x,
                         const float* labels, float rate, uint64_t seed, uint64_t step, float* loss,
                         float* graw, cudaStream_t st) {
  const int P = m->P, F = m->d.F;
  constexpr bool kBf = PathTraits<T>::bf16, kX3 = PathTraits<T>::x3;
  // weight-gradient GEMMs go to the model's side stream (see LcnAux); `wst` is the stream they are enqueued on
  std::lock_guard<std::mutex> aux_lock(m->aux.mu);
  LcnAux* ax;
  int rc = lcn_aux_get(m, &ax);
  if (rc) return rc;
  cudaStream_t wst = ax->st;
  const bool bn_sync = lcn_bn_sync_on(m);
  bool wg_pending[2] = {false, false};
  const int64_t blast = m->L[m->n_lin - 1].b_off;     // last-layer bias gradient: accumulated by k_loss_dout (caller's stream)
  // fork at the very start: the 4 B/parameter clear of the gradient bucket (the weight-gradient GEMMs reduce-add
  // into it) leaves the critical path; the caller's stream only clears what its own first kernels accumulate into
  LCN_CHECK_CUDA(cudaEventRecord(ax->ev_go, st));
  LCN_CHECK_CUDA(cudaStreamWaitEvent(wst, ax->ev_go, 0));
  LCN_CHECK_CUDA(cudaMemsetAsync(graw, 0, sizeof(float) * blast, wst));
  if (blast + 51 < m->n_params)
    LCN_CHECK_CUDA(cudaMemsetAsync(graw + blast + 51, 0, sizeof(float) * (m->n_params - blast - 51), wst));
  LCN_CHECK_CUDA(cudaMemsetAsync(ws + lay.off_dw_last, 0, sizeof(float) * P * 64, wst));
  LCN_CHECK_CUDA(cudaMemsetAsync(ws + lay.off_dw_first, 0, sizeof(float) * 64 * P, wst));
  LCN_CHECK_CUDA(cudaEventRecord(ax->ev_ms, wst));
  LCN_CHECK_CUDA(cudaMemsetAsync(graw + blast, 0, sizeof(float) * 51, st));
  LCN_CHECK_CUDA(cudaMemsetAsync(ws + lay.off_loss, 0, 2 * sizeof(double), st));
  LCN_CHECK_CUDA(cudaMemsetAsync(ws + lay.off_bnsum, 0, sizeof(float) * m->n_bn * (F * 2 + 1), st));   // sums + grid-barrier counters
  float* dout = reinterpret_cast<float*>(ws + lay.off_dout);
  double* lacc = reinterpret_cast<double*>(ws + lay.off_loss);
  __nv_bfloat16* dout16 = kBf ? reinterpret_cast<__nv_bfloat16*>(ws + lay.off_dout16) : nullptr;
  lcn_launch(k_loss_dout, dim3((unsigned)(lay.rows_pad / 16)), dim3(256), 0, st, reinterpret_cast<const float*>(ws + lay.off_out), labels,
                                                             lay.n_rows, dout, dout16,
                                                             kBf ? graw + m->L[m->n_lin - 1].b_off : nullptr, lacc, loss);
  LCN_CHECK_LAUNCH();

  auto D = [&](int i) { return reinterpret_cast<T*>(ws + lay.off_d + (size_t)i * lay.d_stride); };
  auto dZbuf = [&](int l) { return reinterpret_cast<T*>(ws + lay.off_dz + (size_t)(l & 1) * lay.d_stride); };
  int last = m->n_lin - 1;
  int rows_blk = 512;
  while (lay.rows_pad % rows_blk) rows_blk >>= 1;   // rows_pad is a multiple of 128
  int cur = 0;
  if constexpr (kBf) {
    const __nv_bfloat16* Ain = reinterpret_cast<const __nv_bfloat16*>(a_buf(ws, lay, m->n_bn - 1));
    float* dwl = reinterpret_cast<float*>(ws + lay.off_dw_last);
    // the loss gradient (caller's stream) precedes the last layer's weight gradient
    LCN_CHECK_CUDA(cudaEventRecord(ax->ev_loss, st));
    LCN_CHECK_CUDA(cudaStreamWaitEvent(wst, ax->ev_loss, 0));
    rc = lcn_tc_head_dgrad(m, lay, dout16, ws + lay.off_wl16b, reinterpret_cast<__nv_bfloat16*>(D(cur)), st);
    if (rc) return rc;
    rc = lcn_tc_wgrad_last(m, lay, Ain, dout16, dwl, wst);
    if (rc) return rc;
    LCN_CHECK_CUDA(cudaMemcpy2DAsync(graw + m->L[last].w_off, 51 * sizeof(float), dwl, 64 * sizeof(float),
                                     51 * sizeof(float), P, cudaMemcpyDeviceToDevice, wst));
  } else {
    // fp32-parity path: the N = 51 head on CUDA cores.  It accumulates dWm4 / db4 with atomics into the bucket, which the
    // side stream is clearing: wait for that first
    LCN_CHECK_CUDA(cudaStreamWaitEvent(st, ax->ev_ms, 0));
    const T* Ain = reinterpret_cast<const T*>(a_buf(ws, lay, m->n_bn - 1));
    lcn_launch(k_last_layer_bwd<T>, dim3(dim3((unsigned)(lay.rows_pad / rows_blk), (P + 255) / 256)), dim3(256), 0, st, 
        Ain, dout, reinterpret_cast<const float*>(ws + lay.off_wm_last), D(cur), graw + m->L[last].w_off,
        graw + m->L[last].b_off, P, rows_blk);
    LCN_CHECK_LAUNCH();
  }
  const EwGeom ew = ew_geom(m, lay);
  // the weight-gradient GEMM beside these kernels needs the SM's full shared-memory carveout; an SM that holds only
  // BatchNorm blocks keeps that configuration, so a weight-gradient CTA can still join them
  static std::once_flag carveout_once;
  static cudaError_t carveout_rc = cudaSuccess;
  std::call_once(carveout_once, [] {
    const int c = cudaSharedmemCarveoutMaxShared;
    carveout_rc = cudaFuncSetAttribute(k_bn_bwd_reduce<T>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
    if (carveout_rc == cudaSuccess)
      carveout_rc = cudaFuncSetAttribute(k_bn_bwd_apply<T, false>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
    if (carveout_rc == cudaSuccess)
      carveout_rc = cudaFuncSetAttribute(k_bn_bwd_apply<T, true>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  });
  LCN_CHECK_CUDA(carveout_rc);
  LCN_CHECK_CUDA(cudaStreamWaitEvent(st, ax->ev_ms, 0));   // the bucket is clear before this stream stores into it
  for (int l = m->n_bn - 1; l >= 0; --l) {
    const LayerInfo& L = m->L[l];
    const T* Z = reinterpret_cast<const T*>(z_buf(ws, lay, l));
    const float* stat = bn_stat(ws, lay, m, l);
    float* sums = reinterpret_cast<float*>(ws + lay.off_bnsum) + (size_t)l * F * 2;
    const uint16_t* keepbits = reinterpret_cast<const uint16_t*>(ws + lay.off_keep) + (size_t)l * lay.rows_pad * (P / 8);
    T* dZ = dZbuf(l);
    if (wg_pending[l & 1]) {         // the weight gradient of layer l+2 has read this dZ buffer
      LCN_CHECK_CUDA(cudaStreamWaitEvent(st, ax->ev_wg[l & 1], 0));
      wg_pending[l & 1] = false;
    }
    lcn_launch(k_bn_bwd_reduce<T>, dim3(ew.grid), dim3(dim3(P / 8, ew.ewy)), bn_bwd_reduce_smem(P, ew.ewy), st, D(cur), Z, keepbits, stat, sums, P, F,
                                                             lay.bn_group, rate);
    float* gmean = nullptr;            // synchronised BatchNorm: (S1, S2) / N of all ranks, in the layer's accumulator area
    if (bn_sync) {
      LCN_CHECK_LAUNCH();
      gmean = reinterpret_cast<float*>(ws + lay.off_gacc + (size_t)l * lay.gacc_stride);
      rc = lcn_bn_sync(m, m->n_bn + l, LCN_BN_SYNC_SUMS, sums, gmean, lay.n_rows, st);
      if (rc) return rc;
    }
    lcn_launch(bn_sync ? k_bn_bwd_apply<T, true> : k_bn_bwd_apply<T, false>, dim3(ew.grid), dim3(dim3(P / 8, ew.ewy)), bn_bwd_apply_smem(P, ew.ewy), st,
        D(cur), Z, keepbits, stat, params + L.gamma_off, sums, dZ,
        reinterpret_cast<float*>(ws + lay.off_dbpart) + (size_t)l * ew.grid * P, graw + L.gamma_off, graw + L.beta_off, P, F, (int)lay.rows_pad, lay.bn_group, rate,
        gmean);
    LCN_CHECK_LAUNCH();
    // dZ_l is ready: the side stream may start the weight gradient of layer l
    LCN_CHECK_CUDA(cudaEventRecord(ax->ev_dz[l & 1], st));
    LCN_CHECK_CUDA(cudaStreamWaitEvent(wst, ax->ev_dz[l & 1], 0));
    if (l == 0 && kBf) {
      float* dwf = reinterpret_cast<float*>(ws + lay.off_dw_first);
      rc = lcn_tc_wgrad_first(m, lay, reinterpret_cast<const __nv_bfloat16*>(ws + lay.off_x16),
                              reinterpret_cast<const __nv_bfloat16*>(dZ), dwf, wst);
      if (rc) return rc;
      LCN_CHECK_CUDA(cudaMemcpyAsync(graw + L.w_off, dwf, sizeof(float) * L.Kin * P, cudaMemcpyDeviceToDevice, wst));
      break;
    }
    if (l == 0) {
      dim3 grid((unsigned)(lay.rows_pad / rows_blk), (P + 255) / 256);
      if (m->d.in_F == 2) lcn_launch(k_first_wgrad<T, 2>, dim3(grid), dim3(256), 0, st, x, lay.n_rows, dZ, graw + L.w_off, P, rows_blk);
      else lcn_launch(k_first_wgrad<T, 3>, dim3(grid), dim3(256), 0, st, x, lay.n_rows, dZ, graw + L.w_off, P, rows_blk);
      LCN_CHECK_LAUNCH();
      break;
    }
    const T* Ain = reinterpret_cast<const T*>(a_buf(ws, lay, l - 1));
    rc = lcn_tc_wgrad(m, lay, reinterpret_cast<const __nv_bfloat16*>(Ain), reinterpret_cast<const __nv_bfloat16*>(dZ),
                      graw + L.w_off, wst, kX3);
    if (rc) return rc;
    LCN_CHECK_CUDA(cudaEventRecord(ax->ev_wg[l & 1], wst));
    wg_pending[l & 1] = true;
    rc = lcn_dp_exchange_layer(m, graw, l, ax);   // data parallel: dW_l is final on the side stream
    if (rc) return rc;
    // the gradient w.r.t. the layer input goes to the next of the three buffers.  The first layer of a residual block
    // (the one without res_from) adds the block-output gradient, which the block's second layer left in D(cur + 2).
    const T* addend = m->d.residual && L.res_from < 0 ? D((cur + 2) % 3) : nullptr;
    const MidWeights w = mid_weights(m, ws, lay, l, 1);
    rc = lcn_tc_gemm(m, lay, l - 1, 1, reinterpret_cast<const __nv_bfloat16*>(dZ), w.hi, nullptr,
                     reinterpret_cast<const __nv_bfloat16*>(addend), reinterpret_cast<__nv_bfloat16*>(D((cur + 1) % 3)),
                     nullptr, st, nullptr, nullptr, w.lo);
    if (rc) return rc;
    LCN_CHECK_LAUNCH();
    cur = (cur + 1) % 3;
  }
  {
    LinTable lb;
    lb.n = m->n_bn;
    for (int l = 0; l < m->n_bn; ++l) lb.w_off[l] = m->L[l].b_off;
    lcn_launch(k_db_reduce, dim3(dim3((P + 63) / 64, m->n_bn)), dim3(256), 0, st, reinterpret_cast<const float*>(ws + lay.off_dbpart),
                                                              ew.grid, P, graw, lb);
    LCN_CHECK_LAUNCH();
  }
  // join: the caller's stream continues after the last weight gradient
  LCN_CHECK_CUDA(cudaEventRecord(ax->ev_done, wst));
  LCN_CHECK_CUDA(cudaStreamWaitEvent(st, ax->ev_done, 0));
  return lcn_dp_exchange_rest(m, graw, ax, st);   // data parallel: the bucket holds the mean over the ranks after this
}

int lcn_launch_backward(const lcn_model* m, const float* params, char* ws, const WsLayout& lay, const float* x,
                        const float* labels, float dropout_rate, uint64_t seed, uint64_t step, float* loss,
                        float* grads_raw, cudaStream_t st) {
  return m->d.path == LCN_PATH_BF16
             ? backward_impl<__nv_bfloat16>(m, params, ws, lay, x, labels, dropout_rate, seed, step, loss, grads_raw, st)
             : backward_impl<lcn_sp16>(m, params, ws, lay, x, labels, dropout_rate, seed, step, loss, grads_raw, st);
}

// Blocks of each backward BatchNorm kernel that fit on one SM of this device beside one k_tc_wgrad CTA, at the block
// shape and dynamic shared memory backward_impl launches them with for feature width F.  blocks_out[6]:
// k_bn_bwd_reduce, k_bn_bwd_apply<false>, k_bn_bwd_apply<true> on the bf16 path (beside k_tc_wgrad<false>), then the
// same three on the split-bf16 path (beside k_tc_wgrad<true>).  Registers are counted per SM sub-partition, as the CUDA
// occupancy calculator counts them, and every sub-partition is charged as many k_tc_wgrad warps as the fullest one
// holds (2 of its 7).  Shared memory is the SM's maximum: the carveout both kernels prefer (backward_impl) and the one
// the k_tc_wgrad CTA needs.
extern "C" int lcn_debug_bn_bwd_fit(int F, int* blocks_out) {
  LCN_REQUIRE(F == 64 || F == 128, "F=%d: the backward BatchNorm kernels run at F = 64 or 128", F);
  const int P = LCN_J * F, ewy = ew_rows_per_block(P), threads = P / 8 * ewy;
  int dev = 0, sm_regs = 0, sm_smem = 0, reserved = 0, sm_threads = 0, sm_blocks = 0;
  LCN_CHECK_CUDA(cudaGetDevice(&dev));
  LCN_CHECK_CUDA(cudaDeviceGetAttribute(&sm_regs, cudaDevAttrMaxRegistersPerMultiprocessor, dev));
  LCN_CHECK_CUDA(cudaDeviceGetAttribute(&sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
  LCN_CHECK_CUDA(cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev));
  LCN_CHECK_CUDA(cudaDeviceGetAttribute(&sm_threads, cudaDevAttrMaxThreadsPerMultiProcessor, dev));
  LCN_CHECK_CUDA(cudaDeviceGetAttribute(&sm_blocks, cudaDevAttrMaxBlocksPerMultiprocessor, dev));
  constexpr int kSubPartitions = 4, kRegUnit = 256;           // registers are allocated per warp in units of 256
  auto warp_regs = [](const cudaFuncAttributes& a) { return (a.numRegs * 32 + kRegUnit - 1) / kRegUnit * kRegUnit; };
  auto fit = [&](const cudaFuncAttributes& w, size_t w_dyn, int w_threads, const cudaFuncAttributes& k, size_t k_dyn) {
    const int w_warps = (w_threads + 31) / 32, k_warps = (threads + 31) / 32;
    const int sp_left = sm_regs / kSubPartitions - (w_warps + kSubPartitions - 1) / kSubPartitions * warp_regs(w);
    const int by_regs = sp_left / warp_regs(k) * kSubPartitions / k_warps;
    const long smem_left = (long)sm_smem - (long)(w.sharedSizeBytes + w_dyn + reserved);
    const int by_smem = (int)(smem_left / (long)(k.sharedSizeBytes + k_dyn + reserved));
    const int by_threads = (sm_threads - w_warps * 32) / (k_warps * 32);
    return std::max(0, std::min(std::min(by_regs, by_smem), std::min(by_threads, sm_blocks - 1)));
  };
  const size_t reduce_dyn = bn_bwd_reduce_smem(P, ewy), apply_dyn = bn_bwd_apply_smem(P, ewy);
  for (int x3 = 0; x3 < 2; ++x3) {
    cudaFuncAttributes w, k[3];
    size_t w_dyn = 0;
    int w_threads = 0;
    int rc = lcn_tc_wgrad_footprint(x3 != 0, &w, &w_dyn, &w_threads);
    if (rc) return rc;
    if (x3) {
      LCN_CHECK_CUDA(cudaFuncGetAttributes(&k[0], k_bn_bwd_reduce<lcn_sp16>));
      LCN_CHECK_CUDA(cudaFuncGetAttributes(&k[1], k_bn_bwd_apply<lcn_sp16, false>));
      LCN_CHECK_CUDA(cudaFuncGetAttributes(&k[2], k_bn_bwd_apply<lcn_sp16, true>));
    } else {
      LCN_CHECK_CUDA(cudaFuncGetAttributes(&k[0], k_bn_bwd_reduce<__nv_bfloat16>));
      LCN_CHECK_CUDA(cudaFuncGetAttributes(&k[1], k_bn_bwd_apply<__nv_bfloat16, false>));
      LCN_CHECK_CUDA(cudaFuncGetAttributes(&k[2], k_bn_bwd_apply<__nv_bfloat16, true>));
    }
    for (int i = 0; i < 3; ++i) blocks_out[3 * x3 + i] = fit(w, w_dyn, w_threads, k[i], i == 0 ? reduce_dyn : apply_dyn);
  }
  return LCN_OK;
}

template <typename T>
static int layer_gemm_impl(const lcn_model* m, const float* params, char* ws, const WsLayout& lay, int l,
                           int transposed, cudaStream_t st) {
  float* part = reinterpret_cast<float*>(ws + lay.off_part);
  const T* Ain = reinterpret_cast<const T*>(transposed ? ws + lay.off_dz : a_buf(ws, lay, l - 1));
  T* Y = reinterpret_cast<T*>(transposed ? ws + lay.off_d + 2 * lay.d_stride : z_buf(ws, lay, l));
  const MidWeights w = mid_weights(m, ws, lay, l, transposed);
  return lcn_tc_gemm(m, lay, l - 1, transposed, reinterpret_cast<const __nv_bfloat16*>(Ain), w.hi,
                     transposed ? nullptr : params + m->L[l].b_off, nullptr, reinterpret_cast<__nv_bfloat16*>(Y),
                     transposed ? nullptr : part, st, nullptr, nullptr, w.lo);
}
int lcn_launch_layer_gemm(const lcn_model* m, const float* params, char* ws, const WsLayout& lay, int layer,
                          int transposed, cudaStream_t st) {
  return m->d.path == LCN_PATH_BF16 ? layer_gemm_impl<__nv_bfloat16>(m, params, ws, lay, layer, transposed, st)
                                    : layer_gemm_impl<lcn_sp16>(m, params, ws, lay, layer, transposed, st);
}

// ------------------------------------------------------------------------------------------------
// parity taps
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_read_rows(const T* __restrict__ src, float* __restrict__ dst, int64_t n_logical, int P,
                            int bn_group, int gstride) {
  lcn_pdl_prologue();
  int64_t n = n_logical * P;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t lr = e / P;
    int c = (int)(e - lr * P);
    int64_t pr = (lr / bn_group) * gstride + lr % bn_group;
    dst[e] = lcn_ld(src, lcn_off<T>(pr, c, P));
  }
}
// inverse of k_read_rows: dense fp32 rows -> the activation layout of the path (padding rows of a group stay untouched)
template <typename T>
__global__ void k_write_rows(const float* __restrict__ src, T* __restrict__ dst, int64_t n_logical, int P, int bn_group,
                             int gstride) {
  lcn_pdl_prologue();
  int64_t n = n_logical * P;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t lr = e / P;
    int c = (int)(e - lr * P);
    int64_t pr = (lr / bn_group) * gstride + lr % bn_group;
    lcn_st(dst, lcn_off<T>(pr, c, P), src[e]);
  }
}
int lcn_launch_write_tensor(const lcn_model* m, char* ws, const WsLayout& lay, int layer, const float* src,
                            cudaStream_t st) {
  LCN_REQUIRE(lay.training, "activation injection needs a training-mode workspace layout");
  LCN_REQUIRE(layer >= 0 && layer < m->n_bn, "layer %d out of range", layer);
  const int64_t n_logical = (int64_t)lay.n_groups * lay.bn_group;
  char* dst = a_buf(ws, lay, layer);
  LCN_CHECK_CUDA(cudaMemsetAsync(dst, 0, lay.a_stride, st));
  if (m->d.path == LCN_PATH_BF16)
    lcn_launch(k_write_rows<__nv_bfloat16>, dim3(256), dim3(256), 0, st, src, reinterpret_cast<__nv_bfloat16*>(dst), n_logical, m->P, lay.bn_group, lay.gstride);
  else
    lcn_launch(k_write_rows<lcn_sp16>, dim3(256), dim3(256), 0, st, src, reinterpret_cast<lcn_sp16*>(dst), n_logical, m->P, lay.bn_group, lay.gstride);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}
__global__ void k_unpack_mid(const float* __restrict__ wp32, PairTable pt, int nnz, int F, int FC,
                             float* __restrict__ dst) {
  lcn_pdl_prologue();
  int P = LCN_J * F;
  int sb = blockIdx.x;
  int p = sb / (FC * FC), hi = (sb / FC) % FC, ho = sb % FC;
  int i = pt.pi[p], j = pt.pj[p];
  for (int e = threadIdx.x; e < 4096; e += blockDim.x) {
    int fi = e >> 6, fo = e & 63;
    dst[(size_t)(i * F + hi * 64 + fi) * P + j * F + ho * 64 + fo] = wp32[(size_t)sb * 4096 + e];
  }
}

int lcn_launch_read_tensor(const lcn_model* m, char* ws, const WsLayout& lay, int kind, int layer, float* dst,
                           cudaStream_t st) {
  const int P = m->P, F = m->d.F;
  int64_t n_logical = (int64_t)lay.n_groups * lay.bn_group;
  bool bf = m->d.path == LCN_PATH_BF16;
  if (kind == 0 || kind == 1 || kind == 6) {
    LCN_REQUIRE(lay.training, "activation taps need a training-mode workspace layout");
    LCN_REQUIRE(layer >= 0 && layer < m->n_bn, "layer %d out of range", layer);
    const char* src = kind == 0 ? z_buf(ws, lay, layer) : kind == 1 ? a_buf(ws, lay, layer) : ws + lay.off_dz;
    if (bf) lcn_launch(k_read_rows<__nv_bfloat16>, dim3(256), dim3(256), 0, st, reinterpret_cast<const __nv_bfloat16*>(src), dst, n_logical, P, lay.bn_group, lay.gstride);
    else lcn_launch(k_read_rows<lcn_sp16>, dim3(256), dim3(256), 0, st, reinterpret_cast<const lcn_sp16*>(src), dst, n_logical, P, lay.bn_group, lay.gstride);
  } else if (kind == 2) {
    LCN_REQUIRE(layer >= 0 && layer < m->n_lin, "layer %d out of range", layer);
    const LayerInfo& L = m->L[layer];
    if (layer == 0 || layer == m->n_lin - 1) {
      LCN_CHECK_CUDA(cudaMemcpyAsync(dst, ws + (layer == 0 ? lay.off_wm_first : lay.off_wm_last),
                                     sizeof(float) * L.Kin * L.Kout, cudaMemcpyDeviceToDevice, st));
    } else {
      LCN_REQUIRE(!bf, "the mid-layer weight tap needs the fp32-parity path (LCN_PATH_FP32 keeps an fp32 copy of the packed blocks)");
      LCN_CHECK_CUDA(cudaMemsetAsync(dst, 0, sizeof(float) * P * P, st));
      const float* wp = reinterpret_cast<const float*>(ws + lay.off_wp32) + (size_t)(layer - 1) * m->nnz * m->FC * m->FC * 4096;
      lcn_launch(k_unpack_mid, dim3(m->nnz * m->FC * m->FC), dim3(256), 0, st, wp, make_pairs(m), m->nnz, F, m->FC, dst);
    }
  } else if (kind == 3) {
    LCN_CHECK_CUDA(cudaMemcpyAsync(dst, ws + lay.off_mask, sizeof(float) * LCN_J * LCN_J, cudaMemcpyDeviceToDevice, st));
  } else if (kind == 4 || kind == 5) {
    LCN_REQUIRE(layer >= 0 && layer < m->n_bn, "layer %d out of range", layer);
    const float* stat = bn_stat(ws, lay, m, layer);
    LCN_CHECK_CUDA(cudaMemcpy2DAsync(dst, sizeof(float), stat + (kind == 5 ? 1 : 0), 2 * sizeof(float), sizeof(float),
                                     (size_t)lay.n_groups * F, cudaMemcpyDeviceToDevice, st));
  } else {
    lcn_set_error("unknown tensor kind %d", kind);
    return LCN_EINVAL;
  }
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

// dropout keep decisions, exactly as k_bn_act draws them
__global__ void k_dropout_mask(uint64_t seed, uint64_t step, int layer, int64_t n8, float rate, uint8_t* keep) {
  lcn_pdl_prologue();
  const uint32_t thr16 = lcn_keep_thr16(rate);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t kb = lcn_keep8(seed, step, (uint32_t)layer, (uint64_t)i, thr16);
    for (int q = 0; q < 8; ++q) keep[i * 8 + q] = (uint8_t)((kb >> q) & 1u);
  }
}
extern "C" int lcn_dropout_mask(uint64_t seed, uint64_t step, int layer, int64_t rows, int32_t cols, float rate,
                                uint8_t* d_keep, void* stream) {
  LCN_REQUIRE(cols % 8 == 0, "cols must be a multiple of 8");
  lcn_launch(k_dropout_mask, dim3(256), dim3(256), 0, (cudaStream_t)stream, seed, step, layer, rows * cols / 8, rate, d_keep);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

LCN_KTRACE_EXPORT(kernels)
