// Internal definitions shared by the liblcn_b200 translation units (not part of the C ABI).
#pragma once
#include <string.h>

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>
#include <string>
#include <vector>

#include "lcn_b200.h"

#define LCN_J 17
#define LCN_TILE 128          // rows per GEMM tile; BN groups are padded to a multiple of this
#define LCN_CH 64             // channel chunk: joint-pair blocks are handled as 64x64 sub-blocks
#define LCN_MAX_LIN 18        // 2 + 2*num_layers, num_layers <= 8
#define LCN_MAX_TENSORS 80
#define LCN_BN_EPS 1e-3f      // Keras BatchNormalization default epsilon (models_att.py:599)
#define LCN_LRELU 0.2f        // tf.nn.leaky_relu default alpha (models_att.py:526)

// Neighbour lists passed to kernels BY VALUE (no device-side plan allocation).
//   by_out: list a = output joint j  -> idx[j][n] = n-th input joint i of j,  blk = pair id of (i,j)
//   by_in : list a = input joint i   -> idx[i][n] = n-th output joint j of i, blk = pair id of (i,j)
// pair id enumerates the support in (i major, j ascending) order.
struct JointLists {
  uint8_t cnt[LCN_J];
  uint8_t idx[LCN_J][LCN_J];
  int16_t blk[LCN_J][LCN_J];
};

struct SupportBits {            // sup[i] bit j set <=> block (i -> j) exists
  uint32_t row[LCN_J];          // outputs of input joint i
  uint32_t col[LCN_J];          // inputs of output joint j
  int16_t pair[LCN_J][LCN_J];   // pair id or -1
};

struct LayerInfo {
  int Fi, Fo, Kin, Kout;
  int64_t w_off, b_off, gamma_off, beta_off;  // offsets into the flat parameter vector (-1: none)
  int has_bn;                                 // BN + LeakyReLU + dropout follow the linear op
  int res_from;                               // activation index added after this layer, or -1
};

enum { SEG_MASK = 0, SEG_W = 1, SEG_B = 2, SEG_BN = 3 };
struct SegInfo {                // one parameter tensor, for the multi-tensor Adam kernel
  int64_t off, size;
  int32_t kind, layer;
  int32_t chunk_start;          // first Adam chunk (of LCN_ADAM_CHUNK elements) of this tensor
};
#define LCN_ADAM_CHUNK 4096
struct SegTable {
  int n;
  int total_chunks;
  SegInfo s[LCN_MAX_TENSORS];
};

struct TensorMeta {
  std::string name;
  int64_t off;
  int rows, cols;
};

// Side streams of the model.  The weight-gradient GEMM of layer l is off the critical path of the backward pass
// (dZ_l -> dgrad_l -> BN backward of l-1 -> ...), so it is enqueued on a stream owned by the model and joined with
// events (plain fork/join, capturable into the caller's CUDA graph); the weight preparation packs the edge layers
// there too.  Created on first use (lcn_kernels.cu); `mu` serialises the enqueue of concurrent calls on the same model
// (the events are shared).
struct LcnAux {
  std::mutex mu;
  bool ready = false;
  cudaStream_t st = nullptr;
  cudaStream_t xst = nullptr;        // data-parallel exchange of finished weight gradients (lcn_dp.cu), forked from `st`
  cudaEvent_t ev_xdone = nullptr;
  cudaEvent_t ev_go = nullptr, ev_done = nullptr, ev_ms = nullptr, ev_loss = nullptr;
  cudaEvent_t ev_dz[2] = {nullptr, nullptr}, ev_wg[2] = {nullptr, nullptr};
};

void lcn_aux_release(LcnAux& a);   // destroys the streams and events created so far

struct LcnDp;                      // data-parallel exchange buffers mapped across the ranks (lcn_dp.cu); null: single process

struct lcn_model {
  mutable LcnAux aux;
  LcnDp* dp = nullptr;
  lcn_model_desc d;
  int n_lin, n_bn, P, FC, nnz;
  JointLists by_out, by_in;
  SupportBits sup;
  LayerInfo L[LCN_MAX_LIN];
  SegTable segs;
  std::vector<TensorMeta> tensors;
  int64_t n_params, mask_off;
  int sm_count;
};

// Per-layer device scalars (live in the workspace)
struct LayerScalars {
  double norm2;      // ||W||_F^2 of the current weights
  double sdot;       // <dWc, W>
  float inv_norm;    // 1/max(||W||,1)   (1 if !max_norm)
  float coef;        // sdot/||W||^3 if ||W|| > 1 else 0
  float clipped;     // 1 if ||W|| > 1
  float pad;
};

// Workspace layout, a pure function of (model, n_rows, bn_group, training).
struct WsLayout {
  int64_t n_rows, rows_pad;
  int bn_group, gstride, n_groups, tiles, tiles_per_group, training;
  size_t es;                         // activation storage element size
  size_t off_scalars;                // LayerScalars[LCN_MAX_LIN]
  size_t off_mask;                   // float[289] mask values
  size_t off_pairdot;                // float[n_lin][289]  <dWm, W> per support pair
  size_t off_loss;                   // double[2]
  size_t off_wm_first, off_wm_last;  // dense masked fp32 effective weights of the edge layers
  size_t off_wp32;                   // fp32 packed mid-layer blocks  [mid][pair][FC][FC][64][64]
  size_t off_wp16f, off_wp16b;       // bf16 UMMA-layout packed blocks (forward / transposed)
  size_t off_wp16f_lo, off_wp16b_lo; // their lo parts (split-bf16 path only)
  size_t off_wl16f, off_wl16b;       // bf16 packed last-layer weights: per K chunk [64 n][64 k] / per N chunk
  size_t off_wf16;                   // bf16 packed first-layer weights: per N chunk [64 n][64 k (17*in_F used)]
  size_t off_x16, off_dout16;        // bf16 tiles of the 2D input / of dOut (64-column padded), training
  size_t off_dw_first, off_dw_last;  // fp32 padded weight-gradient scratch of the edge layers
  size_t off_part;                   // float[tiles][P][2] BN partials (mean, M2)
  size_t off_bnstat;                 // float[n_bn][n_groups][F][2]  (mean, rstd)
  size_t off_bnsum;                  // float[n_bn][F][2]  backward sums (sum dy, sum dy*xhat)
  size_t off_gacc, gacc_stride;      // per BN layer: double[LCN_GACC_REP][F][2] (sum x, sum x^2) + grid-barrier counter (training)
  size_t off_out;                    // float[rows_pad][51] copy of the prediction (training)
  size_t off_dout;                   // float[rows_pad][51]
  size_t off_z, z_stride; int n_z;   // Z buffers
  size_t off_a, a_stride; int n_a;   // A buffers
  size_t off_d, d_stride; int n_d;   // gradient ping-pong buffers (training)
  size_t off_dz;                     // dZ buffers (training): layer l uses buffer l & 1 (wgrad of l overlaps BN backward of l-1)
  size_t off_dbpart;                 // float[n_bn][2*SMs][P] per-block bias-gradient partial rows (training)
  size_t off_keep;                   // uint8[n_bn][rows_pad][P/8] dropout keep bits (training)
  int fused;                         // inference runs as the fused cluster kernel (lcn_stack_tc.cu)
  size_t off_stack;                  // its per-cluster L2-resident activation scratch
  size_t total;
};

WsLayout lcn_ws_layout(const lcn_model* m, int64_t n_rows, int bn_group, int training);

void lcn_set_error(const char* fmt, ...);
#define LCN_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      lcn_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return LCN_ECUDA;                                                                   \
    }                                                                                     \
  } while (0)
#define LCN_CHECK_LAUNCH() LCN_CHECK_CUDA(cudaGetLastError())

// ---------------------------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  Every kernel of the train / per-layer path starts with lcn_pdl_prologue():
// it lets the NEXT kernel of the stream be scheduled onto SMs as they free up (griddepcontrol.launch_dependents) and
// then waits until the PREVIOUS kernel has completed and flushed its memory (griddepcontrol.wait) before touching
// global memory.  lcn_launch() sets the matching launch attribute.  ~60 short kernels make one train step: this hides
// the per-kernel launch latency and block ramp-up (measured: DESIGN.md section 6).  LCN_DISABLE_PDL=1 turns the
// attribute off (the device-side instructions are then no-ops).
// ---------------------------------------------------------------------------------------------------------------
// -DLCN_KTRACE (profiling build only): block (0,0) of every kernel stamps %globaltimer right after its
// griddepcontrol.wait, i.e. when its predecessor has completed -- the start-to-start distances are the effective
// per-kernel costs of the step as replayed from the CUDA graph (profiles/ktrace_step.py).  One buffer per
// translation unit, read back through lcn_ktrace_read_<tu>().
#ifdef LCN_KTRACE
#define LCN_KTRACE_MAX 8192
static __device__ unsigned long long g_ktrace[2 * LCN_KTRACE_MAX];
static __device__ unsigned g_ktrace_n;
__device__ __forceinline__ void lcn_ktrace_stamp() {
#if defined(__CUDA_ARCH__)
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0 && threadIdx.y == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    unsigned i = atomicAdd(&g_ktrace_n, 1u);
    if (i < LCN_KTRACE_MAX) {
      g_ktrace[2 * i] = t;
      g_ktrace[2 * i + 1] = ((unsigned long long)gridDim.x << 32) | ((unsigned long long)gridDim.y << 20) |
                            ((unsigned long long)blockDim.x << 8) | (unsigned long long)blockDim.y;
    }
  }
#endif
}
#define LCN_KTRACE_EXPORT(tu)                                                                        \
  extern "C" int lcn_ktrace_read_##tu(unsigned long long* h_out, unsigned* h_n, int reset) {        \
    cudaDeviceSynchronize();                                                                         \
    if (cudaMemcpyFromSymbol(h_n, g_ktrace_n, sizeof(unsigned)) != cudaSuccess) return -2;           \
    if (cudaMemcpyFromSymbol(h_out, g_ktrace, sizeof(g_ktrace)) != cudaSuccess) return -2;           \
    if (reset) {                                                                                     \
      unsigned z = 0;                                                                                \
      cudaMemcpyToSymbol(g_ktrace_n, &z, sizeof(z));                                                 \
    }                                                                                                \
    return 0;                                                                                        \
  }
#else
__device__ __forceinline__ void lcn_ktrace_stamp() {}
#define LCN_KTRACE_EXPORT(tu)
#endif
__device__ __forceinline__ void lcn_pdl_prologue() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
  lcn_ktrace_stamp();
}
// split form: trigger at kernel start, wait after the kernel's own setup (barrier init, TMEM allocation)
__device__ __forceinline__ void lcn_pdl_trigger() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
__device__ __forceinline__ void lcn_pdl_wait() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
  lcn_ktrace_stamp();
}
bool lcn_pdl_enabled();
// LCN_TRACE=1 (profiling scripts only, eager launches): CUDA events around every lcn_launch; lcn_debug_trace_dump()
// prints the in-stream duration of each kernel by name (warm caches, unlike an ncu launch list).
bool lcn_trace_enabled();
void lcn_trace_mark(const void* func, cudaStream_t st, int end);
template <typename... KArgs, typename... Args>
static inline void lcn_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = lcn_pdl_enabled() ? 1 : 0;
  const bool trace = lcn_trace_enabled();
  if (trace) lcn_trace_mark(reinterpret_cast<const void*>(kernel), st, 0);
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // errors surface through LCN_CHECK_LAUNCH
  if (trace) lcn_trace_mark(reinterpret_cast<const void*>(kernel), st, 1);
}
#define LCN_REQUIRE(cond, ...)   \
  do {                           \
    if (!(cond)) {               \
      lcn_set_error(__VA_ARGS__); \
      return LCN_EINVAL;         \
    }                            \
  } while (0)

// ---- data-parallel exchange (lcn_dp.cu) ----
int lcn_dp_mode(const lcn_model* m);      // 0: no exchange; 1: streamed behind the weight-gradient GEMMs; 2: one exchange at the end
int lcn_dp_exchange_units(const lcn_model* m, float* graw, int u0, int u1, int s0, int s1, int max_ctas, cudaStream_t st);
int lcn_dp_wait(const lcn_model* m, cudaStream_t st);
void lcn_dp_destroy(lcn_model* m);
// synchronised BatchNorm (lcn_dp_sync_batch_norm): the source of a sync point's local moments
#define LCN_BN_SYNC_GACC 0      // forward, double[LCN_GACC_REP][F][2] (sum x, sum x^2) of the tensor-core GEMM
#define LCN_BN_SYNC_MOMENTS 1   // forward, double[F][3] (n, mean, M2) of k_bn_finalize
#define LCN_BN_SYNC_SUMS 2      // backward, float[F][2] (sum dy, sum dy*xhat) of k_bn_bwd_reduce
bool lcn_bn_sync_on(const lcn_model* m);
int lcn_bn_sync(const lcn_model* m, int point, int kind, const void* src, float* out, int64_t rows, cudaStream_t st);

// ---- launch wrappers implemented in the kernel translation units ----
struct FwdArgs {                 // one call of the forward pass
  const lcn_model* m;
  const float* params;
  char* ws;
  WsLayout lay;
  const float* x;
  float* out;
  float dropout_rate;
  uint64_t seed, step;
  const lcn_step_scalars* dyn;   // device-resident step scalars (overrides `step` when not null)
  cudaStream_t st;
  int layer_begin = 0, layer_end = -1;   // linear layers [begin, end) to run; end < 0: all (lcn_model_forward_layers)
};

int lcn_launch_prepare(const lcn_model* m, const float* params, char* ws, const WsLayout& lay,
                       bool recompute_norm, cudaStream_t st);
int lcn_launch_forward(const FwdArgs& a);
int lcn_launch_backward(const lcn_model* m, const float* params, char* ws, const WsLayout& lay,
                        const float* x, const float* labels, float dropout_rate, uint64_t seed,
                        uint64_t step, float* loss, float* grads_raw, cudaStream_t st);
int lcn_launch_grad_finalize(const lcn_model* m, const float* params, char* ws, const WsLayout& lay,
                             const float* grads_raw, float* grads_out, cudaStream_t st);
int lcn_launch_adam(const lcn_model* m, float* params, float* mm, float* vv, char* ws, const WsLayout& lay,
                    const float* grads_raw, float lr_t, float b1, float b2, float eps, float reg,
                    const lcn_step_scalars* dyn, cudaStream_t st);
int64_t lcn_grad_compact_count(const lcn_model* m);
int lcn_launch_grad_compact(const lcn_model* m, float* graw, float* compact, bool unpack, cudaStream_t st);
int lcn_launch_dp_exchange(const lcn_model* m, float* const* buckets, float* const* stage_at, float* const* stage_local,
                           unsigned long long* pushed_local, unsigned long long* const* pushed_at,
                           unsigned long long* const* done_at, unsigned long long* epoch, unsigned int* ticket, int rank,
                           int world, int u0, int u1, int s0, int s1, int max_ctas, cudaStream_t st);
int lcn_launch_layer_gemm(const lcn_model* m, const float* params, char* ws, const WsLayout& lay, int layer,
                          int transposed, cudaStream_t st);
int lcn_launch_read_tensor(const lcn_model* m, char* ws, const WsLayout& lay, int kind, int layer,
                           float* dst, cudaStream_t st);
int lcn_launch_write_tensor(const lcn_model* m, char* ws, const WsLayout& lay, int layer, const float* src,
                            cudaStream_t st);

// BatchNorm statistics of the forward tensor-core GEMM without a second launch (one BatchNorm group): every CTA adds
// its per-channel (sum x, sum x^2) to fp64 accumulators (LCN_GACC_REP replicas indexed by row tile spread the atomics),
// and k_bn_act_pre derives (mean, rstd) from them in its prologue -- k_bn_finalize is not launched for the layer.
#define LCN_GACC_REP 8
struct TcFuse {
  double* gacc;                      // [LCN_GACC_REP][F][2], zeroed by the caller once per forward pass
  int F;
};
// tcgen05 (bf16) mid-layer kernels, lcn_gemm_tc.cu.  transposed=0: Y = A*Wm (+bias, BN partials);
// transposed=1: dA = dZ*Wm^T (+addend).  fuse != nullptr (forward, one BatchNorm group): *fused = 1 if the statistics
// went to fuse->gacc (the caller skips k_bn_finalize and hands gacc to k_bn_act_pre), 0: per-tile partials as usual.
// x3: split-bf16 operands (A / addend / Y are lcn_sp16 buffers, wpacked_lo holds the lo parts of the packed weights):
// three tensor-core products per block, fp32-parity results.
int lcn_tc_gemm(const lcn_model* m, const WsLayout& lay, int mid_index, int transposed,
                const __nv_bfloat16* A, const char* wpacked, const float* bias, const __nv_bfloat16* addend,
                __nv_bfloat16* Y, float* part, cudaStream_t st, const TcFuse* fuse = nullptr, int* fused = nullptr,
                const char* wpacked_lo = nullptr);
int lcn_tc_wgrad(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* A, const __nv_bfloat16* dZ,
                 float* dW /* dense [P,P] */, cudaStream_t st, bool x3 = false);
int lcn_tc_head(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* A, const char* wpacked,
                const float* bias, const float* x, float* out_user, float* out_ws, cudaStream_t st);
int lcn_tc_head_dgrad(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* dOut16, const char* wpacked,
                      __nv_bfloat16* dA, cudaStream_t st);
int lcn_tc_wgrad_last(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* A, const __nv_bfloat16* dOut16,
                      float* dWpad, cudaStream_t st);
int lcn_tc_wgrad_first(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* X16, const __nv_bfloat16* dZ,
                       float* dWpad, cudaStream_t st);

// fused whole-stack inference kernel (lcn_stack_tc.cu): one thread-block cluster per BatchNorm group
bool lcn_stack_eligible(const lcn_model* m, int bn_group, int training);
size_t lcn_stack_scratch_bytes(const lcn_model* m, int bn_group);
int lcn_stack_forward(const lcn_model* m, const WsLayout& lay, const float* params, char* ws, const float* x,
                      float* out, void* taps /* nullable */, cudaStream_t st);

// ---- device helpers ----
__device__ __forceinline__ float lcn_ld(const float* p, size_t i) { return p[i]; }
__device__ __forceinline__ float lcn_ld(const __nv_bfloat16* p, size_t i) { return __bfloat162float(p[i]); }
__device__ __forceinline__ void lcn_st(float* p, size_t i, float v) { p[i] = v; }
__device__ __forceinline__ void lcn_st(__nv_bfloat16* p, size_t i, float v) { p[i] = __float2bfloat16_rn(v); }

// Activation layouts in HBM.
//  fp32 path: row-major [rows_pad][P].
//  bf16 path: tile-major, each (128-row tile, 64-channel chunk) is ONE contiguous 16 KB block holding the
//  UMMA SWIZZLE_128B image of the tile (row r at r*128 B, 16-byte chunk c stored at c ^ (r & 7)).  A tile
//  therefore moves HBM<->smem with a single 1-D bulk TMA copy and is directly a K-major A operand
//  (forward / dgrad) or an MN-major operand with K = rows (wgrad) of tcgen05.mma.
// `col` multiples of 4 keep 4 consecutive elements contiguous in both layouts.
template <typename T>
__device__ __forceinline__ size_t lcn_off(int64_t row, int col, int P);
template <>
__device__ __forceinline__ size_t lcn_off<float>(int64_t row, int col, int P) {
  return (size_t)row * P + col;
}
template <>
__device__ __forceinline__ size_t lcn_off<__nv_bfloat16>(int64_t row, int col, int P) {
  int r = (int)(row & 127), k = col & 63;
  size_t tile = (size_t)(row >> 7) * (P >> 6) + (col >> 6);
  return (tile * 128 + r) * 64 + ((((k >> 3) ^ (r & 7)) << 3) | (k & 7));
}

// Split-bf16 storage of an fp32 value: v ~ hi + lo with hi = bf16(v), lo = bf16(v - hi) (16 significand bits, relative
// error <= 2^-17).  This is the activation type of the fp32-PARITY tensor-core path (LCN_PATH_FP32): a product
// a * w is formed on the tensor cores as a_hi*w_hi + a_hi*w_lo + a_lo*w_hi with fp32 accumulation in TMEM (the dropped
// lo*lo term is <= 2^-18 relative), which holds the 1e-4 per-layer tolerance of the north_star with two orders of
// magnitude to spare (measured: DESIGN.md section 4.5) where single-pass TF32 (10-bit mantissa) does not.
// Layout: the bf16 tile-major layout with the hi and lo planes of each (128-row tile, 64-channel chunk) block stored
// back to back (hi block at 2b, lo block at 2b+1): a GEMM operand tile is still ONE contiguous bulk copy (32 KB), and
// an element's lo part sits 8192 elements behind its hi part.  The type is a tag: pointers to it index bf16 elements.
struct lcn_sp16 {
  __nv_bfloat16 h;
};
#define LCN_SP_LO 8192        // element distance from the hi part to the lo part
template <>
__device__ __forceinline__ size_t lcn_off<lcn_sp16>(int64_t row, int col, int P) {
  int r = (int)(row & 127), k = col & 63;
  size_t tile = ((size_t)(row >> 7) * (P >> 6) + (col >> 6)) * 2;
  return (tile * 128 + r) * 64 + ((((k >> 3) ^ (r & 7)) << 3) | (k & 7));
}
__device__ __forceinline__ void lcn_sp_split(float v, __nv_bfloat16& h, __nv_bfloat16& l) {
  h = __float2bfloat16_rn(v);
  l = __float2bfloat16_rn(v - __bfloat162float(h));
}
__device__ __forceinline__ float lcn_ld(const lcn_sp16* p, size_t i) {
  const __nv_bfloat16* q = reinterpret_cast<const __nv_bfloat16*>(p);
  return __bfloat162float(q[i]) + __bfloat162float(q[i + LCN_SP_LO]);
}
__device__ __forceinline__ void lcn_st(lcn_sp16* p, size_t i, float v) {
  __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p);
  lcn_sp_split(v, q[i], q[i + LCN_SP_LO]);
}

// 4-wide vector access (16 B for fp32, 8 B for bf16); i is the element index, multiple of 4
__device__ __forceinline__ float4 lcn_ld4(const float* p, size_t i) {
  return *reinterpret_cast<const float4*>(p + i);
}
__device__ __forceinline__ float4 lcn_ld4(const __nv_bfloat16* p, size_t i) {
  uint2 u = *reinterpret_cast<const uint2*>(p + i);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&u.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&u.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void lcn_st4(float* p, size_t i, float4 v) {
  *reinterpret_cast<float4*>(p + i) = v;
}
__device__ __forceinline__ void lcn_st4(__nv_bfloat16* p, size_t i, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
  __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<uint32_t*>(&a);
  u.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p + i) = u;
}

__device__ __forceinline__ float4 lcn_ld4(const lcn_sp16* p, size_t i) {
  const __nv_bfloat16* q = reinterpret_cast<const __nv_bfloat16*>(p);
  float4 a = lcn_ld4(q, i), b = lcn_ld4(q, i + LCN_SP_LO);
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ void lcn_st4(lcn_sp16* p, size_t i, float4 v) {
  __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p);
  __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
  float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
  __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2bfloat162_rn(v.z - f1.x, v.w - f1.y);
  uint2 uh, ul;
  uh.x = *reinterpret_cast<uint32_t*>(&h0); uh.y = *reinterpret_cast<uint32_t*>(&h1);
  ul.x = *reinterpret_cast<uint32_t*>(&l0); ul.y = *reinterpret_cast<uint32_t*>(&l1);
  *reinterpret_cast<uint2*>(q + i) = uh;
  *reinterpret_cast<uint2*>(q + i + LCN_SP_LO) = ul;
}

// 4-wide access into float arrays
template <typename T>
__device__ __forceinline__ void lcn_ldv4(const T* p, size_t i, float v[4]) {
  float4 a = lcn_ld4(p, i);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
template <typename T>
__device__ __forceinline__ void lcn_stv4(T* p, size_t i, const float v[4]) {
  lcn_st4(p, i, make_float4(v[0], v[1], v[2], v[3]));
}
// 8-wide vector access (2 x 16 B for fp32, 16 B for bf16); element offset multiple of 8
__device__ __forceinline__ void lcn_ld8(const float* p, size_t i, float v[8]) {
  float4 a = *reinterpret_cast<const float4*>(p + i), b = *reinterpret_cast<const float4*>(p + i + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void lcn_ld8(const __nv_bfloat16* p, size_t i, float v[8]) {
  uint4 u = *reinterpret_cast<const uint4*>(p + i);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    float2 t = __bfloat1622float2(h[e]);
    v[2 * e] = t.x;
    v[2 * e + 1] = t.y;
  }
}
__device__ __forceinline__ void lcn_st8(float* p, size_t i, const float v[8]) {
  *reinterpret_cast<float4*>(p + i) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + i + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void lcn_st8(__nv_bfloat16* p, size_t i, const float v[8]) {
  uint4 u;
  __nv_bfloat162 b0 = __floats2bfloat162_rn(v[0], v[1]), b1 = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 b2 = __floats2bfloat162_rn(v[4], v[5]), b3 = __floats2bfloat162_rn(v[6], v[7]);
  u.x = *reinterpret_cast<uint32_t*>(&b0);
  u.y = *reinterpret_cast<uint32_t*>(&b1);
  u.z = *reinterpret_cast<uint32_t*>(&b2);
  u.w = *reinterpret_cast<uint32_t*>(&b3);
  *reinterpret_cast<uint4*>(p + i) = u;
}

__device__ __forceinline__ void lcn_ld8(const lcn_sp16* p, size_t i, float v[8]) {
  const __nv_bfloat16* q = reinterpret_cast<const __nv_bfloat16*>(p);
  float lo[8];
  lcn_ld8(q, i, v);
  lcn_ld8(q, i + LCN_SP_LO, lo);
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] += lo[e];
}
__device__ __forceinline__ void lcn_st8(lcn_sp16* p, size_t i, const float v[8]) {
  __nv_bfloat16* q = reinterpret_cast<__nv_bfloat16*>(p);
  uint4 uh, ul;
  uint32_t* ph = reinterpret_cast<uint32_t*>(&uh);
  uint32_t* pl = reinterpret_cast<uint32_t*>(&ul);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
    float2 f = __bfloat1622float2(h);
    __nv_bfloat162 l = __floats2bfloat162_rn(v[2 * e] - f.x, v[2 * e + 1] - f.y);
    ph[e] = *reinterpret_cast<uint32_t*>(&h);
    pl[e] = *reinterpret_cast<uint32_t*>(&l);
  }
  *reinterpret_cast<uint4*>(q + i) = uh;
  *reinterpret_cast<uint4*>(q + i + LCN_SP_LO) = ul;
}

// Philox4x32-10 counter-based generator; one call yields 128 random bits (lcn_keep8: the keep bits of 8 elements).
__device__ __host__ __forceinline__ void lcn_philox4(uint64_t seed, uint64_t step, uint32_t layer, uint64_t idx4,
                                                     uint32_t out[4]) {
  uint32_t c0 = (uint32_t)idx4, c1 = (uint32_t)(idx4 >> 32), c2 = layer, c3 = (uint32_t)step;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ (uint32_t)(step >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// keep decisions of tf.nn.dropout (u >= rate) for the 8 consecutive elements 8*idx8 .. 8*idx8+7: ONE Philox call,
// 16 random bits per element (u = bits / 65536, rate rounded up to a multiple of 2^-16: exact for 0.25 / 0.5);
// bit q of the result = element q kept.  Halves the integer work of the activation kernels, which were bound by
// the instruction count of two Philox calls per 8 elements.
__device__ __host__ __forceinline__ uint32_t lcn_keep_thr16(float rate) {
  float t = rate * 65536.0f;
  uint32_t u = (uint32_t)t;
  if ((float)u < t) ++u;
  return u > 65536u ? 65536u : u;
}
__device__ __host__ __forceinline__ uint32_t lcn_keep8(uint64_t seed, uint64_t step, uint32_t layer, uint64_t idx8,
                                                       uint32_t thr16) {
  uint32_t rb[4];
  lcn_philox4(seed, step, layer, idx8, rb);
  uint32_t kb = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) kb |= ((((rb[q >> 1] >> (16 * (q & 1))) & 0xffffu) >= thr16) ? 1u : 0u) << q;
  return kb;
}
