// Tensor-core kernels of the LCN layers for sm_100a: tcgen05.mma with TMEM accumulators, operands staged by
// 1-D bulk TMA (cp.async.bulk) through mbarrier pipelines.  Two instantiations each: bf16 operands (LCN_PATH_BF16), and
// split-bf16 operands -- (hi, lo) planes, three products per block -- for the fp32-parity path (LCN_PATH_FP32, X3).
//
//   k_tc_gemm  : Y[128-row tile, group of <=6 output chunks] = sum over the input chunks that have a nonzero 64x64
//                block into the group of  A[tile, chunk] (128x64, K-major SW128)  x  Wp(panel of present blocks) --
//                all-zero joint-pair blocks of the mask are never loaded nor multiplied (network/models_att.py:576-586
//                multiplies them densely).  Forward: + bias, BatchNorm statistics per column (models_att.py:588-612;
//                fp64 atomics or per-tile (mean, M2) partials); transposed (dgrad): + residual gradient addend; head
//                mode: the last layer with the xy skip (models_att.py:765-773).
//   k_tc_wgrad : dWm block(i,j) = A[:, i]^T dZ[:, j] for the nonzero blocks only, K = batch rows, both operands MN-major
//                straight out of the tile-major activation layout, M = 128 from pairs of input chunks.
//
// Data layout contracts: activations are tile-major SW128 (lcn_internal.cuh, lcn_off<bf16>), packed weights are
// per-64x64-block SW128 K-major images written by k_pack_mid (lcn_kernels.cu) in the order the panels are consumed, so
// every operand is one contiguous bulk copy -- no tensor maps needed.
//
// Warp roles of k_tc_gemm (352 threads): warp 0 = TMA producer, warps 1-2 = MMA issuers (even / odd iterations; warp 1
// also owns the TMEM allocation), warps 3-10 = epilogue in two teams of four (TMEM -> registers -> swizzled smem tile ->
// bulk store, BatchNorm sums).  k_tc_wgrad (224 threads): producer, two MMA issuers, four epilogue warps.  A kernel
// that allocates TMEM gets ONE resident CTA per SM (cudaOccupancyMaxActiveBlocksPerMultiprocessor reports 1 for any
// kernel containing tcgen05.alloc, profiles/micro/occ.cu), so grids are sized as single waves of <= SM-count CTAs and a
// CTA may use the whole shared memory and all 512 TMEM columns.  What bounds these kernels: DESIGN.md section 4.1.
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <type_traits>
#include <vector>

#include "lcn_internal.cuh"

#define TC_G 4                      // wgrad: max output chunks per unit
#define TC_GMAX 6                   // forward / dgrad: max N-side chunks (of 64 columns) per CTA -> <= 384 of 512 TMEM columns
#define TC_A_BYTES 16384            // 128 rows x 64 bf16
#define TC_B_BYTES 8192             // one 64x64 bf16 block
#define TC_EPI_WARPS 8              // epilogue warps of k_tc_gemm: two per TMEM lane quarter (32 columns of a chunk each)
// Geometry of the two instantiations of k_tc_gemm.  X3 = split-bf16 operands (lcn_sp16, lcn_internal.cuh): every A tile
// and every weight block comes as a (hi, lo) pair and each block costs three MMAs (hi*hi + hi*lo + lo*hi).
template <bool X3>
struct TcGeo {
  static constexpr int PL = X3 ? 2 : 1;                  // planes per operand tile
  static constexpr int A_UNITS = 2 * PL;                 // ring units (8 KB) of the A operand of one iteration
  static constexpr int RING_UNITS = X3 ? 19 : 23;        // operand ring: one K-chunk iteration takes A_UNITS + PL * #blocks units
  static constexpr int RING_BYTES = RING_UNITS * TC_B_BYTES;
  static constexpr int STAGE_BYTES = PL * TC_A_BYTES;    // output staging per epilogue team
  static constexpr int SMEM_BYTES = 1024 + RING_BYTES + 2 * STAGE_BYTES + TC_EPI_WARPS * 64 * 2 * 4;   // + BN partial scratch
};
#define TC_THREADS 192              // wgrad kernel
#define TC_MMA_WARPS 2               // MMA-issuing warps of k_tc_gemm (iteration it is issued by warp it % 2)
#define TC_EPI_T0 (32 + 32 * TC_MMA_WARPS)                  // first epilogue thread
#define TC_GEMM_THREADS (TC_EPI_T0 + 32 * TC_EPI_WARPS)
#define TC_MAX_CHUNKS 34            // 17 joints x (F/64 <= 2) chunks on either side

// optional per-CTA timeline (clock64) for block (0,0): enabled with -DLCN_TC_PROFILE
#ifdef LCN_TC_PROFILE
__device__ unsigned long long g_tc_prof[512];
#define TC_STAMP(i) do { if (blockIdx.x == 0 && blockIdx.y == 0) g_tc_prof[(i)] = clock64(); } while (0)
extern "C" int lcn_debug_read_prof(unsigned long long* h_out) {
  return cudaMemcpyFromSymbol(h_out, g_tc_prof, sizeof(g_tc_prof)) == cudaSuccess ? 0 : -2;
}
#else
#define TC_STAMP(i) do {} while (0)
#endif

enum { TC_MODE_FWD = 0, TC_MODE_DGRAD = 1, TC_MODE_HEAD = 2 };

// One entry of a CTA's schedule (built by the host, tc_fill_schedule): the K chunk of iteration `it`, which of the
// group's N-side chunks have a block under it, where the iteration's operands sit in the shared-memory ring, which
// earlier iteration must have been consumed before that ring space may be overwritten, and which accumulators are
// complete once this iteration's MMAs have retired.
#define TC_S_KC(s) ((s) & 63u)
#define TC_S_BITS(s) (((s) >> 6) & 63u)
#define TC_S_OFF(s) (((s) >> 12) & 31u)
#define TC_S_WAIT(s) ((int)(((s) >> 17) & 127u) - 1)
#define TC_S_DONE(s) (((s) >> 24) & 63u)

struct TcParams {
  uint32_t kmask[LCN_J];            // K-side joint -> bitmask of N-side joints with a block
  int FCK, FCN;                     // 64-chunks per joint on the K side / N side
  int NCK, NCN;                     // chunk counts
  int n_groups;                     // N-side chunk groups (grid.x)
  int P;                            // N-side row width in elements (BN partial indexing)
  int bn_group, gstride;
  int mode;                         // TC_MODE_*
  // head mode (last layer): fp32 output [n_rows, 51] + xy skip from the 2D input
  const float* x;
  int in_F;
  int64_t n_rows;
  float* out_user;
  float* out_ws;
  // Per (N-side chunk group, iteration) schedule.  Lives in the kernel parameters (constant bank) so that the producer /
  // MMA warps index it with uniform loads and keep descriptors in uniform registers (a schedule in shared memory forces
  // an R2UR per tcgen05.mma operand: measured 80-100 cycles per MMA).
  uint32_t sched[TC_MAX_CHUNKS][TC_MAX_CHUNKS];
  // the MMAs of the iteration as runs of adjacent present chunks with equal accumulate state (one tcgen05.mma of
  // N = 64 * len per K = 16 step): 6 bits per run = chunk q (3) | len - 1 (2) | accumulate (1), count in bits 60..63.
  // Precomputed so that the single issuing warp spends its instructions on tcgen05.mma, not on bit scans.
  uint64_t runs[TC_MAX_CHUNKS][TC_MAX_CHUNKS];
  uint16_t gslot[TC_MAX_CHUNKS][TC_MAX_CHUNKS];   // [group][K chunk]: slot of the first present block in the packed panel
  uint8_t gnit[TC_MAX_CHUNKS];                    // iterations of the group (K chunks with a block into it)
  uint8_t gwritten[TC_MAX_CHUNKS];
  uint8_t gdcnt[TC_MAX_CHUNKS][TC_GMAX];          // per chunk of the group: MMA warps that issue into it (arrivals on done[q])
  uint8_t gorder[TC_MAX_CHUNKS][TC_GMAX];         // the group's chunks in the order their accumulators complete
  uint8_t goc0[TC_MAX_CHUNKS + 1];  // group g owns N-side chunks [goc0[g], goc0[g+1]): contiguous, balanced by block count
  int fuse_on;                      // forward only: BatchNorm statistics by fp64 atomics into fuse.gacc (no partials, no k_bn_finalize)
  TcFuse fuse;
};

#include "lcn_tc_ptx.cuh"

// ---------------------------------------------------------------------------------------------
// forward / dgrad / head GEMM.
//   Operand pipeline: a ring of 8 KB units in shared memory; iteration `it` (one K chunk) owns 2 + #blocks units and
//   its own pair of single-use mbarriers (full[it]: bulk copies landed, empty[it]: MMAs retired), so there is no phase
//   bookkeeping and the number of iterations in flight adapts to their size (about five for the knn=3 mask instead of
//   three fixed 64 KB stages: the loop is bound by the L2 -> shared-memory copy rate, profiles/micro/bulk_bw2.csv).
//   Two MMA warps: a tcgen05.mma of N = 64..256 executes in 48..128 cycles but costs the issuing warp about as much in
//   barrier polls, descriptor moves to uniform registers and election (profiles/r1/timeline_tc_gemm.log), and the
//   tensor pipe does not queue far ahead, so one issuer leaves it idle half of the time.  Warp 1 issues the even
//   iterations, warp 2 the odd ones; the accumulators are zeroed by the epilogue warps first (tcgen05.st) so every MMA
//   accumulates and the order in which the two warps reach the tensor pipe does not matter.
//   Epilogue overlap: the host orders each group's K chunks so that its N-side chunks complete one after the other
//   (tc_fill_schedule); the MMA warp commits to done[q] right after the last MMA into chunk q and the four epilogue
//   warps convert / store / reduce that chunk while the remaining MMAs run.  Two 16 KB staging tiles alternate.
// ---------------------------------------------------------------------------------------------
template <bool X3>
__global__ void __launch_bounds__(TC_GEMM_THREADS) k_tc_gemm(const __nv_bfloat16* __restrict__ A,
                                                        const __nv_bfloat16* __restrict__ Wp,
                                                        const __nv_bfloat16* __restrict__ Wp_lo,
                                                        const float* __restrict__ bias,
                                                        const __nv_bfloat16* __restrict__ addend,
                                                        __nv_bfloat16* __restrict__ Y, float* __restrict__ part,
                                                        const __grid_constant__ TcParams p) {
  lcn_pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * TC_MAX_CHUNKS + TC_GMAX];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float bias_s[TC_GMAX * 64];

  uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x, tile = blockIdx.y;
  const int oc0 = p.goc0[g], G = p.goc0[g + 1] - oc0;
  const int n_it = p.gnit[g];
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[TC_MAX_CHUNKS]), done0 = smem_u32(&bars[2 * TC_MAX_CHUNKS]);
  const uint32_t tmem_cols = G <= 1 ? 64u : (G == 2 ? 128u : (G <= 4 ? 256u : 512u));
  using Geo = TcGeo<X3>;
  constexpr int PL = Geo::PL;
  TC_STAMP(0);

  if (threadIdx.x < 2 * TC_MAX_CHUNKS + TC_GMAX) {
    // every barrier is single use: one init each, in parallel.  done[q] collects one commit per MMA warp issuing into q
    const int i = threadIdx.x;
    const uint32_t cnt = i < 2 * TC_MAX_CHUNKS ? 1u : (uint32_t)max(1, (int)p.gdcnt[g][i - 2 * TC_MAX_CHUNKS]);
    mbar_init(full0 + 8 * i, cnt);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (warp > TC_MMA_WARPS) {
    // zero the accumulators: epilogue warp (lane quarter lq, half hh) clears its 32 lanes x half of the G*64 columns
    const int ew0 = warp - 1 - TC_MMA_WARPS;
    for (int c = (ew0 >> 2) * G; c < ((ew0 >> 2) + 1) * G; ++c)
      tmem_st32_zero(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + c * 32);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    tc_fence_before();
  }
  if (warp >= 1) asm volatile("bar.sync 3, %0;" ::"n"(TC_GEMM_THREADS - 32) : "memory");   // MMA + epilogue warps
  lcn_pdl_wait();                 // the previous kernel's outputs are visible from here on
  TC_STAMP(1);

  if (warp == 0) {
    // ===== TMA producer (warp-uniform; one elected lane issues) =====
    const __nv_bfloat16* a_tile = A + (size_t)tile * p.NCK * (8192 * PL);
    for (int it = 0; it < n_it; ++it) {
      const uint32_t s = p.sched[g][it];
      const uint32_t kc = TC_S_KC(s), cnt = (uint32_t)__popc(TC_S_BITS(s));
      const int wait = TC_S_WAIT(s);
      const __nv_bfloat16* wsrc = Wp + (size_t)p.gslot[g][kc] * 4096;
      if (wait >= 0) {                                   // the iterations that occupied this ring space have been consumed:
        mbar_wait(empty0 + 8 * wait, 0u);                // MMAs retire in order per issuing warp, so the newest iteration
        if (wait >= 1) mbar_wait(empty0 + 8 * (wait - 1), 0u);   // of either parity covers all older ones
      }
      if (elect_one()) {
        TC_STAMP(16 + 4 * it);
        const uint32_t sa = sbase + TC_S_OFF(s) * TC_B_BYTES;
        mbar_expect_tx(full0 + 8 * it, PL * (TC_A_BYTES + cnt * TC_B_BYTES));
        bulk_g2s(sa, a_tile + (size_t)kc * (8192 * PL), PL * TC_A_BYTES, full0 + 8 * it);     // X3: hi and lo planes, contiguous
        bulk_g2s(sa + PL * TC_A_BYTES, wsrc, cnt * TC_B_BYTES, full0 + 8 * it);
        if (X3)
          bulk_g2s(sa + PL * TC_A_BYTES + cnt * TC_B_BYTES, Wp_lo + (size_t)p.gslot[g][kc] * 4096, cnt * TC_B_BYTES, full0 + 8 * it);
        TC_STAMP(17 + 4 * it);
      }
      __syncwarp();
    }
  } else if (warp <= TC_MMA_WARPS) {
    // ===== MMA issuers (warp-uniform control flow and operands; one elected lane issues): warp w takes it % 2 == w - 1 =====
    tc_fence_after();
    const uint64_t desc_hi = (uint64_t)((1024u >> 4) & 0x3FFF) << 32 | (1ull << 46) | (2ull << 61) | (1ull << 16);
    const uint32_t idesc0 = umma_idesc(0, 0, 0);
    for (int it = warp - 1; it < n_it; it += TC_MMA_WARPS) {
      const uint32_t s = p.sched[g][it];
      const uint64_t rw = p.runs[g][it];
      const uint32_t bits = TC_S_BITS(s);
      const int nr = (int)(rw >> 60);
      mbar_wait(full0 + 8 * it, 0u);
      tc_fence_after();
      const uint32_t sa = sbase + TC_S_OFF(s) * TC_B_BYTES, sb = sa + PL * TC_A_BYTES;
      const uint32_t sb_lo = sb + (uint32_t)__popc(bits) * TC_B_BYTES;               // X3: the lo parts of the panel's blocks
      const uint64_t ad0 = desc_hi | (uint64_t)((sa >> 4) & 0x3FFF);
      const uint64_t ad0_lo = desc_hi | (uint64_t)(((sa + TC_A_BYTES) >> 4) & 0x3FFF);
      if (lane == 0) TC_STAMP(18 + 4 * it);
#pragma unroll
      for (int r = 0; r < TC_GMAX; ++r) {
        if (r >= nr) break;
        const uint32_t e = (uint32_t)(rw >> (6 * r)) & 63u;
        const uint32_t q = e & 7u, len = ((e >> 3) & 3u) + 1u;
        const uint32_t rank = (uint32_t)__popc(bits & ((1u << q) - 1u));   // blocks of the panel in front of chunk q
        const uint32_t idesc = idesc0 | ((len * 8u) << 17);               // N = 64 * len
        const uint64_t bd0 = desc_hi | (uint64_t)(((sb + rank * TC_B_BYTES) >> 4) & 0x3FFF);
        const uint32_t d = tmem_base + q * 64;
        if (elect_one()) {
          umma_f16(d, ad0, bd0, idesc, 1u);        // K = 64 -> 4 instructions of K = 16 (32 bytes each)
          umma_f16(d, ad0 + 2, bd0 + 2, idesc, 1u);
          umma_f16(d, ad0 + 4, bd0 + 4, idesc, 1u);
          umma_f16(d, ad0 + 6, bd0 + 6, idesc, 1u);
          if (X3) {                                // + a_hi * w_lo + a_lo * w_hi: the fp32-parity products
            const uint64_t bl0 = desc_hi | (uint64_t)(((sb_lo + rank * TC_B_BYTES) >> 4) & 0x3FFF);
#pragma unroll
            for (int k = 0; k < 8; k += 2) umma_f16(d, ad0 + k, bl0 + k, idesc, 1u);
#pragma unroll
            for (int k = 0; k < 8; k += 2) umma_f16(d, ad0_lo + k, bd0 + k, idesc, 1u);
          }
        }
      }
      uint32_t done = TC_S_DONE(s);
      if (elect_one()) {
        umma_commit(empty0 + 8 * it);              // frees the ring space when these MMAs have read it
        while (done) {                             // accumulators that received their last block in this iteration
          const int dq = __ffs(done) - 1;
          done &= done - 1;
          umma_commit(done0 + 8 * dq);
        }
      }
      if (lane == 0) TC_STAMP(19 + 4 * it);
      __syncwarp();
    }
  } else {
    // ===== epilogue: 8 warps; TMEM lane quarter = warp id % 4, column half of the chunk = epilogue warp / 4 =====
    const int lq = warp & 3;
    const int ew = warp - 1 - TC_MMA_WARPS;          // 0..7
    const int hh = ew >> 2;                          // 0: columns 0..31 of a chunk, 1: columns 32..63
    const int row = lq * 32 + lane;
    const int et = threadIdx.x - TC_EPI_T0;          // 0..255
    constexpr int ET = 32 * TC_EPI_WARPS;
    const uint32_t written = p.gwritten[g];
    uint8_t* stage = sgen + Geo::RING_BYTES;         // 2 output staging tiles (head mode: one fp32 tile)
    if (p.mode != TC_MODE_DGRAD) {
      for (int c = et; c < G * 64; c += ET) {
        int col = oc0 * 64 + c;
        bias_s[c] = (p.mode == TC_MODE_HEAD && col >= 51) ? 0.f : bias[col];
      }
      asm volatile("bar.sync 4, 256;" ::: "memory");
    }
    if (!X3 && p.mode == TC_MODE_HEAD) {
      // head mode (last layer, models_att.py:765-773): row geometry and the row's xy inputs are fetched while the main
      // loop runs (independent loads, all in flight before the accumulators are read)
      const int64_t pr = (int64_t)tile * LCN_TILE + row;
      const int64_t grp = pr / p.gstride;
      const int rin = (int)(pr - grp * p.gstride);
      int64_t src = grp * p.bn_group + rin;
      const bool valid = rin < p.bn_group;
      if (!(valid && src < p.n_rows)) src = -1;
      float xr[2 * LCN_J];
#pragma unroll
      for (int j = 0; j < LCN_J; ++j) {
        xr[2 * j] = src >= 0 ? p.x[src * (LCN_J * p.in_F) + j * p.in_F] : 0.f;
        xr[2 * j + 1] = src >= 0 ? p.x[src * (LCN_J * p.in_F) + j * p.in_F + 1] : 0.f;
      }
      if (written & 1u) mbar_wait(done0, 0u);
      if (et == 0) TC_STAMP(2);
      tc_fence_after();
      // 51 valid columns of one chunk -> fp32 prediction rows: through a shared-memory tile (pitch 51 words: conflict
      // free for thread = row), then coalesced stores
      float* stg = reinterpret_cast<float*>(stage);                          // [128][51]
      int64_t* src_s = reinterpret_cast<int64_t*>(stage + 128 * 51 * 4);     // [128]
      if (hh == 0) src_s[row] = valid ? src : -2;                            // -2: tile padding row (out_ws gets zeros)
      {
        uint32_t v[32];
        if (written & 1u) {
          tmem_ld32(tmem_base + ((uint32_t)(lq * 32) << 16) + hh * 32, v);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = 0u;
        }
        // (two compile-time instances of the column loop: xr[] must be indexed with constants to stay in registers)
        auto emit = [&](auto half) {
          constexpr int H = decltype(half)::value;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int c = H * 32 + i;
            if (c < 51) {
              float val = __uint_as_float(v[i]) + bias_s[c];
              const int j = c / 3, cc = c - j * 3;
              if (cc < 2) val += xr[2 * j + cc];
              stg[row * 51 + c] = val;
            }
          }
        };
        if (hh == 0) emit(std::integral_constant<int, 0>{}); else emit(std::integral_constant<int, 1>{});
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int e = et; e < 128 * 51; e += ET) {
        const int r = e / 51, c = e - r * 51;
        const int64_t sr = src_s[r];
        const float val = stg[e];
        if (p.out_ws != nullptr) p.out_ws[(size_t)tile * (LCN_TILE * 51) + e] = sr != -2 ? val : 0.f;
        if (sr >= 0) p.out_user[sr * 51 + c] = val;
      }
    } else {
      // Two teams of four warps (one warp per TMEM lane quarter) take alternate chunks of the completion order, each
      // with its own staging tile, named barrier and reduction scratch: a chunk's epilogue is a chain of latencies
      // (commit -> mbarrier, tcgen05.ld, shared-memory round trips, barriers: ~2.5 k cycles measured whether four or
      // eight warps share it), so two chunks in flight halve the time the accumulators wait for their epilogue.
      const int team = ew >> 2;
      const int tt = et & 127;                                               // thread within the team
      const uint32_t bar_id = 1u + (uint32_t)team;
      const int tig = tile % (p.gstride / LCN_TILE);
      const int nvalid = min(LCN_TILE, p.bn_group - tig * LCN_TILE);
      const float rn = 1.f / (float)nvalid;
      uint8_t* tile_s = stage + team * Geo::STAGE_BYTES;                       // X3: hi tile, then lo tile
      float* red = reinterpret_cast<float*>(stage + 2 * Geo::STAGE_BYTES) + team * (4 * 64 * 2);   // [4 warps][64 columns][s1, s2]
      for (int e = team; e < G; e += 2) {
        const int q = p.gorder[g][e];
        const bool has = (written >> q) & 1u;
        if (e >= 2) {
          // the team's previous bulk store has read the staging tile (its BN partials were read before the last barrier)
          if (tt == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        }
        if (has) {
          mbar_wait(done0 + 8 * q, 0u);
          tc_fence_after();
        }
        if (et == 0 && e == 0) TC_STAMP(2);
        if (tt == 0) TC_STAMP(200 + 8 * e);
        uint32_t v0[32], v1[32];
        if (has) {
          tmem_ld32_nowait(tmem_base + ((uint32_t)(lq * 32) << 16) + q * 64, v0);
          tmem_ld32_nowait(tmem_base + ((uint32_t)(lq * 32) << 16) + q * 64 + 32, v1);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v0[i] = v1[i] = 0u;
        }
        if (tt == 0) TC_STAMP(201 + 8 * e);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float f[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(h ? v1[i] : v0[i]);
          if (p.mode == TC_MODE_FWD) {
            const float4* b4 = reinterpret_cast<const float4*>(bias_s + q * 64 + h * 32);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float4 bv = b4[i];
              f[4 * i] += bv.x; f[4 * i + 1] += bv.y; f[4 * i + 2] += bv.z; f[4 * i + 3] += bv.w;
            }
          } else if (addend != nullptr) {
            const uint8_t* arow = reinterpret_cast<const uint8_t*>(addend) +
                                  ((((size_t)tile * p.NCN + oc0 + q) * PL) * 128 + row) * 128;
#pragma unroll
            for (int pl = 0; pl < PL; ++pl)
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                uint4 u = *reinterpret_cast<const uint4*>(arow + pl * TC_A_BYTES + (((h * 4 + c) ^ (row & 7)) << 4));
                const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  float2 t = __bfloat1622float2(hp[k]);
                  f[c * 8 + 2 * k] += t.x;
                  f[c * 8 + 2 * k + 1] += t.y;
                }
              }
          }
          // pack to bf16 and store the row's 4 sixteen-byte chunks into the swizzled staging tile
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint4 u;
            __nv_bfloat162 b0 = __floats2bfloat162_rn(f[c * 8 + 0], f[c * 8 + 1]);
            __nv_bfloat162 b1 = __floats2bfloat162_rn(f[c * 8 + 2], f[c * 8 + 3]);
            __nv_bfloat162 b2 = __floats2bfloat162_rn(f[c * 8 + 4], f[c * 8 + 5]);
            __nv_bfloat162 b3 = __floats2bfloat162_rn(f[c * 8 + 6], f[c * 8 + 7]);
            u.x = *reinterpret_cast<uint32_t*>(&b0);
            u.y = *reinterpret_cast<uint32_t*>(&b1);
            u.z = *reinterpret_cast<uint32_t*>(&b2);
            u.w = *reinterpret_cast<uint32_t*>(&b3);
            *reinterpret_cast<uint4*>(tile_s + row * 128 + (((h * 4 + c) ^ (row & 7)) << 4)) = u;
            if (X3) {                              // lo = bf16(f - hi): the second plane of the split-bf16 tile
              const float2 h0 = __bfloat1622float2(b0), h1 = __bfloat1622float2(b1), h2 = __bfloat1622float2(b2), h3 = __bfloat1622float2(b3);
              __nv_bfloat162 l0 = __floats2bfloat162_rn(f[c * 8 + 0] - h0.x, f[c * 8 + 1] - h0.y);
              __nv_bfloat162 l1 = __floats2bfloat162_rn(f[c * 8 + 2] - h1.x, f[c * 8 + 3] - h1.y);
              __nv_bfloat162 l2 = __floats2bfloat162_rn(f[c * 8 + 4] - h2.x, f[c * 8 + 5] - h2.y);
              __nv_bfloat162 l3 = __floats2bfloat162_rn(f[c * 8 + 6] - h3.x, f[c * 8 + 7] - h3.y);
              uint4 ul;
              ul.x = *reinterpret_cast<uint32_t*>(&l0);
              ul.y = *reinterpret_cast<uint32_t*>(&l1);
              ul.z = *reinterpret_cast<uint32_t*>(&l2);
              ul.w = *reinterpret_cast<uint32_t*>(&l3);
              *reinterpret_cast<uint4*>(tile_s + TC_A_BYTES + row * 128 + (((h * 4 + c) ^ (row & 7)) << 4)) = ul;
            }
          }
        }
        if (tt == 0) TC_STAMP(202 + 8 * e);
        tc_fence_before();
        fence_proxy_async();                                   // generic smem writes -> bulk-store (async proxy) reads
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");   // the 4 warps of the team
        if (tt == 0) {
          TC_STAMP(203 + 8 * e);
          bulk_s2g(Y + ((size_t)tile * p.NCN + oc0 + q) * (8192 * PL), smem_u32(tile_s), PL * TC_A_BYTES);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        if (p.mode == TC_MODE_FWD && (part != nullptr || p.fuse_on)) {
          // BatchNorm partials of this tile and chunk: per column (mean, M2) over the valid rows, from the bf16 values
          // staged in shared memory (what k_bn_act will read).  Warp w walks rows w, w+4, ...; a lane owns two columns;
          // sums are shifted by the chunk's row-0 value (the same shift in every warp, so the four partial sums add).
          // Constant trip count: all 32 loads of the lane are in flight before the first add.
          const uint32_t coff = (uint32_t)(lane & 3) * 4;
          const int chunk = lane >> 2;
          uint32_t w[32], wl[X3 ? 32 : 1];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int r = lq + 4 * i;
            w[i] = *reinterpret_cast<const uint32_t*>(tile_s + r * 128 + ((chunk ^ (r & 7)) << 4) + coff);
            if (X3) wl[i] = *reinterpret_cast<const uint32_t*>(tile_s + TC_A_BYTES + r * 128 + ((chunk ^ (r & 7)) << 4) + coff);
          }
          // the shift is the row-0 value of the hi plane in both instantiations (any common shift works)
          const uint32_t w0 = *reinterpret_cast<const uint32_t*>(tile_s + (chunk << 4) + coff);
          const float2 sh2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w0));
          float s1a = 0.f, s1b = 0.f, s2a = 0.f, s2b = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (lq + 4 * i < nvalid) {
              float2 t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
              if (X3) {
                const float2 tl = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&wl[i]));
                t.x += tl.x; t.y += tl.y;
              }
              float d0 = t.x - sh2.x, d1 = t.y - sh2.y;
              s1a += d0; s2a = fmaf(d0, d0, s2a);
              s1b += d1; s2b = fmaf(d1, d1, s2b);
            }
          }
          *reinterpret_cast<float4*>(red + ((size_t)lq * 64 + lane * 2) * 2) = make_float4(s1a, s2a, s1b, s2b);
          if (tt == 0) TC_STAMP(204 + 8 * e);
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
          if (tt == 0) TC_STAMP(205 + 8 * e);
          if (tt < 64) {
            const int col = tt;
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int ww = 0; ww < 4; ++ww) {
              const float2 v = *reinterpret_cast<const float2*>(red + ((size_t)ww * 64 + col) * 2);
              s1 += v.x; s2 += v.y;
            }
            const float sh = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(tile_s + ((col >> 3) << 4) + (col & 7) * 2));
            if (p.fuse_on) {
              // unshifted moments in fp64 (sum x = n sh + s1, sum x^2 = s2 + 2 sh s1 + n sh^2) added to this tile's
              // replica of the per-channel accumulators; channel = column within the joint
              const double n = (double)nvalid, shd = (double)sh, d1 = (double)s1;
              const int f = ((oc0 + q) % p.FCN) * 64 + col;
              double* dst = p.fuse.gacc + ((size_t)(tile & (LCN_GACC_REP - 1)) * p.fuse.F + f) * 2;
              atomicAdd(dst, n * shd + d1);
              atomicAdd(dst + 1, (double)s2 + 2.0 * shd * d1 + n * shd * shd);
            } else {
              *reinterpret_cast<float2*>(part + ((size_t)tile * p.P + (oc0 + q) * 64 + col) * 2) =
                  make_float2(fmaf(s1, rn, sh), fmaxf(s2 - s1 * s1 * rn, 0.f));
            }
          }
          if (tt == 0) TC_STAMP(206 + 8 * e);
        }
      }
      if (tt == 0) {
        if (et == 0) TC_STAMP(3);
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem may be released; writes land by grid end
        if (et == 0) TC_STAMP(4);
      }
    }
    if (et == 0) TC_STAMP(5);
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) TC_STAMP(6);
  if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <bool X3>
static int launch_tc_gemm_t(const __nv_bfloat16* A, const __nv_bfloat16* W, const __nv_bfloat16* Wlo, const float* bias,
                            const __nv_bfloat16* addend, __nv_bfloat16* Y, float* part, const TcParams& p, int tiles,
                            cudaStream_t st) {
  static std::once_flag once;              // thread-safe one-time attribute setup (include/lcn_b200.h: re-entrancy)
  static cudaError_t rc = cudaSuccess;
  std::call_once(once, [] {
    rc = cudaFuncSetAttribute(k_tc_gemm<X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcGeo<X3>::SMEM_BYTES);
  });
  LCN_CHECK_CUDA(rc);
  lcn_launch(k_tc_gemm<X3>, dim3(dim3(p.n_groups, tiles)), dim3(TC_GEMM_THREADS), (size_t)TcGeo<X3>::SMEM_BYTES, st, A, W, Wlo,
             bias, addend, Y, part, p);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}
static int launch_tc_gemm(const __nv_bfloat16* A, const __nv_bfloat16* W, const __nv_bfloat16* Wlo, const float* bias,
                          const __nv_bfloat16* addend, __nv_bfloat16* Y, float* part, const TcParams& p, int tiles,
                          cudaStream_t st) {
  return Wlo != nullptr ? launch_tc_gemm_t<true>(A, W, Wlo, bias, addend, Y, part, p, tiles, st)
                        : launch_tc_gemm_t<false>(A, W, nullptr, bias, addend, Y, part, p, tiles, st);
}

// blocks under N-side chunk oc (= K chunks with a block into it)
static int tc_col_blocks(const TcParams& p, int oc) {
  int n = 0;
  for (int ka = 0; ka < p.NCK / p.FCK; ++ka)
    if ((p.kmask[ka] >> (oc / p.FCN)) & 1u) n += p.FCK;
  return n;
}

// contiguous split of the N-side chunks into ng groups of <= TC_GMAX chunks minimising the largest block count
// (a CTA's main-loop time is proportional to its blocks); returns that maximum.  DP over (groups, chunks).
static int tc_partition(const TcParams& p, int ng, uint8_t* goc0) {
  const int NC = p.NCN, INF = 1 << 28;
  static thread_local int best[TC_MAX_CHUNKS + 1][TC_MAX_CHUNKS + 1], from[TC_MAX_CHUNKS + 1][TC_MAX_CHUNKS + 1];
  int pre[TC_MAX_CHUNKS + 1];
  pre[0] = 0;
  for (int c = 0; c < NC; ++c) pre[c + 1] = pre[c] + tc_col_blocks(p, c);
  for (int k = 0; k <= ng; ++k)
    for (int c = 0; c <= NC; ++c) best[k][c] = INF;
  best[0][0] = 0;
  for (int k = 1; k <= ng; ++k)
    for (int c = k; c <= NC; ++c)
      for (int a = 1; a <= TC_GMAX && a <= c; ++a) {
        if (best[k - 1][c - a] >= INF) continue;
        int load = pre[c] - pre[c - a];
        int v = best[k - 1][c - a] > load ? best[k - 1][c - a] : load;
        if (v < best[k][c]) { best[k][c] = v; from[k][c] = a; }
      }
  if (best[ng][NC] >= INF) return INF;
  int c = NC;
  for (int k = ng; k >= 1; --k) {
    goc0[k] = (uint8_t)c;
    c -= from[k][c];
  }
  goc0[0] = 0;
  return best[ng][NC];
}

// Per group: the K-chunk order, the ring placement of every iteration and the completion order of the accumulators.
//   order: greedy -- repeatedly take the N-side chunk with the fewest K chunks still missing and schedule those, so
//          the chunks of a group finish one after the other and their epilogues overlap the remaining MMAs;
//   ring : iteration `it` takes 2 + #blocks units at the running head (wrapping when it does not fit before the end);
//          `wait` = the newest earlier iteration whose units it overwrites (MMAs retire in order, so waiting for that
//          one's empty barrier covers all older ones);
//   slot : position of the iteration's first block in the packed panel (k_pack_mid order).
static void tc_fill_schedule(TcParams& p, bool x3) {
  memset(p.sched, 0, sizeof(p.sched));
  memset(p.runs, 0, sizeof(p.runs));
  memset(p.gslot, 0, sizeof(p.gslot));
  memset(p.gnit, 0, sizeof(p.gnit));
  memset(p.gwritten, 0, sizeof(p.gwritten));
  memset(p.gorder, 0, sizeof(p.gorder));
  memset(p.gdcnt, 0, sizeof(p.gdcnt));
  for (int g = 0; g < p.n_groups; ++g) {
    const int oc0 = p.goc0[g], G = p.goc0[g + 1] - oc0;
    uint32_t kbits[TC_MAX_CHUNKS];                    // per K chunk: present chunks of the group
    for (int kc = 0; kc < p.NCK; ++kc) {
      const int ka = kc / p.FCK, hk = kc - ka * p.FCK;
      const uint32_t km = p.kmask[ka];
      uint32_t bits = 0;
      for (int q = 0; q < G; ++q)
        if ((km >> ((oc0 + q) / p.FCN)) & 1u) bits |= 1u << q;
      kbits[kc] = bits;
      p.gwritten[g] |= (uint8_t)bits;
      if (bits) {
        const int oc = oc0 + __builtin_ctz(bits);
        const int nb = oc / p.FCN, hn = oc - nb * p.FCN;
        int pb = 0;
        for (int q = 0; q < ka; ++q) pb += __builtin_popcount(p.kmask[q]);
        p.gslot[g][kc] = (uint16_t)(p.FCK * p.FCN * pb + hk * (__builtin_popcount(km) * p.FCN) +
                                    __builtin_popcount(km & ((1u << nb) - 1u)) * p.FCN + hn);
      }
    }
    // greedy completion order
    int order[TC_MAX_CHUNKS], n_it = 0, n_done = 0;
    uint32_t done_after[TC_MAX_CHUNKS];               // per iteration: chunks complete after it
    memset(done_after, 0, sizeof(done_after));
    bool used[TC_MAX_CHUNKS] = {false};
    uint32_t finished = 0;
    for (int q = 0; q < G; ++q)
      if (!((p.gwritten[g] >> q) & 1u)) {             // no block at all: nothing to wait for, zeros are stored
        finished |= 1u << q;
        p.gorder[g][n_done++] = (uint8_t)q;
      }
    while (n_done < G) {
      int bq = -1, bmiss = 1 << 30;
      for (int q = 0; q < G; ++q) {
        if ((finished >> q) & 1u) continue;
        int miss = 0;
        for (int kc = 0; kc < p.NCK; ++kc)
          if (!used[kc] && ((kbits[kc] >> q) & 1u)) ++miss;
        if (miss < bmiss) { bmiss = miss; bq = q; }
      }
      for (int kc = 0; kc < p.NCK; ++kc)
        if (!used[kc] && ((kbits[kc] >> bq) & 1u)) {
          used[kc] = true;
          order[n_it++] = kc;
        }
      // every chunk whose K chunks are now all scheduled completes with the last iteration added
      for (int q = 0; q < G; ++q) {
        if ((finished >> q) & 1u) continue;
        bool all = true;
        for (int kc = 0; kc < p.NCK; ++kc)
          if (!used[kc] && ((kbits[kc] >> q) & 1u)) { all = false; break; }
        if (all) {
          finished |= 1u << q;
          p.gorder[g][n_done++] = (uint8_t)q;
        }
      }
    }
    // Completion: MMA warp w issues the iterations it % TC_MMA_WARPS == w and commits to done[q] after its own last
    // iteration touching chunk q; done[q] expects one arrival per warp that touches q.  The epilogue visits the chunks
    // in the order of their overall last iteration.
    {
      int comp[TC_GMAX];
      for (int q = 0; q < G; ++q) {
        comp[q] = -1;
        int cnt = 0;
        for (int w = 0; w < TC_MMA_WARPS; ++w) {
          int last = -1;
          for (int i = w; i < n_it; i += TC_MMA_WARPS)
            if ((kbits[order[i]] >> q) & 1u) last = i;
          if (last >= 0) {
            done_after[last] |= 1u << q;
            ++cnt;
            if (last > comp[q]) comp[q] = last;
          }
        }
        p.gdcnt[g][q] = (uint8_t)cnt;
      }
      int ce[TC_GMAX];
      for (int e = 0; e < G; ++e) ce[e] = comp[p.gorder[g][e]];
      for (int a = 1; a < G; ++a)                     // insertion sort, stable
        for (int b = a; b > 0 && ce[b - 1] > ce[b]; --b) {
          int t = ce[b]; ce[b] = ce[b - 1]; ce[b - 1] = t;
          uint8_t u = p.gorder[g][b]; p.gorder[g][b] = p.gorder[g][b - 1]; p.gorder[g][b - 1] = u;
        }
    }
    p.gnit[g] = (uint8_t)n_it;
    // MMA runs: maximal runs (<= 4 chunks = N 256) of adjacent present chunks (every MMA accumulates: the accumulators
    // are zeroed at kernel start)
    for (int it = 0; it < n_it; ++it) {
      const uint32_t bits = kbits[order[it]];
      uint64_t rw = 0;
      int nr = 0, q = 0;
      while (q < G) {
        if (!((bits >> q) & 1u)) { ++q; continue; }
        int len = 1;
        while (len < 4 && q + len < G && ((bits >> (q + len)) & 1u)) ++len;
        rw |= (uint64_t)((uint32_t)q | ((uint32_t)(len - 1) << 3) | (1u << 5)) << (6 * nr);
        ++nr;
        q += len;
      }
      p.runs[g][it] = rw | ((uint64_t)nr << 60);
    }
    // ring placement
    int head = 0, first_live = 0;
    int off[TC_MAX_CHUNKS], need[TC_MAX_CHUNKS];
    for (int it = 0; it < n_it; ++it) {
      need[it] = x3 ? TcGeo<true>::A_UNITS + 2 * __builtin_popcount(kbits[order[it]])
                    : TcGeo<false>::A_UNITS + __builtin_popcount(kbits[order[it]]);
      if (head + need[it] > (x3 ? TcGeo<true>::RING_UNITS : TcGeo<false>::RING_UNITS)) head = 0;
      off[it] = head;
      int wait = -1;
      for (int j = first_live; j < it; ++j)
        if (off[j] < off[it] + need[it] && off[it] < off[j] + need[j]) wait = j;
      if (wait >= 0) first_live = wait + 1;
      head += need[it];
      p.sched[g][it] = (uint32_t)order[it] | (kbits[order[it]] << 6) | ((uint32_t)off[it] << 12) |
                       ((uint32_t)(wait + 1) << 17) | (done_after[it] << 24);
    }
  }
}

// choose the number of groups (whole waves of sm_count CTAs, minimal waves x per-CTA time), partition, fill the schedule
static void tc_make_schedule(TcParams& p, int tiles, int sm_count, bool x3) {
  int best_ng = p.NCN;
  double best = 1e30;
  uint8_t goc0[TC_MAX_CHUNKS + 1];
  for (int ng = (p.NCN + TC_GMAX - 1) / TC_GMAX; ng <= p.NCN; ++ng) {
    const int maxblk = tc_partition(p, ng, goc0);
    int gmax = 0;
    for (int g = 0; g < ng; ++g) gmax = goc0[g + 1] - goc0[g] > gmax ? goc0[g + 1] - goc0[g] : gmax;
    long ctas = (long)tiles * ng;
    long waves = (ctas + sm_count - 1) / sm_count;
    // per-CTA time ~ main loop (blocks) + the epilogue tail (the last chunks) + fixed cost, in units of one block's MMA time
    double c = (double)waves * (maxblk + 1.5 * gmax + 8.0);
    if (c < best - 1e-9) { best = c; best_ng = ng; }
  }
  p.n_groups = best_ng;
  tc_partition(p, best_ng, p.goc0);
  tc_fill_schedule(p, x3);
}

// Pick the N-side grouping.  One CTA is resident per SM (TMEM kernels), so the grid should be whole waves of
// sm_count CTAs: choose the number of chunk groups that minimises waves x (work per CTA + fixed per-CTA cost).
static int pick_and_launch(const __nv_bfloat16* A, const __nv_bfloat16* W, const __nv_bfloat16* Wlo, const float* bias,
                           const __nv_bfloat16* addend, __nv_bfloat16* Y, float* part, TcParams& p, int tiles,
                           int sm_count, cudaStream_t st) {
  const int force = Wlo != nullptr ? 1 : 0;          // cache key: the ring geometry of the split-bf16 instantiation differs
  // The grouping and its schedule depend only on (mask, chunk geometry, tiles, SM count): computed once, then
  // served from a small cache (the launch path must stay cheap: it runs ~20 times per train step).
  struct Entry { uint32_t kmask[LCN_J]; int FCK, FCN, NCK, NCN, tiles, sm, force; TcParams sched; };
  static std::mutex mu;
  static std::vector<Entry> cache;
  {
    std::lock_guard<std::mutex> lock(mu);
    const Entry* hit = nullptr;
    for (const Entry& e : cache)
      if (e.FCK == p.FCK && e.FCN == p.FCN && e.NCK == p.NCK && e.NCN == p.NCN && e.tiles == tiles && e.sm == sm_count &&
          e.force == force && memcmp(e.kmask, p.kmask, sizeof(e.kmask)) == 0) { hit = &e; break; }
    if (hit == nullptr) {
      Entry e;
      memcpy(e.kmask, p.kmask, sizeof(e.kmask));
      e.FCK = p.FCK; e.FCN = p.FCN; e.NCK = p.NCK; e.NCN = p.NCN; e.tiles = tiles; e.sm = sm_count; e.force = force;
      e.sched = p;
      tc_make_schedule(e.sched, tiles, sm_count, force != 0);
      cache.push_back(e);
      hit = &cache.back();
    }
    p.n_groups = hit->sched.n_groups;
    memcpy(p.sched, hit->sched.sched, sizeof(p.sched));
    memcpy(p.runs, hit->sched.runs, sizeof(p.runs));
    memcpy(p.gslot, hit->sched.gslot, sizeof(p.gslot));
    memcpy(p.gnit, hit->sched.gnit, sizeof(p.gnit));
    memcpy(p.gwritten, hit->sched.gwritten, sizeof(p.gwritten));
    memcpy(p.gorder, hit->sched.gorder, sizeof(p.gorder));
    memcpy(p.gdcnt, hit->sched.gdcnt, sizeof(p.gdcnt));
    memcpy(p.goc0, hit->sched.goc0, sizeof(p.goc0));
  }
  return launch_tc_gemm(A, W, Wlo, bias, addend, Y, part, p, tiles, st);
}

// schedule of the knn-masked mid layer for inspection / tests (host only): returns the number of groups and fills, per
// group, the iteration count; sched_out[g * 34 + it] is the packed entry (TC_S_* fields)
extern "C" int lcn_debug_tc_schedule(const uint32_t* kmask17, int FC, int tiles, int sm_count, uint32_t* sched_out,
                                     uint8_t* nit_out, uint8_t* goc0_out, uint8_t* order_out, uint64_t* runs_out,
                                     uint8_t* dcnt_out) {
  TcParams p;
  memset(&p, 0, sizeof(p));
  for (int a = 0; a < LCN_J; ++a) p.kmask[a] = kmask17[a];
  p.FCK = p.FCN = FC;
  p.NCK = p.NCN = LCN_J * FC;
  tc_make_schedule(p, tiles, sm_count, false);
  memcpy(sched_out, p.sched, sizeof(p.sched));
  memcpy(nit_out, p.gnit, sizeof(p.gnit));
  memcpy(goc0_out, p.goc0, sizeof(p.goc0));
  memcpy(order_out, p.gorder, sizeof(p.gorder));
  if (runs_out) memcpy(runs_out, p.runs, sizeof(p.runs));
  if (dcnt_out) memcpy(dcnt_out, p.gdcnt, sizeof(p.gdcnt));
  return p.n_groups;
}

int lcn_tc_gemm(const lcn_model* m, const WsLayout& lay, int mid_index, int transposed, const __nv_bfloat16* A,
                const char* wpacked, const float* bias, const __nv_bfloat16* addend, __nv_bfloat16* Y, float* part,
                cudaStream_t st, const TcFuse* fuse, int* fused, const char* wpacked_lo) {
  (void)mid_index;
  TcParams p;
  memset(&p, 0, sizeof(p));
  for (int a = 0; a < LCN_J; ++a) p.kmask[a] = transposed ? m->sup.col[a] : m->sup.row[a];
  p.FCK = p.FCN = m->FC;
  p.NCK = p.NCN = LCN_J * m->FC;
  p.P = m->P;
  p.bn_group = lay.bn_group;
  p.gstride = lay.gstride;
  p.mode = transposed ? TC_MODE_DGRAD : TC_MODE_FWD;
  if (fused) *fused = 0;
  if (fuse != nullptr && !transposed && lay.n_groups == 1) {
    p.fuse = *fuse;
    p.fuse_on = 1;
  }
  int rc = pick_and_launch(A, reinterpret_cast<const __nv_bfloat16*>(wpacked), reinterpret_cast<const __nv_bfloat16*>(wpacked_lo),
                           bias, addend, Y, part, p, lay.tiles, m->sm_count, st);
  if (fused) *fused = p.fuse_on;
  return rc;
}

// last layer (17*F -> 51) + output head on the tensor cores: one N-side chunk (51 columns padded to 64),
// every K chunk present; weights packed by k_pack_edges as one 64x64 block per K chunk.
int lcn_tc_head(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* A, const char* wpacked,
                const float* bias, const float* x, float* out_user, float* out_ws, cudaStream_t st) {
  TcParams p;
  memset(&p, 0, sizeof(p));
  for (int a = 0; a < LCN_J; ++a) p.kmask[a] = 1u;
  p.FCK = m->FC;
  p.FCN = 1;
  p.NCK = LCN_J * m->FC;
  p.NCN = 1;
  p.P = 64;
  p.bn_group = lay.bn_group;
  p.gstride = lay.gstride;
  p.mode = TC_MODE_HEAD;
  p.x = x;
  p.in_F = m->d.in_F;
  p.n_rows = lay.n_rows;
  p.out_user = out_user;
  p.out_ws = out_ws;
  return pick_and_launch(A, reinterpret_cast<const __nv_bfloat16*>(wpacked), nullptr, bias, nullptr, nullptr, nullptr, p,
                         lay.tiles, m->sm_count, st);
}

// last layer input gradient dA = dOut * Wm4^T: one K chunk (dOut padded to 64 columns), all N chunks present
int lcn_tc_head_dgrad(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* dOut16, const char* wpacked,
                      __nv_bfloat16* dA, cudaStream_t st) {
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.kmask[0] = (1u << LCN_J) - 1u;
  p.FCK = 1;
  p.FCN = m->FC;
  p.NCK = 1;
  p.NCN = LCN_J * m->FC;
  p.P = m->P;
  p.bn_group = lay.bn_group;
  p.gstride = lay.gstride;
  p.mode = TC_MODE_DGRAD;
  return pick_and_launch(dOut16, reinterpret_cast<const __nv_bfloat16*>(wpacked), nullptr, nullptr, nullptr, dA, nullptr, p,
                         lay.tiles, m->sm_count, st);
}

// ---------------------------------------------------------------------------------------------
// weight gradient of the nonzero blocks: dWm[(i,hi) chunk, (j,ho) chunk] += A[rows, ic]^T dZ[rows, oc]
//   D[M = 128 = two input chunks x 64 channels, N = 64*len output channels] = sum_k A_op[m][k] * B_op[n][k], k = batch row.
//   Both operands are MN-major SW128 tiles exactly as stored in HBM (K = the rows of a tile); the two input chunks of a
//   unit sit 8 KB apart in shared memory, which is the descriptor's leading-dimension stride, like the <=4 output chunks.
//   unit = (pair of input chunks, group of <=4 output chunks out of the union of their neighbourhoods): M = 128 runs the
//   tensor pipe at full rate (M = 64 at half) and halves the number of units; the pairs are matched on the host so that
//   the union wastes as few blocks as possible (knn=3: 218 computed for 175 stored; F=128: the two halves of a joint,
//   no waste).  Blocks of the union that are not in the mask are computed and dropped.  grid.y splits the batch rows.
//   Two MMA-issuing warps (even / odd half tiles) on accumulators zeroed by the epilogue warps, as in k_tc_gemm.
// ---------------------------------------------------------------------------------------------
#define TCW_HALF_BYTES 8192                       // 64 rows x 64 bf16: half of an activation tile
#define TCW_STAGE_BYTES ((2 + TC_G) * TCW_HALF_BYTES)
#define TCW_STAGES 4     // even: a stage is always consumed by the same MMA warp (it % 2 == stage % 2), so each warp sees
                         // the phases of its full barriers in sequence
#define TCW_PITCH 260   // floats per staged output row (1040 B: 16-byte aligned, bank-conflict free)
#define TCW_THREADS (32 + 32 * TC_MMA_WARPS + 128)
#define TCW_MAX_UNITS 160

struct TcwUnit {
  uint8_t ic0, ic1;        // input chunks (ic1 = 0xff: single)
  uint8_t len, pad;
  uint8_t oc[TC_G];        // output chunks
  uint8_t keep[TC_G];      // bit 0: (ic0, oc) is a block of the mask, bit 1: (ic1, oc)
};

struct TcwParams {
  uint32_t row[LCN_J];     // outputs (N-side joints) of input (M-side) joint i
  int FCK, FCN;            // 64-chunks per joint on the A (M) side / dZ (N) side
  int NCK, NCN;            // chunks per row tile of A / dZ
  int ldw;                 // row pitch of dW in floats
  int tiles, tiles_per_cta;
  int n_units;
  TcwUnit unit[TCW_MAX_UNITS];
};

__device__ __forceinline__ void bulk_reduce_add_f32(float* dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(dst), "r"(src),
               "r"(bytes)
               : "memory");
}

// X3 (split-bf16 operands, lcn_internal.cuh): the K loop runs three times per half tile -- (A_hi, dZ_hi), (A_hi, dZ_lo),
// (A_lo, dZ_hi) -- into the same accumulators; the planes of a tile are adjacent in HBM / L2.
template <bool X3>
__global__ void __launch_bounds__(TCW_THREADS) k_tc_wgrad(const __nv_bfloat16* __restrict__ A,
                                                          const __nv_bfloat16* __restrict__ dZ,
                                                          float* __restrict__ dW, const __grid_constant__ TcwParams p) {
  lcn_pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * TCW_STAGES + TC_MMA_WARPS];
  __shared__ uint32_t tmem_base_s;
  uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sgen = smem_raw + (sbase - smem_u32(smem_raw));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const TcwUnit& u = p.unit[blockIdx.x];
  const int ic0 = u.ic0, ic1 = u.ic1, len = u.len;
  const int na = ic1 != 0xff ? 2 : 1;              // input half tiles per stage
  const int t0 = blockIdx.y * p.tiles_per_cta;
  const int t1 = min(t0 + p.tiles_per_cta, p.tiles);
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[TCW_STAGES]), tfull = smem_u32(&bars[2 * TCW_STAGES]);
  const uint32_t tmem_cols = len <= 1 ? 64u : (len == 2 ? 128u : 256u);

  if (threadIdx.x == 0) {
    for (int s = 0; s < TCW_STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    mbar_init(tfull, TC_MMA_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_s), tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (warp > TC_MMA_WARPS) {
    // zero the accumulators (the two MMA warps only accumulate): warp's lane quarter x all columns
    for (int c = 0; c < (int)tmem_cols / 32; ++c) tmem_st32_zero(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + c * 32);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    tc_fence_before();
  }
  if (warp >= 1) asm volatile("bar.sync 3, %0;" ::"n"(TCW_THREADS - 32) : "memory");
  lcn_pdl_wait();                 // the previous kernel's outputs are visible from here on

  constexpr int PL = X3 ? 2 : 1, NPASS = X3 ? 3 : 1;
  const int n_it = NPASS * 2 * (t1 - t0);          // two 64-row half tiles per 128-row tile (x 3 operand-plane passes)
  if (warp == 0) {
    if (lane == 0) {
      for (int it = 0; it < n_it; ++it) {
        int s = it % TCW_STAGES;
        uint32_t ph = (uint32_t)(it / TCW_STAGES) & 1u;
        const int ih = it / NPASS, pass = it - ih * NPASS;
        int t = t0 + (ih >> 1), half = ih & 1;
        const size_t pa = pass == 2 ? 8192 : 0, pz = pass == 1 ? 8192 : 0;   // plane offsets (elements): lo follows hi
        mbar_wait(empty0 + 8 * s, ph ^ 1u);
        uint32_t sa = sbase + s * TCW_STAGE_BYTES;
        mbar_expect_tx(full0 + 8 * s, (na + len) * TCW_HALF_BYTES);
        bulk_g2s(sa, A + ((size_t)t * p.NCK + ic0) * (8192 * PL) + pa + half * 4096, TCW_HALF_BYTES, full0 + 8 * s);
        if (na == 2)
          bulk_g2s(sa + TCW_HALF_BYTES, A + ((size_t)t * p.NCK + ic1) * (8192 * PL) + pa + half * 4096, TCW_HALF_BYTES, full0 + 8 * s);
        for (int q = 0; q < len; ++q)
          bulk_g2s(sa + (2 + q) * TCW_HALF_BYTES, dZ + ((size_t)t * p.NCN + u.oc[q]) * (8192 * PL) + pz + half * 4096,
                   TCW_HALF_BYTES, full0 + 8 * s);
      }
    }
  } else if (warp <= TC_MMA_WARPS) {
    tc_fence_after();
    if (lane == 0) {
      // M = 128, N = 64*len, both operands MN-major.  The stage's empty barrier takes ONE arrival: consecutive
      // iterations alternate between the two warps, and a stage is released by the warp that consumed it.
      uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)((64 * len) >> 3) << 17) |
                       ((uint32_t)(128 >> 4) << 24);
      for (int it = warp - 1; it < n_it; it += TC_MMA_WARPS) {
        int s = it % TCW_STAGES;
        uint32_t ph = (uint32_t)(it / TCW_STAGES) & 1u;
        mbar_wait(full0 + 8 * s, ph);
        tc_fence_after();
        uint32_t sa = sbase + s * TCW_STAGE_BYTES, sb = sa + 2 * TCW_HALF_BYTES;
#pragma unroll
        for (int k16 = 0; k16 < 4; ++k16) {          // 64 rows = 4 MMAs of K = 16
          uint64_t ad = umma_desc_sw128(sa + k16 * 2048, TCW_HALF_BYTES, 1024);
          uint64_t bd = umma_desc_sw128(sb + k16 * 2048, TCW_HALF_BYTES, 1024);
          umma_f16(tmem_base, ad, bd, idesc, 1u);
        }
        umma_commit(empty0 + 8 * s);
      }
      umma_commit(tfull);
    }
  } else {
    const int lq = warp & 3;
    const int et = threadIdx.x - 32 - 32 * TC_MMA_WARPS;          // 0..127
    mbar_wait(tfull, 0);
    tc_fence_after();
    float* out_s = reinterpret_cast<float*>(sgen);
    const int m = lq * 32 + lane;                    // accumulator row: channel m % 64 of input chunk ic0 (m < 64) / ic1
    const int hi = m >> 6;
    for (int q = 0; q < len; ++q)
      for (int h = 0; h < 2; ++h) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(lq * 32) << 16) + q * 64 + h * 32, v);
        float* dst = out_s + m * TCW_PITCH + q * 64 + h * 32;
#pragma unroll
        for (int c = 0; c < 8; ++c)
          *reinterpret_cast<uint4*>(dst + c * 4) = make_uint4(v[c * 4], v[c * 4 + 1], v[c * 4 + 2], v[c * 4 + 3]);
      }
    tc_fence_before();
    fence_proxy_async();
    asm volatile("bar.sync 1, 128;" ::: "memory");
    (void)et;
    if (hi < na) {
      const int ic = hi ? ic1 : ic0;
      for (int q = 0; q < len; ++q)
        if ((u.keep[q] >> hi) & 1u)
          bulk_reduce_add_f32(dW + (size_t)(ic * 64 + (m & 63)) * p.ldw + u.oc[q] * 64, smem_u32(out_s + m * TCW_PITCH + q * 64), 256);
    }
    bulk_commit_wait_read();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

// units of the weight-gradient kernel: input chunks matched in pairs (smallest union of neighbourhoods first), then
// groups of <= TC_G output chunks of the union
static void tcw_build_units(TcwParams& p) {
  const int NI = p.NCK;
  auto outs = [&](int ic, uint8_t* list) {          // output chunks of input chunk ic, ascending
    int n = 0;
    const uint32_t bits = p.row[ic / p.FCK];
    for (int j = 0; j < LCN_J; ++j)
      if ((bits >> j) & 1u)
        for (int ho = 0; ho < p.FCN; ++ho) list[n++] = (uint8_t)(j * p.FCN + ho);
    return n;
  };
  bool used[TC_MAX_CHUNKS] = {false};
  int pa[TC_MAX_CHUNKS], pb[TC_MAX_CHUNKS], np = 0;
  int left = NI;
  while (left > 1) {
    int bi = -1, bk = -1;
    long best = 1L << 60;
    for (int i = 0; i < NI; ++i) {
      if (used[i]) continue;
      for (int k = i + 1; k < NI; ++k) {
        if (used[k]) continue;
        const uint32_t a = p.row[i / p.FCK], b = p.row[k / p.FCK];
        const int un = __builtin_popcount(a | b), waste = 2 * un - __builtin_popcount(a) - __builtin_popcount(b);
        const long key = ((long)waste << 20) | ((long)un << 8) | (long)(k - i);   // least waste, then smallest union, then nearest
        if (key < best) { best = key; bi = i; bk = k; }
      }
    }
    used[bi] = used[bk] = true;
    pa[np] = bi; pb[np] = bk; ++np;
    left -= 2;
  }
  for (int i = 0; i < NI; ++i)
    if (!used[i]) { pa[np] = i; pb[np] = -1; ++np; }
  p.n_units = 0;
  for (int e = 0; e < np; ++e) {
    uint8_t la[TC_MAX_CHUNKS], lb[TC_MAX_CHUNKS], un[2 * TC_MAX_CHUNKS];
    const int na = outs(pa[e], la), nb = pb[e] >= 0 ? outs(pb[e], lb) : 0;
    bool ina[TC_MAX_CHUNKS] = {false}, inb[TC_MAX_CHUNKS] = {false};
    for (int i = 0; i < na; ++i) ina[la[i]] = true;
    for (int i = 0; i < nb; ++i) inb[lb[i]] = true;
    int nu = 0;
    for (int oc = 0; oc < p.NCN; ++oc)
      if (ina[oc] || inb[oc]) un[nu++] = (uint8_t)oc;
    for (int g0 = 0; g0 < nu; g0 += TC_G) {
      if (p.n_units >= TCW_MAX_UNITS) return;       // cannot happen: 17 pairs x ceil(34 / 4) = 153 units at most
      TcwUnit& u = p.unit[p.n_units++];
      memset(&u, 0, sizeof(u));
      u.ic0 = (uint8_t)pa[e];
      u.ic1 = pb[e] >= 0 ? (uint8_t)pb[e] : (uint8_t)0xff;
      u.len = (uint8_t)(nu - g0 < TC_G ? nu - g0 : TC_G);
      for (int q = 0; q < u.len; ++q) {
        u.oc[q] = un[g0 + q];
        u.keep[q] = (uint8_t)((ina[un[g0 + q]] ? 1 : 0) | (inb[un[g0 + q]] ? 2 : 0));
      }
    }
  }
}

// unit table of the weight-gradient kernel for inspection / tests (host only): per unit 12 bytes
// {ic0, ic1, len, 0, oc[4], keep[4]}; returns the number of units
extern "C" int lcn_debug_tcw_units(const uint32_t* row17, int FCK, int FCN, int NCK, int NCN, uint8_t* units_out, int max_units) {
  TcwParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < LCN_J; ++i) p.row[i] = row17[i];
  p.FCK = FCK; p.FCN = FCN; p.NCK = NCK; p.NCN = NCN;
  tcw_build_units(p);
  for (int u = 0; u < p.n_units && u < max_units; ++u) memcpy(units_out + 12 * u, &p.unit[u], 12);
  return p.n_units;
}

// dynamic shared memory of a k_tc_wgrad CTA: the operand ring, plus the alignment slack of its 1024-byte base
static inline size_t tcw_smem_bytes() { return (size_t)TCW_STAGES * TCW_STAGE_BYTES + 1024; }

int lcn_tc_wgrad_footprint(bool x3, cudaFuncAttributes* attr, size_t* dyn_smem, int* threads) {
  LCN_CHECK_CUDA(x3 ? cudaFuncGetAttributes(attr, k_tc_wgrad<true>) : cudaFuncGetAttributes(attr, k_tc_wgrad<false>));
  *dyn_smem = tcw_smem_bytes();
  *threads = TCW_THREADS;
  return LCN_OK;
}

static int launch_tc_wgrad(TcwParams& p, const __nv_bfloat16* A, const __nv_bfloat16* dZ, float* dW, int tiles,
                           int sm_count, cudaStream_t st, bool x3 = false) {
  tcw_build_units(p);
  const int units = p.n_units;
  p.tiles = tiles;
  // One CTA is resident per SM (TMEM kernels: profiles/micro/occ.cu): the row range per CTA is the smallest for which
  // the grid is a single wave.  LCN_TCW_SLOTS overrides the slot count for experiments.
  int slots = sm_count;
  int tpc = 1;
  while (tpc < tiles && (long)units * ((tiles + tpc - 1) / tpc) > slots) ++tpc;
  p.tiles_per_cta = tpc;
  int splits = (tiles + tpc - 1) / tpc;
  const size_t smem = tcw_smem_bytes();
  static std::once_flag once;
  static cudaError_t rc = cudaSuccess;
  std::call_once(once, [smem] {
    rc = cudaFuncSetAttribute(k_tc_wgrad<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (rc == cudaSuccess) rc = cudaFuncSetAttribute(k_tc_wgrad<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  });
  LCN_CHECK_CUDA(rc);
  if (x3) lcn_launch(k_tc_wgrad<true>, dim3(dim3(units, splits)), dim3(TCW_THREADS), smem, st, A, dZ, dW, p);
  else lcn_launch(k_tc_wgrad<false>, dim3(dim3(units, splits)), dim3(TCW_THREADS), smem, st, A, dZ, dW, p);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

// mid layers: dWm (dense [P,P], only the nonzero blocks are touched)
int lcn_tc_wgrad(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* A, const __nv_bfloat16* dZ, float* dW,
                 cudaStream_t st, bool x3) {
  TcwParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < LCN_J; ++i) p.row[i] = m->sup.row[i];
  p.FCK = p.FCN = m->FC;
  p.NCK = p.NCN = LCN_J * m->FC;
  p.ldw = m->P;
  return launch_tc_wgrad(p, A, dZ, dW, lay.tiles, m->sm_count, st, x3);
}
// last layer: dW4pad[P][64] += A_L^T dOut16 (one N chunk: 51 columns padded to 64)
int lcn_tc_wgrad_last(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* A, const __nv_bfloat16* dOut16,
                      float* dWpad, cudaStream_t st) {
  TcwParams p;
  memset(&p, 0, sizeof(p));
  for (int i = 0; i < LCN_J; ++i) p.row[i] = 1u;
  p.FCK = m->FC;
  p.FCN = 1;
  p.NCK = LCN_J * m->FC;
  p.NCN = 1;
  p.ldw = 64;
  return launch_tc_wgrad(p, A, dOut16, dWpad, lay.tiles, m->sm_count, st);
}
// first layer: dW1pad[64][P] += X16^T dZ0 (one M chunk: 17*in_F columns padded to 64)
int lcn_tc_wgrad_first(const lcn_model* m, const WsLayout& lay, const __nv_bfloat16* X16, const __nv_bfloat16* dZ,
                       float* dWpad, cudaStream_t st) {
  TcwParams p;
  memset(&p, 0, sizeof(p));
  p.row[0] = (1u << LCN_J) - 1u;
  p.FCK = 1;
  p.FCN = m->FC;
  p.NCK = 1;
  p.NCN = LCN_J * m->FC;
  p.ldw = m->P;
  return launch_tc_wgrad(p, X16, dZ, dWpad, lay.tiles, m->sm_count, st);
}

LCN_KTRACE_EXPORT(gemm)
