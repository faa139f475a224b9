// Data-parallel gradient exchange inside the library: a two-shot all-reduce written for this bucket, over NVLink peer
// memory (SURVEY 8(e)).  The reference has no distributed code at all (network/models_att.py:155-158: one process, one
// tf.Session); this is the exchange step a data-parallel host needs between optimizer.compute_gradients and
// apply_gradients (:408-409).
//
// One process per GPU.  Every rank owns ONE device allocation [flags | gradient bucket | staging slots] that all peers map
// through CUDA IPC (lcn_dp_export -> the host all-gathers the 64-byte handles -> lcn_dp_connect); lcn_dp_bucket() is the
// pointer the caller passes as d_grads_raw, so the backward pass writes its gradients straight into peer-visible memory.
// At the end of lcn_model_backward (kernels in lcn_kernels.cu, next to the pack kernel whose unit table they share):
//
//   k_dp_push     the units of the bucket -- nonzero joint-pair blocks of the weight gradients, small tensors -- are dealt
//                 round-robin to the ranks; every rank copies its copy of the units it does not own into the owner's staging
//                 slot [sender] with 16-byte peer STORES (posted writes: no NVLink round trip), then publishes
//                 pushed[me] = ++epoch at every peer                                      (st.release.sys over NVLink)
//   k_dp_reduce   the owner waits for pushed[p] >= epoch from every peer, adds its own block and the world-1 staged copies
//                 (local reads, fixed order: every rank ends up with bit-identical gradients) and stores the mean into ALL
//                 `world` buckets, in place (peer stores again); the masked-out 40 % of the bucket never travels; the last
//                 CTA publishes done[me] = epoch at every peer
//   k_dp_wait     waits until done[p] >= epoch for every p: every unit of this rank's bucket holds the mean -- the chain
//                 rule / Adam kernels that follow see averaged gradients
//
// The exchange is STREAMED (backward_impl in lcn_kernels.cu): the units of mid layer l are pushed / reduced on a third stream
// of the model as soon as that layer's weight-gradient GEMM has finished on the side stream, under the rest of the backward
// pass; layer 1 (finishes last), the first / last layer and the small tensors go in one exchange after the join, followed
// by k_dp_wait.  Different layers use disjoint unit sets, hence disjoint staging areas and bucket regions, so consecutive
// exchanges of one step do not interfere; the epoch counts exchanges, not steps.  The last CTA of an exchange kernel
// publishes the epoch with ONE THREAD PER RANK: eight release stores in sequence cost eight NVLink round trips on the
// exposed end of the step (8 GPUs: 0.676 -> 0.630 ms per step together with the streaming, DESIGN.md section 5).
//
// Each gradient byte crosses the NVLink fabric once in each direction, always as a store.  Measured against ncclAllReduce
// of the packed bucket (with its pack / unpack passes, two graph replays), against the same exchange with peer LOADS, and
// against NCCL all-reduces per layer overlapped with the backward pass (SLOWER than no overlap: the NCCL CTAs take SMs
// from single-wave GEMMs and two-blocks-per-SM elementwise kernels): DESIGN.md section 5.
//
// Why this is safe without a cluster-wide barrier: flags only ever grow (epoch numbers), every rank executes the same
// sequence of exchanges, unit sets of different ranks are disjoint (in-place is race free), and the waits order every
// reuse -- an owner overwrites a unit in a peer's bucket only after that peer's pushed(e), i.e. after the peer has read
// it; a rank starts the next backward pass (which overwrites its bucket) and the next push (which overwrites the owners'
// staging slots) only after k_dp_wait(e), i.e. after every owner published done(e), which it does after its last read of
// its staging slots and its last store into this rank's bucket.  All three kernels take only device pointers and read
// the epoch from device memory, so the exchange is captured into the train-step CUDA graph like any other kernel of the
// step.  No kernel needs a peer's kernel to be co-scheduled in order to FINISH its own loads and stores; the waits are on
// flags that the peers' stream-ordered work sets unconditionally, so a late peer delays, never deadlocks.
//
// Synchronised BatchNorm (lcn_dp_sync_batch_norm, off by default): every BatchNorm layer of a training step normalises
// with the moments of the GLOBAL batch.  A step has 2 * n_bn sync points (point l: forward of BN layer l, point n_bn + l:
// its backward), each one launch of k_bn_sync on the caller's stream:
//
//   forward   (n, mean, M2) per channel of this rank's rows x 17 joints (from the GEMM's fp64 sums or from k_bn_finalize)
//             -> merged in rank order (k_bn_finalize's formula, fp64) -> (mean, rstd) of the global batch into the stat
//             buffer that k_bn_act(_pre), the backward pass and read_tensor kinds 4 / 5 read
//   backward  (n, sum dy, sum dy*xhat) per channel from k_bn_bwd_reduce -> summed in rank order (fp64) -> (S1 / N, S2 / N)
//             with N = 17 x global rows, which k_bn_bwd_apply uses instead of its local sums / local count
//
// The BN area behind the staging slots holds, per point, one slot of 3 F doubles per rank and three flag words per rank.
// k_bn_sync: (1) waits until consumed[pt][p] >= e - 1 for every p, (2) stores its payload into slot [pt][me] of every
// rank with peer stores, (3) publishes ready[pt][me] = e at every rank (st.release.sys), (4) waits for ready[pt][p] >= e
// for every p (ld.acquire.sys), merges the `world` slots in rank order -- every rank computes bit-identical statistics --
// and (5) publishes consumed[pt][me] = e at every rank.  e = ++epoch[pt], a local counter in device memory, so the kernel
// is captured into the train-step graph like the gradient exchange.
// Slot-reuse invariant: a rank overwrites slot [pt][me] at rank p (epoch e) only after p has published consumed[pt] = e - 1,
// i.e. after p's last read of that slot for epoch e - 1.  This holds with no gradient exchange between two steps (mode 0,
// eager forward-only calls), because it rests on the point's own flags and not on the order of other kernels.  Every
// rank must run the same sequence of training forward / backward calls while sync is on.
#include <stdlib.h>

#include <algorithm>

#include "lcn_internal.cuh"

#define LCN_DP_MAX_WORLD 8
#define LCN_DP_FLAG_BYTES 4096
#define LCN_DP_STREAMED 1
#define LCN_DP_AT_END 2

struct LcnDpFlags {                       // lives at the start of every rank's exchange allocation
  unsigned long long epoch;               // local: exchanges started by this rank
  unsigned long long pad0[15];
  unsigned long long ready[LCN_DP_MAX_WORLD];   // pushed[p]: written by rank p -- its copies of our units sit in our staging slot p
  unsigned long long pad1[8];
  unsigned long long done[LCN_DP_MAX_WORLD];    // done[p]: written by rank p -- the units it owns hold epoch's mean in our bucket
  unsigned long long pad2[8];
  unsigned int ticket;                    // local: CTAs of k_dp_reduce that have finished
};

// BN area (synchronised BatchNorm), behind the staging slots: LcnBnFlags[points], then double[points][world][3 F]
struct LcnBnFlags {
  unsigned long long ready[LCN_DP_MAX_WORLD];      // ready[p]: written by rank p -- its payload of epoch ready[p] is in slot p here
  unsigned long long consumed[LCN_DP_MAX_WORLD];   // consumed[p]: written by rank p -- it has merged epoch consumed[p]
  unsigned long long epoch;                        // local: uses of the point by this rank
  unsigned long long pad[7];
};

struct LcnDp {
  int rank = 0, world = 1;
  int mode = LCN_DP_STREAMED;             // lcn_dp_enable: 0 off, 1 streamed behind the weight-gradient GEMMs, 2 one exchange at the end
  bool connected = false;
  bool sync_bn = false;                   // lcn_dp_sync_batch_norm
  int64_t count = 0;                      // floats in the bucket (= lcn_model_param_count)
  int64_t packed = 0;                     // floats in one staging slot (= lcn_model_grad_compact_count, 16-byte rounded)
  size_t stage_off = 0, slot_bytes = 0;   // staging: `world` slots behind the bucket
  size_t bn_off = 0, bn_slot_off = 0;     // BN area: flags of the 2 n_bn sync points, then their slots
  int bn_points = 0, F = 0;
  size_t bytes = 0;
  char* base = nullptr;                   // own allocation
  char* peer[LCN_DP_MAX_WORLD] = {};      // mapped allocations (peer[rank] == base)
};

struct DpFlagPtrs {                       // by-value kernel argument
  LcnDpFlags* flags[LCN_DP_MAX_WORLD];
  int rank, world;
};

namespace {

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__global__ void k_dp_wait(DpFlagPtrs d) {
  lcn_pdl_prologue();
  LcnDpFlags* mine = d.flags[d.rank];
  if ((int)threadIdx.x < d.world) {
    const unsigned long long e = mine->epoch;
    unsigned long long spins = 0;
    while (ld_acquire_sys(&mine->done[threadIdx.x]) < e) {
      if (++spins > (1ull << 28)) {        // seconds: a peer died or the ranks disagree on the call sequence
        printf("lcn_dp: wait for a peer's done flag timed out\n");
        __trap();
      }
    }
  }
}

__device__ __forceinline__ void bn_wait_flag(const unsigned long long* p, unsigned long long e, const char* what) {
  unsigned long long spins = 0;
  while (ld_acquire_sys(p) < e) {
    if (++spins > (1ull << 28)) {          // seconds: a peer died or the ranks disagree on the call sequence
      printf("lcn_dp: synchronised BatchNorm: wait for a peer's %s flag timed out\n", what);
      __trap();
    }
  }
}

struct BnSyncArgs {                       // by-value kernel argument: one sync point
  double* slot_at[LCN_DP_MAX_WORLD];      // slot [point][me] at rank p
  unsigned long long* ready_at[LCN_DP_MAX_WORLD];
  unsigned long long* consumed_at[LCN_DP_MAX_WORLD];
  const double* slots;                    // local slots [point][0 .. world)
  LcnBnFlags* mine;                       // local flags of the point
  int rank, world;
};

// One CTA, thread f = channel f (F <= 256).  kind: LCN_BN_SYNC_GACC (src: double[LCN_GACC_REP][F][2] sums of x, x^2),
// LCN_BN_SYNC_MOMENTS (src: double[F][3] (n, mean, M2) of k_bn_finalize) -> out float[F][2] (mean, rstd);
// LCN_BN_SYNC_SUMS (src: float[F][2] (sum dy, sum dy*xhat)) -> out float[F][2] (S1 / N, S2 / N).
__global__ void __launch_bounds__(256) k_bn_sync(BnSyncArgs s, int kind, const void* __restrict__ src,
                                                 float* __restrict__ out, int F, double n_local) {
  lcn_pdl_wait();    // no early trigger: the next kernel's CTAs must not sit on SMs while this one waits for the peers
  __shared__ unsigned long long s_e;
  const int f = threadIdx.x;
  double a = 0.0, b = 0.0;                // forward: (mean, M2); backward: (S1, S2) of this rank's rows
  if (f < F) {
    if (kind == LCN_BN_SYNC_GACC) {
      const double* g = static_cast<const double*>(src);
      double S1 = 0.0, S2 = 0.0;
      for (int rep = 0; rep < LCN_GACC_REP; ++rep) {
        S1 += g[((size_t)rep * F + f) * 2];
        S2 += g[((size_t)rep * F + f) * 2 + 1];
      }
      a = S1 / n_local;
      b = fmax(S2 - S1 * a, 0.0);
    } else if (kind == LCN_BN_SYNC_MOMENTS) {
      const double* mo = static_cast<const double*>(src);
      a = mo[f * 3 + 1];
      b = mo[f * 3 + 2];
    } else {
      const float* su = static_cast<const float*>(src);
      a = (double)su[f * 2];
      b = (double)su[f * 2 + 1];
    }
  }
  if (threadIdx.x == 0) s_e = s.mine->epoch + 1;
  __syncthreads();
  const unsigned long long e = s_e;
  // (1) every rank has merged the previous epoch: its slot [point][me] may be overwritten
  if ((int)threadIdx.x < s.world) bn_wait_flag(&s.mine->consumed[threadIdx.x], e - 1, "consumed");
  __syncthreads();
  // (2) payload into slot [point][me] of every rank, (3) ready = e at every rank
  if (f < F) {
    for (int p = 0; p < s.world; ++p) {
      double* d = s.slot_at[p] + (size_t)f * 3;
      d[0] = n_local;
      d[1] = a;
      d[2] = b;
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < s.world) {
    __threadfence_system();
    st_release_sys(s.ready_at[threadIdx.x], e);
  }
  // (4) every rank's payload of epoch e has landed here; merge in rank order
  if ((int)threadIdx.x < s.world) bn_wait_flag(&s.mine->ready[threadIdx.x], e, "ready");
  __syncthreads();
  if (f < F) {
    const size_t stride = (size_t)F * 3;
    double n = __ldcg(s.slots + (size_t)f * 3), x = __ldcg(s.slots + (size_t)f * 3 + 1), y = __ldcg(s.slots + (size_t)f * 3 + 2);
    for (int p = 1; p < s.world; ++p) {
      const double* q = s.slots + p * stride + (size_t)f * 3;
      const double nq = __ldcg(q), xq = __ldcg(q + 1), yq = __ldcg(q + 2);
      if (kind == LCN_BN_SYNC_SUMS) {
        x += xq;
        y += yq;
        n += nq;
      } else {                             // pairwise merge of (n, mean, M2)
        const double nt = n + nq, d = xq - x;
        x += d * (nq / nt);
        y += yq + d * d * (n * nq / nt);
        n = nt;
      }
    }
    if (kind == LCN_BN_SYNC_SUMS) {
      out[f * 2] = (float)(x / n);
      out[f * 2 + 1] = (float)(y / n);
    } else {
      out[f * 2] = (float)x;
      out[f * 2 + 1] = (float)(1.0 / sqrt(y / n + (double)LCN_BN_EPS));
    }
  }
  // (5) this rank has read every slot of the point for epoch e
  __syncthreads();
  if ((int)threadIdx.x < s.world) st_release_sys(s.consumed_at[threadIdx.x], e);
  if (threadIdx.x == 0) s.mine->epoch = e;
}

}  // namespace

// ---- host side ----------------------------------------------------------------------------------------------------
extern "C" int lcn_dp_export(lcn_model* m, int world, void* h_handle64) {
  LCN_REQUIRE(m != nullptr && h_handle64 != nullptr, "null argument");
  LCN_REQUIRE(m->dp == nullptr, "the model already has an exchange buffer");
  LCN_REQUIRE(world == 2 || world == 4 || world == 8, "world size %d not in {2, 4, 8}", world);
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  static_assert(sizeof(LcnDpFlags) <= LCN_DP_FLAG_BYTES, "flag block");
  LcnDp* dp = new LcnDp();
  dp->world = world;
  dp->count = m->n_params;
  dp->packed = (lcn_grad_compact_count(m) + 3) & ~(int64_t)3;
  dp->stage_off = LCN_DP_FLAG_BYTES + (((size_t)dp->count * 4 + 255) & ~(size_t)255);
  dp->slot_bytes = ((size_t)dp->packed * 4 + 255) & ~(size_t)255;
  dp->bn_points = 2 * m->n_bn;
  dp->F = m->d.F;
  dp->bn_off = dp->stage_off + (size_t)world * dp->slot_bytes;
  dp->bn_slot_off = dp->bn_off + ((sizeof(LcnBnFlags) * dp->bn_points + 255) & ~(size_t)255);
  dp->bytes = dp->bn_slot_off + sizeof(double) * dp->bn_points * world * 3 * dp->F;
  // the one device allocation the library makes: peers have to map it, so it cannot come from the caller's allocator
  cudaError_t e = cudaMalloc(&dp->base, dp->bytes);
  if (e == cudaSuccess) e = cudaMemset(dp->base, 0, dp->bytes);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, dp->base);
  if (e != cudaSuccess) {
    lcn_set_error("lcn_dp_export: %s", cudaGetErrorString(e));
    if (dp->base) cudaFree(dp->base);
    delete dp;
    (void)cudaGetLastError();
    return LCN_ECUDA;
  }
  memcpy(h_handle64, &h, sizeof(h));
  m->dp = dp;
  return LCN_OK;
}

extern "C" float* lcn_dp_bucket(const lcn_model* m) {
  return (m && m->dp) ? reinterpret_cast<float*>(m->dp->base + LCN_DP_FLAG_BYTES) : nullptr;
}

extern "C" int lcn_dp_connect(lcn_model* m, const void* h_handles, int rank, int world) {
  LCN_REQUIRE(m != nullptr && h_handles != nullptr, "null argument");
  LCN_REQUIRE(m->dp != nullptr && !m->dp->connected, "call lcn_dp_export first (once)");
  LCN_REQUIRE(world == m->dp->world && rank >= 0 && rank < world, "rank %d / world %d (exported for world %d)", rank, world,
              m->dp->world);
  LcnDp* dp = m->dp;
  dp->rank = rank;
  for (int p = 0; p < world; ++p) {
    if (p == rank) {
      dp->peer[p] = dp->base;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(h_handles) + (size_t)p * sizeof(h), sizeof(h));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      lcn_set_error("lcn_dp_connect: cudaIpcOpenMemHandle(rank %d) -> %s (are the GPUs NVLink / P2P peers?)", p, cudaGetErrorString(e));
      (void)cudaGetLastError();
      return LCN_ECUDA;
    }
    dp->peer[p] = static_cast<char*>(ptr);
  }
  dp->connected = true;
  return LCN_OK;
}

extern "C" int lcn_dp_world(const lcn_model* m) { return (m && m->dp && m->dp->connected) ? m->dp->world : 1; }

extern "C" int lcn_dp_enable(lcn_model* m, int on) {
  LCN_REQUIRE(m != nullptr, "null model");
  LCN_REQUIRE((m->dp != nullptr && m->dp->connected) || !on, "lcn_dp_enable: the model is not connected (lcn_dp_export / lcn_dp_connect)");
  LCN_REQUIRE(on >= 0 && on <= 2, "lcn_dp_enable: mode %d not in {0, 1, 2}", on);
  if (m->dp) m->dp->mode = on;
  return LCN_OK;
}

extern "C" int lcn_dp_sync_batch_norm(lcn_model* m, int on) {
  LCN_REQUIRE(m != nullptr, "null model");
  LCN_REQUIRE((m->dp != nullptr && m->dp->connected) || !on,
              "lcn_dp_sync_batch_norm: the model is not connected (lcn_dp_export / lcn_dp_connect)");
  if (m->dp) m->dp->sync_bn = on != 0;
  return LCN_OK;
}

bool lcn_bn_sync_on(const lcn_model* m) {
  return m->dp != nullptr && m->dp->connected && m->dp->world > 1 && m->dp->sync_bn;
}

// One sync point (see the header of this file): `rows` = this rank's training batch.
int lcn_bn_sync(const lcn_model* m, int point, int kind, const void* src, float* out, int64_t rows, cudaStream_t st) {
  const LcnDp* dp = m->dp;
  LCN_REQUIRE(point >= 0 && point < dp->bn_points && m->d.F == dp->F, "internal: BatchNorm sync point %d", point);
  BnSyncArgs s;
  memset(&s, 0, sizeof(s));
  const size_t pt_slots = (size_t)dp->world * 3 * dp->F;     // doubles per point
  for (int p = 0; p < dp->world; ++p) {
    LcnBnFlags* fl = reinterpret_cast<LcnBnFlags*>(dp->peer[p] + dp->bn_off) + point;
    s.slot_at[p] = reinterpret_cast<double*>(dp->peer[p] + dp->bn_slot_off) + point * pt_slots + (size_t)dp->rank * 3 * dp->F;
    s.ready_at[p] = &fl->ready[dp->rank];
    s.consumed_at[p] = &fl->consumed[dp->rank];
  }
  s.slots = reinterpret_cast<const double*>(dp->base + dp->bn_slot_off) + point * pt_slots;
  s.mine = reinterpret_cast<LcnBnFlags*>(dp->base + dp->bn_off) + point;
  s.rank = dp->rank;
  s.world = dp->world;
  lcn_launch(k_bn_sync, dim3(1), dim3(256), 0, st, s, kind, src, out, dp->F, (double)rows * LCN_J);
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

void lcn_dp_destroy(lcn_model* m) {
  if (m == nullptr || m->dp == nullptr) return;
  LcnDp* dp = m->dp;
  cudaDeviceSynchronize();
  for (int p = 0; p < dp->world; ++p)
    if (p != dp->rank && dp->peer[p] != nullptr) cudaIpcCloseMemHandle(dp->peer[p]);
  if (dp->base) cudaFree(dp->base);
  (void)cudaGetLastError();
  delete dp;
  m->dp = nullptr;
}

int lcn_dp_mode(const lcn_model* m) {
  return (m->dp != nullptr && m->dp->connected && m->dp->world > 1) ? m->dp->mode : 0;
}

static DpFlagPtrs dp_flag_ptrs(const LcnDp* dp) {
  DpFlagPtrs f;
  memset(&f, 0, sizeof(f));
  f.rank = dp->rank;
  f.world = dp->world;
  for (int p = 0; p < dp->world; ++p) f.flags[p] = reinterpret_cast<LcnDpFlags*>(dp->peer[p]);
  return f;
}

// Average the units [u0, u1) minus [s0, s1) of the raw-gradient bucket over the ranks, in place, on `st` (u1 < 0: to the
// end of the bucket).  Every rank makes the same sequence of calls.  The means have landed in this rank's bucket only after a
// following lcn_dp_wait in stream order.
int lcn_dp_exchange_units(const lcn_model* m, float* graw, int u0, int u1, int s0, int s1, int max_ctas, cudaStream_t st) {
  LcnDp* dp = m->dp;
  LCN_REQUIRE(graw == reinterpret_cast<float*>(dp->base + LCN_DP_FLAG_BYTES),
              "data-parallel model: d_grads_raw must be the peer-mapped bucket returned by lcn_dp_bucket()");
  DpFlagPtrs f = dp_flag_ptrs(dp);
  float *buckets[LCN_DP_MAX_WORLD], *stage_at[LCN_DP_MAX_WORLD], *stage_local[LCN_DP_MAX_WORLD];
  unsigned long long *pushed_at[LCN_DP_MAX_WORLD], *done_at[LCN_DP_MAX_WORLD];
  for (int p = 0; p < dp->world; ++p) {
    buckets[p] = reinterpret_cast<float*>(dp->peer[p] + LCN_DP_FLAG_BYTES);
    stage_at[p] = reinterpret_cast<float*>(dp->peer[p] + dp->stage_off + (size_t)dp->rank * dp->slot_bytes);   // my slot at rank p
    stage_local[p] = reinterpret_cast<float*>(dp->base + dp->stage_off + (size_t)p * dp->slot_bytes);          // sender p's slot here
    pushed_at[p] = &f.flags[p]->ready[dp->rank];
    done_at[p] = &f.flags[p]->done[dp->rank];
  }
  LcnDpFlags* mine = f.flags[dp->rank];
  return lcn_launch_dp_exchange(m, buckets, stage_at, stage_local, mine->ready, pushed_at, done_at, &mine->epoch, &mine->ticket,
                                dp->rank, dp->world, u0, u1, s0, s1, max_ctas, st);
}

// Every exchange enqueued before this call (on streams `st` is ordered after) is complete when this kernel ends.
int lcn_dp_wait(const lcn_model* m, cudaStream_t st) {
  lcn_launch(k_dp_wait, dim3(1), dim3(32), 0, st, dp_flag_ptrs(m->dp));
  LCN_CHECK_LAUNCH();
  return LCN_OK;
}

LCN_KTRACE_EXPORT(dp)
