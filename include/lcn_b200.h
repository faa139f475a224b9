/*
 * lcn_b200.h -- C ABI of liblcn_b200.so: the B200 (sm_100a) implementation of the adgx/lcn-pose
 * LCN hot path.  Plain C, plain pointers and sizes; no torch / TF types.
 *
 * The reference has no FFI or plugin layer (it is TensorFlow graph code + NumPy); the boundary it
 * exposes for this path is the Python class API of network/models_att.py (cgcnn: mask construction,
 * mask_weights, LCN layer stack, loss, Adam, predict batching) and the function API of
 * tools/tools.py (image_to_camera_frame, procrustes/align_to_gt) consumed by evaluate.py.  Each
 * entry point below cites the reference code it replaces (paths relative to the reference root).
 * Host bindings: lcn_pose_b200/_lib.py (ctypes, used here) and the TF custom-op stub shown in
 * INTEGRATION.md (cannot be built in this image: no TensorFlow headers).
 *
 * Conventions
 *  - every pointer named d_* is a DEVICE pointer owned by the caller; h_* is a host pointer.
 *  - every launch-type call takes a cudaStream_t (passed as void*) and only enqueues work; the
 *    library never synchronises the device and never allocates device memory.
 *  - every function returns 0 (LCN_OK) or a negative LCN_E* code; the message is available from
 *    lcn_last_error() (thread local).  No C++ exception crosses the boundary.
 *  - a model handle's tables (block lists, offsets) are immutable after creation.  It also owns two side streams and
 *    a few events, created on first use: the weight-gradient GEMMs of lcn_model_backward and the edge-layer packs of
 *    lcn_model_prepare_weights run on one, forked from and joined to the caller's stream; the data-parallel exchange
 *    of finished weight gradients (lcn_dp_enable mode 1) runs on the other.  A call that cannot create them returns
 *    LCN_ECUDA.  Calls that use them serialise on a mutex inside the handle while they ENQUEUE (never while the GPU
 *    runs), so any number of host threads may call into the same handle with distinct streams and workspaces;
 *    one-time kernel-attribute setup is guarded by std::call_once.
 *  - matrices are row-major; feature index inside a row is joint-major: column j*F + f
 *    (network/models_att.py:582); mask index is [input joint, output joint] (:583).
 */
#ifndef LCN_B200_H_
#define LCN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCN_JOINTS 17

enum {
  LCN_OK = 0,
  LCN_EINVAL = -1,   /* bad argument / unsupported shape */
  LCN_ECUDA = -2,    /* CUDA runtime error (message has the cudaError string) */
  LCN_ENOMEM = -3,   /* workspace too small */
  LCN_ESTATE = -4    /* call order violated (e.g. backward before forward) */
};

/* arithmetic path of the LCN layers -- BOTH run every mid-layer GEMM (forward, input gradient, weight gradient) on the
 * tcgen05 tensor cores with fp32 accumulation in TMEM; they differ in how operands are stored */
enum {
  LCN_PATH_FP32 = 0, /* the 1e-4 parity path ("fp32/TF32 path" of the north_star): activations and packed weights are
                        split-bf16 pairs v = hi + lo (16 significand bits) and every block product is three tensor-core
                        products hi*hi + hi*lo + lo*hi.  Single-pass TF32 (10-bit mantissa) measures 8e-5 per layer, too
                        close to the 1e-4 bar; this measures 5e-7.  The K = 17*in_F first layer and the N = 51 head run
                        on CUDA cores in fp32 (< 1.3 % of the FLOPs, degenerate MMA shapes).                           */
  LCN_PATH_BF16 = 1  /* bf16 operands, one product per block: the 1e-2 path, 3x fewer tensor-core FLOPs, half the bytes */
};

enum {
  LCN_MASK_LOCALLY_CONNECTED = 0, /* trainable softmax(var,axis=0)*support, models_att.py:547-571 */
  LCN_MASK_CONSTANT = 1           /* constant mask values (exponential), models_att.py:573-574     */
};

/* Mirrors the cgcnn constructor kwargs that shape the arithmetic (models_att.py:478-506). */
typedef struct lcn_model_desc {
  int32_t F;            /* channels per joint ("F"), multiple of 64                               */
  int32_t in_F;         /* input features per joint ("in_F"), >= 2                                */
  int32_t num_layers;   /* residual two_linear blocks ("num_layers")                              */
  int32_t mask_kind;    /* LCN_MASK_*                                                             */
  int32_t residual;     /* models_att.py:704                                                      */
  int32_t batch_norm;   /* models_att.py:664 (only 1 is implemented on device)                    */
  int32_t max_norm;     /* tf.clip_by_norm(w, 1) before masking, models_att.py:659                */
  int32_t path;         /* LCN_PATH_*                                                             */
  float support[LCN_JOINTS * LCN_JOINTS];    /* [in_joint, out_joint] != 0 where a block exists    */
  float const_mask[LCN_JOINTS * LCN_JOINTS]; /* mask values when mask_kind == LCN_MASK_CONSTANT    */
} lcn_model_desc;

typedef struct lcn_model lcn_model; /* opaque */

/* ---- library ---- */
const char* lcn_version(void);
const char* lcn_last_error(void);

/* CRC32C (Castagnoli) of HOST memory, continuing from `crc` (0 to start): the checksum TensorFlow's Saver V2 files carry
 * (tools/tf_checkpoint.py reads and writes the reference's checkpoints, models_att.py:256-260,445-463). */
uint32_t lcn_crc32c(const void* h_data, size_t n, uint32_t crc);

/* ---- mask construction on the host, bit exact (tools/params_help.py:8-20, tools/filter_hub.py:4-20,
 *      network/models_att.py:14-69) ---- */
int lcn_neighbour_matrix(int knn, float* h_out /* [17*17] float32 0/1 */);
int lcn_exponential_matrix(float* h_out /* [17*17] float32 */);

/* ---- model handle ---- */
int lcn_model_create(const lcn_model_desc* desc, lcn_model** out);
void lcn_model_destroy(lcn_model* m);

/* Flat fp32 parameter vector (also the layout of Adam m, v and of gradients).  Tensor names follow
 * the reference's TF variable names (SURVEY 8(b)): "mask", "linear_model/w1", ".../b1",
 * "linear_model/two_linear_{i}/w2_{i}", ..., "linear_model/w4", ".../b4",
 * "<bn layer>/gamma", "<bn layer>/beta". */
int64_t lcn_model_param_count(const lcn_model* m);
int lcn_model_num_tensors(const lcn_model* m);
int lcn_model_tensor_info(const lcn_model* m, int index, char* name_buf, int name_buf_len,
                          int64_t* offset, int32_t* rows, int32_t* cols);

/* Row geometry.  A "group" is one BatchNorm batch: `bn_group` consecutive poses share statistics
 * (models_att.py:588-612 reduces over batch x joints; predict() zero-pads the last batch,
 * :92-97, and the zero rows count).  n_rows = number of real poses; the last group is padded with
 * zero inputs up to bn_group.  Training uses one group (bn_group = batch). */
size_t lcn_model_workspace_bytes(const lcn_model* m, int64_t n_rows, int32_t bn_group, int training);

/* (a4) clip_by_norm + mask_weights + pack, for every layer; must run after any parameter change
 * and before forward.  models_att.py:659-660,690-691,726-728,762-764 and :534-586. */
int lcn_model_prepare_weights(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, void* stream);

/* Per-step scalars resident in DEVICE memory.  When the d_dyn argument of lcn_model_forward / lcn_model_adam_step is
 * not NULL, the kernels read `step` (dropout Philox offset) / `lr_t` from it at execution time and ignore the
 * by-value arguments of the same name: a CUDA graph captured around one train step (all calls only enqueue work on
 * the caller's stream, so they are capturable) can then be replayed every step after rewriting these 16 bytes.
 * The reference pays a sess.run feed/launch sequence per step (models_att.py:204-212). */
typedef struct lcn_step_scalars {
  uint64_t step;
  float lr_t;
  float reserved;
} lcn_step_scalars;

/* (a5)-(a8) cgcnn._inference_lcn, models_att.py:707-775.  d_x [n_rows, 17*in_F] fp32,
 * d_out [n_rows, 51] fp32.  dropout_rate 0 reproduces predict() (:102); the keep decision of
 * element e of layer l at step `step` is lcn_dropout_mask()'s. */
int lcn_model_forward(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes,
                      const float* d_x, int64_t n_rows, int32_t bn_group, int training,
                      float dropout_rate, uint64_t seed, uint64_t step, float* d_out,
                      const lcn_step_scalars* d_dyn, void* stream);

/* A sub-range of the stack, for the reference's method-level layer API: runs the linear layers [layer_begin, layer_end)
 * (0 = w1 ... 2*num_layers+1 = w4; each of the first 2*num_layers+1 is followed by its BatchNorm / LeakyReLU / dropout
 * and, where the reference has one, the residual add) on the TRAINING workspace layout, where every layer keeps its
 * own buffers.  The input of layer_begin > 0 is the activation A_{layer_begin-1} already in the workspace (left there
 * by a previous forward, or injected with lcn_model_write_tensor); the output A_{layer_end-1} is read with
 * lcn_model_read_tensor(kind 1).  cgcnn.two_linear(xin, dropout, idx) (models_att.py:630-705) is
 * write_tensor(A_{2 idx}) + forward_layers(2 idx + 1, 2 idx + 3) + read_tensor(A_{2 idx + 2}).  d_x is needed when the
 * range contains the first or the last layer, d_out when it contains the last. */
int lcn_model_forward_layers(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, const float* d_x,
                             int64_t n_rows, int32_t bn_group, float dropout_rate, uint64_t seed, uint64_t step,
                             int layer_begin, int layer_end, float* d_out, void* stream);

/* Same arithmetic, with a parity tap: valid only where inference runs as the fused cluster kernel (bf16 path,
 * F = 64, bn_group <= 256; LCN_EINVAL otherwise).  d_taps receives every layer output A_l (after
 * BN / LeakyReLU / residual) as bf16 in the kernel's tile-major layout: [n_bn][tile][17 chunks][128 rows][64]
 * with the 16-byte chunk c of row r stored at c ^ (r & 7); tile = group * ceil(bn_group/128) + row tile. */
int lcn_model_forward_taps(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes,
                           const float* d_x, int64_t n_rows, int32_t bn_group, float* d_out,
                           void* d_taps, size_t taps_bytes, void* stream);

/* (a9)+(autodiff) base_model.loss models_att.py:352-380 and optimizer.compute_gradients :408.
 * Requires a preceding lcn_model_forward(training=1) on the same workspace.  d_labels [n_rows,51].
 * d_loss: one float (mean squared error).  d_grads_raw: flat, param layout; holds dL/dWm for the
 * weight tensors (gradient w.r.t. the masked effective weight) and true gradients for biases / BN. */
int lcn_model_backward(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes,
                       const float* d_x, const float* d_labels, int64_t n_rows,
                       float dropout_rate, uint64_t seed, uint64_t step,
                       float* d_loss, float* d_grads_raw, void* stream);

/* Chain rule through mask_weights, clip_by_norm and the mask softmax (SURVEY 9-Q5/Q6):
 * reduces <dWm, W> per joint pair, then either writes the true dense gradients (d_grads_out != NULL;
 * used by tests and by data-parallel hosts that want to inspect them) ... */
int lcn_model_finalize_grads(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes,
                             const float* d_grads_raw, float* d_grads_out, void* stream);

/* Data-parallel exchange (SURVEY 8(e): "allreduce of the packed nonzero-block gradient"; the reference has no
 * distributed code, models_att.py:155-158).  The raw-gradient bucket has the parameter layout, so 40 % of it (knn=3) are
 * the never-written zero entries of masked-out joint-pair blocks.  lcn_model_pack_grads gathers what backward actually
 * produces -- the nonzero Fi x Fo blocks of every weight matrix, then every other tensor whole -- into
 * lcn_model_grad_compact_count(m) contiguous floats; the host all-reduces that buffer and lcn_model_unpack_grads
 * scatters it back before lcn_model_adam_step.  Both only enqueue on `stream`. */
int64_t lcn_model_grad_compact_count(const lcn_model* m);
int lcn_model_pack_grads(lcn_model* m, const float* d_grads_raw, float* d_compact, void* stream);
int lcn_model_unpack_grads(lcn_model* m, const float* d_compact, float* d_grads_raw, void* stream);

/* Data-parallel training with the exchange INSIDE the backward pass (csrc/lcn_dp.cu): a two-shot all-reduce of the
 * packed bucket over NVLink peer memory, written for this bucket -- reduce-scatter by peer stores into the owner's staging slots, all-gather
 * by peer stores into every rank's bucket, flags with release / acquire at system scope, no library collective.  One process per GPU (<= 8 GPUs of one
 * NVLink domain; world size 2, 4 or 8).  Setup: every rank calls lcn_dp_export (allocates the rank's gradient bucket -- the
 * ONE device allocation this library makes, because peers must be able to map it -- and returns its 64-byte CUDA IPC
 * handle), the host all-gathers the handles by any means (torch.distributed, MPI, a file), every rank calls
 * lcn_dp_connect with all `world` handles in rank order and from then on passes lcn_dp_bucket(m) as d_grads_raw.
 * lcn_model_backward then leaves the MEAN of the ranks' gradients in the bucket, exchanged in place by the library's own
 * kernel (in stream order; capturable into the caller's CUDA graph like every other call), so
 * lcn_model_adam_step needs no change and a data-parallel step is one graph.  Every rank must issue the same sequence of
 * lcn_model_backward calls.  By default BatchNorm statistics stay per GPU (== the reference at batch B per GPU); see
 * lcn_dp_sync_batch_norm for statistics of the global batch.
 * The exchange is STREAMED: the joint-pair blocks of every mid-layer weight gradient travel on a third stream of the
 * model as soon as that layer's weight-gradient GEMM has finished, under the rest of the backward pass; only the first /
 * last layer and the small tensors (< 2 % of the bucket) are exchanged after it.
 * lcn_dp_enable(m, mode): 1 (default) streamed; 2 one exchange of the whole bucket at the end of the backward pass;
 * 0 no exchange, for calls that want the local gradient (tests, the host-side packed-bucket path above). */
int lcn_dp_export(lcn_model* m, int world, void* h_handle64);
float* lcn_dp_bucket(const lcn_model* m);   /* the rank's peer-mapped gradient bucket: pass it as d_grads_raw */
int lcn_dp_connect(lcn_model* m, const void* h_handles /* world x 64 bytes, rank order */, int rank, int world);
int lcn_dp_world(const lcn_model* m);
int lcn_dp_enable(lcn_model* m, int mode);
/* Synchronised BatchNorm (off by default; on != 0 needs a connected model, off is always accepted).  With it on, every
 * training forward pass (lcn_model_forward(training=1), one BN group = this rank's n_rows) normalises each BatchNorm
 * layer with the mean and biased variance of ALL ranks' rows x 17 joints -- the statistics a single GPU computes on the
 * concatenated batch -- and lcn_model_backward uses the matching global sums: dZ = gamma rstd (d - S1/N - xhat S2/N),
 * S1 = sum over ranks and rows of d, S2 = of d xhat, N = 17 x global rows.  Each rank's gradient is then `world` times
 * its share of the gradient of (1/world) sum_r L_r, so the bucket's mean (any lcn_dp_enable mode, or the host's own
 * all-reduce in mode 0) is that gradient; gamma / beta gradients stay per-rank sums.  Shards may differ in size.  Every
 * rank combines the ranks' moments in rank order in fp64, so the statistics are bit-identical across ranks.  Costs one
 * NVLink flag round trip per BN layer in the forward and in the backward pass.  Inference keeps per-group statistics;
 * lcn_model_forward_layers returns LCN_ESTATE while sync is on.  lcn_model_read_tensor kinds 4 / 5 return the global
 * statistics. */
int lcn_dp_sync_batch_norm(lcn_model* m, int on);

/* (a10) ... or applies TF1 Adam directly from the raw gradients in one fused pass (models_att.py:404-409):
 * lr_t = lr*sqrt(1-b2^t)/(1-b1^t) is computed by the caller (host scalar); theta -= lr_t*m/(sqrt(v)+eps).
 * `regularization` adds reg*theta to the gradient of w* / b* (models_att.py:362-365).  Also re-runs the
 * weight preparation for the next forward. */
int lcn_model_adam_step(lcn_model* m, float* d_params, float* d_m, float* d_v, void* d_ws, size_t ws_bytes,
                        const float* d_grads_raw, float lr_t, float beta1, float beta2, float eps,
                        float regularization, const lcn_step_scalars* d_dyn, void* stream);

/* One LCN linear op in isolation, on the buffers of the last forward (tf.matmul(x, w) + b,
 * models_att.py:662,692): mid layer `layer` (1..2*num_layers) recomputes Z_layer = A_{layer-1} * Wm + b
 * (+ BN partial statistics); transposed != 0 runs the matching input-gradient GEMM dA = dZ * Wm^T into a
 * scratch buffer.  Used by bench.py to time the dominant kernel alone, and by the parity tests. */
int lcn_layer_gemm(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, int64_t n_rows,
                   int32_t bn_group, int layer, int transposed, void* stream);

/* Debug / parity taps: copy an internal tensor of the last forward/backward to dense fp32.
 * kind: 0 = Z_l (pre-BN linear output), 1 = A_l (layer output after BN/act/dropout/residual),
 *       2 = effective masked weight Wm_l (dense [Kin,Kout]), 3 = mask values [17,17],
 *       4 = BN mean [groups,F], 5 = BN rstd [groups,F], 6 = dZ_l. */
int lcn_model_read_tensor(lcn_model* m, void* d_ws, size_t ws_bytes, int kind, int layer,
                          int64_t n_rows, int32_t bn_group, float* d_dst, void* stream);

/* Inverse of the kind-1 tap: d_src dense fp32 [groups*bn_group, 17*F] becomes the layer output A_layer of the
 * training-layout workspace (the input of lcn_model_forward_layers(layer + 1, ...)). */
int lcn_model_write_tensor(lcn_model* m, void* d_ws, size_t ws_bytes, int kind, int layer, int64_t n_rows,
                           int32_t bn_group, const float* d_src, void* stream);

/* ---- the reference's method-level layer API as stand-alone device ops (csrc/lcn_layers.cu) ---- */
/* cgcnn.mask_weights(weights), models_att.py:576-586: d_out = reshape(d_w, [17,Fi,17,Fo]) * d_mask[17,1,17,1];
 * d_w / d_out [rows, cols] with rows, cols multiples of 17; d_mask [17,17] = [in joint, out joint]. */
int lcn_mask_weights(const float* d_w, int32_t rows, int32_t cols, const float* d_mask, float* d_out, void* stream);
/* cgcnn.batch_normalization_warp(y, training, name), models_att.py:588-612: Keras BatchNormalization(axis=-1) on
 * reshape(y, [-1, 17, F]) with BATCH statistics (SURVEY 9-Q2: every entry point of the reference passes
 * training=True): per channel mean / biased variance over rows x 17, gamma (y - mean) / sqrt(var + eps) + beta.
 * d_y / d_out [rows, 17*F]; d_stats [F][2] = (mean, variance), may be NULL. */
int lcn_batch_norm(const float* d_y, int64_t rows, int32_t F, const float* d_gamma, const float* d_beta, float eps,
                   float* d_out, float* d_stats, void* stream);
/* base_model.loss, models_att.py:352-366: d_loss[0] = mean((pred - labels)^2) over n_elems (+ reg_scale * d_reg[0]
 * when d_reg != NULL: the "reg_loss" term, :362-365). */
int lcn_mse_loss(const float* d_pred, const float* d_labels, int64_t n_elems, const float* d_reg, float reg_scale,
                 float* d_loss, void* stream);
/* tf.add_n(self.regularizers), models_att.py:364,465-472: d_out[0] = sum over every w*, b* of sum(v^2)/2.
 * d_scratch16: 16 bytes of device memory, zeroed once by the caller (the kernel leaves them zero). */
int lcn_l2_regularizer(const lcn_model* m, const float* d_params, void* d_scratch16, float* d_out, void* stream);
/* ExponentialMovingAverage(0.9).apply of the loss, run EVERY step by op_loss_average (models_att.py:210-212,370-379):
 * d_ema[0] = decay * d_ema[0] + (1 - decay) * (d_loss[0] + reg_scale * d_reg[0]); d_ema[1] += 1.  The reader applies
 * TF's zero-debias: loss_average = d_ema[0] / (1 - decay^d_ema[1]).  d_reg may be NULL. */
int lcn_loss_ema(const float* d_loss, const float* d_reg, float reg_scale, float decay, float* d_ema, void* stream);

/* ---- data path either side of the stack (SURVEY 8(f) ranks 1 and 3) ---- */
/* Batch gather of base_model.fit (train_data[idx], train_labels[idx], models_att.py:200) from device-resident sets:
 * d_dst_a[b,:] = d_src_a[d_idx[b],:] and, when given, the same for the second row set.  Indices are clamped. */
int lcn_gather_rows(const float* d_src_a, int32_t cols_a, float* d_dst_a, const float* d_src_b, int32_t cols_b,
                    float* d_dst_b, const int64_t* d_idx, int64_t n_idx, int64_t n_src, void* stream);
/* DataReader.read_2d / read_3d "scale" normalisation, tools/data.py:338-445: d_joint_3d_image [n,17,3] (pixels, mm),
 * d_res [n,2] = (res_w, res_h) of each item's camera; d_x2d [n,34] = xy / res_w * 2 - [1, res_h / res_w] (may be
 * NULL), d_y3d [n,51] = the same xy and z / res_w * 2 (may be NULL).  Inverse of lcn_denormalize. */
int lcn_normalize(const float* d_joint_3d_image, const float* d_res, int64_t n, float* d_x2d, float* d_y3d,
                  void* stream);

/* Dropout keep decisions (1 = keep) exactly as the fused kernels draw them: Philox4x32-10 keyed on
 * seed, counter (element/8, layer, step), 16 random bits per element (u = bits/65536, rate rounded up to a
 * multiple of 2^-16).  tf.nn.dropout keeps u >= rate (models_att.py:673).  cols must be a multiple of 8. */
int lcn_dropout_mask(uint64_t seed, uint64_t step, int layer, int64_t rows, int32_t cols, float rate,
                     uint8_t* d_keep, void* stream);

/* ---- (c) evaluation: evaluate.py:53-61 per pose, batched ----
 * d_pred [n,17,3] image-frame predictions (after DataReader.denormalize), d_gt [n,17,3] camera-frame
 * ground truth, d_box [n,4], d_cam [n,4] = (fx, fy, cx, cy), d_root_depth [n], d_action [n] int32 or NULL.
 * tools.image_to_camera_frame (tools/tools.py:183-194) -> optional tools.align_to_gt / procrustes
 * (:96-181,197-202; reflections allowed) -> per-joint L2 error.
 * flags: LCN_EVAL_PROTOCOL2 = Procrustes-align before measuring; LCN_EVAL_CAMERA_FRAME = d_pred is already
 * in the camera frame (skips the un-projection; box / cam / root_depth may be NULL) -- this is what
 * tools.align_to_gt(pose, pose_gt) needs when called on its own.
 * d_err [n,17] per-joint errors in mm, may be NULL.  d_pose_out [n,17,3], may be NULL: the transformed
 * prediction (camera frame; Procrustes-aligned when PROTOCOL2).  d_sums: double [n_actions+1][17+1+1]:
 * per action (row n_actions = all) 17 per-joint error sums, pose count, count(err < 50 mm);
 * accumulated (caller zeroes).  n_actions may be 0. */
#define LCN_EVAL_PROTOCOL2 1
#define LCN_EVAL_CAMERA_FRAME 2
int lcn_eval_mpjpe(const float* d_pred, const float* d_gt, const float* d_box, const float* d_cam,
                   const float* d_root_depth, const int32_t* d_action, int32_t n_actions, int64_t n,
                   int flags, float* d_err, float* d_pose_out, double* d_sums, void* stream);

/* tools.procrustes(A, B, scaling=True, reflection='best') -> (d, Z, tform), tools/tools.py:96-181, for n pose pairs:
 * d_A / d_B [n,17,3] (A = target); reflection: 0 = 'best' (no determinant fix, what align_to_gt uses), 1 = False,
 * 2 = True (:149-157).  d_Z [n,17,3] transformed B (may be NULL); d_tform [n,14] = rotation (9, row major),
 * scale, translation (3), d (may be NULL). */
int lcn_procrustes(const float* d_A, const float* d_B, int64_t n, int scaling, int reflection, float* d_Z,
                   float* d_tform, void* stream);

/* (f) DataReader.denormalize arithmetic, tools/data.py:471-472, fused in front of the evaluator:
 * d_pose [n,17,3] in place; d_res [n,2] = (res_w, res_h). */
int lcn_denormalize(float* d_pose, const float* d_res, int64_t n, void* stream);

/* (f) Pose augmentations of tools/data.py on the device (train.py:85-104, inference.py:75-111 run them on the host):
 * d_src / d_dst [n, 17*k] fp32, k = 2 or 3 coordinates per joint, out of place.
 *   LCN_AUG_FLIP      flip_data        tools/data.py:10-25   (negate x, swap left/right joints)
 *   LCN_AUG_ROTATE    rotate_data      tools/data.py:289-322 (angle_deg about z, pivot = joint 0 of each pose)
 *   LCN_AUG_TRANSLATE translation_data tools/data.py:27-54   (scalar t added to every coordinate) */
#define LCN_AUG_FLIP 1
#define LCN_AUG_ROTATE 2
#define LCN_AUG_TRANSLATE 3
int lcn_augment(const float* d_src, float* d_dst, int64_t n, int k, int op, float angle_deg, float t, void* stream);

/* (f) undo, tools/data.py:269-287 (test-time augmentation of inference.py:110-111): d_preds [(n_ops+1), n, 17, 3];
 * slice_f is un-flipped (:236-249), slice_r rotated by angle_deg about joint 0 (:289-322), slice_t un-translated by t
 * (:205-218); a negative slice index = that operation is absent.  d_out [n, 51] = mean over the n_ops+1 slices. */
int lcn_tta_undo(const float* d_preds, float* d_out, int64_t n, int n_ops, int slice_f, int slice_r, int slice_t,
                 float angle_deg, float t, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LCN_B200_H_ */
