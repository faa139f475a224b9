// C ABI of liblcn_b200.so (see include/lcn_b200.h): model construction, parameter / workspace
// layout, and thin wrappers that enqueue the kernels of lcn_kernels.cu / lcn_gemm_tc.cu / lcn_eval.cu.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include "lcn_internal.cuh"

static thread_local char g_err[512] = "";

void lcn_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* lcn_version(void) { return "lcn_b200 0.1 (sm_100a)"; }
extern "C" const char* lcn_last_error(void) { return g_err; }

// ---- masks on the host, bit exact ------------------------------------------------------------
// 17-joint skeleton, tools/filter_hub.py:4-20 (neighbour_dict_set[0])
static const int kNbr[LCN_J][7] = {
    {1, 4, 7, -1},        {0, 7, 2, -1}, {1, 3, -1},        {2, -1},      {0, 7, 5, -1},  {4, 6, -1},
    {5, -1},              {1, 0, 4, 14, 8, 11, -1},         {7, 9, 11, 14, -1},           {8, 10, -1},
    {9, -1},              {8, 7, 12, -1}, {11, 13, -1},     {12, -1},     {8, 7, 15, -1}, {14, 16, -1},
    {15, -1}};

// tools/params_help.py:8-20: A[i,{i}+nbrs]=1; knn>=2 -> (matrix_power(A,knn) != 0).  All values are
// small exact integers in float32, so an integer matrix power reproduces the float32 result bit for bit.
extern "C" int lcn_neighbour_matrix(int knn, float* h_out) {
  LCN_REQUIRE(knn >= 1 && h_out != nullptr, "knn must be >= 1");
  double a[LCN_J][LCN_J] = {}, acc[LCN_J][LCN_J], tmp[LCN_J][LCN_J];
  for (int i = 0; i < LCN_J; ++i) {
    a[i][i] = 1;
    for (int k = 0; kNbr[i][k] >= 0; ++k) a[i][kNbr[i][k]] = 1;
  }
  memcpy(acc, a, sizeof(a));
  for (int p = 1; p < knn; ++p) {
    for (int i = 0; i < LCN_J; ++i)
      for (int j = 0; j < LCN_J; ++j) {
        double s = 0;
        for (int k = 0; k < LCN_J; ++k) s += acc[i][k] * a[k][j];
        tmp[i][j] = s != 0 ? 1.0 : 0.0;   // only the zero pattern matters; keeps values bounded
      }
    memcpy(acc, tmp, sizeof(acc));
  }
  for (int i = 0; i < LCN_J; ++i)
    for (int j = 0; j < LCN_J; ++j) h_out[i * LCN_J + j] = acc[i][j] != 0 ? 1.0f : 0.0f;
  return LCN_OK;
}

// network/models_att.py:14-69: 18 unit edges -> Floyd-Warshall -> 1/2**dist -> float32
extern "C" int lcn_exponential_matrix(float* h_out) {
  LCN_REQUIRE(h_out != nullptr, "null output");
  static const int e[18][2] = {{0, 1}, {0, 7}, {0, 4}, {4, 5}, {4, 7}, {5, 6}, {1, 7}, {1, 2}, {2, 3},
                               {7, 11}, {7, 8}, {7, 14}, {11, 12}, {12, 13}, {14, 15}, {15, 16}, {8, 9}, {9, 10}};
  double d[LCN_J][LCN_J];
  for (int i = 0; i < LCN_J; ++i)
    for (int j = 0; j < LCN_J; ++j) d[i][j] = i == j ? 0.0 : INFINITY;
  for (auto& p : e) d[p[0]][p[1]] = d[p[1]][p[0]] = 1.0;
  for (int k = 0; k < LCN_J; ++k)
    for (int i = 0; i < LCN_J; ++i)
      for (int j = 0; j < LCN_J; ++j)
        if (d[i][j] > d[i][k] + d[k][j]) d[i][j] = d[i][k] + d[k][j];
  for (int i = 0; i < LCN_J; ++i)
    for (int j = 0; j < LCN_J; ++j) h_out[i * LCN_J + j] = (float)(1.0 / pow(2.0, d[i][j]));
  return LCN_OK;
}

// ---- CRC32C (Castagnoli) of host memory: the checksum of TensorBundle checkpoints (tools/tf_checkpoint.py) ----
// slicing-by-8; tables built once (thread safe: function-local static initialisation)
struct Crc32cTables {
  uint32_t t[8][256];
  Crc32cTables() {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
      t[0][i] = c;
    }
    for (int k = 1; k < 8; ++k)
      for (uint32_t i = 0; i < 256; ++i) t[k][i] = (t[k - 1][i] >> 8) ^ t[0][t[k - 1][i] & 0xFFu];
  }
};
extern "C" uint32_t lcn_crc32c(const void* h_data, size_t n, uint32_t crc) {
  static const Crc32cTables T;
  const uint8_t* p = static_cast<const uint8_t*>(h_data);
  uint32_t c = crc ^ 0xFFFFFFFFu;
  while (n >= 8) {
    uint32_t lo, hi;
    memcpy(&lo, p, 4);
    memcpy(&hi, p + 4, 4);
    lo ^= c;
    c = T.t[7][lo & 0xFF] ^ T.t[6][(lo >> 8) & 0xFF] ^ T.t[5][(lo >> 16) & 0xFF] ^ T.t[4][lo >> 24] ^
        T.t[3][hi & 0xFF] ^ T.t[2][(hi >> 8) & 0xFF] ^ T.t[1][(hi >> 16) & 0xFF] ^ T.t[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n--) c = T.t[0][(c ^ *p++) & 0xFF] ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}

// ---- model -------------------------------------------------------------------------------------
static int64_t align4(int64_t v) { return (v + 3) & ~(int64_t)3; }

extern "C" int lcn_model_create(const lcn_model_desc* desc, lcn_model** out) {
  LCN_REQUIRE(desc && out, "null argument");
  LCN_REQUIRE(desc->F > 0 && desc->F % 64 == 0 && desc->F <= 256, "F=%d: must be a multiple of 64, <= 256", desc->F);
  LCN_REQUIRE(256 % desc->F == 0, "F=%d: must divide 256", desc->F);
  LCN_REQUIRE(desc->in_F == 2 || desc->in_F == 3, "in_F=%d: 2 or 3 supported", desc->in_F);
  LCN_REQUIRE(desc->num_layers >= 0 && desc->num_layers <= 8, "num_layers=%d: 0..8 supported", desc->num_layers);
  LCN_REQUIRE(desc->batch_norm == 1, "batch_norm=False is not implemented on the device path");
  LCN_REQUIRE(desc->mask_kind == LCN_MASK_LOCALLY_CONNECTED || desc->mask_kind == LCN_MASK_CONSTANT, "bad mask_kind");
  LCN_REQUIRE(desc->path == LCN_PATH_FP32 || desc->path == LCN_PATH_BF16, "bad path");
  lcn_model* m = new lcn_model();
  m->d = *desc;
  m->n_lin = 2 + 2 * desc->num_layers;
  m->n_bn = 1 + 2 * desc->num_layers;
  m->P = LCN_J * desc->F;
  m->FC = desc->F / 64;
  // support tables
  memset(&m->by_out, 0, sizeof(JointLists));
  memset(&m->by_in, 0, sizeof(JointLists));
  memset(&m->sup, 0, sizeof(SupportBits));
  int p = 0;
  for (int i = 0; i < LCN_J; ++i)
    for (int j = 0; j < LCN_J; ++j) {
      bool on = desc->support[i * LCN_J + j] != 0.f;
      m->sup.pair[i][j] = on ? (int16_t)p++ : (int16_t)-1;
      if (on) {
        m->sup.row[i] |= 1u << j;
        m->sup.col[j] |= 1u << i;
      }
    }
  m->nnz = p;
  if (p == 0) {
    delete m;
    lcn_set_error("empty mask support");
    return LCN_EINVAL;
  }
  for (int j = 0; j < LCN_J; ++j)
    for (int i = 0; i < LCN_J; ++i)
      if (m->sup.pair[i][j] >= 0) {
        int n = m->by_out.cnt[j]++;
        m->by_out.idx[j][n] = (uint8_t)i;
        m->by_out.blk[j][n] = m->sup.pair[i][j];
      }
  for (int i = 0; i < LCN_J; ++i)
    for (int j = 0; j < LCN_J; ++j)
      if (m->sup.pair[i][j] >= 0) {
        int n = m->by_in.cnt[i]++;
        m->by_in.idx[i][n] = (uint8_t)j;
        m->by_in.blk[i][n] = m->sup.pair[i][j];
      }
  // parameter layout, reference variable names (SURVEY 8(b))
  int64_t off = 0;
  auto add = [&](const std::string& name, int rows, int cols, int kind, int layer) {
    TensorMeta t{name, off, rows, cols};
    m->tensors.push_back(t);
    SegInfo s;
    s.off = off;
    s.size = (int64_t)rows * cols;
    s.kind = kind;
    s.layer = layer;
    s.chunk_start = 0;
    m->segs.s[m->segs.n++] = s;
    int64_t o = off;
    off = align4(off + (int64_t)rows * cols);
    return o;
  };
  m->segs.n = 0;
  m->mask_off = -1;
  if (desc->mask_kind == LCN_MASK_LOCALLY_CONNECTED) m->mask_off = add("mask", LCN_J, LCN_J, SEG_MASK, -1);
  for (int l = 0; l < m->n_lin; ++l) {
    LayerInfo& L = m->L[l];
    L.Fi = l == 0 ? desc->in_F : desc->F;
    L.Fo = l == m->n_lin - 1 ? 3 : desc->F;
    L.Kin = LCN_J * L.Fi;
    L.Kout = LCN_J * L.Fo;
    L.has_bn = l < m->n_lin - 1;
    L.res_from = -1;
    std::string scope = "linear_model/", wn, bn;
    if (l == 0) { wn = "w1"; bn = "b1"; }
    else if (l == m->n_lin - 1) { wn = "w4"; bn = "b4"; }
    else {
      int blk = (l - 1) / 2;
      bool second = ((l - 1) % 2) == 1;
      scope += "two_linear_" + std::to_string(blk) + "/";
      wn = (second ? "w3_" : "w2_") + std::to_string(blk);
      bn = (second ? "b3_" : "b2_") + std::to_string(blk);
      if (second && desc->residual) L.res_from = l - 2;
    }
    L.w_off = add(scope + wn, L.Kin, L.Kout, SEG_W, l);
    L.b_off = add(scope + bn, 1, L.Kout, SEG_B, l);
    L.gamma_off = L.beta_off = -1;
  }
  for (int l = 0; l < m->n_bn; ++l) {
    std::string name = "linear_model/";
    if (l == 0) name += "batch_normalization";
    else {
      int blk = (l - 1) / 2;
      bool second = ((l - 1) % 2) == 1;
      name += "two_linear_" + std::to_string(blk) + "/batch_normalization" + (second ? "2" : "1") + std::to_string(blk);
    }
    m->L[l].gamma_off = add(name + "/gamma", 1, desc->F, SEG_BN, l);
    m->L[l].beta_off = add(name + "/beta", 1, desc->F, SEG_BN, l);
  }
  m->n_params = off;
  int chunks = 0;
  for (int s = 0; s < m->segs.n; ++s) {
    m->segs.s[s].chunk_start = chunks;
    chunks += (int)((m->segs.s[s].size + LCN_ADAM_CHUNK - 1) / LCN_ADAM_CHUNK);
  }
  m->segs.total_chunks = chunks;
  m->sm_count = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) m->sm_count = sms;
  } else {
    (void)cudaGetLastError();
  }
  *out = m;
  return LCN_OK;
}

extern "C" void lcn_model_destroy(lcn_model* m) {
  if (m == nullptr) return;
  lcn_dp_destroy(m);
  lcn_aux_release(m->aux);
  delete m;
}
extern "C" int64_t lcn_model_param_count(const lcn_model* m) { return m ? m->n_params : 0; }
extern "C" int lcn_model_num_tensors(const lcn_model* m) { return m ? (int)m->tensors.size() : 0; }
extern "C" int lcn_model_tensor_info(const lcn_model* m, int index, char* name_buf, int name_buf_len, int64_t* offset,
                                     int32_t* rows, int32_t* cols) {
  LCN_REQUIRE(m && index >= 0 && index < (int)m->tensors.size(), "tensor index out of range");
  const TensorMeta& t = m->tensors[index];
  if (name_buf && name_buf_len > 0) snprintf(name_buf, name_buf_len, "%s", t.name.c_str());
  if (offset) *offset = t.off;
  if (rows) *rows = t.rows;
  if (cols) *cols = t.cols;
  return LCN_OK;
}

// ---- workspace layout ----------------------------------------------------------------------------
WsLayout lcn_ws_layout(const lcn_model* m, int64_t n_rows, int bn_group, int training) {
  WsLayout w;
  memset(&w, 0, sizeof(w));
  w.n_rows = n_rows;
  w.bn_group = bn_group;
  w.gstride = (bn_group + LCN_TILE - 1) / LCN_TILE * LCN_TILE;
  w.n_groups = (int)((n_rows + bn_group - 1) / bn_group);
  w.rows_pad = (int64_t)w.n_groups * w.gstride;
  w.tiles = (int)(w.rows_pad / LCN_TILE);
  w.tiles_per_group = w.gstride / LCN_TILE;
  w.training = training;
  w.es = m->d.path == LCN_PATH_BF16 ? 2 : 4;           // bf16, or a (hi, lo) pair of bf16 (lcn_sp16)
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = (off + bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t P = m->P, F = m->d.F;
  w.off_scalars = take(sizeof(LayerScalars) * LCN_MAX_LIN);
  w.off_mask = take(sizeof(float) * 3 * LCN_J * LCN_J);
  w.off_pairdot = take(sizeof(float) * LCN_MAX_LIN * LCN_J * LCN_J);
  w.off_loss = take(sizeof(double) * 2);
  w.off_wm_first = take(sizeof(float) * m->L[0].Kin * m->L[0].Kout);
  w.off_wm_last = take(sizeof(float) * m->L[m->n_lin - 1].Kin * m->L[m->n_lin - 1].Kout);
  size_t n_mid = m->n_lin - 2;
  size_t sub = (size_t)m->nnz * m->FC * m->FC * 4096;
  const bool x3 = m->d.path == LCN_PATH_FP32;          // fp32 copy for the weight tap, and the lo parts of split bf16
  w.off_wp32 = take(x3 ? sizeof(float) * n_mid * sub : 0);
  w.off_wp16f = take(2 * n_mid * sub);
  w.off_wp16b = take(2 * n_mid * sub);
  w.off_wp16f_lo = take(x3 ? 2 * n_mid * sub : 0);
  w.off_wp16b_lo = take(x3 ? 2 * n_mid * sub : 0);
  w.off_wl16f = take((size_t)LCN_J * m->FC * 8192);
  w.off_wl16b = take((size_t)LCN_J * m->FC * 8192);
  w.off_wf16 = take((size_t)LCN_J * m->FC * 8192);
  w.fused = lcn_stack_eligible(m, bn_group, training) ? 1 : 0;
  w.off_part = take(w.fused ? 0 : sizeof(float) * (size_t)w.tiles * P * 2);
  w.off_bnstat = take(w.fused ? 0 : sizeof(float) * (size_t)m->n_bn * w.n_groups * F * 2);
  w.off_bnsum = take(sizeof(float) * (size_t)m->n_bn * (F * 2 + 1));    // + one grid-barrier counter per BN layer
  w.gacc_stride = sizeof(double) * LCN_GACC_REP * F * 2 + 256;
  w.off_gacc = take(training ? w.gacc_stride * (size_t)m->n_bn : 0);
  w.off_out = take(training ? sizeof(float) * (size_t)w.rows_pad * 51 : 0);
  w.off_dout = take(training ? sizeof(float) * (size_t)w.rows_pad * 51 : 0);
  w.off_x16 = take(training ? (size_t)w.rows_pad * 64 * 2 : 0);
  w.off_dout16 = take(training ? (size_t)w.rows_pad * 64 * 2 : 0);
  w.off_dw_first = take(training ? sizeof(float) * 64 * P : 0);
  w.off_dw_last = take(training ? sizeof(float) * P * 64 : 0);
  size_t act = ((size_t)w.rows_pad * P * w.es + 255) & ~(size_t)255;
  w.n_z = training ? m->n_bn : (w.fused ? 0 : 1);
  w.n_a = training ? m->n_bn : (w.fused ? 0 : 3);
  w.n_d = training ? 3 : 0;
  w.z_stride = w.a_stride = w.d_stride = act;
  w.off_z = take(act * w.n_z);
  w.off_a = take(act * w.n_a);
  w.off_d = take(act * w.n_d);
  w.off_dz = take(training ? 2 * act : 0);
  w.off_dbpart = take(training ? sizeof(float) * (size_t)m->n_bn * 2 * m->sm_count * P : 0);
  w.off_keep = take(training ? sizeof(uint16_t) * (size_t)m->n_bn * w.rows_pad * (P / 8) : 0);
  w.off_stack = take(w.fused ? lcn_stack_scratch_bytes(m, bn_group) : 0);
  w.total = off;
  return w;
}

static int check_geom(const lcn_model* m, int64_t n_rows, int32_t bn_group) {
  LCN_REQUIRE(m != nullptr, "null model");
  LCN_REQUIRE(n_rows > 0 && bn_group > 0, "n_rows=%lld bn_group=%d must be positive", (long long)n_rows, bn_group);
  LCN_REQUIRE(((n_rows + bn_group - 1) / bn_group) * (int64_t)((bn_group + 127) / 128 * 128) < ((int64_t)1 << 31) / 4,
              "too many rows for one call; shard the pose batch");
  return LCN_OK;
}

extern "C" size_t lcn_model_workspace_bytes(const lcn_model* m, int64_t n_rows, int32_t bn_group, int training) {
  if (check_geom(m, n_rows, bn_group)) return 0;
  return lcn_ws_layout(m, n_rows, bn_group, training).total;
}

// *lay = the workspace layout of a call; LCN_ENOMEM when ws_bytes is short of it.  head_only: the call touches only the
// head of the workspace (packed weights, mask, scalars), whose offsets do not depend on the row geometry.
static int ws_layout_for(const lcn_model* m, int64_t n_rows, int bn_group, int training, size_t ws_bytes,
                         bool head_only, WsLayout* lay) {
  *lay = lcn_ws_layout(m, n_rows, bn_group, training);
  const size_t need = head_only ? lay->off_part : lay->total;
  if (ws_bytes < need) {
    lcn_set_error("workspace too small: %zu < %zu", ws_bytes, need);
    return LCN_ENOMEM;
  }
  return LCN_OK;
}

extern "C" int lcn_model_prepare_weights(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, void* stream) {
  LCN_REQUIRE(m && d_params && d_ws, "null argument");
  WsLayout lay;
  int rc = ws_layout_for(m, 128, 128, 0, ws_bytes, true, &lay);
  if (rc) return rc;
  return lcn_launch_prepare(m, d_params, (char*)d_ws, lay, true, (cudaStream_t)stream);
}

bool lcn_pdl_enabled() {
  static const bool v = [] {                       // profiling switch; function-local static: initialised once, thread safe
    const char* e = getenv("LCN_DISABLE_PDL");
    return !(e && e[0] == '1');
  }();
  return v;
}

// ---- LCN_TRACE: per-kernel in-stream durations (debug) ----
#include <map>
#include <mutex>
namespace {
struct TraceRec { const void* func; cudaEvent_t a, b; };
std::vector<TraceRec> g_trace;
std::mutex g_trace_mu;
}
bool lcn_trace_enabled() {
  static const bool v = [] {
    const char* e = getenv("LCN_TRACE");
    return e && e[0] == '1';
  }();
  return v;
}
void lcn_trace_mark(const void* func, cudaStream_t st, int end) {
  std::lock_guard<std::mutex> lock(g_trace_mu);
  if (!end) {
    TraceRec r;
    r.func = func;
    cudaEventCreate(&r.a);
    cudaEventCreate(&r.b);
    cudaEventRecord(r.a, st);
    g_trace.push_back(r);
  } else if (!g_trace.empty()) {
    cudaEventRecord(g_trace.back().b, st);
  }
}
// prints "name launches total_us avg_us" per kernel and clears the trace; returns the number of records
extern "C" int lcn_debug_trace_dump() {
  std::lock_guard<std::mutex> lock(g_trace_mu);
  cudaDeviceSynchronize();
  std::map<std::string, std::pair<int, double>> agg;
  for (const TraceRec& r : g_trace) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, r.a, r.b);
    const char* name = nullptr;
    if (cudaFuncGetName(&name, r.func) != cudaSuccess || name == nullptr) name = "?";
    auto& e = agg[name];
    e.first += 1;
    e.second += ms * 1e3;
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  double tot = 0;
  for (auto& kv : agg) tot += kv.second.second;
  for (auto& kv : agg)
    printf("%-70.70s n=%5d total=%10.1f us avg=%8.2f us share=%5.1f%%\n", kv.first.c_str(), kv.second.first, kv.second.second,
           kv.second.second / kv.second.first, 100.0 * kv.second.second / (tot > 0 ? tot : 1));
  printf("traced launches %zu, total %.1f us\n", g_trace.size(), tot);
  fflush(stdout);
  int n = (int)g_trace.size();
  g_trace.clear();
  return n;
}

// the forward pass of lcn_model_forward / lcn_model_forward_layers once their arguments are checked
static int run_forward(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, const float* d_x,
                       int64_t n_rows, int32_t bn_group, int training, float dropout_rate, uint64_t seed, uint64_t step,
                       float* d_out, const lcn_step_scalars* d_dyn, int layer_begin, int layer_end, void* stream) {
  FwdArgs a;
  int rc = ws_layout_for(m, n_rows, bn_group, training, ws_bytes, false, &a.lay);
  if (rc) return rc;
  a.m = m;
  a.params = d_params;
  a.ws = (char*)d_ws;
  a.x = d_x;
  a.out = d_out;
  a.dropout_rate = dropout_rate;
  a.seed = seed;
  a.step = step;
  a.dyn = d_dyn;
  a.st = (cudaStream_t)stream;
  a.layer_begin = layer_begin;
  a.layer_end = layer_end;
  return lcn_launch_forward(a);
}

extern "C" int lcn_model_forward(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, const float* d_x,
                                 int64_t n_rows, int32_t bn_group, int training, float dropout_rate, uint64_t seed,
                                 uint64_t step, float* d_out, const lcn_step_scalars* d_dyn, void* stream) {
  int rc = check_geom(m, n_rows, bn_group);
  if (rc) return rc;
  LCN_REQUIRE(d_params && d_ws && d_x && d_out, "null argument");
  LCN_REQUIRE(dropout_rate >= 0.f && dropout_rate < 1.f, "dropout rate %f outside [0,1)", dropout_rate);
  return run_forward(m, d_params, d_ws, ws_bytes, d_x, n_rows, bn_group, training, dropout_rate, seed, step, d_out, d_dyn,
                     0, -1, stream);
}

extern "C" int lcn_model_forward_layers(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, const float* d_x,
                                        int64_t n_rows, int32_t bn_group, float dropout_rate, uint64_t seed, uint64_t step,
                                        int layer_begin, int layer_end, float* d_out, void* stream) {
  int rc = check_geom(m, n_rows, bn_group);
  if (rc) return rc;
  LCN_REQUIRE(d_params && d_ws, "null argument");
  LCN_REQUIRE(layer_begin >= 0 && layer_begin < layer_end && layer_end <= m->n_lin, "layer range [%d, %d) outside [0, %d)",
              layer_begin, layer_end, m->n_lin);
  LCN_REQUIRE(d_x != nullptr || (layer_begin > 0 && layer_end < m->n_lin), "the first and the last layer read d_x");
  LCN_REQUIRE(d_out != nullptr || layer_end < m->n_lin, "the last layer writes d_out");
  LCN_REQUIRE(dropout_rate >= 0.f && dropout_rate < 1.f, "dropout rate %f outside [0,1)", dropout_rate);
  if (lcn_bn_sync_on(m)) {   // its per-layer batch statistics would disagree with the global ones of the backward pass
    lcn_set_error("lcn_model_forward_layers: not available while synchronised BatchNorm is on (lcn_dp_sync_batch_norm)");
    return LCN_ESTATE;
  }
  // training layout: every Z_l / A_l has its own buffer
  return run_forward(m, d_params, d_ws, ws_bytes, d_x, n_rows, bn_group, 1, dropout_rate, seed, step, d_out, nullptr,
                     layer_begin, layer_end, stream);
}

extern "C" int lcn_model_write_tensor(lcn_model* m, void* d_ws, size_t ws_bytes, int kind, int layer, int64_t n_rows,
                                      int32_t bn_group, const float* d_src, void* stream) {
  int rc = check_geom(m, n_rows, bn_group);
  if (rc) return rc;
  LCN_REQUIRE(d_ws && d_src, "null argument");
  LCN_REQUIRE(kind == 1, "only kind 1 (layer output A_l) can be injected");
  WsLayout lay;
  rc = ws_layout_for(m, n_rows, bn_group, 1, ws_bytes, false, &lay);
  if (rc) return rc;
  return lcn_launch_write_tensor(m, (char*)d_ws, lay, layer, d_src, (cudaStream_t)stream);
}

extern "C" int lcn_model_forward_taps(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, const float* d_x,
                                      int64_t n_rows, int32_t bn_group, float* d_out, void* d_taps, size_t taps_bytes,
                                      void* stream) {
  int rc = check_geom(m, n_rows, bn_group);
  if (rc) return rc;
  LCN_REQUIRE(d_params && d_ws && d_x && d_out && d_taps, "null argument");
  LCN_REQUIRE(lcn_stack_eligible(m, bn_group, 0), "forward_taps: the fused inference kernel does not cover this model / bn_group");
  WsLayout lay;
  rc = ws_layout_for(m, n_rows, bn_group, 0, ws_bytes, false, &lay);
  if (rc) return rc;
  size_t need = (size_t)m->n_bn * lay.tiles * LCN_J * 8192 * 2;
  LCN_REQUIRE(taps_bytes >= need, "taps buffer too small: %zu < %zu", taps_bytes, need);
  return lcn_stack_forward(m, lay, d_params, (char*)d_ws, d_x, d_out, d_taps, (cudaStream_t)stream);
}

extern "C" int lcn_model_backward(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, const float* d_x,
                                  const float* d_labels, int64_t n_rows, float dropout_rate, uint64_t seed,
                                  uint64_t step, float* d_loss, float* d_grads_raw, void* stream) {
  LCN_REQUIRE(n_rows <= (1 << 24), "training batch too large");
  int rc = check_geom(m, n_rows, (int32_t)n_rows);
  if (rc) return rc;
  LCN_REQUIRE(d_params && d_ws && d_x && d_labels && d_loss && d_grads_raw, "null argument");
  WsLayout lay;
  rc = ws_layout_for(m, n_rows, (int)n_rows, 1, ws_bytes, false, &lay);   // training: the batch is one BN group
  if (rc) return rc;
  return lcn_launch_backward(m, d_params, (char*)d_ws, lay, d_x, d_labels, dropout_rate, seed, step, d_loss,
                             d_grads_raw, (cudaStream_t)stream);
}

extern "C" int lcn_model_finalize_grads(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes,
                                        const float* d_grads_raw, float* d_grads_out, void* stream) {
  LCN_REQUIRE(m && d_params && d_ws && d_grads_raw && d_grads_out, "null argument");
  WsLayout lay;
  int rc = ws_layout_for(m, 128, 128, 0, ws_bytes, true, &lay);
  if (rc) return rc;
  return lcn_launch_grad_finalize(m, d_params, (char*)d_ws, lay, d_grads_raw, d_grads_out, (cudaStream_t)stream);
}

extern "C" int lcn_model_adam_step(lcn_model* m, float* d_params, float* d_m, float* d_v, void* d_ws, size_t ws_bytes,
                                   const float* d_grads_raw, float lr_t, float beta1, float beta2, float eps,
                                   float regularization, const lcn_step_scalars* d_dyn, void* stream) {
  LCN_REQUIRE(m && d_params && d_m && d_v && d_ws && d_grads_raw, "null argument");
  WsLayout lay;
  int rc = ws_layout_for(m, 128, 128, 0, ws_bytes, true, &lay);
  if (rc) return rc;
  return lcn_launch_adam(m, d_params, d_m, d_v, (char*)d_ws, lay, d_grads_raw, lr_t, beta1, beta2, eps, regularization,
                         d_dyn, (cudaStream_t)stream);
}

extern "C" int64_t lcn_model_grad_compact_count(const lcn_model* m) { return m ? lcn_grad_compact_count(m) : 0; }
extern "C" int lcn_model_pack_grads(lcn_model* m, const float* d_grads_raw, float* d_compact, void* stream) {
  LCN_REQUIRE(m != nullptr && d_grads_raw != nullptr && d_compact != nullptr, "null argument");
  return lcn_launch_grad_compact(m, const_cast<float*>(d_grads_raw), d_compact, false, (cudaStream_t)stream);
}
extern "C" int lcn_model_unpack_grads(lcn_model* m, const float* d_compact, float* d_grads_raw, void* stream) {
  LCN_REQUIRE(m != nullptr && d_grads_raw != nullptr && d_compact != nullptr, "null argument");
  return lcn_launch_grad_compact(m, d_grads_raw, const_cast<float*>(d_compact), true, (cudaStream_t)stream);
}

extern "C" int lcn_layer_gemm(lcn_model* m, const float* d_params, void* d_ws, size_t ws_bytes, int64_t n_rows,
                              int32_t bn_group, int layer, int transposed, void* stream) {
  int rc = check_geom(m, n_rows, bn_group);
  if (rc) return rc;
  LCN_REQUIRE(d_params && d_ws, "null argument");
  LCN_REQUIRE(layer >= 1 && layer <= 2 * m->d.num_layers, "layer %d is not a mid layer", layer);
  WsLayout lay;
  rc = ws_layout_for(m, n_rows, bn_group, 1, ws_bytes, false, &lay);
  if (rc) return rc;
  return lcn_launch_layer_gemm(m, d_params, (char*)d_ws, lay, layer, transposed, (cudaStream_t)stream);
}

extern "C" int lcn_model_read_tensor(lcn_model* m, void* d_ws, size_t ws_bytes, int kind, int layer, int64_t n_rows,
                                     int32_t bn_group, float* d_dst, void* stream) {
  int rc = check_geom(m, n_rows, bn_group);
  if (rc) return rc;
  LCN_REQUIRE(d_ws && d_dst, "null argument");
  WsLayout lay;
  rc = ws_layout_for(m, n_rows, bn_group, 1, ws_bytes, kind == 2 || kind == 3, &lay);   // weights / mask live in the head
  if (rc) return rc;
  return lcn_launch_read_tensor(m, (char*)d_ws, lay, kind, layer, d_dst, (cudaStream_t)stream);
}
