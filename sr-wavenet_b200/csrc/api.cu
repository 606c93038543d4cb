// C-ABI entry points: lifetime, weights, workspace sizing, dispatch (include/srwn.h).
#include "common.cuh"
#include "gen_state.cuh"
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

int srwn_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void srwn_count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

extern "C" int srwn_abi_version(void) { return SRWN_ABI_VERSION; }
extern "C" const char* srwn_last_error(void) { return g_err; }
extern "C" int64_t srwn_launch_count(void) { return g_launches.load(); }

// ---- variable table -----------------------------------------------------------------
enum VarKind { V_FRONT_K, V_FRONT_B, V_COND_K, V_COND_B, V_FILT_K, V_FILT_B, V_RES_K, V_RES_B,
               V_SKIP_K, V_SKIP_B, V_HEAD1_K, V_HEAD1_B, V_HEAD2_K, V_HEAD2_B, V_DEAD, V_BAD };

struct VarRef { int stack; VarKind kind; int layer; };

static int var_slot(const srwn_ctx* c, VarKind k, int layer) {
  switch (k) {
    case V_FRONT_K: return 0;
    case V_FRONT_B: return 1;
    case V_HEAD1_K: return 2;
    case V_HEAD1_B: return 3;
    case V_HEAD2_K: return 4;
    case V_HEAD2_B: return 5;
    default: return 6 + layer * 8 + ((int)k - (int)V_COND_K);
  }
}
static int n_slots(const srwn_ctx* c) { return 6 + c->cfg.n_layers * 8; }

static bool var_live(const srwn_ctx* c, VarKind k) {
  if (c->cfg.kind == SRWN_STUDENT)   // student: skip conv is dead (model.py:438-454), one head conv
    return !(k == V_SKIP_K || k == V_SKIP_B || k == V_HEAD2_K || k == V_HEAD2_B);
  return true;
}

// Strips the model scope and classifies a TF variable name (SURVEY.md 8(b) naming table).
static VarRef parse_name(const srwn_ctx* c, const char* full) {
  VarRef r{0, V_BAD, 0};
  const char* s = nullptr;
  if (c->cfg.kind == SRWN_TEACHER) {
    const char* p = strstr(full, "Decoder/");
    s = p ? p + 8 : full;
  } else {
    const char* p = strstr(full, "Flow");
    int f1 = -1, f2 = -1, n = 0;
    if (!p || sscanf(p, "Flow%d/Flow%d/%n", &f1, &f2, &n) < 2 || n == 0 || f1 != f2 ||
        f1 < 0 || f1 >= c->cfg.num_flows)
      return r;
    r.stack = f1;
    s = p + n;
  }
  const int L = c->cfg.n_layers;
  int i = -1, j = -1, n = 0;
  if (!strcmp(s, "causal_conv_Kernel")) { r.kind = V_FRONT_K; return r; }
  if (!strcmp(s, "causal_conv_Bias")) { r.kind = V_FRONT_B; return r; }
  if (sscanf(s, "dilated_conv_%d_filter/dilated_conv_%d_%n", &i, &j, &n) == 2 && n && i == j &&
      i >= 0 && i < L) {
    r.layer = i;
    if (!strcmp(s + n, "Kernel")) r.kind = V_FILT_K;
    else if (!strcmp(s + n, "Bias")) r.kind = V_FILT_B;
    return r;
  }
  n = 0;
  if (sscanf(s, "dilated_conv_%d_gate/dilated_conv_%d_%n", &i, &j, &n) == 2 && n && i == j &&
      i >= 0 && i < L) {
    if (!strcmp(s + n, "Kernel") || !strcmp(s + n, "Bias")) r.kind = V_DEAD;  // ops.py:31-33
    return r;
  }
  int idx = -1;
  const char* tail = nullptr;
  if (!strncmp(s, "conv1d/", 7)) { idx = 0; tail = s + 7; }
  else {
    n = 0;
    if (sscanf(s, "conv1d_%d/%n", &idx, &n) == 1 && n) tail = s + n; else return r;
  }
  bool is_k = !strcmp(tail, "kernel"), is_b = !strcmp(tail, "bias");
  if (!is_k && !is_b) return r;
  if (idx < 0) return r;
  if (idx >= 3 * L) {
    int hj = idx - 3 * L;
    int n_head = c->cfg.kind == SRWN_TEACHER ? 2 : 1;
    if (hj >= n_head) return r;
    r.kind = hj == 0 ? (is_k ? V_HEAD1_K : V_HEAD1_B) : (is_k ? V_HEAD2_K : V_HEAD2_B);
    return r;
  }
  r.layer = idx / 3;
  switch (idx % 3) {
    case 0: r.kind = is_k ? V_COND_K : V_COND_B; break;
    case 1: r.kind = is_k ? V_RES_K : V_RES_B; break;
    default:
      if (c->cfg.kind == SRWN_STUDENT) r.kind = V_DEAD;   // model.py:438-454
      else r.kind = is_k ? V_SKIP_K : V_SKIP_B;
  }
  return r;
}

// expected TF shape + offset inside a stack
static bool var_layout(const srwn_ctx* c, VarKind k, int layer, int64_t* shape, int* ndim,
                       size_t* off, size_t* count) {
  const int R = c->cfg.dilation_channels, S = c->cfg.skip_channels, C = c->cfg.cond_channels,
            K = c->cfg.filter_width, O = 4 * c->cfg.num_mixtures;
  const StackOffsets& o = c->off;
  const bool teacher = c->cfg.kind == SRWN_TEACHER;
  auto set = [&](int nd, int64_t a, int64_t b, int64_t d, size_t base, size_t per_layer) {
    *ndim = nd; shape[0] = a; shape[1] = b; shape[2] = d;
    size_t cnt = (size_t)a * (nd > 1 ? b : 1) * (nd > 2 ? d : 1);
    *count = cnt; *off = base + per_layer * layer;
  };
  switch (k) {
    case V_FRONT_K: set(3, K, 1, R, o.front_k, 0); return true;
    case V_FRONT_B: set(3, 1, 1, R, o.front_b, 0); return true;
    case V_COND_K: set(3, 1, C, R, o.cond_k, (size_t)C * R); return true;
    case V_COND_B: set(1, R, 1, 1, o.cond_b, R); return true;
    case V_FILT_K: set(3, K, R, R, o.filt_k, (size_t)K * R * R); return true;
    case V_FILT_B: set(3, 1, 1, R, o.filt_b, R); return true;
    case V_RES_K: set(3, 1, R, R, o.res_k, (size_t)R * R); return true;
    case V_RES_B: set(1, R, 1, 1, o.res_b, R); return true;
    case V_SKIP_K: set(3, 1, R, S, o.skip_k, (size_t)R * S); return true;
    case V_SKIP_B: set(1, S, 1, 1, o.skip_b, S); return true;
    case V_HEAD1_K: if (teacher) set(3, 1, S, S, o.head1_k, 0); else set(3, 1, R, 2, o.head1_k, 0); return true;
    case V_HEAD1_B: set(1, teacher ? S : 2, 1, 1, o.head1_b, 0); return true;
    case V_HEAD2_K: set(3, 1, S, O, o.head2_k, 0); return teacher;
    case V_HEAD2_B: set(1, O, 1, 1, o.head2_b, 0); return teacher;
    default: return false;
  }
}

struct HostMirror { std::vector<float> w; };
static HostMirror* mirror(srwn_ctx* c);

// the host mirror lives right behind the ctx (kept out of common.cuh on purpose)
struct CtxBox { srwn_ctx ctx; HostMirror host; };
static HostMirror* mirror(srwn_ctx* c) { return &reinterpret_cast<CtxBox*>(c)->host; }

extern "C" int srwn_create(const srwn_config_t* cfg, srwn_handle_t* out) {
  if (!cfg || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_create: null argument");
  *out = nullptr;
  if (cfg->kind != SRWN_TEACHER && cfg->kind != SRWN_STUDENT)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_create: kind must be SRWN_TEACHER or SRWN_STUDENT");
  if (cfg->n_layers <= 0 || cfg->n_layers > 256 || !cfg->dilations)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_create: need 1..256 dilations");
  for (int i = 0; i < cfg->n_layers; i++)
    if (cfg->dilations[i] < 1 || cfg->dilations[i] > (1 << 20))
      return srwn_fail(SRWN_ERR_INVALID, "srwn_create: dilation %d out of range", cfg->dilations[i]);
  if (cfg->filter_width != kK || cfg->dilation_channels != kR ||
      (cfg->kind == SRWN_TEACHER && cfg->skip_channels != kS))
    return srwn_fail(SRWN_ERR_UNSUPPORTED,
                     "kernels are built for filter_width=2, dilation_channels=32, skip_channels=128 "
                     "(teacher.py:55-62); got %d/%d/%d", cfg->filter_width, cfg->dilation_channels,
                     cfg->skip_channels);
  if (cfg->cond_channels < 1 || cfg->cond_channels > kMaxCond)
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "cond_channels must be 1..%d", kMaxCond);
  if (cfg->pool_stride < 1) return srwn_fail(SRWN_ERR_INVALID, "pool_stride must be >= 1");
  if (cfg->kind == SRWN_TEACHER && (cfg->num_mixtures < 1 || 4 * cfg->num_mixtures > kMaxLogit))
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "num_mixtures must be 1..%d", kMaxLogit / 4);
  if (cfg->kind == SRWN_STUDENT && (cfg->num_flows < 1 || cfg->num_flows > 16))
    return srwn_fail(SRWN_ERR_INVALID, "num_flows must be 1..16");

  int dev = 0;
  SRWN_CUDA(cudaGetDevice(&dev));
  CtxBox* box = new (std::nothrow) CtxBox();
  if (!box) return srwn_fail(SRWN_ERR_INVALID, "out of host memory");
  srwn_ctx* c = &box->ctx;
  c->cfg = *cfg;
  c->dilations.assign(cfg->dilations, cfg->dilations + cfg->n_layers);
  c->cfg.dilations = c->dilations.data();
  if (cfg->kind == SRWN_STUDENT) { c->cfg.skip_channels = cfg->skip_channels > 0 ? cfg->skip_channels : kS; c->cfg.num_mixtures = 0; }
  c->n_stacks = cfg->kind == SRWN_TEACHER ? 1 : cfg->num_flows;
  c->device = dev;
  c->committed = false; c->device_dirty = false;
  c->d_weights = nullptr; c->d_dilations = nullptr; c->d_queue_off = nullptr;
  c->d_packed = nullptr; c->packed_bytes = 0; c->d_ar_packed = nullptr;
  c->d_part = nullptr; c->part_B = c->part_T = c->part_out0 = c->part_teams = c->part_G = 0; c->part_team_req = -1;
  c->team_size = 0; c->h_err = nullptr; c->wait_limit_clocks = 1000000000LL;
  c->profiling = 0; c->prof_launches = 0; c->prof_name = "";
  c->prof_ev[0] = c->prof_ev[1] = nullptr;
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, dev);

  const size_t L = cfg->n_layers, R = kR, S = c->cfg.skip_channels, C = cfg->cond_channels,
               K = kK, O = 4 * (size_t)c->cfg.num_mixtures;
  const bool teacher = cfg->kind == SRWN_TEACHER;
  StackOffsets& o = c->off;
  size_t p = 0;
  auto take = [&](size_t n) { size_t r = p; p += (n + 63) & ~(size_t)63; return r; };
  o.front_k = take(K * R); o.front_b = take(R);
  o.cond_k = take(L * C * R); o.cond_b = take(L * R);
  o.filt_k = take(L * K * R * R); o.filt_b = take(L * R);
  o.res_k = take(L * R * R); o.res_b = take(L * R);
  o.skip_k = take(teacher ? L * R * S : 0); o.skip_b = take(teacher ? L * S : 0);
  o.head1_k = take(teacher ? S * S : R * 2); o.head1_b = take(teacher ? S : 2);
  o.head2_k = take(teacher ? S * O : 0); o.head2_b = take(teacher ? O : 0);
  o.skip_b_sum = take(teacher ? S : 0);
  o.end = p;
  c->stack_floats = p;
  c->is_set.assign((size_t)c->n_stacks * n_slots(c), 0);
  box->host.w.assign((size_t)c->n_stacks * p, 0.f);

  std::vector<int32_t> qoff(L);
  int sum = 0;
  for (size_t i = 0; i < L; i++) { qoff[i] = sum; sum += c->dilations[i]; }
  c->sum_dilation = sum;
  cudaError_t e = cudaMalloc(&c->d_weights, (size_t)c->n_stacks * p * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(c->d_weights, 0, (size_t)c->n_stacks * p * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&c->d_dilations, L * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMalloc(&c->d_queue_off, L * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMemcpy(c->d_dilations, c->dilations.data(), L * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(c->d_queue_off, qoff.data(), L * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    c->packed_bytes = fused_packed_bytes(c);
    if (c->packed_bytes) e = cudaMalloc(&c->d_packed, c->packed_bytes);
    if (e == cudaSuccess && c->packed_bytes) e = cudaMalloc(&c->d_part, fused_partition_bytes(c));
  }
  // abort words: every handle has them (a student stream call raises them in either precision)
  if (e == cudaSuccess) e = cudaHostAlloc((void**)&c->h_err, 64, cudaHostAllocMapped);
  if (e == cudaSuccess) memset(c->h_err, 0, 64);
  if (e != cudaSuccess) {
    int rc = srwn_fail(SRWN_ERR_CUDA, "srwn_create: %s", cudaGetErrorString(e));
    srwn_destroy(c);
    return rc;
  }
  *out = c;
  return SRWN_OK;
}

// The abort words [flag, code, a, b] as a status: a fused launch whose pipeline wait expired (code, chunk, cta), or a
// student stream call whose t0 disagreed with its state (kAbortStreamPosition, state t0, call t0).  `clear` lowers them.
static int abort_status(const srwn_ctx* c, const char* fused_lead, const char* stream_lead, bool clear) {
  volatile int* e = c->h_err;
  if (!e || !e[0]) return SRWN_OK;
  const int code = e[1], a = e[2], b = e[3];
  if (clear) { e[0] = 0; e[1] = 0; e[2] = 0; e[3] = 0; }
  if (code == kAbortStreamPosition)
    return srwn_fail(SRWN_ERR_CUDA, "%s: the call passed t0=%d but its state was at t0=%d; results of that call are invalid",
                     stream_lead, b, a);
  return srwn_fail(SRWN_ERR_CUDA, "%s: pipeline wait timed out (code 0x%x, chunk %d, cta %d); results of that call are invalid",
                   fused_lead, code, a, b);
}

// a fused launch or stream call that aborted leaves the abort words raised; every later fused launch and stream call on the
// handle is refused until srwn_check_async_error has reported it
int sticky_error(const srwn_ctx* c) {
  return abort_status(c, "an earlier fused launch aborted", "an earlier call aborted", false);
}

extern "C" int srwn_destroy(srwn_handle_t h) {
  if (!h) return SRWN_OK;
  gen_state_forget(h);
  if (h->prof_ev[0]) { cudaEventDestroy(h->prof_ev[0]); cudaEventDestroy(h->prof_ev[1]); }
  cudaFree(h->d_ar_packed); cudaFree(h->d_part);
  if (h->h_err) cudaFreeHost(h->h_err);
  cudaFree(h->d_weights); cudaFree(h->d_dilations); cudaFree(h->d_queue_off); cudaFree(h->d_packed);
  delete reinterpret_cast<CtxBox*>(h);
  return SRWN_OK;
}

extern "C" int srwn_set_weight(srwn_handle_t h, const char* name, const float* data,
                               const int64_t* shape, int32_t ndim) {
  if (!h || !name || !data || !shape) return srwn_fail(SRWN_ERR_INVALID, "srwn_set_weight: null argument");
  VarRef r = parse_name(h, name);
  if (r.kind == V_BAD) return srwn_fail(SRWN_ERR_WEIGHTS, "unknown variable '%s'", name);
  if (r.kind == V_DEAD) return SRWN_OK;
  int64_t want[3]; int nd; size_t off, cnt;
  if (!var_layout(h, r.kind, r.layer, want, &nd, &off, &cnt))
    return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s' does not exist in this model kind", name);
  bool ok = ndim == nd;
  for (int i = 0; ok && i < nd; i++) ok = shape[i] == want[i];
  if (!ok) {
    return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s': shape mismatch (want ndim %d [%lld,%lld,%lld])",
                     name, nd, (long long)want[0], (long long)(nd > 1 ? want[1] : 1),
                     (long long)(nd > 2 ? want[2] : 1));
  }
  size_t base = (size_t)r.stack * h->stack_floats + off;
  memcpy(mirror(h)->w.data() + base, data, cnt * sizeof(float));
  SRWN_CUDA(cudaMemcpy(h->d_weights + base, data, cnt * sizeof(float), cudaMemcpyHostToDevice));
  h->is_set[(size_t)r.stack * n_slots(h) + var_slot(h, r.kind, r.layer)] = 1;
  h->committed = false;
  return SRWN_OK;
}

extern "C" int srwn_get_weight(srwn_handle_t h, const char* name, float* data, int64_t count) {
  if (!h || !name || !data) return srwn_fail(SRWN_ERR_INVALID, "srwn_get_weight: null argument");
  VarRef r = parse_name(h, name);
  if (r.kind == V_BAD || r.kind == V_DEAD)
    return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s' is not stored (unknown or dead)", name);
  int64_t want[3]; int nd; size_t off, cnt;
  if (!var_layout(h, r.kind, r.layer, want, &nd, &off, &cnt))
    return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s' does not exist in this model kind", name);
  if ((size_t)count != cnt) return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s' has %zu elements", name, cnt);
  SRWN_CUDA(cudaMemcpy(data, h->d_weights + (size_t)r.stack * h->stack_floats + off,
                       cnt * sizeof(float), cudaMemcpyDeviceToHost));
  return SRWN_OK;
}

const float* srwn_host_weights(srwn_ctx* c) { return mirror(c)->w.data(); }

extern "C" int srwn_commit_weights(srwn_handle_t h, void* stream) {
  if (!h) return srwn_fail(SRWN_ERR_INVALID, "srwn_commit_weights: null handle");
  if (h->device_dirty) {     // training steps updated the device copy: refresh the host mirror the packers read
    SRWN_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    SRWN_CUDA(cudaMemcpy(mirror(h)->w.data(), h->d_weights, (size_t)h->n_stacks * h->stack_floats * sizeof(float),
                         cudaMemcpyDeviceToHost));
    h->device_dirty = false;
  }
  static const VarKind kinds[] = {V_FRONT_K, V_FRONT_B, V_HEAD1_K, V_HEAD1_B, V_HEAD2_K, V_HEAD2_B};
  for (int s = 0; s < h->n_stacks; s++) {
    for (VarKind k : kinds)
      if (var_live(h, k) && !h->is_set[(size_t)s * n_slots(h) + var_slot(h, k, 0)])
        return srwn_fail(SRWN_ERR_WEIGHTS, "stack %d: variable kind %d was never set", s, (int)k);
    for (int l = 0; l < h->cfg.n_layers; l++)
      for (int k = V_COND_K; k <= V_SKIP_B; k++)
        if (var_live(h, (VarKind)k) && !h->is_set[(size_t)s * n_slots(h) + var_slot(h, (VarKind)k, l)])
          return srwn_fail(SRWN_ERR_WEIGHTS, "stack %d layer %d: variable kind %d was never set", s, l, k);
  }
  if (h->cfg.kind == SRWN_TEACHER) {   // sum of the skip biases, added once before the head
    float* w = mirror(h)->w.data();
    const int S = h->cfg.skip_channels;
    for (int j = 0; j < S; j++) {
      double acc = 0;
      for (int l = 0; l < h->cfg.n_layers; l++) acc += w[h->off.skip_b + (size_t)l * S + j];
      w[h->off.skip_b_sum + j] = (float)acc;
    }
    SRWN_CUDA(cudaMemcpy(h->d_weights + h->off.skip_b_sum, w + h->off.skip_b_sum, S * sizeof(float),
                         cudaMemcpyHostToDevice));
  }
  int rc = fused_pack_weights(h, (cudaStream_t)stream);
  if (rc != SRWN_OK) return rc;
  if (h->cfg.kind == SRWN_TEACHER) {
    rc = ar_mma_pack_weights(h, (cudaStream_t)stream);
    if (rc != SRWN_OK) return rc;
  }
  h->committed = true;
  return SRWN_OK;
}

// ---- workspace sizing ---------------------------------------------------------------
struct F32Ws { float *h0, *h1, *skip, *cond, *logits, *scales, *means; size_t bytes; };

static F32Ws carve_f32(const srwn_ctx* c, int B, int T, void* ws, size_t cap, bool need_logits) {
  WsCarver w(ws, cap);
  F32Ws r{};
  const size_t n = (size_t)B * T;
  const size_t frames = (size_t)(T / c->cfg.pool_stride);
  r.h0 = w.take<float>(n * kR);
  r.h1 = w.take<float>(n * kR);
  r.cond = w.take<float>((size_t)B * frames * c->cfg.n_layers * kR);
  if (c->cfg.kind == SRWN_TEACHER) {
    r.skip = w.take<float>(n * kS);
    if (need_logits) r.logits = w.take<float>(n * 4 * c->cfg.num_mixtures);
  } else {
    r.scales = w.take<float>(n * c->cfg.num_flows);
    r.means = w.take<float>(n * c->cfg.num_flows);
  }
  r.bytes = w.used;
  return r;
}

size_t student_flows_workspace_bytes(const srwn_ctx* h, int precision, int B, int T) {
  return precision == SRWN_FP16 ? fused_workspace_bytes(h, B, T) : carve_f32(h, B, T, nullptr, 0, false).bytes;
}

// one-call student forward: the flow chain's buffers, then the flows' own workspace
struct StudentWs { float *xa, *xb, *z; void* flows; size_t flows_bytes, bytes; };

static StudentWs carve_student(const srwn_ctx* h, int precision, int B, int T, void* ws, size_t cap) {
  WsCarver w(ws, cap);
  StudentWs r{};
  const size_t n = (size_t)B * T;
  r.xa = w.take<float>(n);
  r.xb = w.take<float>(n);
  if (precision == SRWN_FP32) r.z = w.take<float>(n);   // on-device noise of srwn_student_sample (fp16 draws it in flow 0)
  r.flows_bytes = student_flows_workspace_bytes(h, precision, B, T);
  r.flows = w.take<uint8_t>(r.flows_bytes);
  r.bytes = w.used;
  return r;
}

int check_workspace(const void* ws, size_t have, size_t need) {
  if (!ws || have < need) return srwn_fail(SRWN_ERR_WORKSPACE, "workspace too small: need %zu bytes", need);
  return SRWN_OK;
}

// ---- which op runs at which precision on which handle ------------------------------------
// The handle kind of each op (enum srwn_op) and the kernel that runs its SRWN_FP16 form; every op runs in SRWN_FP32.  The
// fused kernel also limits the batch (fused_check_batch).
enum Fp16Kernel { FP16_NONE, FP16_FUSED, FP16_AR_MMA };
struct OpRule { int kind; Fp16Kernel fp16; };
static const OpRule kOpRules[] = {
    {SRWN_TEACHER, FP16_FUSED},     // SRWN_OP_TEACHER_LOGITS
    {SRWN_TEACHER, FP16_FUSED},     // SRWN_OP_TEACHER_NLL
    {SRWN_TEACHER, FP16_AR_MMA},    // SRWN_OP_TEACHER_GENERATE
    {SRWN_STUDENT, FP16_FUSED},     // SRWN_OP_STUDENT_FORWARD
    {SRWN_STUDENT, FP16_NONE},      // SRWN_OP_STUDENT_TRAIN
    {SRWN_TEACHER, FP16_AR_MMA},    // SRWN_OP_TEACHER_PREFILL
    {SRWN_STUDENT, FP16_FUSED},     // SRWN_OP_STUDENT_STREAM
};
constexpr int kNumOps = sizeof(kOpRules) / sizeof(kOpRules[0]);

// bf16 MMA operands cannot meet the 2e-2 max-abs bound on logits for the 30-layer stack (exact arithmetic on bf16-rounded
// operands already gives 2.45e-2, tools/bf16_emulation.py; the kernel measured 2.5e-2), so the 16-bit path is fp16
// (same tensor rate, 8x finer mantissa, measured 3.6e-3) and SRWN_BF16 is refused rather than shipped with a looser bound.
static int reject_bf16() {
  return srwn_fail(SRWN_ERR_UNSUPPORTED, "SRWN_BF16 is not offered: bf16 operands miss the 2e-2 logit bound on this stack; use SRWN_FP16");
}

// The one rule of which op runs at which precision on which handle, in the refusal order of include/srwn.h: the op's handle
// kind, SRWN_BF16, a value that is no precision, SRWN_FP16 where the op's 16-bit kernel does not cover the configuration
static int check_op(const srwn_ctx* h, int op, int precision) {
  if (op < 0 || op >= kNumOps) return srwn_fail(SRWN_ERR_INVALID, "unknown op %d", op);
  const OpRule& r = kOpRules[op];
  if (h->cfg.kind != r.kind)
    return srwn_fail(SRWN_ERR_INVALID, r.kind == SRWN_TEACHER ? "not a teacher handle" : "not a student handle");
  if (precision == SRWN_BF16) return reject_bf16();
  if (precision != SRWN_FP32 && precision != SRWN_FP16) return srwn_fail(SRWN_ERR_INVALID, "unknown precision %d", precision);
  if (precision == SRWN_FP32) return SRWN_OK;
  switch (r.fp16) {
    case FP16_FUSED: return fused_check_config(h);
    case FP16_AR_MMA: return ar_mma_check_config(h);
    default: return srwn_fail(SRWN_ERR_UNSUPPORTED, "op %d runs in SRWN_FP32 only", op);
  }
}

int check_state(const srwn_ctx* h, int op, int B, int precision) {
  if (int rc = check_op(h, op, precision)) return rc;
  if (B < 1) return srwn_fail(SRWN_ERR_INVALID, "B must be positive");
  return SRWN_OK;
}

// check_op, then B and T, the weights (when `weights`) and the batch limit of the op's 16-bit kernel
static int check_call(const srwn_ctx* h, int op, int B, int T, int precision, bool weights = true) {
  if (int rc = check_op(h, op, precision)) return rc;
  if (B < 1 || T < 1) return srwn_fail(SRWN_ERR_INVALID, "B and T must be positive");
  if (T % h->cfg.pool_stride != 0)
    return srwn_fail(SRWN_ERR_INVALID, "T=%d must be a multiple of pool_stride=%d (model.py:183)", T,
                     h->cfg.pool_stride);
  if (weights && !h->committed) return srwn_fail(SRWN_ERR_WEIGHTS, "weights not committed (srwn_commit_weights)");
  if (precision == SRWN_FP16 && kOpRules[op].fp16 == FP16_FUSED) return fused_check_batch(h, B);
  return SRWN_OK;
}

// check_op's answer without its message
extern "C" int srwn_supports(srwn_handle_t h, int32_t op, int32_t precision) {
  if (!h || op < 0 || op >= kNumOps || h->cfg.kind != kOpRules[op].kind) return 0;
  if (precision == SRWN_FP32) return 1;
  if (precision != SRWN_FP16) return 0;
  switch (kOpRules[op].fp16) {
    case FP16_FUSED: return fused_supported(h) ? 1 : 0;
    case FP16_AR_MMA: return ar_mma_supported(h) ? 1 : 0;
    default: return 0;
  }
}

extern "C" int srwn_set_team_size(srwn_handle_t h, int32_t ctas_per_team) {
  if (!h) return srwn_fail(SRWN_ERR_INVALID, "srwn_set_team_size: null handle");
  if (ctas_per_team < 0 || ctas_per_team > 64) return srwn_fail(SRWN_ERR_INVALID, "team size must be 0 (automatic) .. 64");
  h->team_size = ctas_per_team;
  return SRWN_OK;
}

extern "C" int srwn_set_wait_limit(srwn_handle_t h, int64_t clocks) {
  if (!h || clocks < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_set_wait_limit: bad argument");
  h->wait_limit_clocks = clocks;
  return SRWN_OK;
}

extern "C" int srwn_last_partition(srwn_handle_t h, int32_t* teams, int32_t* ctas_per_team) {
  if (!h || !teams || !ctas_per_team) return srwn_fail(SRWN_ERR_INVALID, "srwn_last_partition: null argument");
  int t = 0, g = 0;
  fused_last_partition(h, &t, &g);
  *teams = t; *ctas_per_team = g;
  return SRWN_OK;
}

extern "C" int srwn_set_profiling(srwn_handle_t h, int32_t enable) {
  if (!h) return srwn_fail(SRWN_ERR_INVALID, "srwn_set_profiling: null handle");
  if (enable && !h->prof_ev[0]) {
    SRWN_CUDA(cudaEventCreate(&h->prof_ev[0]));
    SRWN_CUDA(cudaEventCreate(&h->prof_ev[1]));
  }
  h->profiling = enable ? 1 : 0;
  h->prof_launches = 0;
  return SRWN_OK;
}

extern "C" int srwn_last_kernel_ms(srwn_handle_t h, float* ms, int32_t* launches, const char** name) {
  if (!h || !ms) return srwn_fail(SRWN_ERR_INVALID, "srwn_last_kernel_ms: null argument");
  if (!h->profiling || h->prof_launches == 0)
    return srwn_fail(SRWN_ERR_INVALID, "no profiled call yet (srwn_set_profiling)");
  SRWN_CUDA(cudaEventSynchronize(h->prof_ev[1]));
  SRWN_CUDA(cudaEventElapsedTime(ms, h->prof_ev[0], h->prof_ev[1]));
  if (launches) *launches = h->prof_launches;
  if (name) *name = h->prof_name;
  return SRWN_OK;
}

extern "C" int srwn_check_async_error(srwn_handle_t h, int32_t op, int32_t B, int32_t T, int32_t precision,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  if (!h) return srwn_fail(SRWN_ERR_INVALID, "srwn_check_async_error: null handle");
  if (precision == SRWN_FP32 && op != SRWN_OP_STUDENT_STREAM) {
    SRWN_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return SRWN_OK;
  }
  if (op == SRWN_OP_TEACHER_GENERATE) return ar_mma_check_error(h, B, T, workspace, workspace_bytes, (cudaStream_t)stream);
  SRWN_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return abort_status(h, "fused kernel aborted", "student stream call aborted", true);
}

// The same check without the stream synchronisation, for callers that keep several launches in flight and have already
// waited (on an event) for the launch they ask about: the abort words of the fused kernels live in pinned host memory.
extern "C" int srwn_peek_async_error(srwn_handle_t h) {
  if (!h) return srwn_fail(SRWN_ERR_INVALID, "srwn_peek_async_error: null handle");
  return abort_status(h, "fused kernel aborted", "student stream call aborted", false);
}

extern "C" int srwn_workspace_bytes(srwn_handle_t h, int32_t op, int32_t B, int32_t T,
                                    int32_t precision, size_t* bytes) {
  if (!h || !bytes) return srwn_fail(SRWN_ERR_INVALID, "srwn_workspace_bytes: null argument");
  if (int rc = check_call(h, op, B, T, precision, false)) return rc;
  const bool fp16 = precision == SRWN_FP16;
  switch (op) {
    case SRWN_OP_TEACHER_LOGITS:
    case SRWN_OP_TEACHER_NLL:
      *bytes = fp16 ? fused_workspace_bytes(h, B, T) : carve_f32(h, B, T, nullptr, 0, true).bytes; break;
    case SRWN_OP_TEACHER_GENERATE: *bytes = fp16 ? ar_mma_workspace_bytes(h, B, T) : ar_workspace_bytes(h, B, T); break;
    case SRWN_OP_STUDENT_FORWARD: *bytes = carve_student(h, precision, B, T, nullptr, 0).bytes; break;
    case SRWN_OP_STUDENT_TRAIN: *bytes = train_workspace_bytes(h, B, T); break;
    case SRWN_OP_TEACHER_PREFILL: *bytes = prefill_workspace_bytes(h, B, T, precision); break;
    case SRWN_OP_STUDENT_STREAM: *bytes = student_stream_workspace_bytes(h, B, T, precision); break;
  }
  return SRWN_OK;
}

// ---- teacher --------------------------------------------------------------------------
static int teacher_f32(srwn_ctx* c, const float* x_in, const float* enc, float* logits_dst,
                       int B, int T, const F32Ws& w, cudaStream_t st) {
  float* hf = nullptr;
  int rc = run_stack_f32(c, 0, x_in, enc, B, T, w.h0, w.h1, w.skip, w.cond, &hf, st);
  if (rc) return rc;
  return run_teacher_head_f32(c, w.skip, logits_dst, B, T, st);
}

extern "C" int srwn_teacher_logits(srwn_handle_t h, const float* x, const float* enc, float* logits,
                                   int32_t B, int32_t T, int32_t precision, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  if (!h || !x || !enc || !logits) return srwn_fail(SRWN_ERR_INVALID, "srwn_teacher_logits: null argument");
  if (int rc = check_call(h, SRWN_OP_TEACHER_LOGITS, B, T, precision)) return rc;
  if (precision == SRWN_FP16)
    return run_teacher_fused(h, x, enc, nullptr, nullptr, nullptr, logits, B, T,
                             workspace, workspace_bytes, (cudaStream_t)stream);
  F32Ws w = carve_f32(h, B, T, workspace, workspace_bytes, false);
  if (int rc = check_workspace(workspace, workspace_bytes, w.bytes)) return rc;
  return teacher_f32(h, x, enc, logits, B, T, w, (cudaStream_t)stream);
}

extern "C" int srwn_teacher_nll(srwn_handle_t h, const float* x_in, const float* enc,
                                const float* x_scored, float* nll_out, float* nll_sum,
                                float* logits_out, int32_t B, int32_t T, int32_t precision,
                                void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !x_in || !enc || !x_scored) return srwn_fail(SRWN_ERR_INVALID, "srwn_teacher_nll: null argument");
  int rc = check_call(h, SRWN_OP_TEACHER_NLL, B, T, precision);
  if (rc) return rc;
  if (precision == SRWN_FP16)
    return run_teacher_fused(h, x_in, enc, x_scored, nll_out, nll_sum, logits_out, B, T,
                             workspace, workspace_bytes, (cudaStream_t)stream);
  F32Ws w = carve_f32(h, B, T, workspace, workspace_bytes, logits_out == nullptr);
  if ((rc = check_workspace(workspace, workspace_bytes, w.bytes))) return rc;
  float* lg = logits_out ? logits_out : w.logits;
  rc = teacher_f32(h, x_in, enc, lg, B, T, w, (cudaStream_t)stream);
  if (rc) return rc;
  return run_mol_loss(x_scored, lg, nll_out, nll_sum, B, T, h->cfg.num_mixtures, (cudaStream_t)stream);
}

extern "C" int srwn_teacher_generate(srwn_handle_t h, const float* enc, const float* u1,
                                     const float* u2, float* x_out, float* logits_out, int32_t B,
                                     int32_t T, int32_t precision, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  if (!h || !enc || !u1 || !u2 || !x_out) return srwn_fail(SRWN_ERR_INVALID, "srwn_teacher_generate: null argument");
  if (int rc = check_call(h, SRWN_OP_TEACHER_GENERATE, B, T, precision)) return rc;
  if (precision == SRWN_FP16)
    return run_ar_mma(h, enc, u1, u2, x_out, logits_out, B, T, workspace, workspace_bytes, (cudaStream_t)stream, nullptr,
                      nullptr, 0);
  return run_ar_generate(h, enc, u1, u2, x_out, logits_out, B, T, workspace, workspace_bytes,
                         (cudaStream_t)stream, nullptr, nullptr, 0);
}

// ---- resumable generation (state format: gen_state.cu) ------------------------------------
extern "C" int srwn_teacher_generate_resume(srwn_handle_t h, void* state, const float* enc, const float* u1,
                                            const float* u2, const float* x_prefix, int32_t n_prefix, float* x_out,
                                            float* logits_out, int32_t B, int32_t T, int32_t precision, void* workspace,
                                            size_t workspace_bytes, void* stream) {
  if (!h || !state || !enc || !u1 || !u2 || !x_out)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_teacher_generate_resume: null argument");
  GenState s;
  int rc = check_call(h, SRWN_OP_TEACHER_GENERATE, B, T, precision);
  if (!rc) rc = gen_state_open(h, state, B, precision, &s);
  if (rc) return rc;
  if (n_prefix < 0 || n_prefix > T || (n_prefix > 0 && !x_prefix))
    return srwn_fail(SRWN_ERR_INVALID, "n_prefix=%d must be in [0, T=%d], with x_prefix given when > 0", n_prefix, T);
  if (n_prefix == 0) x_prefix = nullptr;
  if (precision == SRWN_FP16)
    return run_ar_mma(h, enc, u1, u2, x_out, logits_out, B, T, workspace, workspace_bytes, (cudaStream_t)stream, &s,
                      x_prefix, n_prefix);
  return run_ar_generate(h, enc, u1, u2, x_out, logits_out, B, T, workspace, workspace_bytes, (cudaStream_t)stream, &s,
                         x_prefix, n_prefix);
}

extern "C" int srwn_generate_state_prefill(srwn_handle_t h, void* state, const float* x, const float* enc, int32_t n,
                                           int32_t B, int32_t precision, void* workspace, size_t workspace_bytes,
                                           void* stream) {
  if (!h || !state || !x || !enc) return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_prefill: null argument");
  GenState s;
  int rc = check_call(h, SRWN_OP_TEACHER_PREFILL, B, n, precision);   // n % P == 0 keeps t0 on a frame boundary for later calls
  if (!rc) rc = gen_state_open(h, state, B, precision, &s);
  if (rc) return rc;
  return run_prefill(h, s, x, enc, B, n, precision, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- student --------------------------------------------------------------------------
// z supplied (noise.on == 0) or drawn on the device (student.py:104); z_out optionally receives the draws
static int student_forward(srwn_handle_t h, const float* z, NoiseSpec noise, float* z_out, const float* enc, float* out,
                           float* s_tot, float* mu_tot, float* x_last, int32_t B, int32_t T, int32_t precision,
                           void* workspace, size_t workspace_bytes, cudaStream_t st) {
  int rc = check_call(h, SRWN_OP_STUDENT_FORWARD, B, T, precision);
  if (rc) return rc;
  const StudentWs w = carve_student(h, precision, B, T, workspace, workspace_bytes);
  if ((rc = check_workspace(workspace, workspace_bytes, w.bytes))) return rc;
  const size_t n = (size_t)B * T;
  const int F = h->cfg.num_flows;
  if (noise.on && precision == SRWN_FP32) {           // the layer-at-a-time path reads the noise as a tensor
    float* zbuf = z_out ? z_out : w.z;
    rc = run_random_fill(zbuf, (int64_t)n, noise.seed, noise.stream, 1, 0.f, 1.f, st);
    if (rc) return rc;
    z = zbuf; noise.on = 0; z_out = nullptr;
  }
  float* x[17] = {const_cast<float*>(z)};            // flow f reads x[f] and writes x[f + 1] (num_flows <= 16, srwn_create)
  for (int f = 0; f < F; f++) x[f + 1] = (f == F - 1 && x_last) ? x_last : ((f & 1) ? w.xb : w.xa);
  const float *scales = nullptr, *means = nullptr;
  rc = run_student_flows(h, precision, x, noise, enc, B, T, 0, w.flows, w.flows_bytes, &scales, &means, st);
  if (rc) return rc;
  return run_flow_compose(z, noise, z_out, scales, means, F, out, s_tot, mu_tot, (int64_t)n, st);
}

int run_student_flows(srwn_ctx* h, int precision, float* const* x, NoiseSpec noise, const float* enc, int B, int T, int t_out,
                      void* ws, size_t ws_bytes, const float** scales, const float** means, cudaStream_t st) {
  if (precision == SRWN_FP16)
    return run_student_flows_fused(h, x, noise, enc, B, T, t_out, ws, ws_bytes, scales, means, st);
  F32Ws w = carve_f32(h, B, T, ws, ws_bytes, false);
  if (int rc = check_workspace(ws, ws_bytes, w.bytes)) return rc;
  const size_t n = (size_t)B * T;
  for (int f = 0; f < h->cfg.num_flows; f++) {       // model.py:509-513, strictly sequential
    float* hf = nullptr;
    int rc = run_stack_f32(h, f, x[f], enc, B, T, w.h0, w.h1, nullptr, w.cond, &hf, st);
    if (rc) return rc;
    rc = run_flow_head_f32(h, f, hf, x[f], w.scales + (size_t)f * n, w.means + (size_t)f * n, x[f + 1], B, T, st, t_out);
    if (rc) return rc;
  }
  *scales = w.scales; *means = w.means;
  return SRWN_OK;
}

extern "C" int srwn_student_forward(srwn_handle_t h, const float* z, const float* enc, float* out,
                                    float* s_tot, float* mu_tot, float* x_last, int32_t B, int32_t T,
                                    int32_t precision, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  if (!h || !z || !enc || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_forward: null argument");
  return student_forward(h, z, NoiseSpec{0, 0, 0}, nullptr, enc, out, s_tot, mu_tot, x_last, B, T, precision,
                         workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int srwn_student_sample(srwn_handle_t h, uint64_t seed, uint64_t stream_id, const float* enc, float* out,
                                   float* s_tot, float* mu_tot, float* x_last, float* z_out, int32_t B, int32_t T,
                                   int32_t precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !enc || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_sample: null argument");
  return student_forward(h, nullptr, NoiseSpec{seed, stream_id, 1}, z_out, enc, out, s_tot, mu_tot, x_last, B, T,
                         precision, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- student synthesis in chunks through a carried flow state (state format and kernels: student_stream.cu) ----------
extern "C" int srwn_student_forward_resume(srwn_handle_t h, void* state, int64_t t0, const float* z, uint64_t seed,
                                           uint64_t stream_id, const float* enc, float* out, float* s_tot, float* mu_tot,
                                           float* x_last, float* z_out, int32_t B, int32_t S, int32_t precision,
                                           void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !state || !enc || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_forward_resume: null argument");
  if (int rc = check_call(h, SRWN_OP_STUDENT_STREAM, B, S, precision)) return rc;
  if (t0 < 0 || t0 % h->cfg.pool_stride)
    return srwn_fail(SRWN_ERR_INVALID, "t0=%lld must be a non-negative multiple of pool_stride=%d", (long long)t0,
                     h->cfg.pool_stride);
  const NoiseSpec noise{seed, stream_id, z ? 0 : 1};
  return run_student_stream(h, state, t0, z, noise, enc, out, s_tot, mu_tot, x_last, z ? nullptr : z_out, B, S, precision,
                            workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- student distillation step (model.py:356-401) ----------------------------------------------
extern "C" int srwn_param_count(srwn_handle_t h, int64_t* count) {
  if (!h || !count) return srwn_fail(SRWN_ERR_INVALID, "srwn_param_count: null argument");
  *count = (int64_t)h->n_stacks * (int64_t)h->stack_floats;
  return SRWN_OK;
}

extern "C" int srwn_weight_offset(srwn_handle_t h, const char* name, int64_t* offset, int64_t* count) {
  if (!h || !name || !offset || !count) return srwn_fail(SRWN_ERR_INVALID, "srwn_weight_offset: null argument");
  VarRef r = parse_name(h, name);
  if (r.kind == V_BAD || r.kind == V_DEAD)
    return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s' is not stored (unknown or dead)", name);
  int64_t want[3]; int nd; size_t off, cnt;
  if (!var_layout(h, r.kind, r.layer, want, &nd, &off, &cnt))
    return srwn_fail(SRWN_ERR_WEIGHTS, "variable '%s' does not exist in this model kind", name);
  *offset = (int64_t)((size_t)r.stack * h->stack_floats + off);
  *count = (int64_t)cnt;
  return SRWN_OK;
}

extern "C" int srwn_student_forward_train(srwn_handle_t h, const float* z, const float* enc, float* out,
                                          float* s_tot, float* mu_tot, int32_t B, int32_t T, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  if (!h || !z || !enc || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_forward_train: null argument");
  if (int rc = check_call(h, SRWN_OP_STUDENT_TRAIN, B, T, SRWN_FP32)) return rc;
  return run_student_forward_train(h, z, enc, out, s_tot, mu_tot, B, T, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int srwn_student_backward(srwn_handle_t h, const float* z, const float* enc, const float* d_pre,
                                     const float* d_s_extra, float* grads, int32_t B, int32_t T, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  if (!h || !z || !enc || !d_pre || !grads) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_backward: null argument");
  if (int rc = check_call(h, SRWN_OP_STUDENT_TRAIN, B, T, SRWN_FP32)) return rc;
  return run_student_backward(h, z, enc, d_pre, d_s_extra, grads, B, T, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int srwn_mol_loss_grad(const float* x, const float* l, float* dx, float* nll_out, int32_t B, int32_t T,
                                  int32_t M, void* stream) {
  if (!x || !l || !dx) return srwn_fail(SRWN_ERR_INVALID, "srwn_mol_loss_grad: null argument");
  if (B < 1 || T < 1 || M < 1 || M > 8) return srwn_fail(SRWN_ERR_INVALID, "srwn_mol_loss_grad: bad B/T/M");
  return run_mol_nll_grad(x, l, dx, nll_out, B, T, M, (cudaStream_t)stream);
}

int run_stft_workspace_bytes(int B, int T, int N, int step, size_t* bytes);
int run_stft_power(const float* x, float* power, int B, int T, int N, int step, void* ws, size_t cap, cudaStream_t st);
int run_stft_power_loss(const float* truth, const float* out, float gamma, double* loss, float* d_out, int B, int T, int N,
                        int step, void* ws, size_t cap, cudaStream_t st);
int run_distill_loss_grad(const float* z, const float* s_tot, const float* mu_tot, const float* nll, const float* d_ce,
                          const float* d_pow, float alpha, float beta, float inv_norm, float* d_pre, float* d_s, double* sums,
                          int B, int T, cudaStream_t st);

extern "C" int srwn_stft_workspace_bytes(int32_t B, int32_t T, int32_t frame_length, int32_t frame_step, size_t* bytes) {
  if (!bytes) return srwn_fail(SRWN_ERR_INVALID, "srwn_stft_workspace_bytes: null argument");
  return run_stft_workspace_bytes(B, T, frame_length, frame_step, bytes);
}

extern "C" int srwn_stft_power(const float* x, float* power, int32_t B, int32_t T, int32_t frame_length, int32_t frame_step,
                               void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !power || !workspace) return srwn_fail(SRWN_ERR_INVALID, "srwn_stft_power: null argument");
  return run_stft_power(x, power, B, T, frame_length, frame_step, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int srwn_stft_power_loss(const float* truth, const float* out, float gamma, double* loss, float* d_out, int32_t B,
                                    int32_t T, int32_t frame_length, int32_t frame_step, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!truth || !out || !loss || !workspace) return srwn_fail(SRWN_ERR_INVALID, "srwn_stft_power_loss: null argument");
  return run_stft_power_loss(truth, out, gamma, loss, d_out, B, T, frame_length, frame_step, workspace, workspace_bytes,
                             (cudaStream_t)stream);
}

extern "C" int srwn_distill_loss_grad(const float* z, const float* s_tot, const float* mu_tot, const float* nll,
                                      const float* d_ce, const float* d_pow, float alpha, float beta, float inv_norm,
                                      float* d_pre, float* d_s, double* sums, int32_t B, int32_t T, void* stream) {
  if (!z || !s_tot || !mu_tot || !d_ce || !d_pre || !d_s || !sums)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_distill_loss_grad: null argument");
  if (B < 1 || T < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_distill_loss_grad: bad B/T");
  return run_distill_loss_grad(z, s_tot, mu_tot, nll, d_ce, d_pow, alpha, beta, inv_norm, d_pre, d_s, sums, B, T,
                               (cudaStream_t)stream);
}

extern "C" int srwn_weights_flat(srwn_handle_t h, float* buffer, int64_t count, int32_t to_handle, void* stream) {
  if (!h || !buffer) return srwn_fail(SRWN_ERR_INVALID, "srwn_weights_flat: null argument");
  const int64_t n = (int64_t)h->n_stacks * (int64_t)h->stack_floats;
  if (count != n) return srwn_fail(SRWN_ERR_INVALID, "srwn_weights_flat: count %lld != srwn_param_count %lld", (long long)count, (long long)n);
  if (to_handle) {
    SRWN_CUDA(cudaMemcpyAsync(h->d_weights, buffer, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    h->device_dirty = true;        // host mirror and packed operand images are stale until srwn_commit_weights
  } else {
    SRWN_CUDA(cudaMemcpyAsync(buffer, h->d_weights, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  }
  return SRWN_OK;
}

extern "C" int srwn_distill_finish(const double* sums, const double* power, float alpha, float beta, float inv_norm,
                                   float* out2, void* stream) {
  if (!sums || !power || !out2) return srwn_fail(SRWN_ERR_INVALID, "srwn_distill_finish: null argument");
  return run_distill_finish(sums, power, alpha, beta, inv_norm, out2, (cudaStream_t)stream);
}

extern "C" int srwn_clip_by_global_norm(float* grads, int64_t n, float clip_norm, float* scratch, void* stream) {
  if (!grads || !scratch || n < 1 || !(clip_norm > 0.f)) return srwn_fail(SRWN_ERR_INVALID, "srwn_clip_by_global_norm: bad argument");
  return run_clip_by_global_norm(grads, n, clip_norm, scratch, (cudaStream_t)stream);
}

extern "C" int srwn_axpy(float* y, const float* x, float a, int64_t n, void* stream) {
  if (!y || !x || n < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_axpy: bad argument");
  return run_axpy(y, x, a, n, (cudaStream_t)stream);
}

extern "C" int srwn_entropy(const float* s_tot, double* per_example, int32_t B, int32_t T, void* stream) {
  if (!s_tot || !per_example || B < 1 || T < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_entropy: bad argument");
  return run_entropy(s_tot, per_example, B, T, (cudaStream_t)stream);
}

extern "C" int srwn_adam_step(srwn_handle_t h, const float* grads, float* m, float* v, float* scratch, float clip_norm,
                              float lr, float beta1, float beta2, float eps, int32_t step, void* stream) {
  if (!h || !grads || !m || !v || !scratch) return srwn_fail(SRWN_ERR_INVALID, "srwn_adam_step: null argument");
  if (step < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_adam_step: step counts from 1");
  if (!h->committed) return srwn_fail(SRWN_ERR_WEIGHTS, "weights not committed (srwn_commit_weights)");
  h->device_dirty = true;
  return run_adam(h, grads, m, v, scratch, clip_norm, lr, beta1, beta2, eps, step, (cudaStream_t)stream);
}
