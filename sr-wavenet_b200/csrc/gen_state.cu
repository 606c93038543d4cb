// The generation state buffer (gen_state.cuh): its header, layout and sizes, the host registry of owners, the C entry
// points that size, reset and splice it, and the kernels that advance t0 after a call and move utterances between states.
#include "gen_state.cuh"
#include <cstring>
#include <map>
#include <mutex>
#include <vector>

namespace {
struct GenStateHeader {
  long long t0;               // position of the next step (include/srwn.h: the state's first 8 bytes)
  int32_t sig[6];             // B, precision, n_layers, sum of dilations, pool_stride, kStateMagic
};
const int32_t kStateMagic = 0x5357534e;
struct GenStateLayout { size_t xhist, queues, bytes; };

GenStateLayout gen_state_layout(const srwn_ctx* c, int B, int precision) {
  GenStateLayout r;
  r.xhist = 256;                                                        // header, padded to the carving granule
  r.queues = r.xhist + (((size_t)B * 2 * sizeof(float) + 255) & ~(size_t)255);
  r.bytes = r.queues + gen_queue_bytes(c, B, precision);
  return r;
}

void state_signature(const srwn_ctx* c, int B, int precision, int32_t* sig) {
  const int32_t v[6] = {B, precision, c->cfg.n_layers, c->sum_dilation, c->cfg.pool_stride, kStateMagic};
  memcpy(sig, v, sizeof(v));
}

// The signature is also kept on the host, per state buffer, so that a call can refuse a state made for another handle,
// batch size or precision without reading the device copy (which would synchronise the stream).  Generation states and
// the student's synthesis states (student_stream.cu) share the registry; their signatures differ in length and magic.
struct StateOwner { const srwn_ctx* h; std::vector<int32_t> sig; };
std::mutex g_states_mu;
std::map<const void*, StateOwner> g_states;

int check_state_args(const srwn_ctx* h, int B, int precision, const char* fn) {
  if (!h) return srwn_fail(SRWN_ERR_INVALID, "%s: null handle", fn);
  if (h->cfg.kind != SRWN_TEACHER) return srwn_fail(SRWN_ERR_INVALID, "not a teacher handle");
  if (B < 1) return srwn_fail(SRWN_ERR_INVALID, "%s: B must be positive", fn);
  if (precision == SRWN_FP16 && !ar_mma_supported(h))
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "fp16 generation kernel does not cover this configuration");
  if (precision != SRWN_FP32 && precision != SRWN_FP16)
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "generation runs in fp32 (FFMA kernel) or fp16 (tensor-core kernel)");
  return SRWN_OK;
}

// The owner check, then the state's parts (the layout of B utterances in `precision`).
int open_owned(const srwn_ctx* h, void* state, int B, int precision, GenState* s) {
  int32_t sig[6];
  state_signature(h, B, precision, sig);
  const int rc = state_owner_check(h, state, sig, 6, "srwn_generate_state_reset");
  if (rc) return rc;
  uint8_t* base = static_cast<uint8_t*>(state);
  const GenStateLayout lay = gen_state_layout(h, B, precision);
  s->t0 = &reinterpret_cast<GenStateHeader*>(base)->t0;
  s->xhist = reinterpret_cast<float*>(base + lay.xhist);
  s->queues = base + lay.queues;
  return SRWN_OK;
}
}  // namespace

void state_owner_record(const srwn_ctx* h, const void* state, const int32_t* sig, int n) {
  std::lock_guard<std::mutex> lk(g_states_mu);
  StateOwner& o = g_states[state];
  o.h = h;
  o.sig.assign(sig, sig + n);
}

// Refuses a state that was not last reset on this handle with this signature (B and precision first).
int state_owner_check(const srwn_ctx* h, const void* state, const int32_t* sig, int n, const char* reset_fn) {
  std::lock_guard<std::mutex> lk(g_states_mu);
  auto it = g_states.find(state);
  if (it == g_states.end() || it->second.h != h)
    return srwn_fail(SRWN_ERR_INVALID, "state was not reset on this handle (%s)", reset_fn);
  const std::vector<int32_t>& have = it->second.sig;
  if (have.size() != (size_t)n || memcmp(have.data(), sig, n * sizeof(int32_t)))
    return srwn_fail(SRWN_ERR_INVALID, "state was made for B=%d, precision %d; this call has B=%d, precision %d",
                     have.empty() ? 0 : have[0], have.size() < 2 ? 0 : have[1], sig[0], sig[1]);
  return SRWN_OK;
}

// dilation queues of B utterances: fp32, sum_d rows of R floats each; fp16, one block of sum_d slots per group
size_t gen_queue_bytes(const srwn_ctx* c, int B, int precision) {
  if (precision == SRWN_FP16) return (size_t)((B + kGenGroup - 1) / kGenGroup) * c->sum_dilation * kGenSlotBytes;
  return (size_t)B * c->sum_dilation * kR * sizeof(float);
}

void gen_state_forget(const srwn_ctx* h) {
  std::lock_guard<std::mutex> lk(g_states_mu);
  for (auto it = g_states.begin(); it != g_states.end();) it = it->second.h == h ? g_states.erase(it) : std::next(it);
}

int gen_state_open(const srwn_ctx* h, void* state, int B, int T, int precision, GenState* s) {
  int rc = check_state_args(h, B, precision, "generation state");
  if (rc) return rc;
  rc = check_bt(h, B, T);
  if (rc) return rc;
  return open_owned(h, state, B, precision, s);
}

extern "C" int srwn_generate_state_bytes(srwn_handle_t h, int32_t B, int32_t precision, size_t* bytes) {
  if (!bytes) return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_bytes: null argument");
  int rc = check_state_args(h, B, precision, "srwn_generate_state_bytes");
  if (rc) return rc;
  *bytes = gen_state_layout(h, B, precision).bytes;
  return SRWN_OK;
}

extern "C" int srwn_generate_state_reset(srwn_handle_t h, void* state, int32_t B, int32_t precision, void* stream) {
  if (!state) return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_reset: null state");
  int rc = check_state_args(h, B, precision, "srwn_generate_state_reset");
  if (rc) return rc;
  GenStateHeader hdr{};
  state_signature(h, B, precision, hdr.sig);
  const cudaStream_t st = (cudaStream_t)stream;
  uint8_t* base = static_cast<uint8_t*>(state);
  SRWN_CUDA(cudaMemsetAsync(base, 0, gen_state_layout(h, B, precision).bytes, st));      // zero padding of ops.py:9
  // pageable source: the copy is staged before this call returns, so `hdr` may go out of scope
  SRWN_CUDA(cudaMemcpyAsync(base, &hdr, sizeof(hdr), cudaMemcpyHostToDevice, st));
  state_owner_record(h, state, hdr.sig, 6);
  return SRWN_OK;
}

__global__ void k_gen_state_advance(long long* t0, int T) { *t0 += T; }

int run_gen_state_advance(long long* t0, int T, cudaStream_t st) {
  k_gen_state_advance<<<1, 1, 0, st>>>(t0, T);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ---- splice (srwn_generate_state_splice) -----------------------------------------------------------------------------
// Utterance src_rows[r] of one state replaces utterance dst_rows[r] of another.  Both positions are multiples of P
// (gen_state.cuh), so the two states agree on frame boundaries and differ only in each layer's queue phase t0 mod d_l:
// the input at relative position j in [-d_l, 0) moves from slot gen_slot(src.t0, j) to slot gen_slot(dst.t0, j).
constexpr int kSpliceRows = 256;          // row pairs per launch, carried as kernel parameters
constexpr int kSpliceThreads = 256;

struct SpliceParams {
  const uint8_t* src_q; uint8_t* dst_q;   // queues
  const float* src_x; float* dst_x;       // x history [B][2]
  const long long* src_t0; const long long* dst_t0;
  const int32_t* dil; const int32_t* qoff;
  int sum_d;
  int32_t src_rows[kSpliceRows], dst_rows[kSpliceRows];
};

// grid (queue entries of one utterance / threads, row pairs); a thread moves one 16-byte piece of one queue entry
template <bool F16>
__global__ void __launch_bounds__(kSpliceThreads) k_gen_state_splice(const __grid_constant__ SpliceParams p) {
  constexpr int kPieces = F16 ? 4 : kR / 4;         // fp16: the utterance's 4 lane quads of a slot; fp32: 32 floats
  const int sb = p.src_rows[blockIdx.y], db = p.dst_rows[blockIdx.y];
  const int i = blockIdx.x * kSpliceThreads + threadIdx.x;
  if (i == 0) {
    p.dst_x[2 * db] = p.src_x[2 * sb];
    p.dst_x[2 * db + 1] = p.src_x[2 * sb + 1];
  }
  const int e = i / kPieces, q = i % kPieces;       // entry e of the utterance's sum_d queue entries
  if (e >= p.sum_d) return;
  int l = 0;
  while (e >= __ldg(p.qoff + l) + __ldg(p.dil + l)) l++;
  const int d = __ldg(p.dil + l), qoff = __ldg(p.qoff + l);
  const int j = e - qoff - d;                       // relative position in [-d, 0)
  const int ss = gen_slot(p.src_t0, j, d), ds = gen_slot(p.dst_t0, j, d);
  if (F16) {
    *reinterpret_cast<uint4*>(p.dst_q + gen_f16_offset(db, q, p.sum_d, qoff, ds)) =
        *reinterpret_cast<const uint4*>(p.src_q + gen_f16_offset(sb, q, p.sum_d, qoff, ss));
  } else {
    reinterpret_cast<float4*>(reinterpret_cast<float*>(p.dst_q) + gen_f32_row(db, p.sum_d, qoff, ds) * kR)[q] =
        reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.src_q) + gen_f32_row(sb, p.sum_d, qoff, ss) * kR)[q];
  }
}

extern "C" int srwn_generate_state_splice(srwn_handle_t h, void* dst, int32_t dst_B, const int32_t* dst_rows,
                                          const void* src, int32_t src_B, const int32_t* src_rows, int32_t n,
                                          int32_t precision, void* stream) {
  if (!dst || !src) return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_splice: null state");
  int rc = check_state_args(h, dst_B, precision, "srwn_generate_state_splice");
  if (rc) return rc;
  rc = check_state_args(h, src_B, precision, "srwn_generate_state_splice");
  if (rc) return rc;
  if (src == dst) return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_splice: src and dst are the same state");
  if (n < 0 || (n > 0 && (!dst_rows || !src_rows)))
    return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_splice: n=%d must be >= 0, with both row arrays when > 0", n);
  GenState d, s;
  rc = open_owned(h, dst, dst_B, precision, &d);
  if (rc) return rc;
  rc = open_owned(h, const_cast<void*>(src), src_B, precision, &s);
  if (rc) return rc;
  std::vector<uint8_t> named(dst_B, 0);
  for (int i = 0; i < n; i++) {
    if (dst_rows[i] < 0 || dst_rows[i] >= dst_B || src_rows[i] < 0 || src_rows[i] >= src_B)
      return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_splice: row pair %d (%d <- %d) out of range (dst B=%d, src B=%d)",
                       i, dst_rows[i], src_rows[i], dst_B, src_B);
    if (named[dst_rows[i]]++)
      return srwn_fail(SRWN_ERR_INVALID, "srwn_generate_state_splice: destination row %d named twice", dst_rows[i]);
  }
  const cudaStream_t st = (cudaStream_t)stream;
  SpliceParams p;
  p.src_q = static_cast<const uint8_t*>(s.queues); p.dst_q = static_cast<uint8_t*>(d.queues);
  p.src_x = s.xhist; p.dst_x = d.xhist; p.src_t0 = s.t0; p.dst_t0 = d.t0;
  p.dil = h->d_dilations; p.qoff = h->d_queue_off; p.sum_d = h->sum_dilation;
  const int pieces = precision == SRWN_FP16 ? 4 : kR / 4;
  const int grid_x = (h->sum_dilation * pieces + kSpliceThreads - 1) / kSpliceThreads;
  for (int a = 0; a < n; a += kSpliceRows) {
    const int m = n - a < kSpliceRows ? n - a : kSpliceRows;
    memcpy(p.src_rows, src_rows + a, m * sizeof(int32_t));
    memcpy(p.dst_rows, dst_rows + a, m * sizeof(int32_t));
    if (precision == SRWN_FP16) k_gen_state_splice<true><<<dim3(grid_x, m), kSpliceThreads, 0, st>>>(p);
    else k_gen_state_splice<false><<<dim3(grid_x, m), kSpliceThreads, 0, st>>>(p);
    SRWN_LAUNCH_CHECK();
  }
  return SRWN_OK;
}
