// The generation state buffer (gen_state.cuh): its header, layout and sizes, the host registry of owners, the C entry
// points that size and reset it, and the kernel that advances t0 after a call.
#include "gen_state.cuh"
#include <cstring>
#include <map>
#include <mutex>

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
// batch size or precision without reading the device copy (which would synchronise the stream).
struct StateOwner { const srwn_ctx* h; int32_t sig[6]; };
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

// Refuses a state that was not last reset on this handle for this B and precision (host-side signature: no synchronisation).
int check_state_owner(const srwn_ctx* h, const void* state, int B, int precision) {
  int32_t sig[6];
  state_signature(h, B, precision, sig);
  std::lock_guard<std::mutex> lk(g_states_mu);
  auto it = g_states.find(state);
  if (it == g_states.end() || it->second.h != h)
    return srwn_fail(SRWN_ERR_INVALID, "state was not reset on this handle (srwn_generate_state_reset)");
  if (memcmp(it->second.sig, sig, sizeof(sig)))
    return srwn_fail(SRWN_ERR_INVALID, "state was made for B=%d, precision %d; this call has B=%d, precision %d",
                     it->second.sig[0], it->second.sig[1], B, precision);
  return SRWN_OK;
}
}  // namespace

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
  rc = check_state_owner(h, state, B, precision);
  if (rc) return rc;
  uint8_t* base = static_cast<uint8_t*>(state);
  const GenStateLayout lay = gen_state_layout(h, B, precision);
  s->t0 = &reinterpret_cast<GenStateHeader*>(base)->t0;
  s->xhist = reinterpret_cast<float*>(base + lay.xhist);
  s->queues = base + lay.queues;
  return SRWN_OK;
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
  std::lock_guard<std::mutex> lk(g_states_mu);
  StateOwner& o = g_states[state];
  o.h = h;
  memcpy(o.sig, hdr.sig, sizeof(hdr.sig));
  return SRWN_OK;
}

__global__ void k_gen_state_advance(long long* t0, int T) { *t0 += T; }

int run_gen_state_advance(long long* t0, int T, cudaStream_t st) {
  k_gen_state_advance<<<1, 1, 0, st>>>(t0, T);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}
