// Student synthesis in chunks through a carried flow state (srwn_student_state_*, srwn_student_forward_resume).
//
// An output sample of a flow depends on that flow's input over the (K-1) * sum(d) + K = sum(d) + 2 rows before and at
// it (front conv on x[t-1], x[t-2], then the dilated layers: stack_f32.cu:45), and on the frames of those rows.  The
// state keeps, per flow, the last H of those inputs, H being that window rounded up to a multiple of pool_stride P, and
// the last H/P conditioning frames.  A call of S samples at position t0 runs each flow over a buffer of Heff + S rows,
// Heff = min(t0, H): the carried rows first, then the new ones, and keeps the outputs of rows >= Heff.  Row 0 of the
// buffer is the true start of the utterance (t0 <= H) or lies a whole window before the first output row (t0 > H), so
// the zero padding every kernel applies before row 0 is exactly right: the outputs are bit for bit those of one call over
// the whole clip, in both precisions and for any work partition.  The carried rows are recomputed (not their layer
// activations), which costs about (Heff + S) / S of the one-call rate.
//
// State buffer: header (t0, signature) | x history [F][B][H] fp32 at byte 256 | frame history [B][H/P][C] fp32.
#include "common.cuh"
#include "gen_state.cuh"
#include "philox.cuh"
#include <cstring>

namespace {
constexpr int kSigLen = 8;
const int32_t kStreamMagic = 0x53545245;
struct StreamHeader {
  long long t0;               // position of the next sample (the state's first 8 bytes)
  int32_t sig[kSigLen];       // B, precision, flows, layers, sum of dilations, pool_stride, cond_channels, kStreamMagic
};
struct StreamLayout { size_t xhist, fhist, bytes; };

// H: the flow's dependency window (filter_width - 1) * sum(d) + filter_width, rounded up to a multiple of pool_stride
int history_rows(const srwn_ctx* c) {
  const int P = c->cfg.pool_stride, need = (c->cfg.filter_width - 1) * c->sum_dilation + c->cfg.filter_width;
  return (need + P - 1) / P * P;
}

StreamLayout layout(const srwn_ctx* c, int B) {
  const size_t H = history_rows(c), F = c->cfg.num_flows, C = c->cfg.cond_channels;
  StreamLayout r;
  r.xhist = 256;
  r.fhist = r.xhist + ((F * B * H * sizeof(float) + 255) & ~(size_t)255);
  r.bytes = r.fhist + (((size_t)B * (H / c->cfg.pool_stride) * C * sizeof(float) + 255) & ~(size_t)255);
  return r;
}

void signature(const srwn_ctx* c, int B, int precision, int32_t* sig) {
  const int32_t v[kSigLen] = {B, precision, c->cfg.num_flows, c->cfg.n_layers, c->sum_dilation, c->cfg.pool_stride,
                              c->cfg.cond_channels, kStreamMagic};
  memcpy(sig, v, sizeof(v));
}

// one call: the flows' input buffers [B][N] (x[F] = the last flow's output), the frames of the buffer, the state
struct StreamArgs {
  float* x[17];               // num_flows <= 16 (srwn_create)
  float* ebuf;                // [B][N/P][C]
  float* xhist;               // state [F][B][H]
  float* fhist;               // state [B][H/P][C]
  long long* t0;              // state header
  int* valid;                 // workspace: the state was at t0_call (written by assemble, read by commit)
  int* err;                   // the handle's abort words (pinned, mapped)
  long long t0_call;
  int B, S, N, H, Heff, F, C, P;
};

constexpr int kThreads = 256;

// The carried rows of every flow and frame ahead of the new ones; the new noise into flow 0's buffer (copied, or the
// logistic draw of element b*S + s of this call's Philox stream).  Thread 0 compares the state's t0 with the caller's and
// raises the handle's abort words on a mismatch: the call's outputs are then invalid and the commit leaves the state.
__global__ void __launch_bounds__(kThreads) k_stream_assemble(const __grid_constant__ StreamArgs a, const float* __restrict__ z,
                                                              NoiseSpec noise, const float* __restrict__ enc) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i == 0) {
    const long long t0 = *a.t0;
    *a.valid = t0 == a.t0_call;
    if (t0 != a.t0_call) {
      volatile int* e = a.err;
      e[1] = kAbortStreamPosition; e[2] = (int)t0; e[3] = (int)a.t0_call;
      __threadfence_system();
      e[0] = 1;
    }
  }
  const int Hf = a.H / a.P, Nf = a.N / a.P, hf = a.Heff / a.P;
  const int64_t n_hist = (int64_t)a.F * a.B * a.Heff, n_new = (int64_t)a.B * a.S, n_frames = (int64_t)a.B * Nf * a.C;
  if (i < n_hist) {
    const int f = (int)(i / ((int64_t)a.B * a.Heff));
    const int64_t r = i % ((int64_t)a.B * a.Heff);
    const int b = (int)(r / a.Heff), t = (int)(r % a.Heff);
    a.x[f][(size_t)b * a.N + t] = a.xhist[((size_t)f * a.B + b) * a.H + a.H - a.Heff + t];
  } else if (i < n_hist + n_new) {
    const int64_t j = i - n_hist;
    const int b = (int)(j / a.S), s = (int)(j % a.S);
    a.x[0][(size_t)b * a.N + a.Heff + s] = noise.on ? philox::logistic_at(noise.seed, noise.stream, (uint64_t)j) : z[j];
  } else if (i < n_hist + n_new + n_frames) {
    const int64_t j = i - n_hist - n_new;
    const int b = (int)(j / ((int64_t)Nf * a.C));
    const int fr = (int)(j / a.C % Nf), ch = (int)(j % a.C);
    a.ebuf[j] = fr < hf ? a.fhist[((size_t)b * Hf + Hf - hf + fr) * a.C + ch]
                        : enc[((size_t)b * (Nf - hf) + fr - hf) * a.C + ch];
  }
}

// out = clip(z*s_tot + mu_tot, -1, 1) for the rows >= Heff, into [B][S] (k_flow_compose's arithmetic: flow_compose_at)
__global__ void __launch_bounds__(kThreads) k_stream_compose(const __grid_constant__ StreamArgs a, const float* __restrict__ scales,
                                                             const float* __restrict__ means, float* __restrict__ out,
                                                             float* __restrict__ s_tot, float* __restrict__ mu_tot,
                                                             float* __restrict__ x_last, float* __restrict__ z_out) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= (int64_t)a.B * a.S) return;
  const int64_t row = i / a.S * a.N + a.Heff + i % a.S;
  const float zi = a.x[0][row];
  if (z_out) z_out[i] = zi;
  float st, mt;
  flow_compose_at(scales, means, a.F, (int64_t)a.B * a.N, row, st, mt);
  if (s_tot) s_tot[i] = st;
  if (mu_tot) mu_tot[i] = mt;
  if (x_last) x_last[i] = a.x[a.F][row];
  out[i] = fminf(fmaxf(fmaf(zi, st, mt), -1.f), 1.f);
}

// The last H rows of each flow's input and the last H/P frames of [old history | this call] into the state, t0 += S.
// Row j of the new history is position j + S of that sequence: a buffer row, or (only while t0 + S < H) a position
// before the utterance's start, which is zero.
__global__ void __launch_bounds__(kThreads) k_stream_commit(const __grid_constant__ StreamArgs a) {
  if (!*a.valid) return;
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i == 0) *a.t0 = a.t0_call + a.S;
  const int Hf = a.H / a.P, Nf = a.N / a.P, hf = a.Heff / a.P, Sf = a.S / a.P;
  const int64_t n_x = (int64_t)a.F * a.B * a.H, n_f = (int64_t)a.B * Hf * a.C;
  if (i < n_x) {
    const int f = (int)(i / ((int64_t)a.B * a.H));
    const int64_t r = i % ((int64_t)a.B * a.H);
    const int b = (int)(r / a.H), j = (int)(r % a.H);
    const int src = j + a.S - (a.H - a.Heff);
    a.xhist[i] = src >= 0 ? a.x[f][(size_t)b * a.N + src] : 0.f;
  } else if (i < n_x + n_f) {
    const int64_t k = i - n_x;
    const int b = (int)(k / ((int64_t)Hf * a.C));
    const int j = (int)(k / a.C % Hf), ch = (int)(k % a.C);
    const int src = j + Sf - (Hf - hf);
    a.fhist[k] = src >= 0 ? a.ebuf[((size_t)b * Nf + src) * a.C + ch] : 0.f;
  }
}

// workspace: flow buffers [F+1][B][H+S] | frames [B][(H+S)/P][C] | valid word | the flows' own workspace for (B, H+S)
struct StreamWs { float* x[17]; float* ebuf; int* valid; uint8_t* inner; size_t inner_bytes, bytes; };

StreamWs carve(const srwn_ctx* c, int B, int S, int precision, void* ws, size_t cap) {
  WsCarver w(ws, cap);
  StreamWs r{};
  const int Nmax = history_rows(c) + S;
  for (int f = 0; f <= c->cfg.num_flows; f++) r.x[f] = w.take<float>((size_t)B * Nmax);
  r.ebuf = w.take<float>((size_t)B * (Nmax / c->cfg.pool_stride) * c->cfg.cond_channels);
  r.valid = w.take<int>(1);
  r.inner_bytes = student_flows_workspace_bytes(c, precision, B, Nmax);
  r.inner = w.take<uint8_t>(r.inner_bytes);
  r.bytes = w.used;
  return r;
}
}  // namespace

size_t student_stream_workspace_bytes(const srwn_ctx* h, int B, int S, int precision) {
  return carve(h, B, S, precision, nullptr, 0).bytes;
}

extern "C" int srwn_student_state_bytes(srwn_handle_t h, int32_t B, int32_t precision, size_t* bytes) {
  if (!h || !bytes) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_state_bytes: null argument");
  if (int rc = check_state(h, SRWN_OP_STUDENT_STREAM, B, precision)) return rc;
  *bytes = layout(h, B).bytes;
  return SRWN_OK;
}

extern "C" int srwn_student_state_reset(srwn_handle_t h, void* state, int32_t B, int32_t precision, void* stream) {
  if (!h || !state) return srwn_fail(SRWN_ERR_INVALID, "srwn_student_state_reset: null argument");
  if (int rc = check_state(h, SRWN_OP_STUDENT_STREAM, B, precision)) return rc;
  StreamHeader hdr{};
  signature(h, B, precision, hdr.sig);
  const cudaStream_t st = (cudaStream_t)stream;
  SRWN_CUDA(cudaMemsetAsync(state, 0, layout(h, B).bytes, st));          // silence before the utterance (ops.py:9)
  // pageable source: the copy is staged before this call returns, so `hdr` may go out of scope
  SRWN_CUDA(cudaMemcpyAsync(state, &hdr, sizeof(hdr), cudaMemcpyHostToDevice, st));
  state_owner_record(h, state, hdr.sig, kSigLen);
  return SRWN_OK;
}

int run_student_stream(srwn_ctx* h, void* state, long long t0, const float* z, NoiseSpec noise, const float* enc, float* out,
                       float* s_tot, float* mu_tot, float* x_last, float* z_out, int B, int S, int precision, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  int32_t sig[kSigLen];
  signature(h, B, precision, sig);
  int rc = state_owner_check(h, state, sig, kSigLen, "srwn_student_state_reset");
  if (rc) return rc;
  const StreamWs w = carve(h, B, S, precision, ws, ws_bytes);
  if ((rc = check_workspace(ws, ws_bytes, w.bytes))) return rc;
  rc = sticky_error(h);
  if (rc) return rc;
  StreamArgs a;
  const int F = h->cfg.num_flows, H = history_rows(h);
  memcpy(a.x, w.x, sizeof(a.x));
  a.ebuf = w.ebuf; a.valid = w.valid; a.err = h->h_err;
  uint8_t* base = static_cast<uint8_t*>(state);
  const StreamLayout lay = layout(h, B);
  a.t0 = &reinterpret_cast<StreamHeader*>(base)->t0;
  a.xhist = reinterpret_cast<float*>(base + lay.xhist);
  a.fhist = reinterpret_cast<float*>(base + lay.fhist);
  a.t0_call = t0;
  a.B = B; a.S = S; a.H = H; a.Heff = (int)(t0 < H ? t0 : H); a.N = a.Heff + S; a.F = F;
  a.C = h->cfg.cond_channels; a.P = h->cfg.pool_stride;

  const int64_t n_in = (int64_t)F * B * a.Heff + (int64_t)B * S + (int64_t)B * (a.N / a.P) * a.C;
  k_stream_assemble<<<(unsigned)((n_in + kThreads - 1) / kThreads), kThreads, 0, st>>>(a, z, noise, enc);
  SRWN_LAUNCH_CHECK();
  const float *scales = nullptr, *means = nullptr;
  rc = run_student_flows(h, precision, a.x, NoiseSpec{0, 0, 0}, a.ebuf, B, a.N, a.Heff, w.inner, w.inner_bytes, &scales, &means, st);
  if (rc) return rc;
  const int64_t n_out = (int64_t)B * S;
  k_stream_compose<<<(unsigned)((n_out + kThreads - 1) / kThreads), kThreads, 0, st>>>(a, scales, means, out, s_tot, mu_tot,
                                                                                       x_last, z_out);
  SRWN_LAUNCH_CHECK();
  const int64_t n_state = (int64_t)F * B * H + (int64_t)B * (H / a.P) * a.C;
  k_stream_commit<<<(unsigned)((n_state + kThreads - 1) / kThreads), kThreads, 0, st>>>(a);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}
