// Spectral power loss of the distillation objective (model.py:360-371) and the elementwise loss glue of
// model.py:356-379, on the device.
//
//   stft   = tf.contrib.signal.stft(x, frame_length N = 512, frame_step = 256): periodic Hann window,
//            fft_length = N, no padding -> F = 1 + (T - N) / step frames of N/2 + 1 bins      (model.py:360-361)
//   s(x)   = mean over frames of |stft|^2, [B, N/2 + 1]                                        (model.py:366-367)
//   loss   = gamma * sum_{b,k} (s(truth) - s(out))^2                                           (model.py:369-371)
//
// Forward: one CTA per (frame, utterance, signal) runs a radix-2 Stockham FFT of the windowed frame in shared
// memory and stores |X_k|^2 (and X_k itself for `out`, the signal that is differentiated).  Frame means and the loss
// are summed in a fixed order (deterministic).  Backward: with a_k = dLoss/d|X_{f,k}|^2 = -2 gamma (s1 - s2)_k / F,
//   dLoss/dx_frame[n] = 2 w[n] sum_{k=0}^{N/2} a_k Re(X_k e^{+2 pi i k n / N}) = w[n] * IDFT_N(Z)[n],
// Z the Hermitian extension of a_k X_k with the k = 0 and k = N/2 bins doubled (IDFT unnormalised), evaluated
// with the same FFT routine on conj(Z); frames are overlap-added by a gather, again in a fixed order.
// The problem is tiny (B * F frames of 512 points; 2 MB of spectra at 4 x 64000) next to the flows' backward pass.
#include "common.cuh"

namespace stftk {

// Stockham autosort radix-2 FFT (forward, e^{-i...}) of N = 2^lg points held in `a`; `b` is the ping-pong buffer,
// `tw[j] = exp(-2 pi i j / N)` for j < N/2.  Returns the buffer that holds the result (natural order).
__device__ __forceinline__ float2* fft_pow2(float2* a, float2* b, const float2* tw, int N, int lg) {
  float2 *x = a, *y = b;
  int s = 1;                                  // stride; sub-transform length n = N / s
  for (int st = 0; st < lg; st++, s <<= 1) {
    const int m = (N / s) >> 1;
    for (int i = threadIdx.x; i < N / 2; i += blockDim.x) {
      const int p = i / s, q = i - p * s;
      const float2 w = tw[p * s];
      const float2 u = x[q + s * p], v = x[q + s * (p + m)];
      const float dr = u.x - v.x, di = u.y - v.y;
      y[q + s * (2 * p)] = make_float2(u.x + v.x, u.y + v.y);
      y[q + s * (2 * p + 1)] = make_float2(dr * w.x - di * w.y, dr * w.y + di * w.x);
    }
    __syncthreads();
    float2* t = x; x = y; y = t;
  }
  return x;
}

__device__ __forceinline__ void make_twiddles(float2* tw, int N) {
  for (int j = threadIdx.x; j < N / 2; j += blockDim.x) {
    float sn, cs;
    sincospif(2.0f * (float)j / (float)N, &sn, &cs);
    tw[j] = make_float2(cs, -sn);
  }
}
__device__ __forceinline__ float hann_periodic(int n, int N) { return 0.5f - 0.5f * cospif(2.0f * (float)n / (float)N); }

// grid (F, B, nsig).  P [nsig][B][F][K] = |X|^2; spec [B][F][K] = X of the LAST signal (may be null).
__global__ void k_frames(const float* __restrict__ sig0, const float* __restrict__ sig1, float* __restrict__ P,
                         float2* __restrict__ spec, int B, int T, int N, int lg, int step, int F) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* a = reinterpret_cast<float2*>(smem_raw);
  float2* b = a + N;
  float2* tw = b + N;
  const int f = blockIdx.x, bi = blockIdx.y, sg = blockIdx.z, K = N / 2 + 1;
  const float* x = (sg == 0 ? sig0 : sig1) + (size_t)bi * T + (size_t)f * step;
  make_twiddles(tw, N);
  for (int n = threadIdx.x; n < N; n += blockDim.x) a[n] = make_float2(x[n] * hann_periodic(n, N), 0.f);
  __syncthreads();
  const float2* X = fft_pow2(a, b, tw, N, lg);
  const size_t row = (((size_t)sg * B + bi) * F + f) * K;
  const bool keep = spec != nullptr && sg == (int)gridDim.z - 1;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const float2 v = X[k];
    P[row + k] = v.x * v.x + v.y * v.y;
    if (keep) spec[((size_t)bi * F + f) * K + k] = v;
  }
}

// mean over frames in a fixed order: grid (B, nsig), thread per bin.
__global__ void k_frame_mean(const float* __restrict__ P, float* __restrict__ mean, int B, int F, int K) {
  const int bi = blockIdx.x, sg = blockIdx.y;
  const float* p = P + ((size_t)sg * B + bi) * F * K;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    double acc = 0;
    for (int f = 0; f < F; f++) acc += (double)p[(size_t)f * K + k];
    mean[((size_t)sg * B + bi) * K + k] = (float)(acc / F);
  }
}

// g = s(truth) - s(out) [B*K]; loss = gamma * sum g^2 (one CTA, fixed order).
__global__ void k_power_loss(const float* __restrict__ mean, float* __restrict__ g, double* __restrict__ loss, int n, float gamma) {
  __shared__ double red[256];
  double acc = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float d = mean[i] - mean[n + i];
    g[i] = d;
    acc += (double)d * d;
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s >= 1; s >>= 1) { if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s]; __syncthreads(); }
  if (threadIdx.x == 0) *loss = (double)gamma * red[0];
}

// grid (F, B): fr [B][F][N] = dLoss/d(frame samples), before the overlap-add.
__global__ void k_grad_frames(const float2* __restrict__ spec, const float* __restrict__ g, float* __restrict__ fr,
                              int N, int lg, int F, float coef /* -2 gamma / F */) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* a = reinterpret_cast<float2*>(smem_raw);
  float2* b = a + N;
  float2* tw = b + N;
  const int f = blockIdx.x, bi = blockIdx.y, K = N / 2 + 1;
  const float2* X = spec + ((size_t)bi * F + f) * K;
  const float* gb = g + (size_t)bi * K;
  make_twiddles(tw, N);
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const float ak = coef * gb[k];
    const float2 v = X[k];
    if (k == 0 || k == N / 2) a[k] = make_float2(2.f * ak * v.x, 0.f);        // X_0, X_{N/2} are real for a real frame
    else {
      a[k] = make_float2(ak * v.x, -ak * v.y);                                // conj(Z_k)
      a[N - k] = make_float2(ak * v.x, ak * v.y);                             // conj(Z_{N-k}) = Z_k
    }
  }
  __syncthreads();
  const float2* R = fft_pow2(a, b, tw, N, lg);                                // DFT(conj Z) = conj(IDFT(Z)); real
  float* o = fr + ((size_t)bi * F + f) * N;
  for (int n = threadIdx.x; n < N; n += blockDim.x) o[n] = hann_periodic(n, N) * R[n].x;
}

// d_out[b][t] = sum over the frames that contain t, lowest frame first.
__global__ void k_overlap_add(const float* __restrict__ fr, float* __restrict__ d_out, int B, int T, int N, int step, int F) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * T) return;
  const int bi = (int)(i / T), t = (int)(i - (int64_t)bi * T);
  int f_lo = t - N + 1 <= 0 ? 0 : (t - N + step) / step;                       // ceil((t - N + 1) / step)
  int f_hi = t / step;
  if (f_hi > F - 1) f_hi = F - 1;
  float acc = 0.f;
  for (int f = f_lo; f <= f_hi; f++) acc += fr[((size_t)bi * F + f) * N + (t - f * step)];
  d_out[i] = acc;
}

// ---- loss glue (model.py:356, 374-379, 535) ------------------------------------------------------------------
// pre = z s_tot + mu_tot;  d_pre = (beta d_ce + d_pow) [|pre| <= 1] / norm  (tf.clip_by_value passes the gradient
// inside the interval);  d_s = -(alpha / norm) / s_tot (entropy sum(log s_tot + 2));  sums: sum nll, sum(log s_tot + 2).
constexpr int kGlueBlocks = 296;
__global__ void __launch_bounds__(256)
k_loss_glue(const float* __restrict__ z, const float* __restrict__ s_tot, const float* __restrict__ mu_tot,
            const float* __restrict__ nll, const float* __restrict__ d_ce, const float* __restrict__ d_pow,
            float alpha, float beta, float inv_norm, float* __restrict__ d_pre, float* __restrict__ d_s,
            double* __restrict__ partial, int64_t n) {
  __shared__ double red[2][256];
  double a_nll = 0, a_ent = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float s = s_tot[i];
    const float pre = __fadd_rn(__fmul_rn(z[i], s), mu_tot[i]);
    const float m = (pre >= -1.f && pre <= 1.f) ? inv_norm : 0.f;
    const float dp = d_pow ? d_pow[i] : 0.f;
    d_pre[i] = __fmaf_rn(beta, d_ce[i], dp) * m;
    d_s[i] = -(alpha * inv_norm) / s;
    if (nll) a_nll += (double)nll[i];
    a_ent += (double)(logf(s) + 2.f);
  }
  red[0][threadIdx.x] = a_nll; red[1][threadIdx.x] = a_ent;
  __syncthreads();
  for (int st = 128; st >= 1; st >>= 1) {
    if (threadIdx.x < st) { red[0][threadIdx.x] += red[0][threadIdx.x + st]; red[1][threadIdx.x] += red[1][threadIdx.x + st]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = red[0][0]; partial[2 * blockIdx.x + 1] = red[1][0]; }
}
__global__ void k_glue_final(const double* __restrict__ partial, double* __restrict__ sums, int blocks) {
  if (threadIdx.x < 2) {
    double acc = 0;
    for (int i = 0; i < blocks; i++) acc += partial[2 * i + threadIdx.x];
    sums[threadIdx.x] = acc;
  }
}

}  // namespace stftk

struct StftWs { float* P; float2* spec; float* mean; float* g; float* fr; size_t bytes; };
static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }
static StftWs carve_stft(int B, int N, int F, void* ws) {
  const size_t K = N / 2 + 1;
  char* p = (char*)ws;
  StftWs w;
  size_t o = 0;
  w.P = (float*)(p + o); o += al256(2 * (size_t)B * F * K * sizeof(float));
  w.spec = (float2*)(p + o); o += al256((size_t)B * F * K * sizeof(float2));
  w.mean = (float*)(p + o); o += al256(2 * (size_t)B * K * sizeof(float));
  w.g = (float*)(p + o); o += al256((size_t)B * K * sizeof(float));
  w.fr = (float*)(p + o); o += al256((size_t)B * F * N * sizeof(float));
  w.bytes = o;
  return w;
}

static int stft_shape(int B, int T, int N, int step, int* lg, int* F, const char* who) {
  int l = 0;
  while ((1 << l) < N) l++;
  if (B < 1 || T < 1 || N < 8 || N > 4096 || (1 << l) != N || step < 1)
    return srwn_fail(SRWN_ERR_INVALID, "%s: frame_length must be a power of two in [8, 4096], frame_step >= 1", who);
  if (T < N) return srwn_fail(SRWN_ERR_INVALID, "%s: T = %d is shorter than one frame (%d): the reference's mean over frames is empty", who, T, N);
  *lg = l;
  *F = 1 + (T - N) / step;
  return SRWN_OK;
}

int run_stft_workspace_bytes(int B, int T, int N, int step, size_t* bytes) {
  int lg, F;
  if (int rc = stft_shape(B, T, N, step, &lg, &F, "srwn_stft_workspace_bytes")) return rc;
  *bytes = carve_stft(B, N, F, nullptr).bytes;
  return SRWN_OK;
}

int run_stft_power(const float* x, float* power, int B, int T, int N, int step, void* ws, size_t cap, cudaStream_t st) {
  int lg, F;
  if (int rc = stft_shape(B, T, N, step, &lg, &F, "srwn_stft_power")) return rc;
  StftWs w = carve_stft(B, N, F, ws);
  if (int rc = check_workspace(ws, cap, w.bytes)) return rc;
  const int K = N / 2 + 1, thr = N / 2 < 32 ? 32 : (N / 2 > 256 ? 256 : N / 2);
  const size_t smem = (size_t)(2 * N + N / 2) * sizeof(float2);
  if (smem > 48 * 1024) SRWN_CUDA(cudaFuncSetAttribute(stftk::k_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  stftk::k_frames<<<dim3(F, B, 1), thr, smem, st>>>(x, x, w.P, nullptr, B, T, N, lg, step, F);
  SRWN_LAUNCH_CHECK();
  stftk::k_frame_mean<<<dim3(B, 1), 256, 0, st>>>(w.P, w.mean, B, F, K);
  SRWN_LAUNCH_CHECK();
  SRWN_CUDA(cudaMemcpyAsync(power, w.mean, (size_t)B * K * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return SRWN_OK;
}

int run_stft_power_loss(const float* truth, const float* out, float gamma, double* loss, float* d_out, int B, int T, int N,
                        int step, void* ws, size_t cap, cudaStream_t st) {
  int lg, F;
  if (int rc = stft_shape(B, T, N, step, &lg, &F, "srwn_stft_power_loss")) return rc;
  StftWs w = carve_stft(B, N, F, ws);
  if (int rc = check_workspace(ws, cap, w.bytes)) return rc;
  const int K = N / 2 + 1, thr = N / 2 < 32 ? 32 : (N / 2 > 256 ? 256 : N / 2);
  const size_t smem = (size_t)(2 * N + N / 2) * sizeof(float2);
  if (smem > 48 * 1024) {
    SRWN_CUDA(cudaFuncSetAttribute(stftk::k_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SRWN_CUDA(cudaFuncSetAttribute(stftk::k_grad_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  stftk::k_frames<<<dim3(F, B, 2), thr, smem, st>>>(truth, out, w.P, w.spec, B, T, N, lg, step, F);
  SRWN_LAUNCH_CHECK();
  stftk::k_frame_mean<<<dim3(B, 2), 256, 0, st>>>(w.P, w.mean, B, F, K);
  SRWN_LAUNCH_CHECK();
  stftk::k_power_loss<<<1, 256, 0, st>>>(w.mean, w.g, loss, B * K, gamma);
  SRWN_LAUNCH_CHECK();
  if (d_out) {
    stftk::k_grad_frames<<<dim3(F, B), thr, smem, st>>>(w.spec, w.g, w.fr, N, lg, F, -2.f * gamma / (float)F);
    SRWN_LAUNCH_CHECK();
    const int64_t n = (int64_t)B * T;
    stftk::k_overlap_add<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w.fr, d_out, B, T, N, step, F);
    SRWN_LAUNCH_CHECK();
  }
  return SRWN_OK;
}

int run_distill_loss_grad(const float* z, const float* s_tot, const float* mu_tot, const float* nll, const float* d_ce,
                          const float* d_pow, float alpha, float beta, float inv_norm, float* d_pre, float* d_s, double* sums,
                          int B, int T, cudaStream_t st) {
  const int64_t n = (int64_t)B * T;
  stftk::k_loss_glue<<<stftk::kGlueBlocks, 256, 0, st>>>(z, s_tot, mu_tot, nll, d_ce, d_pow, alpha, beta, inv_norm, d_pre, d_s,
                                                         sums + 2, n);
  SRWN_LAUNCH_CHECK();
  stftk::k_glue_final<<<1, 32, 0, st>>>(sums + 2, sums, stftk::kGlueBlocks);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}
