// Stateless, shape-generic versions of the ops.py building blocks.  These back the
// Python mirror of ops.py (any channel count / kernel size); the model paths use the
// specialised kernels in stack_f32.cu / fused.cu / ar_generate.cu instead.
#include "common.cuh"

// ops.py:6-20: out[b,t,co] = bias[co] + sum_k sum_ci x[b, t - d*(K-1-k), ci] * w[k,ci,co]
__global__ void k_conv_generic(const float* __restrict__ x, const float* __restrict__ w,
                               const float* __restrict__ bias, float* __restrict__ y, int T, int Cin,
                               int Cout, int K, int d) {
  const int b = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)T * Cout) return;
  const int t = (int)(idx / Cout), co = (int)(idx % Cout);
  float acc = bias ? bias[co] : 0.f;
  for (int k = 0; k < K; k++) {
    const int tt = t - d * (K - 1 - k);
    if (tt < 0) continue;
    const float* xr = x + ((size_t)b * T + tt) * Cin;
    const float* wk = w + (size_t)k * Cin * Cout + co;
    for (int ci = 0; ci < Cin; ci++) acc = fmaf(xr[ci], wk[(size_t)ci * Cout], acc);
  }
  y[((size_t)b * T + t) * Cout + co] = acc;
}

extern "C" int srwn_dilated_causal_conv1d(const float* x, const float* filters, const float* bias,
                                          float* y, int32_t B, int32_t T, int32_t Cin, int32_t Cout,
                                          int32_t K, int32_t dilation, void* stream) {
  if (!x || !filters || !y) return srwn_fail(SRWN_ERR_INVALID, "srwn_dilated_causal_conv1d: null argument");
  if (B < 0 || T < 0 || Cin < 1 || Cout < 1 || K < 1 || dilation < 1 || B > 65535)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_dilated_causal_conv1d: bad shape");
  if (B == 0 || T == 0) return SRWN_OK;
  dim3 grid((unsigned)(((int64_t)T * Cout + 255) / 256), B);
  k_conv_generic<<<grid, 256, 0, (cudaStream_t)stream>>>(x, filters, bias, y, T, Cin, Cout, K, dilation);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// tf.layers.conv1d(padding='SAME', strides=1) as the non-causal layers use it (ops.py:48-57): TensorFlow pads
// (K - 1) / 2 on the left and the rest on the right, so out[b,t,co] = bias[co] + sum_k sum_ci act(x[b, t + k - (K-1)/2, ci]) w[k,ci,co];
// flags: bit 0 = relu on the input (ops.py:49,52), bit 1 = relu on the output
__global__ void k_conv_same(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                            float* __restrict__ y, int T, int Cin, int Cout, int K, int flags) {
  const int b = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)T * Cout) return;
  const int t = (int)(idx / Cout), co = (int)(idx % Cout), left = (K - 1) / 2;
  float acc = bias ? bias[co] : 0.f;
  for (int k = 0; k < K; k++) {
    const int tt = t + k - left;
    if (tt < 0 || tt >= T) continue;
    const float* xr = x + ((size_t)b * T + tt) * Cin;
    const float* wk = w + (size_t)k * Cin * Cout + co;
    if (flags & 1) { for (int ci = 0; ci < Cin; ci++) acc = fmaf(fmaxf(xr[ci], 0.f), wk[(size_t)ci * Cout], acc); }
    else { for (int ci = 0; ci < Cin; ci++) acc = fmaf(xr[ci], wk[(size_t)ci * Cout], acc); }
  }
  y[((size_t)b * T + t) * Cout + co] = (flags & 2) ? fmaxf(acc, 0.f) : acc;
}

extern "C" int srwn_conv1d_same(const float* x, const float* filters, const float* bias, float* y, int32_t B, int32_t T,
                                int32_t Cin, int32_t Cout, int32_t K, int32_t flags, void* stream) {
  if (!x || !filters || !y) return srwn_fail(SRWN_ERR_INVALID, "srwn_conv1d_same: null argument");
  if (B < 0 || T < 0 || Cin < 1 || Cout < 1 || K < 1 || B > 65535) return srwn_fail(SRWN_ERR_INVALID, "srwn_conv1d_same: bad shape");
  if (B == 0 || T == 0) return SRWN_OK;
  dim3 grid((unsigned)(((int64_t)T * Cout + 255) / 256), B);
  k_conv_same<<<grid, 256, 0, (cudaStream_t)stream>>>(x, filters, bias, y, T, Cin, Cout, K, flags);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ops.py:111-122: log_prob_from_logits (mode 0: y [rows][C] = x - max - log sum exp(x - max)) and log_sum_exp
// (mode 1: y [rows] = max + log sum exp(x - max)) over the last axis
__global__ void k_log_softmax_rows(const float* __restrict__ x, float* __restrict__ y, int64_t rows, int C, int mode) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* xr = x + r * C;
  float m = xr[0];
  for (int c = 1; c < C; c++) m = fmaxf(m, xr[c]);
  float sum = 0.f;
  for (int c = 0; c < C; c++) sum += expf(xr[c] - m);
  const float ls = logf(sum);
  if (mode == 1) { y[r] = m + ls; return; }
  for (int c = 0; c < C; c++) y[r * C + c] = xr[c] - m - ls;
}
extern "C" int srwn_log_softmax(const float* x, float* y, int64_t rows, int32_t C, int32_t reduce, void* stream) {
  if (!x || !y || rows < 1 || C < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_log_softmax: bad argument");
  k_log_softmax_rows<<<(unsigned)((rows + 127) / 128), 128, 0, (cudaStream_t)stream>>>(x, y, rows, C, reduce ? 1 : 0);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ops.py:23-46 for generic R / S / K.  8 time steps per CTA; gate activations staged in smem.
constexpr int kGenRows = 8;
__global__ void __launch_bounds__(128)
k_block_generic(const float* __restrict__ x, const float* __restrict__ fk, const float* __restrict__ fb,
                const float* __restrict__ rk, const float* __restrict__ rb, const float* __restrict__ sk,
                const float* __restrict__ sb, float* __restrict__ dense, float* __restrict__ skip,
                int T, int R, int S, int K, int d) {
  extern __shared__ float s_c[];   // [kGenRows][R]
  const int b = blockIdx.y, t0 = blockIdx.x * kGenRows;
  for (int o = threadIdx.x; o < kGenRows * R; o += blockDim.x) {
    const int row = o / R, r = o % R, t = t0 + row;
    float v = 0.f;
    if (t < T) {
      float acc = fb ? fb[r] : 0.f;
      for (int k = 0; k < K; k++) {
        const int tt = t - d * (K - 1 - k);
        if (tt < 0) continue;
        const float* xr = x + ((size_t)b * T + tt) * R;
        const float* wk = fk + (size_t)k * R * R + r;
        for (int ci = 0; ci < R; ci++) acc = fmaf(xr[ci], wk[(size_t)ci * R], acc);
      }
      const float f = tanhf(acc);                       // ops.py:28
      v = f * (1.0f / (1.0f + expf(-f)));               // ops.py:33,36 (gate is sigmoid of the tanh)
    }
    s_c[o] = v;
  }
  __syncthreads();
  for (int o = threadIdx.x; o < kGenRows * R; o += blockDim.x) {
    const int row = o / R, r = o % R, t = t0 + row;
    if (t >= T) continue;
    float acc = rb[r];
    for (int k = 0; k < R; k++) acc = fmaf(s_c[row * R + k], rk[(size_t)k * R + r], acc);
    const size_t at = ((size_t)b * T + t) * R + r;
    dense[at] = (x[at] + acc) * SRWN_SQRT_HALF;          // ops.py:40
  }
  if (skip) {
    for (int o = threadIdx.x; o < kGenRows * S; o += blockDim.x) {
      const int row = o / S, j = o % S, t = t0 + row;
      if (t >= T) continue;
      float acc = sb[j];
      for (int k = 0; k < R; k++) acc = fmaf(s_c[row * R + k], sk[(size_t)k * S + j], acc);
      skip[((size_t)b * T + t) * S + j] = acc;           // ops.py:44
    }
  }
}

extern "C" int srwn_residual_dilation_layer(const float* x, const float* filt_k, const float* filt_b,
                                            const float* res_k, const float* res_b,
                                            const float* skip_k, const float* skip_b, float* dense,
                                            float* skip, int32_t B, int32_t T, int32_t R, int32_t S,
                                            int32_t K, int32_t dilation, void* stream) {
  if (!x || !filt_k || !res_k || !res_b || !dense)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_residual_dilation_layer: null argument");
  if (skip && (!skip_k || !skip_b)) return srwn_fail(SRWN_ERR_INVALID, "skip output needs skip_k and skip_b");
  if (B < 0 || T < 0 || R < 1 || (skip && S < 1) || K < 1 || dilation < 1 || B > 65535 || R > 1024)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_residual_dilation_layer: bad shape");
  if (B == 0 || T == 0) return SRWN_OK;
  dim3 grid((T + kGenRows - 1) / kGenRows, B);
  k_block_generic<<<grid, 128, kGenRows * R * sizeof(float), (cudaStream_t)stream>>>(
      x, filt_k, filt_b, res_k, res_b, skip_k, skip_b, dense, skip, T, R, S, K, dilation);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ops.py:78-80
__global__ void k_right_shift(const float* __restrict__ x, float* __restrict__ y, int T, int C, int shift) {
  const int b = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)T * C) return;
  const int t = (int)(idx / C), c = (int)(idx % C);
  y[((size_t)b * T + t) * C + c] = t >= shift ? x[((size_t)b * T + t - shift) * C + c] : 0.f;
}

extern "C" int srwn_right_shift(const float* x, float* y, int32_t B, int32_t T, int32_t C,
                                int32_t shift, void* stream) {
  if (!x || !y) return srwn_fail(SRWN_ERR_INVALID, "srwn_right_shift: null argument");
  if (B < 0 || T < 0 || C < 1 || shift < 0 || B > 65535) return srwn_fail(SRWN_ERR_INVALID, "srwn_right_shift: bad shape");
  if (B == 0 || T == 0) return SRWN_OK;
  dim3 grid((unsigned)(((int64_t)T * C + 255) / 256), B);
  k_right_shift<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, T, C, shift);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ops.py:64-74: resize_nearest_neighbor(align_corners=False): src = min(floor(dst*L/out), L-1)
__global__ void k_resize_nearest(const float* __restrict__ x, float* __restrict__ y, int L, int C, int out) {
  const int b = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)out * C) return;
  const int t = (int)(idx / C), c = (int)(idx % C);
  int src = (int)(((int64_t)t * L) / out);
  if (src > L - 1) src = L - 1;
  y[((size_t)b * out + t) * C + c] = x[((size_t)b * L + src) * C + c];
}

extern "C" int srwn_resize_nearest(const float* x, float* y, int32_t B, int32_t L, int32_t C,
                                   int32_t out_size, void* stream) {
  if (!x || !y) return srwn_fail(SRWN_ERR_INVALID, "srwn_resize_nearest: null argument");
  if (B < 0 || L < 1 || C < 1 || out_size < 0 || B > 65535) return srwn_fail(SRWN_ERR_INVALID, "srwn_resize_nearest: bad shape");
  if (B == 0 || out_size == 0) return SRWN_OK;
  dim3 grid((unsigned)(((int64_t)out_size * C + 255) / 256), B);
  k_resize_nearest<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, L, C, out_size);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ---- pieces of the classification / embedding heads (model.py:33-57, 692-713): relu, average pooling over a window of time
// steps (tf.nn.pool AVG, VALID), softmax over the channels, Euclidean distance of two embeddings (model.py:735)
__global__ void k_relu(float* __restrict__ x, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = fmaxf(x[i], 0.f);
}
extern "C" int srwn_relu(float* x, int64_t n, void* stream) {
  if (!x || n < 0) return srwn_fail(SRWN_ERR_INVALID, "srwn_relu: bad argument");
  if (n == 0) return SRWN_OK;
  k_relu<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, n);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// y[b][o][c] = mean over w < window of x[b][o + w][c]; one CTA per (o, b), the threads split the window, fixed-order sum
__global__ void __launch_bounds__(256) k_avg_pool_time(const float* __restrict__ x, float* __restrict__ y, int T, int C, int window, int out) {
  extern __shared__ double s_part[];                 // [parts][C]
  const int o = blockIdx.x, b = blockIdx.y, parts = blockDim.x / C > 0 ? blockDim.x / C : 1;
  const int c = threadIdx.x % C, part = threadIdx.x / C;
  if (part < parts && threadIdx.x < parts * C) {
    double acc = 0.0;
    for (int w = part; w < window; w += parts) acc += (double)x[((size_t)b * T + o + w) * C + c];
    s_part[part * C + c] = acc;
  }
  __syncthreads();
  for (int cc = threadIdx.x; cc < C; cc += blockDim.x) {
    double t = 0.0;
    for (int k = 0; k < parts; k++) t += s_part[k * C + cc];
    y[((size_t)b * out + o) * C + cc] = (float)(t / window);
  }
}
extern "C" int srwn_avg_pool_time(const float* x, float* y, int32_t B, int32_t T, int32_t C, int32_t window, void* stream) {
  if (!x || !y) return srwn_fail(SRWN_ERR_INVALID, "srwn_avg_pool_time: null argument");
  if (B < 1 || T < 1 || C < 1 || C > 256 || window < 1 || window > T || B > 65535)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_avg_pool_time: needs 1 <= window <= T, 1 <= C <= 256");
  const int out = T - window + 1, parts = 256 / C > 0 ? 256 / C : 1;
  k_avg_pool_time<<<dim3(out, B), 256, (size_t)parts * C * sizeof(double), (cudaStream_t)stream>>>(x, y, T, C, window, out);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

__global__ void k_softmax_rows(const float* __restrict__ x, float* __restrict__ y, int64_t rows, int C) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* xr = x + r * C;
  float m = xr[0];
  for (int c = 1; c < C; c++) m = fmaxf(m, xr[c]);
  float sum = 0.f;
  for (int c = 0; c < C; c++) sum += expf(xr[c] - m);
  for (int c = 0; c < C; c++) y[r * C + c] = expf(xr[c] - m) / sum;
}
extern "C" int srwn_softmax(const float* x, float* y, int64_t rows, int32_t C, void* stream) {
  if (!x || !y || rows < 1 || C < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_softmax: bad argument");
  k_softmax_rows<<<(unsigned)((rows + 127) / 128), 128, 0, (cudaStream_t)stream>>>(x, y, rows, C);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// d[b] = sqrt(1e-8 + sum_k (a[b][k] - c[b][k])^2)   (model.py:735, the 1e-8 keeps the gradient finite)
__global__ void k_pair_distance(const float* __restrict__ a, const float* __restrict__ c, float* __restrict__ d, int B, int D) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float s = 0.f;
  for (int k = 0; k < D; k++) { const float t = a[(size_t)b * D + k] - c[(size_t)b * D + k]; s = fmaf(t, t, s); }
  d[b] = sqrtf(1e-8f + s);
}
extern "C" int srwn_pair_distance(const float* a, const float* b, float* d, int32_t B, int32_t D, void* stream) {
  if (!a || !b || !d || B < 1 || D < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_pair_distance: bad argument");
  k_pair_distance<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a, b, d, B, D);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

extern "C" int srwn_mol_loss(const float* x, const float* l, float* nll_out, float* nll_sum, int32_t B,
                             int32_t T, int32_t M, void* stream) {
  if (!x || !l || (!nll_out && !nll_sum)) return srwn_fail(SRWN_ERR_INVALID, "srwn_mol_loss: null argument");
  if (B < 1 || T < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_mol_loss: bad shape");
  return run_mol_loss(x, l, nll_out, nll_sum, B, T, M, (cudaStream_t)stream);
}

extern "C" int srwn_mol_sample(const float* l, const float* u1, const float* u2, float* out,
                               int32_t* idx_out, int32_t B, int32_t T, int32_t M, void* stream) {
  if (!l || !u1 || !u2 || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_mol_sample: null argument");
  if (B < 1 || T < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_mol_sample: bad shape");
  return run_mol_sample(l, u1, u2, out, idx_out, B, T, M, (cudaStream_t)stream);
}
