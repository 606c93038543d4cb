// Student distillation step, device side (fp32 grade): forward that keeps every layer input, and the backward pass
// of the IAF flows (model.py:415-535) given the gradient of the loss (model.py:356-379) with respect to the
// network output.  Layer at a time; activations and their gradients round-trip HBM in fp32.  The forward is the
// fp32-grade stack of stack_f32.cu, run so that it keeps every layer input; the two backward layer kernels are tcgen05
// kernels (train_tc.cu).  This file holds the elementwise kernels around them and the host sequence.
//
//   forward (per flow f):  x_0 = front(x_{f-1}) + cond_0;  x_{l+1} = (x_l + Wr c_l + br) sqrt(1/2) + cond_{l+1},
//                          c_l = f sigmoid(f), f = tanh(W0 x_l[t-d] + W1 x_l[t] + bf)          (ops.py:23-46, F1-F3)
//                          p = relu(x_L) Wh + bh;  s_f = exp(p0), mu_f = p1, x_f = x_{f-1} s_f + mu_f (model.py:479-482)
//   compose:               S = prod s_f,  M = sum_f mu_f prod_{j>f} s_j,  out = clip(z S + M)   (model.py:517-535)
//   backward:              reverse of the above; weight gradients are reduced per CTA (registers -> one partial
//                          row per CTA) and summed by a second kernel in a fixed order (deterministic).
#include "common.cuh"
#include "mol.cuh"
#include "train_tc.cuh"

namespace train {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// sums `rows` partial rows (row pitch `pitch`) of width w1 + w2 into dst1 [w1] and dst2 [w2] (+=) in a fixed order:
// 32 columns per CTA, the rows split over the 8 warps (independent loads in flight), then a fixed-order sum of the 8 parts
__global__ void __launch_bounds__(256)
k_reduce_partials(const float* __restrict__ partial, int rows, int pitch, int w1, float* __restrict__ dst1, int w2,
                  float* __restrict__ dst2, size_t layer_stride = 0, int dst1_stride = 0, int dst2_stride = 0) {
  __shared__ float red[8][33];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5, j = blockIdx.x * 32 + x, w = w1 + w2;
  partial += blockIdx.y * layer_stride;              // blockIdx.y = layer: every layer's partial rows are reduced by one launch
  dst1 += (size_t)blockIdx.y * dst1_stride;
  dst2 += (size_t)blockIdx.y * dst2_stride;
  float acc = 0.f;
  if (j < w) {
#pragma unroll 8
    for (int r = y; r < rows; r += 8) acc += partial[(size_t)r * pitch + j];
  }
  red[y][x] = acc;
  __syncthreads();
  if (y == 0 && j < w) {
    float t = red[0][x];
#pragma unroll
    for (int k = 1; k < 8; k++) t += red[k][x];
    if (j < w1) dst1[j] += t; else dst2[j - w1] += t;
  }
}
static inline unsigned reduce_grid(int w) { return (unsigned)((w + 31) / 32); }

// ---- flow head backward (model.py:451-452, 479-482) ---------------------------------------------------
// inputs per sample: d_scale, d_mean (from the composition), d_xout (from the next flow's front conv), x_prev, scale;
// outputs: d x_L [n][32], d x_prev (direct term) [n]; head weight gradients through per-CTA partials [64 + 2].
__global__ void __launch_bounds__(256)
k_bwd_flow_head(const float* __restrict__ h, const float* __restrict__ x_prev, const float* __restrict__ scale,
                const float* __restrict__ d_scale, const float* __restrict__ d_mean, const float* __restrict__ d_xout,
                const float* __restrict__ hk, float* __restrict__ dh, float* __restrict__ dx_prev,
                float* __restrict__ partial, int64_t n) {
  __shared__ float s_red[8][66];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float k0 = hk[lane * 2], k1 = hk[lane * 2 + 1];
  float g0 = 0.f, g1 = 0.f, gb0 = 0.f, gb1 = 0.f;          // dW[lane][0..1], db
  for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < n; row += (int64_t)gridDim.x * 8) {
    const float sc = scale[row];
    const float dxo = d_xout ? d_xout[row] : 0.f;
    const float ds = d_scale[row] + dxo * x_prev[row];      // x_f = x_{f-1} s_f + mu_f
    const float dm = d_mean[row] + dxo;
    const float dp0 = ds * sc, dp1 = dm;                    // s = exp(p0), mu = p1
    const float hv = h[row * kR + lane];
    const float e = fmaxf(hv, 0.f);
    dh[row * kR + lane] = hv > 0.f ? fmaf(k0, dp0, k1 * dp1) : 0.f;
    g0 = fmaf(e, dp0, g0); g1 = fmaf(e, dp1, g1);
    if (lane == 0) { dx_prev[row] = dxo * sc; gb0 += dp0; gb1 += dp1; }
  }
  s_red[warp][lane * 2] = g0; s_red[warp][lane * 2 + 1] = g1;
  if (lane == 0) { s_red[warp][64] = gb0; s_red[warp][65] = gb1; }
  __syncthreads();
  if (tid < 66) {
    float tot = 0.f;
    for (int w = 0; w < 8; w++) tot += s_red[w][tid];
    partial[(size_t)blockIdx.x * 66 + tid] = tot;
  }
}

// ---- front backward (RightShift + K=2 causal conv on one channel, model.py:172-173/423-424) -------------
// h_0[t][r] = x[t-2] k0[r] + x[t-1] k1[r] + b[r] + cond_0;  dx[t] = sum_r dh0[t+2][r] k0[r] + dh0[t+1][r] k1[r]
__global__ void __launch_bounds__(256)
k_bwd_front(const float* __restrict__ x_in, const float* __restrict__ dh0, const float* __restrict__ fk,
            float* __restrict__ dx_in,                 // += (accumulates onto the direct term), may be null
            float* __restrict__ partial,               // [gridDim.x][96]: dk0 | dk1 | db
            int B, int T) {
  __shared__ float s_red[8][96];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float k0 = fk[lane], k1 = fk[kR + lane];
  float g0 = 0.f, g1 = 0.f, gb = 0.f;
  const int64_t n = (int64_t)B * T;
  for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < n; row += (int64_t)gridDim.x * 8) {
    const int t = (int)(row % T);
    const float dv = dh0[row * kR + lane];
    const float xm2 = t >= 2 ? x_in[row - 2] : 0.f, xm1 = t >= 1 ? x_in[row - 1] : 0.f;
    g0 = fmaf(xm2, dv, g0); g1 = fmaf(xm1, dv, g1); gb += dv;
    if (dx_in) {
      float v = (t + 2 < T ? dh0[(row + 2) * kR + lane] * k0 : 0.f) + (t + 1 < T ? dh0[(row + 1) * kR + lane] * k1 : 0.f);
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) dx_in[row] += v;
    }
  }
  s_red[warp][lane] = g0; s_red[warp][32 + lane] = g1; s_red[warp][64 + lane] = gb;
  __syncthreads();
  if (tid < 96) {
    float tot = 0.f;
    for (int w = 0; w < 8; w++) tot += s_red[w][tid];
    partial[(size_t)blockIdx.x * 96 + tid] = tot;
  }
}

// conditioning 1x1 (model.py:431): cond[bf][l][r] = enc[bf][:] Wc_l[:, r] + bc_l[r]
// dWc_l[c][r] += sum_bf enc[bf][c] dcond_l[bf][r];  dbc_l[r] += sum_bf dcond_l[bf][r].   grid = (L, C + 1), block = 256:
// CTA (l, c) owns the 32 outputs of input channel c (c == C: the bias); lane = r, the 8 warps split the frames, and
// their parts are added in a fixed order
__global__ void __launch_bounds__(256)
k_bwd_cond(const float* __restrict__ enc, const float* __restrict__ dcond,   // dcond [L][BF][32]
           float* __restrict__ dWc, float* __restrict__ dbc, int BF, int C) {
  __shared__ float red[8][kR];
  const int l = blockIdx.x, c = blockIdx.y, r = threadIdx.x & 31, y = threadIdx.x >> 5;
  const float* dl = dcond + (size_t)l * BF * kR;
  float acc = 0.f;
  if (c < C) {
#pragma unroll 4
    for (int bf = y; bf < BF; bf += 8) acc = fmaf(enc[(size_t)bf * C + c], dl[(size_t)bf * kR + r], acc);
  } else {
#pragma unroll 4
    for (int bf = y; bf < BF; bf += 8) acc += dl[(size_t)bf * kR + r];
  }
  red[y][r] = acc;
  __syncthreads();
  if (y == 0) {
    float t = red[0][r];
#pragma unroll
    for (int k = 1; k < 8; k++) t += red[k][r];
    if (c < C) dWc[((size_t)l * C + c) * kR + r] += t; else dbc[(size_t)l * kR + r] += t;
  }
}

// ---- composition backward (model.py:517-535) ----------------------------------------------------------
// pre = z S + M;  given d_pre (already masked by the clip) and d_S_extra (entropy term): d s_f, d mu_f.
__global__ void k_bwd_compose(const float* __restrict__ z, const float* __restrict__ scales, const float* __restrict__ means,
                              const float* __restrict__ d_pre, const float* __restrict__ d_s_extra, int F,
                              float* __restrict__ d_scales, float* __restrict__ d_means, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s[16], mu[16];
  for (int f = 0; f < F; f++) { s[f] = scales[(size_t)f * n + i]; mu[f] = means[(size_t)f * n + i]; }
  float S = 1.f;
  for (int f = 0; f < F; f++) S *= s[f];
  const float dM = d_pre[i];
  const float dS = fmaf(dM, z[i], d_s_extra ? d_s_extra[i] : 0.f);
  for (int f = 0; f < F; f++) {
    float tail = 1.f;                                   // prod_{j>f} s_j
    for (int j = f + 1; j < F; j++) tail *= s[j];
    d_means[(size_t)f * n + i] = dM * tail;
    float others = 1.f;                                 // S / s_f without dividing
    for (int j = 0; j < F; j++) if (j != f) others *= s[j];
    float acc = dS * others;
    for (int k = 0; k < f; k++) {                       // mu_k prod_{j>k, j != f} s_j
      float pr = mu[k];
      for (int j = k + 1; j < F; j++) if (j != f) pr *= s[j];
      acc = fmaf(dM, pr, acc);
    }
    d_scales[(size_t)f * n + i] = acc;
  }
}

// ---- loss pieces ----------------------------------------------------------------------------------------
// d/dx of the mixture-of-logistics negative log-likelihood (ops.py:124-175) for fixed logits; nll optional.
__global__ void k_mol_nll_grad(const float* __restrict__ x, const float* __restrict__ l, float* __restrict__ dx,
                               float* __restrict__ nll, int64_t n, int M) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float xv = x[i];
  const float* lg = l + i * 4 * M;
  float mx = lg[0];
  for (int m = 1; m < M; m++) mx = fmaxf(mx, lg[m]);
  float se = 0.f;
  for (int m = 0; m < M; m++) se += expf(lg[m] - mx);
  const float lse_p = mx + logf(se);
  float lp[8], dv[8], best = -INFINITY;
  for (int m = 0; m < M; m++) {
    const float mean = lg[M + m], ls = fmaxf(lg[2 * M + m], -7.f), inv = expf(-ls), c = xv - mean;
    const float plus = inv * (c + 1.f / 255.f), mn = inv * (c - 1.f / 255.f), mid = inv * c;
    float v, d;
    if (xv < -0.999f) { v = plus - srwn_softplus(plus); d = inv * train::sigmoidf_(-plus); }
    else if (xv > 0.999f) { v = -srwn_softplus(mn); d = -inv * train::sigmoidf_(mn); }
    else {
      float a = plus, bb = mn;
      if (mid > 0.f) { a = -mn; bb = -plus; }
      const float ea = expf(a), eb = expf(bb);
      const float delta = -ea * expm1f(bb - a) / ((1.f + ea) * (1.f + eb));
      if (delta > 1e-5f) {
        v = logf(fmaxf(delta, 1e-12f));
        // d/dx log(sig(plus) - sig(min)) = inv (sig'(plus) - sig'(min)) / delta, and sig' = sig - sig^2 gives
        // sig'(plus) - sig'(min) = delta (1 - sig(plus) - sig(min)): no division, no cancellation
        d = inv * (train::sigmoidf_(-plus) - train::sigmoidf_(mn));
      } else {
        v = mid - ls - 2.f * srwn_softplus(mid) - 4.8481163902538321f;
        d = inv * (1.f - 2.f * train::sigmoidf_(mid));
      }
    }
    lp[m] = v + lg[m] - lse_p; dv[m] = d;
    best = fmaxf(best, lp[m]);
  }
  float ssum = 0.f, dsum = 0.f;
  for (int m = 0; m < M; m++) { const float e = expf(lp[m] - best); ssum += e; dsum = fmaf(e, dv[m], dsum); }
  dx[i] = -dsum / ssum;
  if (nll) nll[i] = -(best + logf(ssum));
}

// Adam as tf.train.AdamOptimizer applies it (model.py:382, 401): lr_t = lr sqrt(1-b2^t)/(1-b1^t);
// m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; w -= lr_t m / (sqrt(v) + eps).  `scale` = clip_by_global_norm factor.
__global__ void k_adam(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                       const float* __restrict__ gnorm_sq, float clip, float lr_t, float b1, float b2, float eps, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gn = sqrtf(*gnorm_sq);
  const float scale = clip > 0.f ? clip / fmaxf(gn, clip) : 1.f;      // tf.clip_by_global_norm (model.py:385)
  const float gi = g[i] * scale;
  const float mi = fmaf(b1, m[i], (1.f - b1) * gi);
  const float vi = fmaf(b2, v[i], (1.f - b2) * gi * gi);
  m[i] = mi; v[i] = vi;
  w[i] -= lr_t * mi / (sqrtf(vi) + eps);
}

__global__ void __launch_bounds__(1024) k_sumsq(const float* __restrict__ g, int64_t n, float* __restrict__ out) {
  __shared__ double s_red[1024];
  double acc = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += (double)g[i] * g[i];
  s_red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 512; s >= 1; s >>= 1) { if (threadIdx.x < s) s_red[threadIdx.x] += s_red[threadIdx.x + s]; __syncthreads(); }
  if (threadIdx.x == 0) *out = (float)s_red[0];
}

// loss = (beta * H(Ps,Pt) - alpha * H(Ps) + power) / B   (model.py:374-379); out2 = {loss, power_loss} as the reference returns them
__global__ void k_distill_finish(const double* __restrict__ sums, const double* __restrict__ power, float alpha, float beta,
                                 float inv_norm, float* __restrict__ out2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    out2[0] = (float)(((double)beta * sums[0] - (double)alpha * sums[1] + *power) * (double)inv_norm);
    out2[1] = (float)*power;
  }
}

// tf.clip_by_global_norm(grads, clip) in place: g *= clip / max(||g||, clip)   (model.py:385)
__global__ void k_clip_scale(float* __restrict__ g, const float* __restrict__ gnorm_sq, float clip, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  g[i] *= clip / fmaxf(sqrtf(*gnorm_sq), clip);
}

__global__ void k_axpy(float* __restrict__ y, const float* __restrict__ x, float a, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = fmaf(a, x[i], y[i]);
}

// per-example entropy term sum_t (log s_tot + 2)   (model.py:356, 578-593); one CTA per example, fixed summation order
__global__ void __launch_bounds__(1024) k_entropy(const float* __restrict__ s_tot, double* __restrict__ out, int T) {
  __shared__ double s_red[1024];
  const float* s = s_tot + (size_t)blockIdx.x * T;
  double acc = 0;
  for (int t = threadIdx.x; t < T; t += blockDim.x) acc += (double)logf(s[t]) + 2.0;
  s_red[threadIdx.x] = acc;
  __syncthreads();
  for (int k = 512; k >= 1; k >>= 1) { if (threadIdx.x < k) s_red[threadIdx.x] += s_red[threadIdx.x + k]; __syncthreads(); }
  if (threadIdx.x == 0) out[blockIdx.x] = s_red[0];
}

}  // namespace train

int run_distill_finish(const double* sums, const double* power, float alpha, float beta, float inv_norm, float* out2, cudaStream_t st) {
  train::k_distill_finish<<<1, 32, 0, st>>>(sums, power, alpha, beta, inv_norm, out2);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

int run_clip_by_global_norm(float* grads, int64_t n, float clip, float* scratch1, cudaStream_t st) {
  train::k_sumsq<<<1, 1024, 0, st>>>(grads, n, scratch1);
  SRWN_LAUNCH_CHECK();
  train::k_clip_scale<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(grads, scratch1, clip, n);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

int run_axpy(float* y, const float* x, float a, int64_t n, cudaStream_t st) {
  train::k_axpy<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(y, x, a, n);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

int run_entropy(const float* s_tot, double* per_example, int B, int T, cudaStream_t st) {
  train::k_entropy<<<B, 1024, 0, st>>>(s_tot, per_example, T);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ---- host ----------------------------------------------------------------------------------------------
struct TrainWs {
  float *acts, *cond, *scales, *means, *xs, *g0, *g1, *da, *dcond, *d_scales, *d_means, *dxa, *dxb, *partial, *partial_gate, *partial_conv;
  size_t bytes; int grid, grid_tc;
};

static TrainWs carve_train(const srwn_ctx* c, int B, int T, void* ws, size_t cap) {
  WsCarver w(ws, cap);
  TrainWs r{};
  const size_t n = (size_t)B * T, L = c->cfg.n_layers, F = c->cfg.num_flows, frames = T / c->cfg.pool_stride;
  r.grid = 3 * (c->sm_count > 0 ? c->sm_count : 148);     // elementwise kernels of the step (heads, front)
  r.grid_tc = c->sm_count > 0 ? c->sm_count : 148;         // tensor-core layer kernels: one persistent CTA per SM (shared memory)
  r.acts = w.take<float>(F * (L + 1) * n * kR);
  r.cond = w.take<float>((size_t)B * frames * L * kR);
  r.scales = w.take<float>(F * n);
  r.means = w.take<float>(F * n);
  r.xs = w.take<float>(F * n);                              // flow outputs x_f
  r.g0 = w.take<float>(n * kR);
  r.g1 = w.take<float>(n * kR);
  r.da = w.take<float>(n * kR);
  r.dcond = w.take<float>(L * (size_t)B * frames * kR);     // [L][B*frames][32] of the current flow
  r.d_scales = w.take<float>(F * n);
  r.d_means = w.take<float>(F * n);
  r.dxa = w.take<float>(n);
  r.dxb = w.take<float>(n);
  r.partial = w.take<float>((size_t)r.grid * (2 * kR * kR + kR));
  r.partial_gate = w.take<float>(L * (size_t)r.grid * (kR * kR + kR));           // [L][grid][dWr | dbr]
  r.partial_conv = w.take<float>(L * (size_t)r.grid * (2 * kR * kR + kR));       // [L][grid][dWf | dbf]
  r.bytes = w.used;
  return r;
}

size_t train_workspace_bytes(const srwn_ctx* c, int B, int T) { return carve_train(c, B, T, nullptr, 0).bytes; }

// forward of all flows in fp32, keeping every layer input (model.py:489-535): acts of flow f is [L+1][B][T][R]
int run_student_forward_train(srwn_ctx* c, const float* z, const float* enc, float* out, float* s_tot,
                              float* mu_tot, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st) {
  TrainWs w = carve_train(c, B, T, ws, ws_bytes);
  if (int rc = check_workspace(ws, ws_bytes, w.bytes)) return rc;
  const size_t n = (size_t)B * T;
  const int F = c->cfg.num_flows, L = c->cfg.n_layers;
  const float* xin = z;
  for (int f = 0; f < F; f++) {
    float* hL = nullptr;
    int rc = run_stack_f32(c, f, xin, enc, B, T, w.acts + (size_t)f * (L + 1) * n * kR, nullptr, nullptr, w.cond, &hL, st);
    if (rc) return rc;
    rc = run_flow_head_f32(c, f, hL, xin, w.scales + (size_t)f * n, w.means + (size_t)f * n, w.xs + (size_t)f * n, B, T, st);
    if (rc) return rc;
    xin = w.xs + (size_t)f * n;
  }
  return run_flow_compose(z, NoiseSpec{0, 0, 0}, nullptr, w.scales, w.means, F, out, s_tot, mu_tot, (int64_t)n, st);
}

// backward: d_pre [B,T] = dLoss/d(z S + M) (caller applies the clip mask), d_s_extra [B,T] = extra dLoss/dS (entropy);
// grads: flat buffer in the layout of the weight arena (n_stacks x stack_floats), overwritten.
int run_student_backward(srwn_ctx* c, const float* z, const float* enc, const float* d_pre, const float* d_s_extra,
                         float* grads, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st) {
  using namespace train;
  TrainWs w = carve_train(c, B, T, ws, ws_bytes);
  if (int rc = check_workspace(ws, ws_bytes, w.bytes)) return rc;
  const size_t n = (size_t)B * T;
  const int F = c->cfg.num_flows, L = c->cfg.n_layers, P = c->cfg.pool_stride, frames = T / P, C = c->cfg.cond_channels;
  const int BF = B * frames;
  const StackOffsets& o = c->off;
  SRWN_CUDA(cudaFuncSetAttribute(traintc::k_bwd_gate_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::gate_smem_bytes()));
  SRWN_CUDA(cudaFuncSetAttribute(traintc::k_bwd_conv_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::conv_smem_bytes()));
  SRWN_CUDA(cudaMemsetAsync(grads, 0, (size_t)c->n_stacks * c->stack_floats * sizeof(float), st));
  k_bwd_compose<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(z, w.scales, w.means, d_pre, d_s_extra, F, w.d_scales, w.d_means, (int64_t)n);
  SRWN_LAUNCH_CHECK();
  const int grid = w.grid, gtc = w.grid_tc;
  ProfScope prof(c, st, "k_bwd_gate_tc+k_bwd_conv_tc (student backward)", F * L * 2);
  float* dx_next = nullptr;                  // dLoss/dx_f arriving from flow f+1's front conv (null for the last flow)
  float* dx_cur = w.dxa;
  for (int f = F - 1; f >= 0; f--) {
    const float* sw = stack_w(c, f);
    float* gs = grads + (size_t)f * c->stack_floats;
    const float* acts = w.acts + (size_t)f * (L + 1) * n * kR;
    const float* x_prev = f == 0 ? z : w.xs + (size_t)(f - 1) * n;
    // head: d x_L, direct d x_{f-1}
    k_bwd_flow_head<<<grid, 256, 0, st>>>(acts + (size_t)L * n * kR, x_prev, w.scales + (size_t)f * n, w.d_scales + (size_t)f * n,
                                          w.d_means + (size_t)f * n, dx_next, sw + o.head1_k, w.g0, dx_cur, w.partial, (int64_t)n);
    SRWN_LAUNCH_CHECK();
    k_reduce_partials<<<reduce_grid(66), 256, 0, st>>>(w.partial, grid, 66, 64, gs + o.head1_k, 2, gs + o.head1_b);
    SRWN_LAUNCH_CHECK();
    SRWN_CUDA(cudaMemsetAsync(w.dcond, 0, (size_t)L * BF * kR * sizeof(float), st));
    float* g = w.g0;
    float* gn = w.g1;
    for (int l = L - 1; l >= 0; l--) {
      const float* x_l = acts + (size_t)l * n * kR;
      const int d = c->dilations[l];
      // per-CTA weight-gradient partials of every layer are kept ([L][grid][...]) and reduced by ONE launch per flow
      float* pg = w.partial_gate + (size_t)l * gtc * (kR * kR + kR);
      float* pc = w.partial_conv + (size_t)l * gtc * (2 * kR * kR + kR);
      SRWN_CUDA(launch_dependent(traintc::k_bwd_gate_tc, gtc, traintc::kThreads, (size_t)traintc::gate_smem_bytes(), st, x_l, (const float*)g, w.da,
                                 sw + o.filt_k + (size_t)l * 2 * kR * kR, sw + o.filt_b + (size_t)l * kR,
                                 sw + o.res_k + (size_t)l * kR * kR, pg, B, T, d));
      SRWN_LAUNCH_CHECK();
      // x_l carries cond_l (added before the block, model.py:183; for l = 0 by the front): dcond_l = sum over the frame of dx_l
      SRWN_CUDA(launch_dependent(traintc::k_bwd_conv_tc, gtc, traintc::kThreads, (size_t)traintc::conv_smem_bytes(), st, x_l, (const float*)g, (const float*)w.da, gn,
                                 sw + o.filt_k + (size_t)l * 2 * kR * kR, pc, w.dcond + (size_t)l * BF * kR, B, T, d, P, frames));
      SRWN_LAUNCH_CHECK();
      float* tmp = g; g = gn; gn = tmp;
    }
    k_reduce_partials<<<dim3(reduce_grid(kR * kR + kR), L), 256, 0, st>>>(w.partial_gate, gtc, kR * kR + kR, kR * kR, gs + o.res_k, kR,
                                                                         gs + o.res_b, (size_t)gtc * (kR * kR + kR), kR * kR, kR);
    SRWN_LAUNCH_CHECK();
    k_reduce_partials<<<dim3(reduce_grid(2 * kR * kR + kR), L), 256, 0, st>>>(w.partial_conv, gtc, 2 * kR * kR + kR, 2 * kR * kR,
                                                                             gs + o.filt_k, kR, gs + o.filt_b,
                                                                             (size_t)gtc * (2 * kR * kR + kR), 2 * kR * kR, kR);
    SRWN_LAUNCH_CHECK();
    // g = dLoss/dx_0 (front output incl. cond_0)
    k_bwd_front<<<grid, 256, 0, st>>>(x_prev, g, sw + o.front_k, f > 0 ? dx_cur : nullptr, w.partial, B, T);
    SRWN_LAUNCH_CHECK();
    k_reduce_partials<<<reduce_grid(96), 256, 0, st>>>(w.partial, grid, 96, 64, gs + o.front_k, 32, gs + o.front_b);
    SRWN_LAUNCH_CHECK();
    // conditioning: every layer's dcond -> dWc, dbc
    k_bwd_cond<<<dim3(L, C + 1), 256, 0, st>>>(enc, w.dcond, gs + o.cond_k, gs + o.cond_b, BF, C);
    SRWN_LAUNCH_CHECK();
    dx_next = dx_cur;
    dx_cur = dx_cur == w.dxa ? w.dxb : w.dxa;
  }
  return SRWN_OK;
}

int run_mol_nll_grad(const float* x, const float* l, float* dx, float* nll, int B, int T, int M, cudaStream_t st) {
  const int64_t n = (int64_t)B * T;
  train::k_mol_nll_grad<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, l, dx, nll, n, M);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

int run_adam(srwn_ctx* c, const float* grads, float* m, float* v, float* scratch1, float clip, float lr, float b1, float b2,
             float eps, int step, cudaStream_t st) {
  const int64_t n = (int64_t)c->n_stacks * c->stack_floats;
  train::k_sumsq<<<1, 1024, 0, st>>>(grads, n, scratch1);
  SRWN_LAUNCH_CHECK();
  const float lr_t = lr * sqrtf(1.f - powf(b2, (float)step)) / (1.f - powf(b1, (float)step));
  train::k_adam<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(c->d_weights, grads, m, v, scratch1, clip, lr_t, b1, b2, eps, n);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}
