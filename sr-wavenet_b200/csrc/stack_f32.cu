// fp32-grade path of the residual stack (parity path, <= 1e-4 relative vs the oracle).
//
// One launch per layer; the residual stream (and the teacher's skip sum) round-trips through HBM as fp32.  The layer
// GEMMs run on the tensor cores with split TF32 operands (train::k_fwd_layer, three MMAs per product), conditioning,
// front conv and the output heads are FFMA kernels.  This is the reference-grade path and the GPU-side cross-check for
// the fused fp16 tcgen05 kernel (fused.cu), which is the one the benchmark times.
//
// Stored tensor convention: `hc_i` = the block input of layer i = h_i + upsampled
// conditioning of layer i (model.py:183 adds it before ResidualDilationLayer, so it also
// feeds the `inputs + residual` term at ops.py:40 and is zero-padded like the rest).
#include "common.cuh"
#include "philox.cuh"

// cond[b][frame][layer][r] = enc[b][frame][:] @ cond_k[layer] + cond_b[layer]   (model.py:180/431)
__global__ void k_cond(const float* __restrict__ enc, const float* __restrict__ cond_k,
                       const float* __restrict__ cond_b, float* __restrict__ cond,
                       int frames_total, int L, int C) {
  __shared__ float s_enc[kMaxCond];
  const int bf = blockIdx.x;
  if (threadIdx.x < C) s_enc[threadIdx.x] = enc[(size_t)bf * C + threadIdx.x];
  __syncthreads();
  for (int o = threadIdx.x; o < L * kR; o += blockDim.x) {
    const int l = o / kR, r = o % kR;
    const float* wk = cond_k + (size_t)l * C * kR + r;
    float acc = cond_b[l * kR + r];
    for (int c = 0; c < C; c++) acc = fmaf(s_enc[c], wk[(size_t)c * kR], acc);
    cond[(size_t)bf * L * kR + o] = acc;
  }
}

// hc_0[b][t][r] = x[t-2]*k[0][r] + x[t-1]*k[1][r] + b[r] + cond[b][t/P][0][r]
// (RightShift ops.py:78-80, then the K=2, d=1 causal conv model.py:173/424)
__global__ void k_front(const float* __restrict__ x, const float* __restrict__ fk,
                        const float* __restrict__ fb, const float* __restrict__ cond,
                        float* __restrict__ hc, int T, int P, int L, int frames) {
  const int b = blockIdx.y;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over T*R
  if (idx >= (int64_t)T * kR) return;
  const int t = (int)(idx / kR), r = (int)(idx % kR);
  const float* xb = x + (size_t)b * T;
  const float xm2 = t >= 2 ? xb[t - 2] : 0.f, xm1 = t >= 1 ? xb[t - 1] : 0.f;
  float v = fmaf(xm2, fk[r], fmaf(xm1, fk[kR + r], fb[r]));
  v += cond[(((size_t)b * frames + t / P) * L + 0) * kR + r];
  hc[((size_t)b * T + t) * kR + r] = v;
}

// The residual blocks (ops.py:23-46) run in train::k_fwd_layer (train_f32.cu): 64-step tiles, 3xTF32 tensor-core GEMMs.
int run_layer_tf32x3(srwn_ctx* c, bool with_skip, const float* x_l, float* x_next, float* skip, const float* filt_k,
                     const float* filt_b, const float* res_k, const float* res_b, const float* skip_k, const float* skip_b,
                     const float* cond_next, int B, int T, int d, int P, int L, int frames, int skip_init, cudaStream_t st);

int run_stack_f32(srwn_ctx* c, int stack, const float* xin, const float* enc, int B, int T,
                  float* h0, float* h1, float* skip, float* cond, float** h_final,
                  cudaStream_t st) {
  const float* w = stack_w(c, stack);
  const StackOffsets& o = c->off;
  const int L = c->cfg.n_layers, P = c->cfg.pool_stride, C = c->cfg.cond_channels;
  const int frames = T / P;
  const bool with_skip = c->cfg.kind == SRWN_TEACHER;
  k_cond<<<B * frames, 256, 0, st>>>(enc, w + o.cond_k, w + o.cond_b, cond, B * frames, L, C);
  SRWN_LAUNCH_CHECK();
  {
    dim3 grid((unsigned)(((int64_t)T * kR + 255) / 256), B);
    k_front<<<grid, 256, 0, st>>>(xin, w + o.front_k, w + o.front_b, cond, h0, T, P, L, frames);
    SRWN_LAUNCH_CHECK();
  }
  float* cur = h0;
  float* nxt = h1;
  ProfScope prof(c, st, with_skip ? "k_fwd_layer<skip> (3xTF32)" : "k_fwd_layer (3xTF32)", L);
  for (int l = 0; l < L; l++) {
    const float* cond_next = l + 1 < L ? cond + (size_t)(l + 1) * kR : nullptr;
    int rc = run_layer_tf32x3(c, with_skip, cur, nxt, skip, w + o.filt_k + (size_t)l * 2 * kR * kR, w + o.filt_b + (size_t)l * kR,
                              w + o.res_k + (size_t)l * kR * kR, w + o.res_b + (size_t)l * kR,
                              with_skip ? w + o.skip_k + (size_t)l * kR * kS : nullptr, with_skip ? w + o.skip_b + (size_t)l * kS : nullptr,
                              cond_next, B, T, c->dilations[l], P, L, frames, l == 0, st);
    if (rc) return rc;
    float* tmp = cur; cur = nxt; nxt = tmp;
  }
  *h_final = cur;
  return SRWN_OK;
}

// ---- teacher head: relu -> 1x1 S->S -> relu -> 1x1 S->4M (model.py:191-196) ------------
constexpr int kHT = 64;
__global__ void __launch_bounds__(256)
k_head_f32(const float* __restrict__ skip, const float* __restrict__ w1, const float* __restrict__ b1,
           const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ logits,
           int64_t n_rows, int O) {
  __shared__ __align__(16) float s_a[kHT][kS + 4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t row0 = (int64_t)blockIdx.x * kHT;
  for (int i = tid; i < kHT * (kS / 4); i += 256) {
    const int row = i / (kS / 4), q = i % (kS / 4);
    float4 v = make_float4(0, 0, 0, 0);
    if (row0 + row < n_rows) v = *reinterpret_cast<const float4*>(skip + (row0 + row) * kS + q * 4);
    v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
    *reinterpret_cast<float4*>(&s_a[row][q * 4]) = v;
  }
  __syncthreads();
  const int r0 = warp * 8;
  float acc[8][4];
#pragma unroll
  for (int r = 0; r < 8; r++)
#pragma unroll
    for (int j = 0; j < 4; j++) acc[r][j] = b1[lane + 32 * j];
  for (int k4 = 0; k4 < kS / 4; k4++) {
    float w[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; kk++)
#pragma unroll
      for (int j = 0; j < 4; j++) w[kk][j] = __ldg(w1 + (size_t)(k4 * 4 + kk) * kS + lane + 32 * j);
#pragma unroll
    for (int r = 0; r < 8; r++) {
      const float4 a = *reinterpret_cast<const float4*>(&s_a[r0 + r][k4 * 4]);
#pragma unroll
      for (int j = 0; j < 4; j++) {
        acc[r][j] = fmaf(a.x, w[0][j], acc[r][j]); acc[r][j] = fmaf(a.y, w[1][j], acc[r][j]);
        acc[r][j] = fmaf(a.z, w[2][j], acc[r][j]); acc[r][j] = fmaf(a.w, w[3][j], acc[r][j]);
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 8; r++)
#pragma unroll
    for (int j = 0; j < 4; j++) s_a[r0 + r][lane + 32 * j] = fmaxf(acc[r][j], 0.f);
  __syncwarp();
  float lg[8];
  const int oc = lane < O ? lane : 0;
#pragma unroll
  for (int r = 0; r < 8; r++) lg[r] = b2[oc];
  for (int k4 = 0; k4 < kS / 4; k4++) {
    const float w0 = __ldg(w2 + (size_t)(k4 * 4 + 0) * O + oc), w1v = __ldg(w2 + (size_t)(k4 * 4 + 1) * O + oc),
                w2v = __ldg(w2 + (size_t)(k4 * 4 + 2) * O + oc), w3 = __ldg(w2 + (size_t)(k4 * 4 + 3) * O + oc);
#pragma unroll
    for (int r = 0; r < 8; r++) {
      const float4 a = *reinterpret_cast<const float4*>(&s_a[r0 + r][k4 * 4]);
      lg[r] = fmaf(a.x, w0, lg[r]); lg[r] = fmaf(a.y, w1v, lg[r]);
      lg[r] = fmaf(a.z, w2v, lg[r]); lg[r] = fmaf(a.w, w3, lg[r]);
    }
  }
  if (lane < O) {
#pragma unroll
    for (int r = 0; r < 8; r++)
      if (row0 + r0 + r < n_rows) logits[(row0 + r0 + r) * O + lane] = lg[r];
  }
}

int run_teacher_head_f32(srwn_ctx* c, const float* skip, float* logits, int B, int T, cudaStream_t st) {
  const float* w = stack_w(c, 0);
  const StackOffsets& o = c->off;
  const int64_t n = (int64_t)B * T;
  k_head_f32<<<(unsigned)((n + kHT - 1) / kHT), 256, 0, st>>>(
      skip, w + o.head1_k, w + o.head1_b, w + o.head2_k, w + o.head2_b, logits, n,
      4 * c->cfg.num_mixtures);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// ---- student flow head + affine (model.py:451-452, 479-482) ---------------------------------
// params = relu(h) @ W[R][2] + b; scale = exp(p0); mean = p1; out = x*scale + mean
__global__ void k_flow_head(const float* __restrict__ h, const float* __restrict__ xin,
                            const float* __restrict__ hk, const float* __restrict__ hb,
                            float* __restrict__ scale, float* __restrict__ mean,
                            float* __restrict__ xout, int64_t n) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t row = gid >> 3;          // 8 lanes per time step
  const int q = (int)(gid & 7);
  float p0 = 0.f, p1 = 0.f;
  if (row < n) {
    const float4 v = *reinterpret_cast<const float4*>(h + row * kR + q * 4);
    const float e[4] = {fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f)};
#pragma unroll
    for (int i = 0; i < 4; i++) {
      p0 = fmaf(e[i], hk[(q * 4 + i) * 2 + 0], p0);
      p1 = fmaf(e[i], hk[(q * 4 + i) * 2 + 1], p1);
    }
  }
#pragma unroll
  for (int s = 4; s >= 1; s >>= 1) {
    p0 += __shfl_xor_sync(0xffffffffu, p0, s);
    p1 += __shfl_xor_sync(0xffffffffu, p1, s);
  }
  if (row < n && q == 0) {
    const float sc = expf(p0 + hb[0]);       // no clamp on the log-scale (model.py:479)
    const float mu = p1 + hb[1];
    scale[row] = sc; mean[row] = mu;
    xout[row] = fmaf(xin[row], sc, mu);      // model.py:482
  }
}

int run_flow_head_f32(srwn_ctx* c, int stack, const float* h, const float* xin, float* scale,
                      float* mean, float* xout, int B, int T, cudaStream_t st) {
  const float* w = stack_w(c, stack);
  const int64_t n = (int64_t)B * T;
  k_flow_head<<<(unsigned)((n * 8 + 255) / 256), 256, 0, st>>>(h, xin, w + c->off.head1_k,
                                                               w + c->off.head1_b, scale, mean, xout, n);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// s_tot = prod s_f; mu_tot = sum_f mu_f * prod_{j>f} s_j in the reference's loop order
// (model.py:517-533); out = clip(z*s_tot + mu_tot, -1, 1) (model.py:535)
__global__ void k_flow_compose(const float* __restrict__ z, NoiseSpec noise, float* __restrict__ z_out,
                               const float* __restrict__ scales,
                               const float* __restrict__ means, int F, float* __restrict__ out,
                               float* __restrict__ s_tot, float* __restrict__ mu_tot, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // the student's input noise (student.py:104): supplied, or the same Philox draw the flow kernel evaluated
  const float zi = noise.on ? philox::logistic_at(noise.seed, noise.stream, (uint64_t)i) : z[i];
  if (z_out) z_out[i] = zi;
  float st = 1.f, mt = 0.f;
  for (int f = 0; f < F; f++) {
    st *= scales[(size_t)f * n + i];
    float mu = means[(size_t)f * n + i];
    for (int j = f + 1; j < F; j++) mu *= scales[(size_t)j * n + i];
    mt += mu;
  }
  if (s_tot) s_tot[i] = st;
  if (mu_tot) mu_tot[i] = mt;
  out[i] = fminf(fmaxf(fmaf(zi, st, mt), -1.f), 1.f);
}

int run_flow_compose(const float* z, NoiseSpec noise, float* z_out, const float* scales, const float* means, int F, float* out,
                     float* s_tot, float* mu_tot, int64_t n, cudaStream_t st) {
  k_flow_compose<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(z, noise, z_out, scales, means, F, out, s_tot, mu_tot, n);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}
