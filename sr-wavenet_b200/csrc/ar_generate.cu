// Autoregressive teacher generation with per-layer dilation queues (fp32).
//
// Restates the O(T^2) loop of teacher.py:153-170 (one full decoder pass per sample) as an
// O(T) recurrence: layer i keeps a ring of its last d_i block inputs, so sample t needs one
// pop + one push of R floats per layer (SURVEY.md 3.2 / 8(d) cfg4).  One persistent CTA owns
// U utterances for all T steps; weights stay in L2 and are streamed every step.
#include "common.cuh"
#include "gen_state.cuh"
#include "mol.cuh"

struct ArParams {
  const float* w;            // stack weights (fp32 arena)
  StackOffsets off;
  const int32_t* dil;        // [L]
  const int32_t* qoff;       // [L] prefix sums of dilations
  float* queues;             // [B][sum_d][R], zero-initialised == zero padding of ops.py:9
  const float* cond;         // [B][frames][L][R]
  const float* u1;           // [B][T][M]
  const float* u2;           // [B][T]
  float* x_out;              // [B][T]
  float* logits_out;         // [B][T][4M] or null
  int B, T, L, P, frames, M, sum_d;
  // resumable generation (RESUME): `queues` is then the caller's state, and so are these
  const long long* t0;       // position of step 0 of this call: slot of layer l at step t is (t0 + t) mod d_l
  float* xhist;              // [B][2] x[t-1], x[t-2] before step 0; rewritten with those of step T on exit
  const float* x_prefix;     // [B][n_prefix]: for t < n_prefix, x[t] is this sample instead of a draw
  int n_prefix;
};

template <int U, bool RESUME>
__global__ void __launch_bounds__(256, 1) k_ar_generate(const ArParams p) {
  __shared__ float s_cur[U][kR], s_tap[U][kR], s_c[U][kR];
  __shared__ float s_part[8][U][kR];
  __shared__ float s_skip[U][kS], s_hid[U][kS];
  __shared__ float s_part2[2][U][kS];
  __shared__ float s_logit[U][kMaxLogit];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b0 = blockIdx.x * U;
  const int O = 4 * p.M;
  const float* W = p.w;
  const StackOffsets& o = p.off;

  // role of the first U warps: warp u owns utterance b0+u's residual stream element `lane`
  const bool own = warp < U && (b0 + warp) < p.B;
  const int ub = b0 + (warp < U ? warp : 0);
  float xm1 = 0.f, xm2 = 0.f;            // x[t-1], x[t-2] (RightShift + K=2 front conv)
  if (RESUME && own) { xm1 = p.xhist[2 * ub]; xm2 = p.xhist[2 * ub + 1]; }
  const long long t0 = RESUME ? *p.t0 : 0;
  float skipacc[U];

  for (int t = 0; t < p.T; t++) {
    const int frame = t / p.P;
    float hreg = 0.f;                    // block input of the next layer, element (u=warp, lane)
    if (warp < U) {
      if (own) {
        hreg = fmaf(xm2, W[o.front_k + lane], fmaf(xm1, W[o.front_k + kR + lane], W[o.front_b + lane]));
        hreg += p.cond[(((size_t)ub * p.frames + frame) * p.L + 0) * kR + lane];
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) skipacc[u] = 0.f;

    for (int l = 0; l < p.L; l++) {
      // pop h[t-d] / push h[t] on this layer's ring (slot t mod d)
      if (warp < U) {
        float tap = 0.f;
        if (own) {
          const int d = p.dil[l];
          const int slot = RESUME ? (int)((t0 + t) % d) : t % d;
          float* q = p.queues + gen_f32_row(ub, p.sum_d, p.qoff[l], slot) * kR + lane;
          tap = *q;
          *q = hreg;
        }
        s_cur[warp][lane] = hreg;
        s_tap[warp][lane] = tap;
      }
      __syncthreads();
      // filter conv as a 64->32 GEMV, K split over the 8 warps (ops.py:6-10: W[0]~x[t-d], W[1]~x[t])
      {
        const float* wf = W + o.filt_k + (size_t)l * 2 * kR * kR + (size_t)(warp * 8) * kR + lane;
        float wv[8];
#pragma unroll
        for (int kk = 0; kk < 8; kk++) wv[kk] = __ldg(wf + kk * kR);
#pragma unroll
        for (int u = 0; u < U; u++) {
          const float* a = warp < 4 ? &s_tap[u][warp * 8] : &s_cur[u][(warp - 4) * 8];
          float acc = 0.f;
#pragma unroll
          for (int kk = 0; kk < 8; kk++) acc = fmaf(a[kk], wv[kk], acc);
          s_part[warp][u][lane] = acc;
        }
      }
      __syncthreads();
      if (warp < U) {
        float f = W[o.filt_b + l * kR + lane];
#pragma unroll
        for (int kq = 0; kq < 8; kq++) f += s_part[kq][warp][lane];
        f = tanhf(f);                                        // ops.py:28
        s_c[warp][lane] = f * (1.0f / (1.0f + expf(-f)));    // ops.py:33,36
      }
      __syncthreads();
      if (warp < U) {
        // residual 1x1 + dense (ops.py:39-40), then next layer's conditioning (model.py:183)
        const float* wr = W + o.res_k + (size_t)l * kR * kR + lane;
        float acc = W[o.res_b + l * kR + lane];
#pragma unroll 8
        for (int k = 0; k < kR; k++) acc = fmaf(s_c[warp][k], __ldg(wr + k * kR), acc);
        hreg = (hreg + acc) * SRWN_SQRT_HALF;
        if (own && l + 1 < p.L)
          hreg += p.cond[(((size_t)ub * p.frames + frame) * p.L + (l + 1)) * kR + lane];
      } else if (warp >= 4) {
        // skip 1x1 (ops.py:44), summed over layers in registers (model.py:190)
        const int j = tid - 128;
        const float* ws = W + o.skip_k + (size_t)l * kR * kS + j;
        float acc[U];
#pragma unroll
        for (int u = 0; u < U; u++) acc[u] = 0.f;
#pragma unroll 8
        for (int k = 0; k < kR; k++) {
          const float wv = __ldg(ws + k * kS);
#pragma unroll
          for (int u = 0; u < U; u++) acc[u] = fmaf(s_c[u][k], wv, acc[u]);
        }
#pragma unroll
        for (int u = 0; u < U; u++) skipacc[u] += acc[u];
      }
      // no barrier needed here: the next writes to s_cur/s_tap come from the warps that just
      // finished reading s_c, and s_c is rewritten only after two more barriers
    }

    // head: relu -> S->S -> relu -> S->4M (model.py:191-196)
    if (warp >= 4) {
      const int j = tid - 128;
      const float bsum = W[o.skip_b_sum + j];
#pragma unroll
      for (int u = 0; u < U; u++) s_skip[u][j] = fmaxf(skipacc[u] + bsum, 0.f);
    }
    __syncthreads();
    {
      const int half = tid >> 7, j = tid & 127;
      const float* w1 = W + o.head1_k + (size_t)(half * 64) * kS + j;
      float acc[U];
#pragma unroll
      for (int u = 0; u < U; u++) acc[u] = 0.f;
#pragma unroll 8
      for (int k = 0; k < 64; k++) {
        const float wv = __ldg(w1 + (size_t)k * kS);
#pragma unroll
        for (int u = 0; u < U; u++) acc[u] = fmaf(s_skip[u][half * 64 + k], wv, acc[u]);
      }
#pragma unroll
      for (int u = 0; u < U; u++) s_part2[half][u][j] = acc[u];
    }
    __syncthreads();
    if (tid < kS) {
      const float b1 = W[o.head1_b + tid];
#pragma unroll
      for (int u = 0; u < U; u++) s_hid[u][tid] = fmaxf(b1 + s_part2[0][u][tid] + s_part2[1][u][tid], 0.f);
    }
    __syncthreads();
    {
      const int oc = lane < O ? lane : 0;
      const float* w2 = W + o.head2_k + (size_t)(warp * 16) * O + oc;
      float acc[U];
#pragma unroll
      for (int u = 0; u < U; u++) acc[u] = 0.f;
#pragma unroll 8
      for (int k = 0; k < 16; k++) {
        const float wv = __ldg(w2 + (size_t)k * O);
#pragma unroll
        for (int u = 0; u < U; u++) acc[u] = fmaf(s_hid[u][warp * 16 + k], wv, acc[u]);
      }
#pragma unroll
      for (int u = 0; u < U; u++) s_part[warp][u][lane] = acc[u];
    }
    __syncthreads();
    if (warp < U) {
      float lg = lane < O ? W[o.head2_b + lane] : 0.f;
#pragma unroll
      for (int kq = 0; kq < 8; kq++) lg += s_part[kq][warp][lane];
      s_logit[warp][lane] = lg;
      if (own && p.logits_out && lane < O) p.logits_out[((size_t)ub * p.T + t) * O + lane] = lg;
      __syncwarp();
      float xs = 0.f;
      if (own && lane == 0) {
        float uu[kMaxLogit / 4];
        for (int m = 0; m < p.M; m++) uu[m] = p.u1[((size_t)ub * p.T + t) * p.M + m];
        int k;
        xs = mol_sample_one(s_logit[warp], uu, p.u2[(size_t)ub * p.T + t], p.M, &k);   // ops.py:178-201
        if (RESUME && t < p.n_prefix) xs = p.x_prefix[(size_t)ub * p.n_prefix + t];
        p.x_out[(size_t)ub * p.T + t] = xs;
      }
      xs = __shfl_sync(0xffffffffu, xs, 0);
      xm2 = xm1; xm1 = xs;
    }
    __syncthreads();   // s_part / s_logit reuse in the next step
  }
  if (RESUME && own && lane == 0) { p.xhist[2 * ub] = xm1; p.xhist[2 * ub + 1] = xm2; }
}

size_t ar_workspace_bytes(const srwn_ctx* c, int B, int T) {
  WsCarver w(nullptr, 0);
  w.take<uint8_t>(gen_queue_bytes(c, B, SRWN_FP32));
  w.take<float>((size_t)B * (T / c->cfg.pool_stride) * c->cfg.n_layers * kR);
  return w.used;
}

int run_ar_generate(srwn_ctx* c, const float* enc, const float* u1, const float* u2, float* x_out,
                    float* logits_out, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st, const GenState* rs,
                    const float* x_prefix, int n_prefix) {
  if (!ws || ws_bytes < ar_workspace_bytes(c, B, T))
    return srwn_fail(SRWN_ERR_WORKSPACE, "workspace too small: need %zu bytes", ar_workspace_bytes(c, B, T));
  WsCarver w(ws, ws_bytes);
  const int frames = T / c->cfg.pool_stride;
  const size_t queue_bytes = gen_queue_bytes(c, B, SRWN_FP32);
  void* queues = w.take<uint8_t>(queue_bytes);
  float* cond = w.take<float>((size_t)B * frames * c->cfg.n_layers * kR);
  if (!rs) SRWN_CUDA(cudaMemsetAsync(queues, 0, queue_bytes, st));
  const GenState s = rs ? *rs : GenState{nullptr, nullptr, queues};   // one call from silence: the zeroed workspace queues
  const float* sw = stack_w(c, 0);
  k_cond<<<B * frames, 256, 0, st>>>(enc, sw + c->off.cond_k, sw + c->off.cond_b, cond, B * frames,
                                     c->cfg.n_layers, c->cfg.cond_channels);
  SRWN_LAUNCH_CHECK();
  ArParams p;
  p.w = sw; p.off = c->off; p.dil = c->d_dilations; p.qoff = c->d_queue_off;
  p.queues = static_cast<float*>(s.queues); p.cond = cond; p.u1 = u1; p.u2 = u2; p.x_out = x_out; p.logits_out = logits_out;
  p.B = B; p.T = T; p.L = c->cfg.n_layers; p.P = c->cfg.pool_stride; p.frames = frames;
  p.M = c->cfg.num_mixtures; p.sum_d = c->sum_dilation;
  p.t0 = s.t0; p.xhist = s.xhist; p.x_prefix = x_prefix; p.n_prefix = n_prefix;
  {
    ProfScope prof(c, st, "k_ar_generate", 1);
    const bool two = B > c->sm_count;
    const dim3 grid = two ? (B + 1) / 2 : B;
    if (rs) {
      if (two) k_ar_generate<2, true><<<grid, 256, 0, st>>>(p); else k_ar_generate<1, true><<<grid, 256, 0, st>>>(p);
    } else {
      if (two) k_ar_generate<2, false><<<grid, 256, 0, st>>>(p); else k_ar_generate<1, false><<<grid, 256, 0, st>>>(p);
    }
    SRWN_LAUNCH_CHECK();
  }
  return rs ? run_gen_state_advance(s.t0, T, st) : SRWN_OK;
}
