// fp32-grade path of the residual stack (parity path, <= 1e-4 relative vs the oracle).
//
// One launch per layer; the residual stream (and the teacher's skip sum) round-trips through HBM as fp32.  The layer
// GEMMs run on the tensor cores with split TF32 operands (three MMAs per product): the teacher's layers in
// tf32x3::k_fwd_layer below (mma.sync, with the skip output), the student's in traintc::k_fwd_layer_tc (train_tc.cu,
// tcgen05).  Conditioning, front conv and the output heads are FFMA kernels.  This is the reference-grade path, the
// GPU-side cross-check for the fused fp16 tcgen05 kernel (fused.cu), which is the one the benchmark times, and the
// forward of the distillation step (train_f32.cu), which keeps every layer input: the training step differentiates
// exactly what this file computes.
//
// Stored tensor convention: `hc_i` = the block input of layer i = h_i + upsampled
// conditioning of layer i (model.py:183 adds it before ResidualDilationLayer, so it also
// feeds the `inputs + residual` term at ops.py:40 and is zero-padded like the rest).
#include "common.cuh"
#include "philox.cuh"
#include "train_tc.cuh"

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

// ---- teacher layer: residual block with the skip output, 3xTF32 on mma.sync -----------------------------------------
// x_{l+1} = (x_l + c Wr + br) sqrt(1/2) + cond_{l+1},  c = f sigmoid(f),  f = tanh([x_l[t-d] | x_l[t]] Wf + bf),
// skip (+)= c Ws + bs   (ops.py:23-46, model.py:190).  64 time steps per tile, persistent CTAs, weights staged once.  The
// GEMMs run on the tensor cores at fp32 grade: every operand is split into two TF32 numbers (x = hi + lo,
// |lo| <= 2^-11 |hi|) and a product is three MMAs, lo*hi + hi*lo + hi*hi, small terms first (the dropped lo*lo term is
// 2^-22 relative).
namespace tf32x3 {

constexpr int kTT = 64;             // time steps per tile
constexpr int kAP = kR + 4;         // padded pitch
constexpr int kThreads = 256;

// ---- warp-level TF32 tensor-core helpers (mma.sync.m16n8k8, fp32 accumulate) ------------------------------
// Fragment layouts (g = lane >> 2, q = lane & 3):  A 16x8 row-major: a0 (g, q) a1 (g+8, q) a2 (g, q+4) a3 (g+8, q+4);
// B 8x8: b0 (k = q, n = g) b1 (k = q+4, n = g);  C 16x8: c0 (g, 2q) c1 (g, 2q+1) c2 (g+8, 2q) c3 (g+8, 2q+1).
__device__ __forceinline__ void mma_tf32(float (&d)[4], float a0, float a1, float a2, float a3, float b0, float b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(__float_as_uint(a0)), "r"(__float_as_uint(a1)), "r"(__float_as_uint(a2)), "r"(__float_as_uint(a3)),
                 "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}
constexpr int kWP = kR + 8;         // pitch of B operands read as (k = q, n = g): banks 8q + g
// A fragment (16 rows x 8 tf32) with one ldmatrix: a 8x8 b16 matrix is 8 rows of 16 bytes = 8 rows x 4 tf32 words, and thread
// (g, q) receives row g, word q -- the m16n8k8 A layout.  Lane l passes the row address of matrix l >> 3:
// {rows 0-7 | rows 8-15} x {words 0-3 | words 4-7} -> a0, a1, a2, a3.  Rows are 144 bytes apart: conflict-free.
__device__ __forceinline__ void ldsm_a(float (&a)[4], const float* lane_row_ptr) {
  uint32_t r0, r1, r2, r3;
  const uint32_t addr = (uint32_t)__cvta_generic_to_shared(lane_row_ptr);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
  a[0] = __uint_as_float(r0); a[1] = __uint_as_float(r1); a[2] = __uint_as_float(r2); a[3] = __uint_as_float(r3);
}

constexpr int kSP = kS + 8;         // pitch of the skip weights: banks 8q + g
// the skip weights join the resident set and the gate output c takes over the tap rows, which are dead once the filter
// conv has run, so that two CTAs still fit one SM
struct Smem {
  float tap_h[kTT][kAP], tap_l[kTT][kAP], cur_h[kTT][kAP], cur_l[kTT][kAP];
  float wf_h[2 * kR][kWP], wf_l[2 * kR][kWP], wr_h[kR][kWP], wr_l[kR][kWP], bf[kR], br[kR];
  float ws_h[kR][kSP], ws_l[kR][kSP], bs[kS];
};
// x = hi + lo with both parts valid TF32 numbers (low 13 mantissa bits clear).  Truncation instead of cvt.rna: hi is off by
// up to 2^-10 |x| but x - hi is exact, and truncating lo costs 2^-10 |lo| <= 2^-20 |x|; two LOP3 + one FADD, where
// cvt.rna.tf32.f32 expands to ~5 instructions each on sm_100a (FSETP / VIADD / SEL / LOP3).
// (train_tc.cu keeps all of lo's bits instead: the two splits give different results.)
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  lo = __uint_as_float(__float_as_uint(x - hi) & 0xFFFFE000u);
}
__device__ __forceinline__ void split_store4(float* h, float* l, float4 v) {
  float4 vh, vl;
  split_tf32(v.x, vh.x, vl.x); split_tf32(v.y, vh.y, vl.y); split_tf32(v.z, vh.z, vl.z); split_tf32(v.w, vh.w, vl.w);
  *reinterpret_cast<float4*>(h) = vh;
  *reinterpret_cast<float4*>(l) = vl;
}

__global__ void __launch_bounds__(kThreads)
k_fwd_layer(const float* __restrict__ x_l, float* __restrict__ x_next, const float* __restrict__ filt_k,
            const float* __restrict__ filt_b, const float* __restrict__ res_k, const float* __restrict__ res_b,
            const float* __restrict__ cond_next,     // cond + (l + 1) * R of layout [B][frames][L][R], or null after the last layer
            int B, int T, int d, int P, int L, int frames,
            const float* __restrict__ skip_k, const float* __restrict__ skip_b, float* __restrict__ skip, int skip_init) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw);
  float (*c_h)[kAP] = s.tap_h;
  float (*c_l)[kAP] = s.tap_l;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  for (int i = tid; i < kR * kS; i += kThreads) split_tf32(skip_k[i], s.ws_h[i / kS][i % kS], s.ws_l[i / kS][i % kS]);
  if (tid < kS) s.bs[tid] = skip_b[tid];
  for (int i = tid; i < 2 * kR * kR; i += kThreads) split_tf32(filt_k[i], s.wf_h[i / kR][i % kR], s.wf_l[i / kR][i % kR]);
  for (int i = tid; i < kR * kR; i += kThreads) split_tf32(res_k[i], s.wr_h[i / kR][i % kR], s.wr_l[i / kR][i % kR]);
  if (tid < kR) { s.bf[tid] = filt_b[tid]; s.br[tid] = res_b[tid]; }
  const int tiles_per_b = (T + kTT - 1) / kTT;
  const int n_tiles = B * tiles_per_b;
  const int mt = warp & 3, nh = warp >> 2, r0 = mt * 16;
  const int lrow = r0 + (lane & 7) + ((lane >> 3) & 1) * 8, lcol = (lane >> 4) * 4;      // this lane's row address inside an ldmatrix A tile
  grid_dependency_wait();                            // weights are staged; the activations come from the previous launch
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kTT;
    const float* xb = x_l + (size_t)b * T * kR;
    __syncthreads();
    for (int i = tid; i < kTT * (kR / 4); i += kThreads) {
      const int row = i / (kR / 4), c4 = i % (kR / 4);
      const int t = t0 + row;
      float4 cur = make_float4(0, 0, 0, 0), tap = cur;
      if (t < T) {
        cur = *reinterpret_cast<const float4*>(xb + (size_t)t * kR + c4 * 4);
        if (t - d >= 0) tap = *reinterpret_cast<const float4*>(xb + (size_t)(t - d) * kR + c4 * 4);
      }
      split_store4(&s.cur_h[row][c4 * 4], &s.cur_l[row][c4 * 4], cur);
      split_store4(&s.tap_h[row][c4 * 4], &s.tap_l[row][c4 * 4], tap);
    }
    __syncthreads();
    // filter conv (ops.py:6-20): W[0] pairs with x[t-d], W[1] with x[t]
    float acc[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; nt++) {
      const int n0 = nh * 16 + nt * 8 + 2 * q;
      acc[nt][0] = acc[nt][2] = s.bf[n0]; acc[nt][1] = acc[nt][3] = s.bf[n0 + 1];
    }
#pragma unroll
    for (int ks = 0; ks < 8; ks++) {
      const float (*XH)[kAP] = ks < 4 ? s.tap_h : s.cur_h;
      const float (*XL)[kAP] = ks < 4 ? s.tap_l : s.cur_l;
      const int kc = (ks & 3) * 8;
      float ah[4], al[4];
      ldsm_a(ah, &XH[lrow][kc + lcol]);
      ldsm_a(al, &XL[lrow][kc + lcol]);
#pragma unroll
      for (int nt = 0; nt < 2; nt++) {
        const int n0 = nh * 16 + nt * 8 + g;
        const float bh0 = s.wf_h[ks * 8 + q][n0], bh1 = s.wf_h[ks * 8 + q + 4][n0];
        const float bl0 = s.wf_l[ks * 8 + q][n0], bl1 = s.wf_l[ks * 8 + q + 4][n0];
        mma_tf32(acc[nt], al[0], al[1], al[2], al[3], bh0, bh1);
        mma_tf32(acc[nt], ah[0], ah[1], ah[2], ah[3], bl0, bl1);
        mma_tf32(acc[nt], ah[0], ah[1], ah[2], ah[3], bh0, bh1);
      }
    }
    __syncthreads();                                   // every warp is done with the tap rows: c may take their place
    // gate: tanh, sigmoid OF THE TANH, product (ops.py:28,33,36)
#pragma unroll
    for (int nt = 0; nt < 2; nt++) {
      const int n0 = nh * 16 + nt * 8 + 2 * q;
      float cv[4], ch[4], cl[4];
#pragma unroll
      for (int e = 0; e < 4; e++) { const float f = tanhf(acc[nt][e]); cv[e] = f * (1.0f / (1.0f + expf(-f))); split_tf32(cv[e], ch[e], cl[e]); }
      *reinterpret_cast<float2*>(&c_h[r0 + g][n0]) = make_float2(ch[0], ch[1]);
      *reinterpret_cast<float2*>(&c_h[r0 + g + 8][n0]) = make_float2(ch[2], ch[3]);
      *reinterpret_cast<float2*>(&c_l[r0 + g][n0]) = make_float2(cl[0], cl[1]);
      *reinterpret_cast<float2*>(&c_l[r0 + g + 8][n0]) = make_float2(cl[2], cl[3]);
    }
    __syncthreads();
    // residual 1x1 (ops.py:39), dense = (inputs + residual) * sqrt(1/2) (ops.py:40), next layer's conditioning (model.py:183)
#pragma unroll
    for (int nt = 0; nt < 2; nt++) {
      const int n0 = nh * 16 + nt * 8 + 2 * q;
      acc[nt][0] = acc[nt][2] = s.br[n0]; acc[nt][1] = acc[nt][3] = s.br[n0 + 1];
    }
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      const int kc = ks * 8;
      float ah[4], al[4];
      ldsm_a(ah, &c_h[lrow][kc + lcol]);
      ldsm_a(al, &c_l[lrow][kc + lcol]);
      const float h0 = ah[0], h1 = ah[1], h2 = ah[2], h3 = ah[3], l0 = al[0], l1 = al[1], l2 = al[2], l3 = al[3];
#pragma unroll
      for (int nt = 0; nt < 2; nt++) {
        const int n0 = nh * 16 + nt * 8 + g;
        const float bh0 = s.wr_h[kc + q][n0], bh1 = s.wr_h[kc + q + 4][n0];
        const float bl0 = s.wr_l[kc + q][n0], bl1 = s.wr_l[kc + q + 4][n0];
        mma_tf32(acc[nt], l0, l1, l2, l3, bh0, bh1);
        mma_tf32(acc[nt], h0, h1, h2, h3, bl0, bl1);
        mma_tf32(acc[nt], h0, h1, h2, h3, bh0, bh1);
      }
    }
    const int ta = t0 + r0 + g, tb = ta + 8;
#pragma unroll
    for (int nt = 0; nt < 2; nt++) {
      const int n0 = nh * 16 + nt * 8 + 2 * q;
      if (ta < T) {
        const size_t at = ((size_t)b * T + ta) * kR + n0;
        const float2 xv = *reinterpret_cast<const float2*>(x_l + at);
        float2 v = make_float2((xv.x + acc[nt][0]) * SRWN_SQRT_HALF, (xv.y + acc[nt][1]) * SRWN_SQRT_HALF);
        if (cond_next) { const float2 cn = *reinterpret_cast<const float2*>(cond_next + ((size_t)b * frames + ta / P) * L * kR + n0); v.x += cn.x; v.y += cn.y; }
        *reinterpret_cast<float2*>(x_next + at) = v;
      }
      if (tb < T) {
        const size_t at = ((size_t)b * T + tb) * kR + n0;
        const float2 xv = *reinterpret_cast<const float2*>(x_l + at);
        float2 v = make_float2((xv.x + acc[nt][2]) * SRWN_SQRT_HALF, (xv.y + acc[nt][3]) * SRWN_SQRT_HALF);
        if (cond_next) { const float2 cn = *reinterpret_cast<const float2*>(cond_next + ((size_t)b * frames + tb / P) * L * kR + n0); v.x += cn.x; v.y += cn.y; }
        *reinterpret_cast<float2*>(x_next + at) = v;
      }
    }
    // skip 1x1 (ops.py:44) accumulated over layers in global memory (model.py:190); warp (mt, nh): rows 16 mt.., channels 64 nh..
    float sk[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      const int n0 = nh * 64 + nt * 8 + 2 * q;
      sk[nt][0] = sk[nt][2] = s.bs[n0]; sk[nt][1] = sk[nt][3] = s.bs[n0 + 1];
    }
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      const int kc = ks * 8;
      float ah[4], al[4];
      ldsm_a(ah, &c_h[lrow][kc + lcol]);
      ldsm_a(al, &c_l[lrow][kc + lcol]);
      const float h0 = ah[0], h1 = ah[1], h2 = ah[2], h3 = ah[3], l0 = al[0], l1 = al[1], l2 = al[2], l3 = al[3];
#pragma unroll
      for (int nt = 0; nt < 8; nt++) {
        const int n0 = nh * 64 + nt * 8 + g;
        const float bh0 = s.ws_h[kc + q][n0], bh1 = s.ws_h[kc + q + 4][n0];
        const float bl0 = s.ws_l[kc + q][n0], bl1 = s.ws_l[kc + q + 4][n0];
        mma_tf32(sk[nt], l0, l1, l2, l3, bh0, bh1);
        mma_tf32(sk[nt], h0, h1, h2, h3, bl0, bl1);
        mma_tf32(sk[nt], h0, h1, h2, h3, bh0, bh1);
      }
    }
#pragma unroll
    for (int nt = 0; nt < 8; nt++) {
      const int n0 = nh * 64 + nt * 8 + 2 * q;
      if (ta < T) {
        float2* dst = reinterpret_cast<float2*>(skip + ((size_t)b * T + ta) * kS + n0);
        float2 v = make_float2(sk[nt][0], sk[nt][1]);
        if (!skip_init) { const float2 pv = *dst; v.x += pv.x; v.y += pv.y; }
        *dst = v;
      }
      if (tb < T) {
        float2* dst = reinterpret_cast<float2*>(skip + ((size_t)b * T + tb) * kS + n0);
        float2 v = make_float2(sk[nt][2], sk[nt][3]);
        if (!skip_init) { const float2 pv = *dst; v.x += pv.x; v.y += pv.y; }
        *dst = v;
      }
    }
  }
}

}  // namespace tf32x3

// cond, front, then one launch per layer.  The layers ping-pong between h0 and h1; with h1 == nullptr, h0 is
// [L+1][B][T][R] and keeps every layer input (h0[l] = block input of layer l, h0[L] = stack output), which is what the
// backward of the distillation step reads.  That forward opens no ProfScope, so that the step's timing names the backward.
int run_stack_f32(srwn_ctx* c, int stack, const float* xin, const float* enc, int B, int T,
                  float* h0, float* h1, float* skip, float* cond, float** h_final,
                  cudaStream_t st) {
  const float* w = stack_w(c, stack);
  const StackOffsets& o = c->off;
  const int L = c->cfg.n_layers, P = c->cfg.pool_stride, C = c->cfg.cond_channels;
  const int frames = T / P;
  const size_t n = (size_t)B * T;
  const bool with_skip = c->cfg.kind == SRWN_TEACHER;
  const int sms = c->sm_count > 0 ? c->sm_count : 148;
  k_cond<<<B * frames, 256, 0, st>>>(enc, w + o.cond_k, w + o.cond_b, cond, B * frames, L, C);
  SRWN_LAUNCH_CHECK();
  {
    dim3 grid((unsigned)(((int64_t)T * kR + 255) / 256), B);
    k_front<<<grid, 256, 0, st>>>(xin, w + o.front_k, w + o.front_b, cond, h0, T, P, L, frames);
    SRWN_LAUNCH_CHECK();
  }
  if (with_skip)
    SRWN_CUDA(cudaFuncSetAttribute(tf32x3::k_fwd_layer, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tf32x3::Smem)));
  else
    SRWN_CUDA(cudaFuncSetAttribute(traintc::k_fwd_layer_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::fwd_smem_bytes()));
  ProfScope prof(c, st, !h1 ? nullptr : with_skip ? "k_fwd_layer<skip> (3xTF32)" : "k_fwd_layer (3xTF32)", L);
  float* cur = h0;
  for (int l = 0; l < L; l++) {
    float* nxt = !h1 ? cur + n * kR : cur == h0 ? h1 : h0;
    const float* cond_next = l + 1 < L ? cond + (size_t)(l + 1) * kR : nullptr;
    const float *filt_k = w + o.filt_k + (size_t)l * 2 * kR * kR, *filt_b = w + o.filt_b + (size_t)l * kR;
    const float *res_k = w + o.res_k + (size_t)l * kR * kR, *res_b = w + o.res_b + (size_t)l * kR;
    const int d = c->dilations[l];
    if (with_skip)      // two CTAs per SM (64-step tiles)
      SRWN_CUDA(launch_dependent(tf32x3::k_fwd_layer, 2 * sms, tf32x3::kThreads, sizeof(tf32x3::Smem), st, cur, nxt, filt_k,
                                 filt_b, res_k, res_b, cond_next, B, T, d, P, L, frames, w + o.skip_k + (size_t)l * kR * kS,
                                 w + o.skip_b + (size_t)l * kS, skip, l == 0));
    else                // one CTA per SM (128-step tiles, tensor memory)
      SRWN_CUDA(launch_dependent(traintc::k_fwd_layer_tc, sms, traintc::kThreads, (size_t)traintc::fwd_smem_bytes(), st, cur,
                                 nxt, filt_k, filt_b, res_k, res_b, cond_next, B, T, d, P, L, frames));
    SRWN_LAUNCH_CHECK();
    cur = nxt;
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
                            float* __restrict__ xout, int64_t n, int T, int t_out) {
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
    if (t_out == 0 || row % T >= t_out) xout[row] = fmaf(xin[row], sc, mu);      // model.py:482
  }
}

int run_flow_head_f32(srwn_ctx* c, int stack, const float* h, const float* xin, float* scale,
                      float* mean, float* xout, int B, int T, cudaStream_t st, int t_out) {
  const float* w = stack_w(c, stack);
  const int64_t n = (int64_t)B * T;
  k_flow_head<<<(unsigned)((n * 8 + 255) / 256), 256, 0, st>>>(h, xin, w + c->off.head1_k,
                                                               w + c->off.head1_b, scale, mean, xout, n, T, t_out);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// s_tot, mu_tot (flow_compose_at); out = clip(z*s_tot + mu_tot, -1, 1) (model.py:535)
__global__ void k_flow_compose(const float* __restrict__ z, NoiseSpec noise, float* __restrict__ z_out,
                               const float* __restrict__ scales,
                               const float* __restrict__ means, int F, float* __restrict__ out,
                               float* __restrict__ s_tot, float* __restrict__ mu_tot, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // the student's input noise (student.py:104): supplied, or the same Philox draw the flow kernel evaluated
  const float zi = noise.on ? philox::logistic_at(noise.seed, noise.stream, (uint64_t)i) : z[i];
  if (z_out) z_out[i] = zi;
  float st, mt;
  flow_compose_at(scales, means, F, n, i, st, mt);
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
