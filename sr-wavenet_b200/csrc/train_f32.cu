// Student distillation step, device side (fp32 grade): forward that keeps every layer input, and the backward pass
// of the IAF flows (model.py:415-535) given the gradient of the loss (model.py:356-379) with respect to the
// network output.  Layer at a time; activations and their gradients round-trip HBM in fp32.  The three per-layer
// kernels are tcgen05 kernels (train_tc.cu); this file holds the elementwise kernels around them, the teacher's
// fp32-grade layer kernel (mma.sync, with the skip output) and the host sequence.
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
#include <type_traits>

namespace train {

constexpr int kTT = 64;             // time steps per tile
constexpr int kAP = kR + 4;         // padded pitch
constexpr int kThreads = 256;

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
// Programmatic dependent launch: the layer kernels are launched so that a kernel's CTAs may start (and stage their weights) while
// the previous layer's kernel drains; everything the previous launch wrote is visible after this wait (no-op in a plain launch).
// The trigger right after it lets the NEXT launch's CTAs take the SM slots this grid frees as its CTAs exit (all of this grid's
// CTAs are resident from the start, so nothing of it can be starved).
__device__ __forceinline__ void grid_dependency_wait() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ---- warp-level TF32 tensor-core helpers (mma.sync.m16n8k8, fp32 accumulate) ------------------------------
// Used by the teacher's fp32-grade layer kernel below (operands pre-split into hi + lo TF32 parts, three MMAs per product).
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

// ---- forward layer of the training pass ---------------------------------------------------------------
// x_{l+1} = (x_l + c Wr + br) sqrt(1/2) + cond_{l+1},  c = f sigmoid(f),  f = tanh([x_l[t-d] | x_l[t]] Wf + bf)   (ops.py:23-46)
// Same tiling as the backward kernels (64 time steps, persistent CTAs, weights staged once).  The GEMMs run on the
// tensor cores at fp32 grade: every operand is split into two TF32 numbers (x = hi + lo, |lo| <= 2^-11 |hi|) and a
// product is three MMAs, lo*hi + hi*lo + hi*hi, small terms first (the dropped lo*lo term is 2^-22 relative).  The
// stored activations are what the backward pass differentiates, so they stay within the fp32 path's 1e-4 of the oracle.
constexpr int kSP = kS + 8;         // pitch of the skip weights: banks 8q + g
struct FwdSmem {
  float tap_h[kTT][kAP], tap_l[kTT][kAP], cur_h[kTT][kAP], cur_l[kTT][kAP], c_h[kTT][kAP], c_l[kTT][kAP];
  float wf_h[2 * kR][kWP], wf_l[2 * kR][kWP], wr_h[kR][kWP], wr_l[kR][kWP], bf[kR], br[kR];
};
// teacher layers (skip 1x1, ops.py:44): the skip weights join the resident set and the gate output c takes over the
// tap rows, which are dead once the filter conv has run, so that two CTAs still fit one SM
struct FwdSmemSkip {
  float tap_h[kTT][kAP], tap_l[kTT][kAP], cur_h[kTT][kAP], cur_l[kTT][kAP];
  float wf_h[2 * kR][kWP], wf_l[2 * kR][kWP], wr_h[kR][kWP], wr_l[kR][kWP], bf[kR], br[kR];
  float ws_h[kR][kSP], ws_l[kR][kSP], bs[kS];
};
// x = hi + lo with both parts valid TF32 numbers (low 13 mantissa bits clear).  Truncation instead of cvt.rna: hi is off by
// up to 2^-10 |x| but x - hi is exact, and truncating lo costs 2^-10 |lo| <= 2^-20 |x|; two LOP3 + one FADD, where
// cvt.rna.tf32.f32 expands to ~5 instructions each on sm_100a (FSETP / VIADD / SEL / LOP3: half of k_bwd_gate's ALU work).
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

template <bool SKIP>
__global__ void __launch_bounds__(kThreads)
k_fwd_layer(const float* __restrict__ x_l, float* __restrict__ x_next, const float* __restrict__ filt_k,
            const float* __restrict__ filt_b, const float* __restrict__ res_k, const float* __restrict__ res_b,
            const float* __restrict__ cond_next,     // cond + (l + 1) * R of layout [B][frames][L][R], or null after the last layer
            int B, int T, int d, int P, int L, int frames,
            const float* __restrict__ skip_k, const float* __restrict__ skip_b, float* __restrict__ skip, int skip_init) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  typedef typename std::conditional<SKIP, FwdSmemSkip, FwdSmem>::type Smem;
  Smem& s = *reinterpret_cast<Smem*>(smem_raw);
  float (*c_h)[kAP];
  float (*c_l)[kAP];
  if constexpr (SKIP) { c_h = s.tap_h; c_l = s.tap_l; } else { c_h = s.c_h; c_l = s.c_l; }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  if constexpr (SKIP) {
    for (int i = tid; i < kR * kS; i += kThreads) split_tf32(skip_k[i], s.ws_h[i / kS][i % kS], s.ws_l[i / kS][i % kS]);
    if (tid < kS) s.bs[tid] = skip_b[tid];
  }
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
    if constexpr (SKIP) __syncthreads();               // every warp is done with the tap rows: c may take their place
    // gate: tanh, sigmoid OF THE TANH, product (ops.py:28,33,36)
#pragma unroll
    for (int nt = 0; nt < 2; nt++) {
      const int n0 = nh * 16 + nt * 8 + 2 * q;
      float cv[4], ch[4], cl[4];
#pragma unroll
      for (int e = 0; e < 4; e++) { const float f = tanhf(acc[nt][e]); cv[e] = f * sigmoidf_(f); split_tf32(cv[e], ch[e], cl[e]); }
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
    if constexpr (SKIP) {
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
}

// The per-layer kernels of the student's training pass (forward keeping activations, gate backward, conv backward) live in
// train_tc.cu (tcgen05 kind::tf32); k_fwd_layer<true> above remains for the teacher's fp32-grade path, whose layers also
// produce the skip output.

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
#ifdef SRWN_TC_GRID
  r.grid_tc = SRWN_TC_GRID;                                // tuning builds: few CTAs, so that small test shapes give every CTA several tiles
#endif
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

// forward of all flows in fp32, keeping every layer input (model.py:489-535)
template <typename... KArgs, typename... Args>
static cudaError_t launch_dependent(void (*kern)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
#ifdef SRWN_NO_PDL
  cfg.numAttrs = 0;                        // tuning builds: plain stream order
#endif
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// one layer of the fp32-grade path (stack_f32.cu): x_l -> x_next, teacher layers also accumulate their skip output
int run_layer_tf32x3(srwn_ctx* c, bool with_skip, const float* x_l, float* x_next, float* skip, const float* filt_k,
                     const float* filt_b, const float* res_k, const float* res_b, const float* skip_k, const float* skip_b,
                     const float* cond_next, int B, int T, int d, int P, int L, int frames, int skip_init, cudaStream_t st) {
  const int grid = 2 * (c->sm_count > 0 ? c->sm_count : 148);
  if (with_skip) {
    SRWN_CUDA(cudaFuncSetAttribute(train::k_fwd_layer<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(train::FwdSmemSkip)));
    SRWN_CUDA(launch_dependent(train::k_fwd_layer<true>, grid, train::kThreads, sizeof(train::FwdSmemSkip), st,
        x_l, x_next, filt_k, filt_b, res_k, res_b, cond_next, B, T, d, P, L, frames, skip_k, skip_b, skip, skip_init));
  } else {
    SRWN_CUDA(cudaFuncSetAttribute(traintc::k_fwd_layer_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::fwd_smem_bytes()));
    SRWN_CUDA(launch_dependent(traintc::k_fwd_layer_tc, grid / 2, traintc::kThreads, (size_t)traintc::fwd_smem_bytes(), st,
        x_l, x_next, filt_k, filt_b, res_k, res_b, cond_next, B, T, d, P, L, frames));
  }
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

// forward of one flow keeping every layer input: acts [L+1][B][T][R], acts[l] = block input of layer l, acts[L] = stack output
static int run_stack_train_acts(srwn_ctx* c, int stack, const float* xin, const float* enc, int B, int T, float* acts,
                                float* cond, int grid, cudaStream_t st) {
  const float* w = stack_w(c, stack);
  const StackOffsets& o = c->off;
  const int L = c->cfg.n_layers, P = c->cfg.pool_stride, C = c->cfg.cond_channels, frames = T / P;
  const size_t n = (size_t)B * T;
  k_cond<<<B * frames, 256, 0, st>>>(enc, w + o.cond_k, w + o.cond_b, cond, B * frames, L, C);
  SRWN_LAUNCH_CHECK();
  {
    dim3 g((unsigned)(((int64_t)T * kR + 255) / 256), B);
    k_front<<<g, 256, 0, st>>>(xin, w + o.front_k, w + o.front_b, cond, acts, T, P, L, frames);
    SRWN_LAUNCH_CHECK();
  }
  SRWN_CUDA(cudaFuncSetAttribute(traintc::k_fwd_layer_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::fwd_smem_bytes()));
  for (int l = 0; l < L; l++) {
    const float* cond_next = l + 1 < L ? cond + (size_t)(l + 1) * kR : nullptr;
    SRWN_CUDA(launch_dependent(traintc::k_fwd_layer_tc, grid, traintc::kThreads, (size_t)traintc::fwd_smem_bytes(), st,
        acts + (size_t)l * n * kR, acts + (size_t)(l + 1) * n * kR, w + o.filt_k + (size_t)l * 2 * kR * kR,
        w + o.filt_b + (size_t)l * kR, w + o.res_k + (size_t)l * kR * kR, w + o.res_b + (size_t)l * kR, cond_next,
        B, T, c->dilations[l], P, L, frames));
    SRWN_LAUNCH_CHECK();
  }
  return SRWN_OK;
}

int run_student_forward_train(srwn_ctx* c, const float* z, const float* enc, float* out, float* s_tot,
                              float* mu_tot, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st) {
  TrainWs w = carve_train(c, B, T, ws, ws_bytes);
  if (!ws || w.bytes > ws_bytes) return srwn_fail(SRWN_ERR_WORKSPACE, "workspace too small: need %zu bytes", w.bytes);
  const size_t n = (size_t)B * T;
  const int F = c->cfg.num_flows, L = c->cfg.n_layers;
  const float* xin = z;
  for (int f = 0; f < F; f++) {
    float* acts = w.acts + (size_t)f * (L + 1) * n * kR;
    int rc = run_stack_train_acts(c, f, xin, enc, B, T, acts, w.cond, w.grid_tc, st);
    if (rc) return rc;
    rc = run_flow_head_f32(c, f, acts + (size_t)L * n * kR, xin, w.scales + (size_t)f * n, w.means + (size_t)f * n,
                           w.xs + (size_t)f * n, B, T, st);
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
  if (!ws || w.bytes > ws_bytes) return srwn_fail(SRWN_ERR_WORKSPACE, "workspace too small: need %zu bytes", w.bytes);
  const size_t n = (size_t)B * T;
  const int F = c->cfg.num_flows, L = c->cfg.n_layers, P = c->cfg.pool_stride, frames = T / P, C = c->cfg.cond_channels;
  const int BF = B * frames;
  const StackOffsets& o = c->off;
  static bool attr_done = false;
  if (!attr_done) {
    SRWN_CUDA(cudaFuncSetAttribute(traintc::k_bwd_gate_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::gate_smem_bytes()));
    SRWN_CUDA(cudaFuncSetAttribute(traintc::k_bwd_conv_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, traintc::conv_smem_bytes()));
    attr_done = true;
  }
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
