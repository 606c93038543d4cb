// Teacher encoder (SURVEY.md 8(f)-1): model.py:137-155 createEncoder built from ops.py:48-57
// ResidualDilationLayerNC.  Per layer: a = relu(h); y = relu(a[t]*W0 + a[t+1]*W1 + b) (K=2, SAME padding,
// not causal, not dilated); h' = y*Wr + br (no skip connection); skip = y*Ws + bs.  encoding =
// avgpool_P((sum of skips)*Wl + bl).
//
// Two paths behind srwn_teacher_encode:
//  * fp32 (parity grade): FFMA GEMM kernels, activations and the skip sum in fp32 in the workspace.
//  * fp16 operands on tcgen05 tensor cores, one launch per layer (k_enc_layer):
//      - activations travel between layers as the 16-bit image of relu(h) in the UMMA K-major
//        no-swizzle layout, one contiguous block [16 kc][129 rows][8] per tile of 128 time steps (row 128
//        repeats row 0 of the next tile), so a tile is loaded with two bulk copies and the a[t+1] tap is the
//        same shared-memory buffer addressed one row (16 B) later;
//      - persistent CTAs keep the layer's weights (conv 64 KB + residual 32 KB) in shared memory and
//        stream tiles: conv GEMM [128x256]x[256x128] -> relu epilogue -> residual GEMM [128x128]x[128x128]
//        -> relu epilogue -> 16-bit store, double-buffered in TMEM (4 x 128 columns);
//      - the skip path is never materialised: average pooling, the skip 1x1 and the latent 1x1 are all
//        linear, so avgpool((sum_l y_l Ws_l + bs_l) Wl + bl) = sum_l avgpool(y_l) (Ws_l Wl) + const.  The
//        kernel only emits the column sums of y over each tile (one pooling window when P = 128); a
//        small finishing kernel applies the folded [L*128 x latent] matrix.  This removes a quarter of
//        the FLOPs and every O(B*T*S) skip tensor.
#include "common.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>
#include <cstring>
#include <cstdio>
#include <map>
#include <new>
#include <string>
#include <vector>

using namespace umma;

namespace enc {

constexpr int kE = 128;            // encoder_channels the tensor-core path is built for (teacher.py default)
constexpr int kTile = 128;
constexpr int kTileBytes = kTile * kE * 2;        // 32768: one y operand tile
constexpr int kConvImg = 2 * kE * kE * 2;         // 65536
constexpr int kResImg = kE * kE * 2;              // 32768
constexpr int kLayerImg = kConvImg + kResImg + 2 * kE * 4;   // + conv bias + res bias (fp32)
constexpr int kFrontImg = kResImg + 4 * kE * 4;   // res image | front_k[2][E] | front_b[E] | res bias[E]
constexpr int kARows = kTile + 1;                 // rows per k-chunk of an A stage (tile + the t+1 halo row)
constexpr int kAStage = 16 * kARows * 16;         // 33024: one activation tile, in HBM and in shared memory
constexpr int kStages = 3;

struct Smem {
  static constexpr int w = 0;                                  // conv image | res image   (front: res image only)
  static constexpr int bias = w + kConvImg + kResImg;          // 4 x [128] fp32
  static constexpr int a = bias + 4 * kE * 4;                  // kStages A stages [16][129][16 B]
  static constexpr int y = a + kStages * kAStage;              // y operand buffer [16][128][16 B]
  static constexpr int bars = y + kTileBytes;
  static constexpr int n_bars = 18;
  static constexpr int misc = bars + n_bars * 8;
  static constexpr int total = misc + 16;
};
static_assert(Smem::total <= 232448, "shared memory budget");

enum Bar { B_W = 0, B_AF = 1, B_AE = 4, B_D1F = 7, B_D1E = 9, B_YF = 11, B_YE = 12, B_D2F = 13, B_D2E = 15 };

struct LayerParams {
  const uint8_t* img;        // this layer's packed image
  const uint8_t* in;         // blocked 16-bit activations (null for the front layer)
  const float* x;            // [B][T] audio (front layer)
  uint8_t* out;              // blocked 16-bit activations of the next layer (null: last layer)
  float* pooled;             // [n_tiles][128] column sums of y (null: front layer)
  int* err;
  int n_tiles, tiles_per_utt, T;
  int reverse;               // walk the tiles from the end: the tail of the previous layer's output is still in L2
};

__device__ __forceinline__ uint32_t pack2_relu(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));   // saturating: no inf in an operand image
  return r;
}
__device__ __forceinline__ float2 unpack2(uint32_t v) { return __half22float2(*reinterpret_cast<const __half2*>(&v)); }

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

constexpr int kThreads = 10 * 32;   // warp 0 loader, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue 1, warps 6-9 epilogue 2

template <bool FRONT>
__global__ void __launch_bounds__(kThreads, 1) k_enc_layer(const LayerParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t sbase = smem_u32(smem);
  auto bar = [&](int i) { return sbase + Smem::bars + i * 8; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Smem::misc);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(smem + Smem::misc + 8);
  const bool do_res = p.out != nullptr, do_pool = p.pooled != nullptr;

  if (tid == 0) {
    mbar_init(bar(B_W), 1);
    for (int i = 0; i < kStages; i++) { mbar_init(bar(B_AF + i), 1); mbar_init(bar(B_AE + i), 1); }
    for (int i = 0; i < 2; i++) {
      mbar_init(bar(B_D1F + i), 1); mbar_init(bar(B_D1E + i), 1);
      mbar_init(bar(B_D2F + i), 1); mbar_init(bar(B_D2E + i), 1);
    }
    mbar_init(bar(B_YF), 1); mbar_init(bar(B_YE), do_res ? 2 : 1);   // y free: residual MMAs retired + pooling reads done
    abort_flag[0] = 0; abort_flag[1] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int n_my = p.n_tiles > (int)blockIdx.x ? (p.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  auto tile_of = [&](int k) { const int i = (int)blockIdx.x + k * (int)gridDim.x; return p.reverse ? p.n_tiles - 1 - i : i; };
  constexpr uint32_t idesc = make_idesc(0, 128, 128);      // fp16 operands
  constexpr int w_bytes = FRONT ? kFrontImg : kLayerImg;
  constexpr int res_off = FRONT ? 0 : kConvImg;               // residual image inside the shared weight area
  float* s_bias = reinterpret_cast<float*>(smem + Smem::bias);

  if (warp == 0) {
    // ================= loader ============================================================
    if (lane == 0) {
      mbar_expect_tx(bar(B_W), w_bytes);
      constexpr int img_bytes = FRONT ? kResImg : kConvImg + kResImg;      // 16-bit images, then the fp32 tail -> bias area
      for (int o = 0; o < img_bytes; o += 16384) bulk_g2s(sbase + Smem::w + o, p.img + o, 16384, bar(B_W));
      bulk_g2s(sbase + Smem::bias, p.img + img_bytes, w_bytes - img_bytes, bar(B_W));
      if (!FRONT) {
        for (int k = 0; k < n_my; k++) {
          const int s = k % kStages;
          const int tile = tile_of(k);
          if (!mbar_wait(bar(B_AE + s), ((k / kStages) & 1) ^ 1, abort_flag, 0x100 | s)) break;
          const uint32_t dst = sbase + Smem::a + s * kAStage;
          const uint8_t* src = p.in + (size_t)tile * kAStage;
          mbar_expect_tx(bar(B_AF + s), kAStage);
          bulk_g2s(dst, src, kAStage / 2, bar(B_AF + s));
          bulk_g2s(dst + kAStage / 2, src + kAStage / 2, kAStage / 2, bar(B_AF + s));
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================= MMA issuer ========================================================
    if (lane == 0) {
      bool ok = mbar_wait(bar(B_W), 0, abort_flag, 0x200);
      const uint32_t wb_lo = ((sbase + Smem::w) >> 4) + (128u << 16);                 // conv image: LBO = 128 rows
      const uint32_t rb_lo = ((sbase + Smem::w + res_off) >> 4) + (128u << 16);
      for (int k = 0; k <= n_my && ok; k++) {
        if (!FRONT && k < n_my) {
          const int s = k % kStages, d = k & 1;
          ok = ok && mbar_wait(bar(B_AF + s), (k / kStages) & 1, abort_flag, 0x210 | s);
          ok = ok && mbar_wait(bar(B_D1E + d), ((k >> 1) & 1) ^ 1, abort_flag, 0x220 | d);
          if (!ok) break;
          tc_fence_after();
          const uint32_t a_lo = ((sbase + Smem::a + s * kAStage) >> 4) + ((uint32_t)kARows << 16);
          const uint32_t d1 = tmem + d * 128;
#pragma unroll
          for (int ks = 0; ks < 16; ks++) {
            // k-steps 0..7: a[t] x W[0]; 8..15: a[t+1] x W[1] (same buffer, one row later)
            const uint32_t al = a_lo + (uint32_t)((ks & 7) * 2 * kARows) + (ks >= 8 ? 1u : 0u);
            const uint32_t bl = wb_lo + (uint32_t)(ks * 256);
            if (ks == 0) tc_mma<0>(d1, desc_from_lo(al), desc_from_lo(bl), idesc);
            else tc_mma<1>(d1, desc_from_lo(al), desc_from_lo(bl), idesc);
          }
          tc_commit(bar(B_D1F + d));
          tc_commit(bar(B_AE + s));
        }
        if (k >= 1) {
          const int j = k - 1, yb = j & 1;
          if (do_res) {
            ok = ok && mbar_wait(bar(B_YF), j & 1, abort_flag, 0x230);
            ok = ok && mbar_wait(bar(B_D2E + yb), ((j >> 1) & 1) ^ 1, abort_flag, 0x240 | yb);
            if (!ok) break;
            tc_fence_after();
            const uint32_t y_lo = ((sbase + Smem::y) >> 4) + ((uint32_t)kTile << 16);
            const uint32_t d2 = tmem + 256 + yb * 128;
#pragma unroll
            for (int ks = 0; ks < 8; ks++) {
              const uint32_t al = y_lo + (uint32_t)(ks * 2 * kTile), bl = rb_lo + (uint32_t)(ks * 256);
              if (ks == 0) tc_mma<0>(d2, desc_from_lo(al), desc_from_lo(bl), idesc);
              else tc_mma<1>(d2, desc_from_lo(al), desc_from_lo(bl), idesc);
            }
            tc_commit(bar(B_D2F + yb));
            tc_commit(bar(B_YE));
          }
        }
      }
    }
    __syncwarp();
  } else if (warp < 6) {
    // ================= epilogue 1: conv accumulator -> y = relu(. + b) as the 16-bit A operand ==========
    const int q = warp & 3, row = q * 32 + lane;
    bool ok = mbar_wait(bar(B_W), 0, abort_flag, 0x300);       // biases / front weights landed
    const float* cbias = FRONT ? s_bias + 2 * kE : s_bias;     // front image tail: fk[2][E] | fb[E] | res bias[E]
    uint8_t* yb = smem + Smem::y;
    for (int k = 0; k < n_my; k++) {
      const int d = k & 1;
      const int tile = tile_of(k);
      float a0 = 0.f, a1 = 0.f;
      if (FRONT) {
        const int b = tile / p.tiles_per_utt, t = (tile % p.tiles_per_utt) * kTile + row;
        a0 = fmaxf(__ldg(p.x + (size_t)b * p.T + t), 0.f);                              // ops.py:49 relu on the raw audio
        a1 = t + 1 < p.T ? fmaxf(__ldg(p.x + (size_t)b * p.T + t + 1), 0.f) : 0.f;
      } else {
        ok = ok && mbar_wait(bar(B_D1F + d), (k >> 1) & 1, abort_flag, 0x310 | d);
      }
      tc_fence_after();
      uint32_t w[64];                     // the row's 128 channels, packed: computed before the y buffer is free
#pragma unroll
      for (int c2 = 0; c2 < 2; c2++) {
        float v[64];
        if (!FRONT && ok) {
          const uint32_t ta = tmem + d * 128 + c2 * 64 + ((uint32_t)(q * 32) << 16);
          tc_ld32(ta, v);
          tc_ld32(ta + 32, v + 32);
          tc_wait_ld();
        }
#pragma unroll
        for (int j = 0; j < 32; j++) {
          const int c = c2 * 64 + 2 * j;
          float lo, hi;
          if (FRONT) {
            lo = fmaf(a0, s_bias[c], fmaf(a1, s_bias[kE + c], cbias[c]));
            hi = fmaf(a0, s_bias[c + 1], fmaf(a1, s_bias[kE + c + 1], cbias[c + 1]));
          } else {
            lo = v[2 * j] + cbias[c];
            hi = v[2 * j + 1] + cbias[c + 1];
          }
          w[c2 * 32 + j] = pack2_relu(lo, hi);
        }
      }
      if (!FRONT) {                       // accumulator drained: the conv GEMM of tile k+2 may overwrite it
        tc_fence_before();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (warp == 2 && lane == 0) mbar_arrive(bar(B_D1E + d));
      }
      ok = ok && mbar_wait(bar(B_YE), (k & 1) ^ 1, abort_flag, 0x320);
#pragma unroll
      for (int j = 0; j < 16; j++)
        *reinterpret_cast<uint4*>(yb + (j * kTile + row) * 16) = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
      fence_async_smem();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (warp == 2 && lane == 0) mbar_arrive(bar(B_YF));
    }
  } else {
    // ================= epilogue 2: pooling of y; residual accumulator -> relu(h') 16-bit image in HBM =====
    const int q = warp & 3, row = q * 32 + lane, gt = tid - 6 * 32;
    bool ok = mbar_wait(bar(B_W), 0, abort_flag, 0x400);
    const float* rbias = FRONT ? s_bias + 3 * kE : s_bias + kE;
    for (int k = 0; k < n_my; k++) {
      const int s = k & 1;
      const int tile = tile_of(k);
      ok = ok && mbar_wait(bar(B_YF), k & 1, abort_flag, 0x410);
      if (do_pool && ok) {
        // column sums of the tile's y (16-bit image in shared memory): thread = (k-chunk, row residue mod 8)
        const int kc = gt >> 3, sub = gt & 7;
        const uint8_t* yb = smem + Smem::y + (kc * kTile + sub) * 16;
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; e++) acc[e] = 0.f;
#pragma unroll 4
        for (int i = 0; i < 16; i++) {
          const uint4 u = *reinterpret_cast<const uint4*>(yb + i * 8 * 16);
          const float2 f0 = unpack2(u.x), f1 = unpack2(u.y), f2 = unpack2(u.z), f3 = unpack2(u.w);
          acc[0] += f0.x; acc[1] += f0.y; acc[2] += f1.x; acc[3] += f1.y;
          acc[4] += f2.x; acc[5] += f2.y; acc[6] += f3.x; acc[7] += f3.y;
        }
#pragma unroll
        for (int o = 1; o < 8; o <<= 1)
#pragma unroll
          for (int e = 0; e < 8; e++) acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], o);
        if (sub == 0) {
          float4* dst = reinterpret_cast<float4*>(p.pooled + (size_t)tile * kE + kc * 8);
          dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
          dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (warp == 6 && lane == 0) mbar_arrive(bar(B_YE));
      if (do_res) {
        ok = ok && mbar_wait(bar(B_D2F + s), (k >> 1) & 1, abort_flag, 0x420 | s);
        tc_fence_after();
        // HBM tile block = the A stage image [16][129][16 B]: row 128 is row 0 of the next tile (written by that
        // tile's row-0 thread) or the SAME-padding zero row at the end of an utterance (ops.py:51)
        uint8_t* og = p.out + (size_t)tile * kAStage;
        const int tpos = tile % p.tiles_per_utt;
        const bool dup = row == 0 && tpos != 0, zero_tail = row == kTile - 1 && tpos == p.tiles_per_utt - 1;
#pragma unroll 1
        for (int c2 = 0; c2 < 2 && ok; c2++) {
          float v[64];
          const uint32_t ta = tmem + 256 + s * 128 + c2 * 64 + ((uint32_t)(q * 32) << 16);
          tc_ld32(ta, v);
          tc_ld32(ta + 32, v + 32);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 8; j++) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
              const int c = c2 * 64 + j * 8 + 2 * e;
              w[e] = pack2_relu(v[j * 8 + 2 * e] + rbias[c], v[j * 8 + 2 * e + 1] + rbias[c + 1]);   // ops.py:49 of the next layer
            }
            const uint4 u = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(og + ((c2 * 8 + j) * kARows + row) * 16) = u;
            if (dup) *reinterpret_cast<uint4*>(og - kAStage + ((c2 * 8 + j) * kARows + kTile) * 16) = u;
            if (zero_tail) *reinterpret_cast<uint4*>(og + ((c2 * 8 + j) * kARows + kTile) * 16) = make_uint4(0, 0, 0, 0);
          }
        }
        tc_fence_before();
        asm volatile("bar.sync 2, 128;" ::: "memory");
        if (warp == 6 && lane == 0) mbar_arrive(bar(B_D2E + s));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0 && abort_flag[0]) { p.err[0] = 1; p.err[1] = abort_flag[1]; }
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
  }
}

// encoding[b, f, c] = bias'[c] + (1/P) * sum_l sum_ch (sum over the window's tiles of pooled[l][tile][ch]) * Wf[l][ch][c]
// One block per pooling window: the window's L*128 column sums are staged in shared memory (coalesced rows of 128
// floats), then 8 partial dot products per output channel.
__global__ void __launch_bounds__(256) k_enc_finish(const float* __restrict__ pooled, const float* __restrict__ wf,
                                                    const float* __restrict__ bf, float* __restrict__ out, int L, size_t n_tiles,
                                                    int tiles_per_utt, int frames, int tiles_per_win, int C, float inv_p) {
  extern __shared__ float sp[];                 // [L * 128]
  __shared__ float red[8][64];
  const int win = blockIdx.x, c0 = threadIdx.x & 31, part = threadIdx.x >> 5;
  const size_t tile0 = (size_t)(win / frames) * tiles_per_utt + (size_t)(win % frames) * tiles_per_win;
  for (int k = threadIdx.x; k < L * kE; k += 256) {
    const int l = k / kE, ch = k % kE;
    float s = 0.f;
    for (int j = 0; j < tiles_per_win; j++) s += __ldg(pooled + ((size_t)l * n_tiles + tile0 + j) * kE + ch);
    sp[k] = s;
  }
  __syncthreads();
  float acc0 = 0.f, acc1 = 0.f;
  const bool two = c0 + 32 < C;
  const int cc = c0 < C ? c0 : 0;
#pragma unroll 4
  for (int k = part; k < L * kE; k += 8) {
    const float s = sp[k];
    acc0 = fmaf(s, __ldg(wf + (size_t)k * C + cc), acc0);
    if (two) acc1 = fmaf(s, __ldg(wf + (size_t)k * C + c0 + 32), acc1);
  }
  red[part][c0] = acc0; red[part][c0 + 32] = acc1;
  __syncthreads();
  if (threadIdx.x < C) {
    float s = 0.f;
    for (int i = 0; i < 8; i++) s += red[i][threadIdx.x];
    out[(size_t)win * C + threadIdx.x] = fmaf(s, inv_p, bf[threadIdx.x]);
  }
}

// ---- fp32 parity path ----------------------------------------------------------------------------------
// y[row][c] = relu(relu(x[t]) * fk[0][c] + relu(x[t+1]) * fk[1][c] + fb[c])   (nc_conv, ops.py:49-52)
__global__ void k_enc_front_f32(const float* __restrict__ x, const float* __restrict__ fk, const float* __restrict__ fb,
                                float* __restrict__ y, size_t rows, int T, int E) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * E) return;
  const size_t r = i / E; const int c = (int)(i % E), t = (int)(r % T);
  const float a0 = fmaxf(x[r], 0.f), a1 = t + 1 < T ? fmaxf(x[r + 1], 0.f) : 0.f;
  y[i] = fmaxf(fmaf(a0, fk[c], fmaf(a1, fk[E + c], fb[c])), 0.f);
}

// out[row][n] (+)= sum_tap sum_k f(in[row + tap][k]) W[tap][k][n] + bias[n]; rows are (utterance, time) pairs and
// row + 1 exists only inside the same utterance.  64 rows x 64 columns per block, 256 threads, 4 x 4 per thread.
template <bool RELU_IN, int TAPS, bool RELU_OUT, bool ACCUM>
__global__ void __launch_bounds__(256) k_enc_gemm_f32(const float* __restrict__ in, const float* __restrict__ W,
                                                      const float* __restrict__ bias, float* __restrict__ out,
                                                      size_t rows, int T, int K, int N) {
  __shared__ float sa[16][64 + 4];
  __shared__ float sw[16][64 + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const size_t r0 = (size_t)blockIdx.x * 64;
  const int n0 = blockIdx.y * 64;
  float acc[4][4] = {};
  for (int tap = 0; tap < TAPS; tap++) {
    for (int k0 = 0; k0 < K; k0 += 16) {
      for (int i = threadIdx.x; i < 64 * 16; i += 256) {
        const int rr = i >> 4, kk = i & 15;
        const size_t r = r0 + rr;
        float v = 0.f;
        if (r < rows && k0 + kk < K) {
          const int t = (int)(r % T);
          if (t + tap < T) v = in[(r + tap) * K + k0 + kk];
          if (RELU_IN) v = fmaxf(v, 0.f);
        }
        sa[kk][rr] = v;
      }
      for (int i = threadIdx.x; i < 16 * 64; i += 256) {
        const int kk = i >> 6, nn = i & 63;
        sw[kk][nn] = (k0 + kk < K && n0 + nn < N) ? W[((size_t)tap * K + k0 + kk) * N + n0 + nn] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < 16; kk++) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { a[i] = sa[kk][ty * 4 + i]; b[i] = sw[kk][tx * 4 + i]; }
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  for (int i = 0; i < 4; i++) {
    const size_t r = r0 + ty * 4 + i;
    if (r >= rows) continue;
    for (int j = 0; j < 4; j++) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] + bias[n];
      if (RELU_OUT) v = fmaxf(v, 0.f);
      if (ACCUM) v += out[r * N + n];
      out[r * N + n] = v;
    }
  }
}

// encoding[b,f,:] = mean over the window of skipsum rows, then the latent 1x1 (model.py:152-154; both linear)
__global__ void k_enc_latent_pool_f32(const float* __restrict__ skipsum, const float* __restrict__ lk, const float* __restrict__ lb,
                                      float* __restrict__ enc, int T, int P, int frames, int S, int C) {
  extern __shared__ float mean[];
  const int b = blockIdx.x / frames, f = blockIdx.x % frames;
  const float* src = skipsum + ((size_t)b * T + (size_t)f * P) * S;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    float a = 0.f;
    for (int t = 0; t < P; t++) a += src[(size_t)t * S + s];
    mean[s] = a / (float)P;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = lb[c];
    for (int s = 0; s < S; s++) a = fmaf(mean[s], lk[(size_t)s * C + c], a);
    enc[((size_t)b * frames + f) * C + c] = a;
  }
}

}  // namespace enc

// ---- handle -------------------------------------------------------------------------------------------
struct srwn_encoder {
  srwn_encoder_config_t cfg;
  int L, E, S, C, P;
  // host copies, TF layout
  std::vector<float> front_k, front_b, conv_k, conv_b, res_k, res_b, skip_k, skip_b, lat_k, lat_b;
  std::vector<uint8_t> is_set;
  float* d_f32;                    // fp32 arena: all of the above, in that order
  size_t o_front_k, o_front_b, o_conv_k, o_conv_b, o_res_k, o_res_b, o_skip_k, o_skip_b, o_lat_k, o_lat_b, o_wf, o_bf, n_f32;
  uint8_t* d_img;                  // fp16 operands: front image | L layer images
  size_t img_bytes;
  bool committed;
  int sm_count;
  int profiling;
  cudaEvent_t ev[2];
};

static bool enc_tc_supported(const srwn_encoder* e) {
  return e->E == enc::kE && e->cfg.filter_width == 2 && e->P % enc::kTile == 0 && e->C <= 64;
}

extern "C" int srwn_encoder_create(const srwn_encoder_config_t* cfg, srwn_encoder_t* out) {
  if (!cfg || !out) return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_create: null argument");
  *out = nullptr;
  if (cfg->n_layers < 1 || cfg->n_layers > 256) return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_create: need 1..256 layers");
  if (cfg->filter_width != 2)
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "encoder kernels are built for filter_width=2 (teacher.py:59); got %d", cfg->filter_width);
  if (cfg->encoder_channels < 1 || cfg->encoder_channels > 1024 || cfg->skip_channels < 1 || cfg->skip_channels > 1024 ||
      cfg->latent_channels < 1 || cfg->latent_channels > 1024 || cfg->pool_stride < 1)
    return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_create: channel counts must be 1..1024 and pool_stride >= 1");
  srwn_encoder* e = new (std::nothrow) srwn_encoder();
  if (!e) return srwn_fail(SRWN_ERR_INVALID, "out of host memory");
  e->cfg = *cfg;
  e->L = cfg->n_layers; e->E = cfg->encoder_channels; e->S = cfg->skip_channels; e->C = cfg->latent_channels; e->P = cfg->pool_stride;
  const size_t L = e->L, E = e->E, S = e->S, C = e->C;
  e->front_k.assign(2 * E, 0.f); e->front_b.assign(E, 0.f);
  e->conv_k.assign(L * 2 * E * E, 0.f); e->conv_b.assign(L * E, 0.f);
  e->res_k.assign((L + 1) * E * E, 0.f); e->res_b.assign((L + 1) * E, 0.f);
  e->skip_k.assign(L * E * S, 0.f); e->skip_b.assign(L * S, 0.f);
  e->lat_k.assign(S * C, 0.f); e->lat_b.assign(C, 0.f);
  e->is_set.assign(2 + 2 * L + 2 * (L + 1) + 2 * L + 2, 0);
  size_t p = 0;
  auto take = [&](size_t n) { size_t r = p; p += (n + 63) & ~(size_t)63; return r; };
  e->o_front_k = take(2 * E); e->o_front_b = take(E);
  e->o_conv_k = take(L * 2 * E * E); e->o_conv_b = take(L * E);
  e->o_res_k = take((L + 1) * E * E); e->o_res_b = take((L + 1) * E);
  e->o_skip_k = take(L * E * S); e->o_skip_b = take(L * S);
  e->o_lat_k = take(S * C); e->o_lat_b = take(C);
  e->o_wf = take(L * E * C); e->o_bf = take(C);
  e->n_f32 = p;
  e->d_f32 = nullptr; e->d_img = nullptr; e->committed = false; e->profiling = 0; e->ev[0] = e->ev[1] = nullptr;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaMalloc(&e->d_f32, p * sizeof(float)) != cudaSuccess) {
    cudaGetLastError();
    delete e;
    return srwn_fail(SRWN_ERR_CUDA, "srwn_encoder_create: no CUDA device / allocation failed (there is no CPU fallback)");
  }
  cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, dev);
  e->img_bytes = (size_t)enc::kFrontImg + (size_t)e->L * enc::kLayerImg;
  if (enc_tc_supported(e) && cudaMalloc(&e->d_img, e->img_bytes) != cudaSuccess) {
    cudaGetLastError(); cudaFree(e->d_f32); delete e;
    return srwn_fail(SRWN_ERR_CUDA, "srwn_encoder_create: allocation failed");
  }
  cudaEventCreate(&e->ev[0]); cudaEventCreate(&e->ev[1]);
  *out = e;
  return SRWN_OK;
}

extern "C" int srwn_encoder_destroy(srwn_encoder_t e) {
  if (!e) return SRWN_OK;
  cudaFree(e->d_f32); cudaFree(e->d_img);
  if (e->ev[0]) cudaEventDestroy(e->ev[0]);
  if (e->ev[1]) cudaEventDestroy(e->ev[1]);
  delete e;
  return SRWN_OK;
}

// slot layout of is_set: 0 front_k, 1 front_b, 2+2i conv_k/conv_b (i<L), then res (L+1 pairs), skip (L pairs), latent pair
extern "C" int srwn_encoder_set_weight(srwn_encoder_t e, const char* name, const float* data, const int64_t* shape, int32_t ndim) {
  if (!e || !name || !data || !shape) return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_set_weight: null argument");
  const char* p = strstr(name, "/Encoder/");                  // "WaveNetAutoEncoder/Encoder/<variable>"
  const char* s = p ? p + 9 : (!strncmp(name, "Encoder/", 8) ? name + 8 : name);
  const int L = e->L, E = e->E, S = e->S, C = e->C;
  float* dst = nullptr; int64_t want[3] = {0, 0, 0}; int nd = 0; int slot = -1; size_t count = 0;
  auto kernel = [&](float* d, int64_t a, int64_t b, int64_t c, int sl) { dst = d; want[0] = a; want[1] = b; want[2] = c; nd = 3; slot = sl; count = (size_t)(a * b * c); };
  auto bias = [&](float* d, int64_t a, int sl) { dst = d; want[0] = a; nd = 1; slot = sl; count = (size_t)a; };
  int i = -1, n = 0;
  const int base_res = 2 + 2 * L, base_skip = base_res + 2 * (L + 1), base_lat = base_skip + 2 * L;
  if (!strcmp(s, "nc_conv_NC/conv1d/kernel")) kernel(e->front_k.data(), 2, 1, E, 0);
  else if (!strcmp(s, "nc_conv_NC/conv1d/bias")) bias(e->front_b.data(), E, 1);
  else if (sscanf(s, "dilated_conv_%d_NC/conv1d/%n", &i, &n) == 1 && n && i >= 0 && i < L) {
    if (!strcmp(s + n, "kernel")) kernel(e->conv_k.data() + (size_t)i * 2 * E * E, 2, E, E, 2 + 2 * i);
    else if (!strcmp(s + n, "bias")) bias(e->conv_b.data() + (size_t)i * E, E, 3 + 2 * i);
  } else {
    int idx = -1; const char* tail = nullptr;
    if (!strncmp(s, "conv1d/", 7)) { idx = 0; tail = s + 7; }
    else { n = 0; if (sscanf(s, "conv1d_%d/%n", &idx, &n) == 1 && n) tail = s + n; }
    if (tail && idx >= 0) {
      const bool is_k = !strcmp(tail, "kernel"), is_b = !strcmp(tail, "bias");
      if (is_k || is_b) {
        if (idx == 2 * (L + 1)) {
          if (is_k) kernel(e->lat_k.data(), 1, S, C, base_lat); else bias(e->lat_b.data(), C, base_lat + 1);
        } else if (idx < 2 * (L + 1)) {
          const int j = idx / 2;
          if (idx % 2 == 0) {
            if (is_k) kernel(e->res_k.data() + (size_t)j * E * E, 1, E, E, base_res + 2 * j);
            else bias(e->res_b.data() + (size_t)j * E, E, base_res + 2 * j + 1);
          } else if (j == 0) {
            return SRWN_OK;        // skip conv of nc_conv: created by the reference, discarded (model.py:141)
          } else {
            if (is_k) kernel(e->skip_k.data() + (size_t)(j - 1) * E * S, 1, E, S, base_skip + 2 * (j - 1));
            else bias(e->skip_b.data() + (size_t)(j - 1) * S, S, base_skip + 2 * (j - 1) + 1);
          }
        }
      }
    }
  }
  if (!dst) return srwn_fail(SRWN_ERR_WEIGHTS, "unknown encoder variable '%s'", name);
  bool shape_ok = ndim == nd;
  for (int d = 0; shape_ok && d < nd; d++) shape_ok = shape[d] == want[d];
  if (!shape_ok && nd == 1 && ndim == 3 && shape[0] == 1 && shape[1] == 1 && shape[2] == want[0]) shape_ok = true;
  if (!shape_ok) return srwn_fail(SRWN_ERR_WEIGHTS, "encoder variable '%s': unexpected shape", name);
  memcpy(dst, data, count * sizeof(float));
  e->is_set[slot] = 1;
  e->committed = false;
  return SRWN_OK;
}

static uint16_t enc_to_bits(float f) {
  __half h = __float2half_rn(f);
  return *reinterpret_cast<uint16_t*>(&h);
}
static inline size_t enc_kmajor(int n, int k, int rows) { return ((size_t)(k / 8) * rows + n) * 8 + (k % 8); }

extern "C" int srwn_encoder_commit(srwn_encoder_t e, void* stream) {
  if (!e) return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_commit: null handle");
  for (size_t i = 0; i < e->is_set.size(); i++)
    if (!e->is_set[i]) return srwn_fail(SRWN_ERR_WEIGHTS, "encoder variable slot %d was never set (model.py:137-155)", (int)i);
  cudaStream_t st = (cudaStream_t)stream;
  const int L = e->L, E = e->E, S = e->S, C = e->C;
  std::vector<float> host(e->n_f32, 0.f);
  auto put = [&](size_t off, const std::vector<float>& v) { memcpy(host.data() + off, v.data(), v.size() * sizeof(float)); };
  put(e->o_front_k, e->front_k); put(e->o_front_b, e->front_b); put(e->o_conv_k, e->conv_k); put(e->o_conv_b, e->conv_b);
  put(e->o_res_k, e->res_k); put(e->o_res_b, e->res_b); put(e->o_skip_k, e->skip_k); put(e->o_skip_b, e->skip_b);
  put(e->o_lat_k, e->lat_k); put(e->o_lat_b, e->lat_b);
  // folded skip -> latent matrices: Wf[l][ch][c] = sum_s Ws_l[ch][s] Wl[s][c];  bf[c] = bl[c] + sum_s (sum_l bs_l[s]) Wl[s][c]
  for (int l = 0; l < L; l++)
    for (int ch = 0; ch < E; ch++)
      for (int c = 0; c < C; c++) {
        double a = 0;
        for (int s = 0; s < S; s++) a += (double)e->skip_k[((size_t)l * E + ch) * S + s] * e->lat_k[(size_t)s * C + c];
        host[e->o_wf + ((size_t)l * E + ch) * C + c] = (float)a;
      }
  for (int c = 0; c < C; c++) {
    double a = e->lat_b[c];
    for (int s = 0; s < S; s++) {
      double bs = 0;
      for (int l = 0; l < L; l++) bs += e->skip_b[(size_t)l * S + s];
      a += bs * e->lat_k[(size_t)s * C + c];
    }
    host[e->o_bf + c] = (float)a;
  }
  SRWN_CUDA(cudaMemcpyAsync(e->d_f32, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  std::vector<uint8_t> img;
  if (e->d_img) {
    img.assign(e->img_bytes, 0);
    {  // front: res image | front_k[2][E] | front_b[E] | res bias[E]
      uint16_t* ri = reinterpret_cast<uint16_t*>(img.data());
      for (int k = 0; k < E; k++)
        for (int n = 0; n < E; n++) ri[enc_kmajor(n, k, E)] = enc_to_bits(e->res_k[(size_t)k * E + n]);
      float* f = reinterpret_cast<float*>(img.data() + enc::kResImg);
      memcpy(f, e->front_k.data(), 2 * E * sizeof(float));
      memcpy(f + 2 * E, e->front_b.data(), E * sizeof(float));
      memcpy(f + 3 * E, e->res_b.data(), E * sizeof(float));
    }
    for (int l = 0; l < L; l++) {
      uint8_t* lb = img.data() + enc::kFrontImg + (size_t)l * enc::kLayerImg;
      uint16_t* ci = reinterpret_cast<uint16_t*>(lb);
      uint16_t* ri = reinterpret_cast<uint16_t*>(lb + enc::kConvImg);
      const float* ck = e->conv_k.data() + (size_t)l * 2 * E * E;        // [tap][Cin][Cout]
      for (int k = 0; k < 2 * E; k++)
        for (int n = 0; n < E; n++) ci[enc_kmajor(n, k, E)] = enc_to_bits(ck[(size_t)k * E + n]);
      const float* rk = e->res_k.data() + (size_t)(l + 1) * E * E;
      for (int k = 0; k < E; k++)
        for (int n = 0; n < E; n++) ri[enc_kmajor(n, k, E)] = enc_to_bits(rk[(size_t)k * E + n]);
      float* f = reinterpret_cast<float*>(lb + enc::kConvImg + enc::kResImg);
      memcpy(f, e->conv_b.data() + (size_t)l * E, E * sizeof(float));
      memcpy(f + E, e->res_b.data() + (size_t)(l + 1) * E, E * sizeof(float));
    }
    SRWN_CUDA(cudaMemcpyAsync(e->d_img, img.data(), img.size(), cudaMemcpyHostToDevice, st));
  }
  SRWN_CUDA(cudaStreamSynchronize(st));
  e->committed = true;
  return SRWN_OK;
}

extern "C" int srwn_encoder_supports(srwn_encoder_t e, int32_t precision) {
  if (!e) return 0;
  if (precision == SRWN_FP32) return 1;
  return precision == SRWN_FP16 && enc_tc_supported(e) ? 1 : 0;   // bf16 operands are not offered (see srwn.h)
}

static size_t enc_ws_bytes(const srwn_encoder* e, int B, int T, int precision) {
  WsCarver w(nullptr, 0);
  const size_t rows = (size_t)B * T;
  if (precision == SRWN_FP32) {
    w.take<float>(rows * e->E); w.take<float>(rows * e->E); w.take<float>(rows * e->S);
  } else {
    const size_t n_tiles = rows / enc::kTile;
    w.take<uint8_t>(n_tiles * enc::kAStage); w.take<uint8_t>(n_tiles * enc::kAStage);
    w.take<float>((size_t)e->L * n_tiles * enc::kE);
    w.take<int>(64);
  }
  return w.used;
}

// what srwn_teacher_encode refuses of a precision (srwn_encoder_workspace_bytes refuses the same)
static int check_encode_precision(srwn_encoder_t e, int T, int precision) {
  if (!srwn_encoder_supports(e, precision))
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "encoder precision %d needs encoder_channels=128, pool_stride %% 128 == 0, latent <= 64", precision);
  if (precision != SRWN_FP32 && T % enc::kTile != 0)
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "the encoder's tensor-core path needs T %% 128 == 0 (got %d); use SRWN_FP32", T);
  return SRWN_OK;
}

extern "C" int srwn_encoder_workspace_bytes(srwn_encoder_t e, int32_t B, int32_t T, int32_t precision, size_t* bytes) {
  if (!e || !bytes || B < 1 || T < 1) return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_workspace_bytes: bad argument");
  if (int rc = check_encode_precision(e, T, precision)) return rc;
  *bytes = enc_ws_bytes(e, B, T, precision);
  return SRWN_OK;
}

template <bool FRONT>
static int launch_layer(const srwn_encoder* e, const enc::LayerParams& p, cudaStream_t st) {
  SRWN_CUDA(cudaFuncSetAttribute(enc::k_enc_layer<FRONT>, cudaFuncAttributeMaxDynamicSharedMemorySize, enc::Smem::total));
  const int grid = p.n_tiles < e->sm_count ? p.n_tiles : e->sm_count;
  enc::k_enc_layer<FRONT><<<grid, enc::kThreads, enc::Smem::total, st>>>(p);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

/* encode(inputs) (model.py:250-255): x [B,T] -> encoding [B, T/P, latent]. */
extern "C" int srwn_teacher_encode(srwn_encoder_t e, const float* x, float* enc_out, int32_t B, int32_t T, int32_t precision,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  if (!e || !x || !enc_out) return srwn_fail(SRWN_ERR_INVALID, "srwn_teacher_encode: null argument");
  if (!e->committed) return srwn_fail(SRWN_ERR_WEIGHTS, "srwn_teacher_encode: weights not committed");
  if (B < 1 || T < e->P) return srwn_fail(SRWN_ERR_INVALID, "srwn_teacher_encode: need B >= 1 and T >= pool_stride");
  if (int rc = check_encode_precision(e, T, precision)) return rc;
  if (int rc = check_workspace(workspace, workspace_bytes, enc_ws_bytes(e, B, T, precision))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int L = e->L, E = e->E, S = e->S, C = e->C, P = e->P, frames = T / P;
  const size_t rows = (size_t)B * T;
  const float* W = e->d_f32;
  WsCarver w(workspace, workspace_bytes);
  if (e->profiling) cudaEventRecord(e->ev[0], st);
  if (precision == SRWN_FP32) {
    float* h = w.take<float>(rows * E); float* y = w.take<float>(rows * E); float* skip = w.take<float>(rows * S);
    const unsigned rb = (unsigned)((rows + 63) / 64);
    enc::k_enc_front_f32<<<(unsigned)((rows * E + 255) / 256), 256, 0, st>>>(x, W + e->o_front_k, W + e->o_front_b, y, rows, T, E);
    SRWN_LAUNCH_CHECK();
    enc::k_enc_gemm_f32<false, 1, false, false><<<dim3(rb, (E + 63) / 64), 256, 0, st>>>(y, W + e->o_res_k, W + e->o_res_b, h, rows, T, E, E);
    SRWN_LAUNCH_CHECK();
    for (int l = 0; l < L; l++) {
      enc::k_enc_gemm_f32<true, 2, true, false><<<dim3(rb, (E + 63) / 64), 256, 0, st>>>(
          h, W + e->o_conv_k + (size_t)l * 2 * E * E, W + e->o_conv_b + (size_t)l * E, y, rows, T, E, E);
      SRWN_LAUNCH_CHECK();
      if (l + 1 < L) {   // the last layer's residual output is never read (model.py:147-151)
        enc::k_enc_gemm_f32<false, 1, false, false><<<dim3(rb, (E + 63) / 64), 256, 0, st>>>(
            y, W + e->o_res_k + (size_t)(l + 1) * E * E, W + e->o_res_b + (size_t)(l + 1) * E, h, rows, T, E, E);
        SRWN_LAUNCH_CHECK();
      }
      if (l == 0)
        enc::k_enc_gemm_f32<false, 1, false, false><<<dim3(rb, (S + 63) / 64), 256, 0, st>>>(
            y, W + e->o_skip_k, W + e->o_skip_b, skip, rows, T, E, S);
      else
        enc::k_enc_gemm_f32<false, 1, false, true><<<dim3(rb, (S + 63) / 64), 256, 0, st>>>(
            y, W + e->o_skip_k + (size_t)l * E * S, W + e->o_skip_b + (size_t)l * S, skip, rows, T, E, S);
      SRWN_LAUNCH_CHECK();
    }
    enc::k_enc_latent_pool_f32<<<B * frames, 128, S * sizeof(float), st>>>(skip, W + e->o_lat_k, W + e->o_lat_b, enc_out, T, P, frames, S, C);
    SRWN_LAUNCH_CHECK();
  } else {
    if (precision != SRWN_FP16) return srwn_fail(SRWN_ERR_UNSUPPORTED, "the tensor-core encoder is built for fp16 operands only; use SRWN_FP16 or SRWN_FP32");
    const size_t n_tiles = rows / enc::kTile;
    uint8_t* act0 = w.take<uint8_t>(n_tiles * enc::kAStage);
    uint8_t* act1 = w.take<uint8_t>(n_tiles * enc::kAStage);
    float* pooled = w.take<float>((size_t)L * n_tiles * enc::kE);
    int* err = w.take<int>(64);
    SRWN_CUDA(cudaMemsetAsync(err, 0, 64 * sizeof(int), st));
    const uint8_t* img = e->d_img;
    enc::LayerParams p;
    p.err = err; p.n_tiles = (int)n_tiles; p.tiles_per_utt = T / enc::kTile; p.T = T;
    p.img = img; p.in = nullptr; p.x = x; p.out = act0; p.pooled = nullptr; p.reverse = 0;
    int rc = launch_layer<true>(e, p, st);
    if (rc) return rc;
    uint8_t* cur = act0; uint8_t* nxt = act1;
    for (int l = 0; l < L; l++) {
      p.img = img + enc::kFrontImg + (size_t)l * enc::kLayerImg;
      p.in = cur; p.x = nullptr; p.out = l + 1 < L ? nxt : nullptr; p.pooled = pooled + (size_t)l * n_tiles * enc::kE;
      p.reverse = (l & 1) ^ 1;
      rc = launch_layer<false>(e, p, st);
      if (rc) return rc;
      uint8_t* t = cur; cur = nxt; nxt = t;
    }
    if ((size_t)L * enc::kE * sizeof(float) > 48 * 1024)
      SRWN_CUDA(cudaFuncSetAttribute(enc::k_enc_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, L * enc::kE * (int)sizeof(float)));
    enc::k_enc_finish<<<B * frames, 256, (size_t)L * enc::kE * sizeof(float), st>>>(pooled, W + e->o_wf, W + e->o_bf, enc_out, L, n_tiles, T / enc::kTile, frames, P / enc::kTile, C, 1.f / (float)P);
    SRWN_LAUNCH_CHECK();
  }
  if (e->profiling) cudaEventRecord(e->ev[1], st);
  return SRWN_OK;
}

/* Synchronises `stream` and reports whether a tensor-core encoder launch that used this workspace aborted. */
extern "C" int srwn_encoder_check_async_error(srwn_encoder_t e, int32_t B, int32_t T, int32_t precision, void* workspace,
                                              size_t workspace_bytes, void* stream) {
  if (!e || !workspace) return srwn_fail(SRWN_ERR_INVALID, "srwn_encoder_check_async_error: null argument");
  SRWN_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  if (precision == SRWN_FP32) return SRWN_OK;
  WsCarver w(workspace, workspace_bytes);
  const size_t n_tiles = (size_t)B * T / enc::kTile;
  w.take<uint8_t>(n_tiles * enc::kAStage); w.take<uint8_t>(n_tiles * enc::kAStage);
  w.take<float>((size_t)e->L * n_tiles * enc::kE);
  int* err = w.take<int>(64);
  int h[2] = {0, 0};
  SRWN_CUDA(cudaMemcpy(h, err, sizeof(h), cudaMemcpyDeviceToHost));
  if (h[0]) return srwn_fail(SRWN_ERR_CUDA, "encoder kernel aborted: a pipeline wait expired (code 0x%x)", h[1]);
  return SRWN_OK;
}

extern "C" int srwn_encoder_set_profiling(srwn_encoder_t e, int32_t enable) {
  if (!e) return srwn_fail(SRWN_ERR_INVALID, "null handle");
  e->profiling = enable;
  return SRWN_OK;
}
/* Elapsed time of the last srwn_teacher_encode call (all its launches), when profiling is enabled. */
extern "C" int srwn_encoder_last_ms(srwn_encoder_t e, float* ms) {
  if (!e || !ms) return srwn_fail(SRWN_ERR_INVALID, "null argument");
  SRWN_CUDA(cudaEventSynchronize(e->ev[1]));
  SRWN_CUDA(cudaEventElapsedTime(ms, e->ev[0], e->ev[1]));
  return SRWN_OK;
}
