// Autoregressive teacher generation on tensor cores (fp16 operands, fp32 accumulate / residual stream).
//
// Same recurrence as ar_generate.cu (the queue restatement of teacher.py:153-170), organised for the
// per-sample latency chain x[t] -> 30 gated layers -> head -> sampler -> x[t+1], which is what bounds
// this workload (BASELINE.json configs[3]: 256 utterances x 16000 strictly sequential steps):
//   * one CTA owns 8 utterances (rows 0..7 of the m16n8k16 tiles) for all T steps;
//   * CHAIN warp: the whole layer chain for those rows with warp-level mma.sync -- filter conv
//     [8x64]x[64x32], gate, residual 1x1 [8x32]x[32x32] -- with every chain weight (B fragments, 6 KB per
//     layer, 184 KB) resident in shared memory; accumulator fragments turn into the next A fragments in
//     registers, so a layer costs two short MMA bursts and one gate, no shared-memory round trip;
//   * SKIP warps (8): the skip 1x1 (ops.py:44) is off the chain -- the chain warp drops the gate output
//     c_l into a per-layer slot, the skip warps multiply it by Ws_l (16 skip channels per warp) and keep
//     the sum over layers (model.py:190) in accumulator registers; they then run the head's S->S conv
//     (model.py:193) cooperatively;
//   * PRODUCER warp: streams the skip / head weights (280 KB per step, L2 resident) through a 3-stage
//     cp.async.bulk ring;
//   * the chain warp finishes the head (S->4M), and 8 of its lanes run the mixture-of-logistics sampler
//     (ops.py:178-201) and feed x[t] back;
//   * dilation queues (fp16 images of each layer's input, 64 B per utterance and slot) live in global
//     memory / L2; the pop of layer l+2 is prefetched while layer l runs.
#include "common.cuh"
#include "mol.cuh"
#include <cuda_fp16.h>
#include <vector>
#include <cstdio>

const float* srwn_host_weights(srwn_ctx* c);
__global__ void k_cond(const float* __restrict__ enc, const float* __restrict__ cond_k,
                       const float* __restrict__ cond_b, float* __restrict__ cond,
                       int frames_total, int L, int C);
namespace fused {
__global__ void k_fold_bias(const float* __restrict__ cond, const float* __restrict__ front_b,
                            const float* __restrict__ res_b, float* __restrict__ cb, int L);
}

namespace armma {

constexpr int kU = 8;                         // utterances per CTA
constexpr int kMaxL = 30;                     // chain weights of 30 layers fill shared memory
constexpr int kChainLayerBytes = 4096 + 2048 + 128;   // Wf fragments | Wr fragments | filter bias (fp32)
constexpr int kItemBytes = 8192;              // one ring item: skip weights of a layer / a quarter of H1 / H2
constexpr int kStages = 3;
constexpr int kSlotBytes = 512;               // gate output of one layer: [lane][4 x b32]
constexpr int kThreads = 9 * 32;
constexpr int kChainWarps = 4, kProducerWarp = 4, kSkipWarps = 4;   // warps 0..3: chain (one per SMSP), 4: producer, 5..8: skip warps

struct Smem {
  static constexpr int chain = 0;
  static constexpr int ring = chain + kMaxL * kChainLayerBytes;          // 188160
  static constexpr int cslots = ring + kStages * kItemBytes;             // 212736
  static constexpr int misc = cslots + kMaxL * kSlotBytes;               // 228096
  // misc: front fk[64] fb.. (256 B) | head biases bsum[128] b1[128] b2[32] (1152 B) | logits [8][24] (768 B) | barriers
  static constexpr int front = misc;
  static constexpr int hbias = front + 256;
  static constexpr int logits = hbias + 1152;
  static constexpr int bars = logits + 768;
  static constexpr int n_bars = 2 * kStages + kMaxL + 2;
  static constexpr int flags = bars + n_bars * 8 + 16;     // per-layer step counters: gate slot l holds step (flag - 1)
  static constexpr int xslot = flags + kMaxL * 4;           // x[t] of the 8 utterances, chain warp 0 -> chain warps 1..3
  static constexpr int qofs = xslot + 64;                   // queue slot byte offsets, [2 step parities][kMaxL] ints
  static constexpr int tmem = qofs + 2 * kMaxL * 4;         // TMEM base address (tcgen05.alloc)
  static constexpr int hslot = (tmem + 16 + 15) / 16 * 16;  // residual-stream image of the current layer: [lane][4 x b32], one word per chain warp
  static constexpr int total = hslot + kSlotBytes;
};
static_assert(Smem::total <= 232448, "shared memory budget");

struct Params {
  const uint8_t* chain_w;     // [L][kChainLayerBytes]
  const uint8_t* stream;      // [L + 5][kItemBytes]
  const float* fixed;         // fk[64] | bsum[128] b1[128] b2[32]
  const float* cb;            // [B][frames][L+1][32] folded biases + conditioning (fused::k_fold_bias)
  uint8_t* queues;            // [grid][sum_d][kSlotBytes]
  const float* g1;            // [B][T][M]  -log(-log(u1))           (k_sampler_noise)
  const float* lg2;           // [B][T]     log(u2) - log(1 - u2)
  float* x_out;               // [B][T]
  float* logits_out;          // [B][T][4M] or null
  int* err;
  int B, T, L, P, frames, M, sum_d;
  int dil[kMaxL];
  int qoff[kMaxL];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool mbar_try(uint32_t a, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
               "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(a), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: a stuck pipeline raises the abort flag instead of hanging the GPU
__device__ __forceinline__ bool mbar_wait(uint32_t a, uint32_t parity, volatile int* abort_flag) {
  if (mbar_try(a, parity)) return true;
  const long long t0 = clock64();
  while (true) {
    if (mbar_try(a, parity)) return true;
    if (*abort_flag) return false;
    if (clock64() - t0 > 2000000000LL) { *abort_flag = 1; return false; }
  }
}
__device__ __forceinline__ void mbar_arrive(uint32_t a) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
// D(16x8, fp32) += A(16x16, fp16, row) * B(16x8, fp16, col); rows 8..15 of A are zero padding (a1 = a3 = 0)
__device__ __forceinline__ void mma8(float (&d)[2], uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  float z0 = 0.f, z1 = 0.f;
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(z0), "+f"(z1)
               : "r"(a0), "r"(0u), "r"(a2), "r"(0u), "r"(b0), "r"(b1));
}
// Same instruction with all four A registers named by the caller.  Rows 8..15 of A only reach rows 8..15 of D, which
// nobody reads, so a1 / a3 may hold anything: passing registers that already sit next to a0 / a2 (the neighbours
// inside a 128-bit load, or a quad the caller keeps alive) saves the moves that zero padding would cost.
__device__ __forceinline__ void mma8q(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// ops.py:28,33,36: f = tanh(a); f * sigmoid(f), sigmoid on [-1,1] as 0.5 + f*P(f^2) (error 1.5e-6)
__device__ __forceinline__ float gate(float a) {
  const float f = tanh_fast(a);
  const float s = f * f;
  float t = fmaf(s, 0.0017294071149080992f, -0.020638039335608482f);
  t = fmaf(s, t, 0.2499687224626541f);
  return fmaf(f, 0.5f, s * t);
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
// resident, read-only after setup: the compiler may hoist these loads (no volatile, no memory clobber)
__device__ __forceinline__ uint4 lds128_ro(uint32_t a) {
  uint4 v;
  asm("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}

// Tensor memory as a per-lane scratchpad (mma.sync leaves it unused): each chain warp keeps the folded bias +
// conditioning table of the current latent frame, 8 floats per lane and layer, in its own 32-lane quarter.
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float2 (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "f"(v[0].x), "f"(v[0].y), "f"(v[1].x), "f"(v[1].y), "f"(v[2].x), "f"(v[2].y), "f"(v[3].x), "f"(v[3].y) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float2 (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[2].x), "=f"(v[2].y), "=f"(v[3].x), "=f"(v[3].y)
               : "r"(taddr) : "memory");
}
// wait for the warp's tcgen05.ld; the operands tie the loaded registers to the wait so no use moves above it
__device__ __forceinline__ void tmem_wait_ld(float2 (&v)[4]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(v[0].x), "+f"(v[0].y), "+f"(v[1].x), "+f"(v[1].y), "+f"(v[2].x), "+f"(v[2].y), "+f"(v[3].x), "+f"(v[3].y)
               :: "memory");
}
constexpr int kTmemCols = 256;                 // (kMaxL + 1) * 8 = 248 columns used
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, float2& v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld2(float2& v) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(v.x), "+f"(v.y) :: "memory");
}
#ifdef SRWN_AR_TIMING
__device__ __forceinline__ long long clk_after(uint32_t dep) {      // clock read ordered after the value `dep` is ready
  long long t;
  asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "r"(dep) : "memory");
  return t;
}
#define AR_T(var, dep) const long long var = clk_after(dep)
#define AR_ACC(acc, expr) acc += (expr)
#else
#define AR_T(var, dep)
#define AR_ACC(acc, expr)
#endif

// The sampler's noise transforms (ops.py:187,197) do not depend on the logits: one elementwise pass ahead of the
// sequential kernel takes ~12 logarithms per sample off the per-step dependency chain.  Same operations and order
// as mol_sample_one (mol.cuh), so the samples are bit-identical to it.
__global__ void k_sampler_noise(const float* __restrict__ u1, const float* __restrict__ u2, float* __restrict__ g1,
                                float* __restrict__ lg2, int64_t n, int M) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n * M) g1[i] = -logf(-logf(u1[i]));
  if (i < n) { const float u = u2[i]; lg2[i] = logf(u) - logf(1.f - u); }
}

__global__ void __launch_bounds__(kThreads, 1) k_ar_mma(const Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, q = lane & 3;              // fragment row / column-pair index
  const int L = p.L, O = 4 * p.M;
  const int n_items = L;                              // ring items per step: the skip weights of each layer
  // hidden-layer exchange tiles (16 x 256 B used): behind the gate slots when there is room, else on top of
  // slots 0..15, which every skip warp has left by then (the 3-stage ring keeps them within 3 layers of each other)
  const int hid_slot = (L + 16 <= kMaxL) ? L : 0;
  volatile int* abort_flag = reinterpret_cast<volatile int*>(smem + Smem::bars + Smem::n_bars * 8);
  auto bar = [&](int i) { return sbase + Smem::bars + i * 8; };
  // barrier indices: wfull[3] | wempty[3] | cfull[L] | hid1 | hid2
  const int B_WFULL = 0, B_WEMPTY = kStages, B_CFULL = 2 * kStages, B_HID1 = 2 * kStages + kMaxL, B_HID2 = B_HID1 + 1;

  if (tid == 0) {
    for (int s = 0; s < kStages; s++) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(B_WFULL + s)), "r"(1));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(B_WEMPTY + s)), "r"(kSkipWarps));
    }
    for (int l = 0; l < kMaxL; l++) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(B_CFULL + l)), "r"(1));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(B_HID1)), "r"(kSkipWarps * 32));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar(B_HID2)), "r"(kSkipWarps * 32));
    *abort_flag = 0;
    for (int i = 0; i < 9; i++) reinterpret_cast<volatile float*>(smem + Smem::xslot)[i] = 0.f;
    for (int l = 0; l < kMaxL; l++) reinterpret_cast<volatile int*>(smem + Smem::flags)[l] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {  // resident chain weights + small constants
    const uint4* src = reinterpret_cast<const uint4*>(p.chain_w);
    uint4* dst = reinterpret_cast<uint4*>(smem + Smem::chain);
    for (int i = tid; i < L * kChainLayerBytes / 16; i += kThreads) dst[i] = src[i];
    float* sf = reinterpret_cast<float*>(smem + Smem::front);
    for (int i = tid; i < 64; i += kThreads) sf[i] = p.fixed[i];
    float* sh = reinterpret_cast<float*>(smem + Smem::hbias);
    for (int i = tid; i < 288; i += kThreads) sh[i] = p.fixed[64 + i];
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sbase + Smem::tmem), "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + Smem::tmem);

  const int b0 = blockIdx.x * kU;
  const bool pow2 = p.sum_d < 0;      // host encodes "all dilations are powers of two" in the sign
  const int sum_d = pow2 ? -p.sum_d : p.sum_d;

  if (warp == kProducerWarp) {
    // ================= producer: skip / head weights, L2 -> shared ring ===========================
    if (lane == 0) {
      long long it = 0;
      for (int t = 0; t < p.T; t++) {
        for (int i = 0; i < n_items; i++, it++) {
          const int s = (int)(it % kStages);
          if (!mbar_wait(bar(B_WEMPTY + s), (uint32_t)(((it / kStages) & 1) ^ 1), abort_flag)) { t = p.T; break; }
          asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar(B_WFULL + s)), "r"(kItemBytes) : "memory");
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(sbase + Smem::ring + s * kItemBytes), "l"(p.stream + (size_t)i * kItemBytes),
                         "r"(kItemBytes), "r"(bar(B_WFULL + s)) : "memory");
        }
      }
    }
    return;
  }
  if (warp < kChainWarps) {
    // ================= chain warps: warp j owns channels 8j..8j+7 (n-tile j) of the filter conv, the gate, the residual
    // conv and the fp32 residual stream; the warps exchange the stream's 16-bit image once per layer
    const int j = warp;
    const int cpos = (j == 1 ? 2 : j == 2 ? 1 : j) * 4;   // n-tile j's word inside a lane's 16 bytes of a gate slot: order {0, 2, 1, 3}
    auto chain_sync = [&]() { asm volatile("bar.sync 1, 128;" ::: "memory"); };
    const int bg = min(b0 + g, p.B - 1);               // utterance of fragment row g (clamped: padding rows repeat the last one)
    const float* cb_b = p.cb + (size_t)bg * p.frames * (L + 1) * 32 + 2 * q;
    uint8_t* qbase = p.queues + (size_t)blockIdx.x * sum_d * kSlotBytes + lane * 16;
    const float* sf = reinterpret_cast<const float*>(smem + Smem::front);
    volatile int* sq = reinterpret_cast<volatile int*>(smem + Smem::qofs);      // [2][kMaxL]: queue slot byte offsets, by step parity
    volatile float* sx = reinterpret_cast<volatile float*>(smem + Smem::xslot);
    float xm1 = 0.f, xm2 = 0.f;                         // x[t-1], x[t-2] of utterance g
    float h[4][2];                                      // layer-0 input (front conv): n-tile i, columns 8i+2q, 8i+2q+1 of row g
    uint32_t hA[4];                                     // its fp16 image, n-tile i = channels 8i+2q, 8i+2q+1 (A fragments: kt0 (0,1), kt1 (2,3))
    uint32_t hB[2];                                     // second copy of hA[2], hA[3]: a0 / a2 of the k-tile 1 quad
    uint32_t dm[6];                                     // don't-care registers that complete the k-tile 1 quads
#pragma unroll
    for (int i = 0; i < 6; i++) asm volatile("mov.u32 %0, %%laneid;" : "=r"(dm[i]));   // opaque to ptxas: a constant would be re-materialised per use
    long long it_base = 0;                              // ring item counter at the start of the step
    const int ub = b0 + lane;                           // sampler lanes 0..7 of warp 0: utterance b0+lane
    const bool samp = j == 0 && lane < kU && ub < p.B;
    bool ok = true;
    long long tm_a = 0, tm_b = 0, tm_c = 0, tm_d = 0;
    [[maybe_unused]] long long tl_conv = 0, tl_gate = 0, tl_sync = 0, tl_res = 0, tl_top = 0;

    // Queue pops (L2) run three layers ahead of their use, in three register sets that the layer loop (unrolled by
    // three) addresses by name: nothing is rotated through register moves, and a set is reloaded right after its
    // value is consumed, so whenever the warp waits for a pop every load in flight is at least a layer old (loads
    // share scoreboards: waiting for an old one also waits for the newest).
    // The folded bias + conditioning terms (8 floats per lane and layer) change once per latent frame: they live in
    // tensor memory, one table per chain warp, and come back with tcgen05.ld a layer ahead of their use.
    struct Pre { uint4 tap; int ofs; };
    Pre S0, S1, S2;
    uint4 h2w[4];                                       // H2 B fragments of logit n-tile j (warps 0..2), k-tile pairs 0..3
#pragma unroll
    for (int kp = 0; kp < 4; kp++)
      h2w[kp] = j < 3 ? *reinterpret_cast<const uint4*>(p.stream + (size_t)(L + 4) * kItemBytes + ((j * 4 + kp) * 512) + lane * 16)
                      : make_uint4(0u, 0u, 0u, 0u);
    float2 cb0[4];                                      // folded term of layer 0 (front bias + conditioning)
    const uint32_t tm = tmem_base + ((uint32_t)(j * 32) << 16);
    auto slot_of = [&](int l, int t) {
      const int d = p.dil[l];
      return (p.qoff[l] + (pow2 ? (t & (d - 1)) : (t % d))) * kSlotBytes;
    };
    auto prefetch = [&](Pre& S, int l, const volatile int* sqt) {      // pop of layer l: the slot holds h_l[t - d]
      S.ofs = sqt[l];
      S.tap = *reinterpret_cast<const uint4*>(qbase + S.ofs);
    };
    auto load_frame_table = [&](int frame) {            // cb [frame][0..L][32] of utterance g -> TMEM columns 8 li..8 li + 7
      const float* cbf = cb_b + (size_t)frame * (L + 1) * 32;
      for (int li = 0; li <= L; li++) {
        float2 v[4];
#pragma unroll
        for (int i = 0; i < 4; i++) v[i] = *reinterpret_cast<const float2*>(cbf + li * 32 + 8 * i);
        tmem_st8(tm + li * 8, v);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    };
    if (j == 0 && lane < L) sq[lane] = slot_of(lane, 0);
    chain_sync();
    prefetch(S0, 0, sq);
    prefetch(S1, 1, sq);
    prefetch(S2, 2, sq);

    for (int t = 0; t < p.T; t++, it_base += n_items) {
      const long long c0 = clock64();
      const volatile int* sqt = sq + (t & 1) * kMaxL;
      if (t % p.P == 0) load_frame_table(t / p.P);
      tmem_ld8(tm, cb0);
      // sampler noise of this step, already transformed (k_sampler_noise); latency hidden behind the layer chain
      float g1v[8], lg2v = 0.f;
#pragma unroll
      for (int m = 0; m < 8; m++) g1v[m] = (samp && m < p.M) ? __ldg(p.g1 + ((size_t)ub * p.T + t) * p.M + m) : 0.f;
      if (samp) lg2v = __ldg(p.lg2 + (size_t)ub * p.T + t);
      // queue slots of the next step, one lane per layer (read after the barriers of this step)
      if (j == 0 && lane < L) sq[((t + 1) & 1) * kMaxL + lane] = slot_of(lane, t + 1);
      // front: RightShift + K=2 causal conv on one channel (model.py:172-173) + bias + conditioning of layer 0
      tmem_wait_ld(cb0);
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const int c = 8 * i + 2 * q;
        h[i][0] = fmaf(xm2, sf[c], fmaf(xm1, sf[32 + c], cb0[i].x));
        h[i][1] = fmaf(xm2, sf[c + 1], fmaf(xm1, sf[32 + c + 1], cb0[i].y));
      }
#pragma unroll
      for (int i = 0; i < 4; i++) hA[i] = pack_h2(h[i][0], h[i][1]);
      hB[0] = pack_h2(h[2][0], h[2][1]); hB[1] = pack_h2(h[3][0], h[3][1]);
      float hj0 = j == 0 ? h[0][0] : j == 1 ? h[1][0] : j == 2 ? h[2][0] : h[3][0];      // this warp's part of the fp32 stream
      float hj1 = j == 0 ? h[0][1] : j == 1 ? h[1][1] : j == 2 ? h[2][1] : h[3][1];
      // filter-conv B fragments of this warp's n-tile: [taps k-tiles 0,1 | current k-tiles 2,3]
      uint4 wft = lds128_ro(sbase + Smem::chain + lane * 16 + (2 * j) * 512);
      uint4 wfc = lds128_ro(sbase + Smem::chain + lane * 16 + (2 * j + 1) * 512);

      // Register quads of the A operands (a0, a1, a2, a3); a1 / a3 are don't-care (see mma8q).  The 16 bytes a lane
      // keeps per queue slot / gate slot are ordered {k-tile 0: a0, k-tile 1: a0, k-tile 0: a2, k-tile 1: a2}, so the
      // 128-bit value IS the quad of k-tile 0 and the quad of k-tile 1 is two moves.
      auto layer = [&](const int l, Pre& S) {
        const uint32_t wl = sbase + Smem::chain + l * kChainLayerBytes + lane * 16;
        AR_T(t_0, hA[0]);
        float2 cbj;                                      // term added after this layer (index l + 1), this warp's two channels
        if (l + 1 < L) tmem_ld2(tm + (l + 1) * 8 + 2 * j, cbj);
        // ---- filter conv (ops.py:6-10), n-tile j: taps (W[0] on h[t-d]) and current (W[1] on h[t]) as two
        //      independent accumulation chains
        float acc[4] = {0.f, 0.f, 0.f, 0.f}, acc2[4] = {0.f, 0.f, 0.f, 0.f};
        mma8q(acc2, hA[0], hA[2], hA[1], hA[3], wfc.x, wfc.y);
        mma8q(acc, S.tap.x, S.tap.y, S.tap.z, S.tap.w, wft.x, wft.y);
        mma8q(acc2, hB[0], dm[0], hB[1], dm[1], wfc.z, wfc.w);
        mma8q(acc, S.tap.y, dm[2], S.tap.w, dm[3], wft.z, wft.w);
        AR_T(t_1, S.tap.x);
        AR_T(t_2, __float_as_uint(acc[0] + acc2[0]));
        const uint4 wrj = lds128_ro(wl + 4096 + j * 512); // residual B fragments of n-tile j: land while the gate runs
        // push h[t] (the slot held h[t-d] until now); every chain warp holds the same image
        if (j == 0) *reinterpret_cast<uint4*>(qbase + S.ofs) = make_uint4(hA[0], hA[2], hA[1], hA[3]);
        if (l + 3 < L) prefetch(S, l + 3, sqt);          // this set's next use: layer l + 3
        // ---- gate (ops.py:28,33,36) of this warp's 8 channels -> one word of the A fragments of the residual / skip convs
        {
          const float2 b = *reinterpret_cast<const float2*>(reinterpret_cast<const float*>(smem + Smem::chain + l * kChainLayerBytes + 6144) + 8 * j + 2 * q);
          const uint32_t cj = pack_h2(gate(acc[0] + acc2[0] + b.x), gate(acc[1] + acc2[1] + b.y));
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(sbase + Smem::cslots + l * kSlotBytes + lane * 16 + cpos), "r"(cj) : "memory");
        }
        AR_T(t_3, 0u);
        if (l + 1 < L) {                                 // next layer's filter-conv fragments
          wft = lds128_ro(wl + kChainLayerBytes + (2 * j) * 512);
          wfc = lds128_ro(wl + kChainLayerBytes + (2 * j + 1) * 512);
        }
        chain_sync();                                    // the four words of every lane's slot are in place
        AR_T(t_4, 0u);
        if (j == 0 && lane == 0) mbar_arrive(bar(B_CFULL + l));      // release: the skip warps may read the slot
        // The output of the last layer is not used (model.py:183-190: only the skips reach the head), so its residual conv
        // is skipped.  Otherwise warp j computes n-tile j of the residual conv (two dependent MMAs instead of eight),
        // updates its two channels of the fp32 stream and the four warps exchange the 16-bit image through one slot.
        if (l + 1 < L) {
          const uint4 cA = lds128(sbase + Smem::cslots + l * kSlotBytes + lane * 16);     // {c n-tile 0, 2, 1, 3}
          float r[4] = {0.f, 0.f, 0.f, 0.f};
          mma8q(r, cA.x, cA.y, cA.z, cA.w, wrj.x, wrj.y);
          mma8q(r, cA.y, dm[4], cA.w, dm[5], wrj.z, wrj.w);
          tmem_wait_ld2(cbj);
          hj0 = fmaf(hj0 + r[0], SRWN_SQRT_HALF, cbj.x);
          hj1 = fmaf(hj1 + r[1], SRWN_SQRT_HALF, cbj.y);
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(sbase + Smem::hslot + lane * 16 + cpos), "r"(pack_h2(hj0, hj1)) : "memory");
          chain_sync();
          const uint4 hq = lds128(sbase + Smem::hslot + lane * 16);                       // {h n-tile 0, 2, 1, 3}
          hA[0] = hq.x; hA[2] = hq.y; hA[1] = hq.z; hA[3] = hq.w; hB[0] = hq.y; hB[1] = hq.w;
        }
        AR_T(t_5, hA[0] ^ hA[3]);
        AR_ACC(tl_top, t_1 - t_0); AR_ACC(tl_conv, t_2 - t_1); AR_ACC(tl_gate, t_3 - t_2); AR_ACC(tl_sync, t_4 - t_3); AR_ACC(tl_res, t_5 - t_4);
      };
      {
        int l = 0;
        for (; l + 3 <= L; l += 3) { layer(l, S0); layer(l + 1, S1); layer(l + 2, S2); }
        if (l < L) { layer(l, S0); if (l + 1 < L) layer(l + 1, S1); }
      }
      // pops of the next step's first three layers: their latency hides behind the head
      if (t + 1 < p.T) {
        const volatile int* sqn = sq + ((t + 1) & 1) * kMaxL;
        prefetch(S0, 0, sqn);
        prefetch(S1, 1, sqn);
        prefetch(S2, 2, sqn);
      }

      // ---- head, last stage: relu(hidden) @ H2 -> logits (model.py:194-196), chain warp i < 3 owns logit n-tile i with
      //      its H2 fragments resident in registers (nothing to fetch on the critical path); then the sampler ----------
      float xs = 0.f;
      const long long c1 = clock64();
      long long c2 = c1;
      if (j < 3) {
        ok = ok && mbar_wait(bar(B_HID2), (uint32_t)(t & 1), abort_flag);
        c2 = clock64();
        float lgA[4] = {0.f, 0.f, 0.f, 0.f}, lgB[4] = {0.f, 0.f, 0.f, 0.f};      // two accumulation chains
        const uint32_t hb = sbase + Smem::cslots + (hid_slot + 8) * kSlotBytes + lane * 8;   // hid2 tiles
#pragma unroll
        for (int kp = 0; kp < 4; kp++) {
          const uint2 a0 = lds64(hb + (2 * kp) * kSlotBytes), a1 = lds64(hb + (2 * kp + 1) * kSlotBytes);
          if (kp & 1) {
            mma8q(lgB, a0.x, dm[0], a0.y, dm[1], h2w[kp].x, h2w[kp].y);
            mma8q(lgB, a1.x, dm[2], a1.y, dm[3], h2w[kp].z, h2w[kp].w);
          } else {
            mma8q(lgA, a0.x, dm[0], a0.y, dm[1], h2w[kp].x, h2w[kp].y);
            mma8q(lgA, a1.x, dm[2], a1.y, dm[3], h2w[kp].z, h2w[kp].w);
          }
        }
        const float* b2 = reinterpret_cast<const float*>(smem + Smem::hbias) + 256;
        float* slw = reinterpret_cast<float*>(smem + Smem::logits) + g * 24 + 8 * j + 2 * q;
        slw[0] = (lgA[0] + lgB[0]) + b2[8 * j + 2 * q];
        slw[1] = (lgA[1] + lgB[1]) + b2[8 * j + 2 * q + 1];
      }
      chain_sync();                                       // the three logit n-tiles are in shared memory
      if (j == 0) {
        if (samp) {
          // ops.py:178-201 on the transformed noise: Gumbel-argmax mixture pick, logistic inverse CDF, clip
          const float* sl = reinterpret_cast<const float*>(smem + Smem::logits) + lane * 24;
          int k = 0;
          float best = -INFINITY;
#pragma unroll
          for (int m = 0; m < 8; m++) {
            if (m < p.M) {
              const float v = sl[m] + g1v[m];                             // ops.py:187
              if (v > best) { best = v; k = m; }
            }
          }
          const float mean = sl[p.M + k];
          const float ls = fmaxf(sl[2 * p.M + k], -7.f);                  // ops.py:192
          xs = fminf(fmaxf(fmaf(expf(ls), lg2v, mean), -1.f), 1.f);       // ops.py:197-199
          p.x_out[(size_t)ub * p.T + t] = xs;
          if (p.logits_out) {
            float* dst = p.logits_out + ((size_t)ub * p.T + t) * O;
            for (int i = 0; i < O; i++) dst[i] = sl[i];
          }
        }
        if (lane < kU) sx[lane] = xs;
        if (!ok) sx[8] = -1.f;                            // tells the other chain warps to stop
      }
      const long long c3 = clock64();
      chain_sync();
      xm2 = xm1;
      xm1 = sx[g];
      tm_a += c1 - c0; tm_b += c2 - c1; tm_c += c3 - c2; tm_d += clock64() - c3;
      if (sx[8] < 0.f) break;
    }
#ifdef SRWN_AR_TIMING
    if (lane == 0 && blockIdx.x == 0) {
      printf("chain warp %d: layers %lld clk/step, wait hid2 %lld, head+sampler %lld, final sync %lld\n", j, tm_a / p.T, tm_b / p.T, tm_c / p.T, tm_d / p.T);
      const long long n = (long long)p.T * L;
      printf("chain warp %d per layer: wait tap %lld, conv mma %lld, gate+store %lld, sync %lld, residual %lld\n", j, tl_top / n, tl_conv / n, tl_gate / n, tl_sync / n, tl_res / n);
    }
#endif
    if (j == 0 && lane == 0 && *abort_flag) atomicExch(p.err, 1);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    chain_sync();
    if (j == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols));
    }
    return;
  }

  // ================= skip warps: skip 1x1 summed over layers, then the S->S conv of the head =========
  // Transposed GEMMs: the WEIGHTS are the A operand (16 output channels x 16 inputs: every row of the tile is used) and the
  // 8 utterances are the N dimension, so a warp owns 32 output channels with 2 MMAs per k-tile and no padded rows --
  // half the tensor-pipe work of the row-major form, on pipes the chain warps share.  The B fragment of c^T is the same
  // register pair as the A fragment of c (b0 = a0, b1 = a2), so the gate slot is read as it is.
  const int sw = warp - 5;                                // warps 5..8 -> 0..3: skip / hidden channels 32 sw .. 32 sw + 31
  const float* shb = reinterpret_cast<const float*>(smem + Smem::hbias);
  long long it = 0;
  uint4 h1a[2][8];                                        // H1^T A fragments of this warp's two m-tiles, resident: [m-tile][k-tile]
#pragma unroll
  for (int mt = 0; mt < 2; mt++)
#pragma unroll
    for (int kt = 0; kt < 8; kt++)
      h1a[mt][kt] = *reinterpret_cast<const uint4*>(p.stream + (size_t)L * kItemBytes + (size_t)(((sw * 2 + mt) * 8 + kt) * 512) + lane * 16);
  // where a value (channel c = 16 kt + cc, utterance u) goes inside k-tile kt of a hidden-layer exchange tile so that lane
  // (g', q') of a consumer finds {(k = 2q', 2q'+1; u = g'), (k = 2q'+8, 2q'+9; u = g')}: the B fragment of hidden^T and,
  // equally, the (a0, a2) pair of the row-major A fragment the chain warps use for the last conv
  auto hid_ofs = [&](int c, int u) { const int cc = c & 15; return (c >> 4) * kSlotBytes + (u * 4 + ((cc & 7) >> 1)) * 8 + (cc >> 3) * 4 + (cc & 1) * 2; };
  for (int t = 0; t < p.T; t++) {
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};   // skip sum (model.py:190): [m-tile]{(ch g, utt 2q), (g, 2q+1), (g+8, 2q), (g+8, 2q+1)}
    bool ok = true;
    for (int l = 0; l < L && ok; l++, it++) {
      const int st = (int)(it % kStages);
      ok = mbar_wait(bar(B_WFULL + st), (uint32_t)((it / kStages) & 1), abort_flag) &&
           mbar_wait(bar(B_CFULL + l), (uint32_t)(t & 1), abort_flag);      // suspended, not spinning: the chain warps share the SMSPs
      if (!ok) break;
      const uint4 c = lds128(sbase + Smem::cslots + l * kSlotBytes + lane * 16);   // gate output, n-tiles {0, 2, 1, 3}
      const uint32_t wb = sbase + Smem::ring + st * kItemBytes + sw * 2048 + lane * 16;   // [m-tile][k-tile][lane][16 B]
      const uint4 w00 = lds128(wb), w01 = lds128(wb + 512), w10 = lds128(wb + 1024), w11 = lds128(wb + 1536);
      mma8q(acc[0], w00.x, w00.y, w00.z, w00.w, c.x, c.z);
      mma8q(acc[1], w10.x, w10.y, w10.z, w10.w, c.x, c.z);
      mma8q(acc[0], w01.x, w01.y, w01.z, w01.w, c.y, c.w);
      mma8q(acc[1], w11.x, w11.y, w11.z, w11.w, c.y, c.w);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(B_WEMPTY + st));
    }
    if (!ok) break;
    // relu(sum of skips + summed skip biases) -> hidden^T tiles of the S->S conv (model.py:190-193)
    {
      uint8_t* hb1 = smem + Smem::cslots + hid_slot * kSlotBytes;
#pragma unroll
      for (int mt = 0; mt < 2; mt++) {
        const int c0 = 32 * sw + 16 * mt + g;
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int ch = c0 + (e >> 1) * 8, u = 2 * q + (e & 1);
          *reinterpret_cast<__half*>(hb1 + hid_ofs(ch, u)) = __float2half_rn(fmaxf(acc[mt][e] + shb[ch], 0.f));
        }
      }
      mbar_arrive(bar(B_HID1));
    }
    if (!mbar_wait(bar(B_HID1), (uint32_t)(t & 1), abort_flag)) break;
    float hd[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}}, he[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
    for (int kt = 0; kt < 8; kt++) {                    // S -> S conv of the head (model.py:193): two chains per m-tile
      const uint2 b = lds64(sbase + Smem::cslots + (hid_slot + kt) * kSlotBytes + lane * 8);
      if (kt & 1) {
        mma8q(he[0], h1a[0][kt].x, h1a[0][kt].y, h1a[0][kt].z, h1a[0][kt].w, b.x, b.y);
        mma8q(he[1], h1a[1][kt].x, h1a[1][kt].y, h1a[1][kt].z, h1a[1][kt].w, b.x, b.y);
      } else {
        mma8q(hd[0], h1a[0][kt].x, h1a[0][kt].y, h1a[0][kt].z, h1a[0][kt].w, b.x, b.y);
        mma8q(hd[1], h1a[1][kt].x, h1a[1][kt].y, h1a[1][kt].z, h1a[1][kt].w, b.x, b.y);
      }
    }
    {
      uint8_t* hb2 = smem + Smem::cslots + (hid_slot + 8) * kSlotBytes;
#pragma unroll
      for (int mt = 0; mt < 2; mt++) {
        const int c0 = 32 * sw + 16 * mt + g;
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int ch = c0 + (e >> 1) * 8, u = 2 * q + (e & 1);
          *reinterpret_cast<__half*>(hb2 + hid_ofs(ch, u)) = __float2half_rn(fmaxf(hd[mt][e] + he[mt][e] + shb[128 + ch], 0.f));
        }
      }
      mbar_arrive(bar(B_HID2));
    }
  }
}

}  // namespace armma

// ---- host -------------------------------------------------------------------------------------------
static inline uint16_t h16(float f) { __half h = __float2half_rn(f); return *reinterpret_cast<uint16_t*>(&h); }

// B fragment pair of W [K][N] (row stride ld) for n-tile nt and k-tiles kt, kt+1, as the 16 bytes lane (g,q) loads:
// {b0(kt), b1(kt), b0(kt+1), b1(kt+1)}, b0 = (W[16kt+2q][n], W[16kt+2q+1][n]), b1 = rows +8, n = 8nt+g
static void pack_frag_pair(uint8_t* dst, const float* W, int ld, int K, int N, int kt, int nt) {
  uint16_t* o = reinterpret_cast<uint16_t*>(dst);
  for (int lane = 0; lane < 32; lane++) {
    const int g = lane >> 2, q = lane & 3, n = 8 * nt + g;
    for (int half = 0; half < 2; half++) {
      const int k0 = 16 * (kt + half) + 2 * q;
      const int ks[4] = {k0, k0 + 1, k0 + 8, k0 + 9};
      for (int e = 0; e < 4; e++) {
        const float v = (ks[e] < K && n < N) ? W[(size_t)ks[e] * ld + n] : 0.f;
        o[lane * 8 + half * 4 + e] = h16(v);
      }
    }
  }
}

// A fragment of W^T for the transposed GEMMs (W is [K][N], row stride ld): m-tile = output channels ch0 .. ch0 + 15,
// k-tile kt; the 16 bytes lane (g, q) loads are {a0, a1, a2, a3} = {(row g, k 2q..2q+1), (row g+8, same k),
// (row g, k 2q+8..2q+9), (row g+8, same k)} with A[row][k] = W[16 kt + k][ch0 + row]
static void pack_frag_a_t(uint8_t* dst, const float* W, int ld, int kt, int ch0) {
  uint16_t* o = reinterpret_cast<uint16_t*>(dst);
  for (int lane = 0; lane < 32; lane++) {
    const int g = lane >> 2, q = lane & 3;
    const int rows[4] = {g, g + 8, g, g + 8}, ks[4] = {2 * q, 2 * q, 2 * q + 8, 2 * q + 8};
    for (int r = 0; r < 4; r++)
      for (int e = 0; e < 2; e++) o[lane * 8 + r * 2 + e] = h16(W[(size_t)(16 * kt + ks[r] + e) * ld + ch0 + rows[r]]);
  }
}

bool ar_mma_supported(const srwn_ctx* c) {
  return c->cfg.kind == SRWN_TEACHER && c->cfg.n_layers >= 3 && c->cfg.n_layers <= armma::kMaxL && (c->cfg.n_layers <= armma::kMaxL - 16 || c->cfg.n_layers >= 20) && 4 * c->cfg.num_mixtures <= 24 &&
         c->cfg.num_mixtures <= 8;
}

static size_t ar_mma_image_bytes(const srwn_ctx* c) {
  return (size_t)c->cfg.n_layers * armma::kChainLayerBytes + (size_t)(c->cfg.n_layers + 5) * armma::kItemBytes + 352 * 4;
}

int ar_mma_pack_weights(srwn_ctx* c, cudaStream_t st) {
  if (!ar_mma_supported(c)) return SRWN_OK;
  const int L = c->cfg.n_layers, O = 4 * c->cfg.num_mixtures;
  const size_t n = ar_mma_image_bytes(c);
  if (!c->d_ar_packed) SRWN_CUDA(cudaMalloc(&c->d_ar_packed, n));
  std::vector<uint8_t> host(n, 0);
  const float* w = srwn_host_weights(c);
  const StackOffsets& o = c->off;
  uint8_t* chain = host.data();
  uint8_t* stream = chain + (size_t)L * armma::kChainLayerBytes;
  float* fixed = reinterpret_cast<float*>(stream + (size_t)(L + 5) * armma::kItemBytes);
  for (int l = 0; l < L; l++) {
    uint8_t* cl = chain + (size_t)l * armma::kChainLayerBytes;
    const float* fk = w + o.filt_k + (size_t)l * 2 * kR * kR;      // [2][Cin][Cout] = K 64 x N 32
    for (int j = 0; j < 4; j++) {
      pack_frag_pair(cl + (2 * j) * 512, fk, kR, 64, 32, 0, j);
      pack_frag_pair(cl + (2 * j + 1) * 512, fk, kR, 64, 32, 2, j);
    }
    const float* rk = w + o.res_k + (size_t)l * kR * kR;
    for (int j = 0; j < 4; j++) pack_frag_pair(cl + 4096 + j * 512, rk, kR, 32, 32, 0, j);
    memcpy(cl + 6144, w + o.filt_b + (size_t)l * kR, 32 * 4);
    uint8_t* it = stream + (size_t)l * armma::kItemBytes;           // skip weights, transposed: [warp][m-tile][k-tile]
    const float* sk = w + o.skip_k + (size_t)l * kR * kS;
    for (int sw = 0; sw < 4; sw++)
      for (int mt = 0; mt < 2; mt++)
        for (int kt = 0; kt < 2; kt++) pack_frag_a_t(it + ((sw * 2 + mt) * 2 + kt) * 512, sk, kS, kt, 32 * sw + 16 * mt);
  }
  {                                                                  // H1, transposed: [warp][m-tile][k-tile], 32 KB = items L..L+3
    uint8_t* it = stream + (size_t)L * armma::kItemBytes;
    for (int sw = 0; sw < 4; sw++)
      for (int mt = 0; mt < 2; mt++)
        for (int kt = 0; kt < 8; kt++) pack_frag_a_t(it + ((sw * 2 + mt) * 8 + kt) * 512, w + o.head1_k, kS, kt, 32 * sw + 16 * mt);
  }
  {                                                                  // H2: [n-tile][k-tile pair]
    uint8_t* it = stream + (size_t)(L + 4) * armma::kItemBytes;
    for (int j = 0; j < 3; j++)
      for (int kp = 0; kp < 4; kp++) pack_frag_pair(it + (j * 4 + kp) * 512, w + o.head2_k, O, 128, O, 2 * kp, j);
  }
  memcpy(fixed, w + o.front_k, 64 * 4);
  memcpy(fixed + 64, w + o.skip_b_sum, 128 * 4);
  memcpy(fixed + 192, w + o.head1_b, 128 * 4);
  for (int j = 0; j < O; j++) fixed[320 + j] = w[o.head2_b + j];
  SRWN_CUDA(cudaMemcpyAsync(c->d_ar_packed, host.data(), n, cudaMemcpyHostToDevice, st));
  SRWN_CUDA(cudaStreamSynchronize(st));
  return SRWN_OK;
}

struct ArMmaWs { uint8_t* queues; float *cond, *cb, *g1, *lg2; int* err; size_t bytes; int grid; };

static ArMmaWs carve_ar_mma(const srwn_ctx* c, int B, int T, void* ws, size_t cap) {
  WsCarver w(ws, cap);
  ArMmaWs r{};
  const size_t frames = T / c->cfg.pool_stride, L = c->cfg.n_layers;
  r.grid = (B + armma::kU - 1) / armma::kU;
  r.queues = w.take<uint8_t>((size_t)r.grid * c->sum_dilation * armma::kSlotBytes);
  r.cond = w.take<float>((size_t)B * frames * L * 32);
  r.cb = w.take<float>((size_t)B * frames * (L + 1) * 32);
  r.g1 = w.take<float>((size_t)B * T * c->cfg.num_mixtures);
  r.lg2 = w.take<float>((size_t)B * T);
  r.err = w.take<int>(4);
  r.bytes = w.used;
  return r;
}

size_t ar_mma_workspace_bytes(const srwn_ctx* c, int B, int T) { return carve_ar_mma(c, B, T, nullptr, 0).bytes; }

int run_ar_mma(srwn_ctx* c, const float* enc, const float* u1, const float* u2, float* x_out,
               float* logits_out, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (!ar_mma_supported(c) || !c->d_ar_packed)
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "fp16 generation kernel supports up to %d layers and 6 mixtures", armma::kMaxL);
  ArMmaWs w = carve_ar_mma(c, B, T, ws, ws_bytes);
  if (!ws || w.bytes > ws_bytes) return srwn_fail(SRWN_ERR_WORKSPACE, "workspace too small: need %zu bytes", w.bytes);
  const int L = c->cfg.n_layers, frames = T / c->cfg.pool_stride;
  SRWN_CUDA(cudaMemsetAsync(w.queues, 0, (size_t)w.grid * c->sum_dilation * armma::kSlotBytes, st));   // zero padding of ops.py:9
  SRWN_CUDA(cudaMemsetAsync(w.err, 0, 16, st));
  const float* sw = stack_w(c, 0);
  k_cond<<<B * frames, 256, 0, st>>>(enc, sw + c->off.cond_k, sw + c->off.cond_b, w.cond, B * frames, L, c->cfg.cond_channels);
  SRWN_LAUNCH_CHECK();
  fused::k_fold_bias<<<B * frames, 256, 0, st>>>(w.cond, sw + c->off.front_b, sw + c->off.res_b, w.cb, L);
  SRWN_LAUNCH_CHECK();
  {
    const int64_t n = (int64_t)B * T, nm = n * c->cfg.num_mixtures;
    armma::k_sampler_noise<<<(unsigned)((nm + 255) / 256), 256, 0, st>>>(u1, u2, w.g1, w.lg2, n, c->cfg.num_mixtures);
    SRWN_LAUNCH_CHECK();
  }
  armma::Params p;
  memset(&p, 0, sizeof(p));
  const uint8_t* img = reinterpret_cast<const uint8_t*>(c->d_ar_packed);
  p.chain_w = img;
  p.stream = img + (size_t)L * armma::kChainLayerBytes;
  p.fixed = reinterpret_cast<const float*>(p.stream + (size_t)(L + 5) * armma::kItemBytes);
  p.cb = w.cb; p.queues = w.queues; p.g1 = w.g1; p.lg2 = w.lg2; p.x_out = x_out; p.logits_out = logits_out; p.err = w.err;
  p.B = B; p.T = T; p.L = L; p.P = c->cfg.pool_stride; p.frames = frames; p.M = c->cfg.num_mixtures;
  bool pow2 = true;
  int off = 0;
  for (int l = 0; l < L; l++) {
    p.dil[l] = c->dilations[l]; p.qoff[l] = off; off += c->dilations[l];
    if (c->dilations[l] & (c->dilations[l] - 1)) pow2 = false;
  }
  p.sum_d = pow2 ? -c->sum_dilation : c->sum_dilation;
  SRWN_CUDA(cudaFuncSetAttribute(armma::k_ar_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, armma::Smem::total));
  ProfScope prof(c, st, "k_ar_mma", 1);
  armma::k_ar_mma<<<w.grid, armma::kThreads, armma::Smem::total, st>>>(p);
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

int ar_mma_check_error(const srwn_ctx* c, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st) {
  ArMmaWs w = carve_ar_mma(c, B, T, ws, ws_bytes);
  int flag = 0;
  SRWN_CUDA(cudaStreamSynchronize(st));
  SRWN_CUDA(cudaMemcpy(&flag, w.err, sizeof(int), cudaMemcpyDeviceToHost));
  if (flag) return srwn_fail(SRWN_ERR_CUDA, "generation kernel aborted: pipeline wait timed out");
  return SRWN_OK;
}
