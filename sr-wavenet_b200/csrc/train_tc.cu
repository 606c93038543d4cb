// Student training pass, layer kernels on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM).
//
// The three per-layer kernels of the distillation step (model.py:356-401 differentiates model.py:415-535; block = ops.py:23-46):
//   k_fwd_layer_tc   x_{l+1} = (x_l + c Wr + br) sqrt(1/2) + cond_{l+1},  c = f sigmoid(f),  f = tanh([x_l[t-d] | x_l[t]] Wf + bf)
//   k_bwd_gate_tc    da = dL/da (a = pre-activation of the filter conv), dWr, dbr        (recomputes a, f, c from x_l)
//   k_bwd_conv_tc    dx_l = g sqrt(1/2) + da W1^T + da[t+d] W0^T, dWf, dbf, dcond_l
//
// Tile = 128 time steps = the M of one MMA; 512 worker threads (thread = (row, quarter of the 32 channels): four warps per
// scheduler hide the latencies of the epilogue math) plus two issuing warps (a tcgen05.mma costs its issuing thread 60-120
// clocks: 16-40 instructions per tile would otherwise sit on the workers' critical path); one persistent CTA per SM.
// fp32 grade on TF32 tensor cores: every operand is split x = hi + lo into two TF32 numbers by truncation (x - hi is exact)
// and a product is hi*hi + hi*lo + lo*hi.  The two terms that share the A operand come out of ONE instruction by stacking
// [W_hi ; W_lo] along N (N = 64), so a GEMM costs two instruction chains instead of three:
//     D[:, 0:32] = A_hi W_hi    D[:, 32:64] = A_hi W_lo    D[:, 64:96] = A_lo W_hi      (summed by the epilogue)
// The two chains write separate accumulator columns (the first instruction of each overwrites), so they need no order
// between them; the pipe takes ~47 (N = 32) / ~57 (N = 64) clocks per instruction (tools/umma_tf32_probe.cu) -- the time to
// read its 5-6 KB of operands from shared memory, which is what bounds these kernels (DESIGN.md 4.5).
// Weight gradients contract over TIME: both operands are needed transposed, [channel][time].  MN-major TF32 operands only
// exist for the 128B_BASE32B swizzle (the probe's no-swizzle MN-major descriptors return zeros), so the threads write
// transposed copies themselves: thread = row, the 32 lanes of a warp hit 32 different banks with a chunk stride of
// 16 * rows + 16 bytes.  [c_hi ; c_lo]^T (M) x [g_hi ; g_lo]^T (N = 64) is again one instruction per 8 time steps for all
// four partial products, accumulated in TMEM over every tile of the CTA and read once at the end.
//
// Global memory is only touched with coalesced accesses (8 consecutive lanes = one 128-byte row: a thread-per-row LDG.128
// touches 32 lines per instruction and the L1 tag stage, one line per clock, became the bound of the first version);
// whatever a thread needs per ROW (TMEM lane) goes through shared memory in the operand layout, where both mappings are
// conflict-free.
//
// Operand layouts (no swizzle, K-major, 8 x 16-byte core matrices; cute::UMMA canonical INTERLEAVE layout):
//   activation operand (rows = time):    (row, ch)  at (ch / 4) * kCHS + row * 16 + (ch % 4) * 4      LBO = kCHS,  SBO = 128
//   weight operand (rows = out channel): (n, k)     at (k / 4) * kWCH + n * 16 + (k % 4) * 4          LBO = kWCH,  SBO = 128
//   transposed operand (rows = channel): (ch, t)    at (t / 4) * kTC* + ch * 16 + (t % 4) * 4         LBO = kTC*,  SBO = 128
#include "common.cuh"
#include "umma.cuh"
#include "train_tc.cuh"

#ifdef SRWN_TUNING
// per-phase clock stamps of CTA 0's worker thread 0 on its fourth tile (tools/tc_trace.py)
__device__ long long g_tc_trace[3][16];
#define TC_STAMP(k, it, slot) do { if (blockIdx.x == 0 && threadIdx.x == 0 && (it) == 3) g_tc_trace[k][slot] = clock64(); } while (0)
extern "C" int srwn_debug_tc_trace(long long* out) { return (int)cudaMemcpyFromSymbol(out, g_tc_trace, sizeof(g_tc_trace)); }
#else
#define TC_STAMP(k, it, slot) do { } while (0)
#endif

namespace traintc {
using namespace umma;

constexpr int kRows = 128;
constexpr int kCHS = kRows * 16 + 16;        // 2064
constexpr int kTC64 = 64 * 16 + 16;          // 1040
constexpr int kTC128 = 128 * 16 + 16;        // 2064
constexpr int kWCH = 64 * 16;                // 1024
constexpr uint32_t kTmemCols = 256;

__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
  // cute::UMMA::InstrDescriptor: c = F32 (bit 4), a / b format TF32 = 2 (bits 7, 10), K-major, N >> 3 at 17, M >> 4 at 24
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// issued by a whole (converged) warp: the instruction itself is predicated on the elected lane, so the descriptors stay in
// uniform registers and the compiler emits no per-thread election loop around it
__device__ __forceinline__ void mma_tf32_elect(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
// the same with the A operand in tensor memory (row = lane, one TF32 element per column: K = 8 is 8 columns)
__device__ __forceinline__ void mma_tf32_ts_elect(uint32_t d_tmem, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem), "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const float* v) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_commit_elect(uint32_t bar) {
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
               "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar) : "memory");
}
constexpr int kWorkers = 512;                 // warps 0..15: operand staging and epilogues; warp 16: GEMM issue; warp 17: weight-gradient issue
__device__ __forceinline__ void worker_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kWorkers) : "memory"); }
__device__ __forceinline__ void tc_ld8(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
// x = hi + lo: hi is a valid TF32 number (low 13 mantissa bits clear) and x - hi is exact.  lo is stored with all its bits:
// the tensor core reads the top 19 of them, and whether it truncates or rounds the rest moves the product by 2^-21 |x| at most.
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  lo = x - hi;
}
__device__ __forceinline__ void split4(float4 v, float4& h, float4& l) {
  split_tf32(v.x, h.x, l.x); split_tf32(v.y, h.y, l.y); split_tf32(v.z, h.z, l.z); split_tf32(v.w, h.w, l.w);
}
__device__ __forceinline__ void split_store4(unsigned char* hi, unsigned char* lo, float4 v) {
  float4 h, l;
  split4(v, h, l);
  *reinterpret_cast<float4*>(hi) = h;
  *reinterpret_cast<float4*>(lo) = l;
}
// ex2.approx + rcp.approx (one MUFU each, ~1 ulp): ~2e-7 absolute on outputs in [-1, 1] (tanh.approx alone is 5e-4).
// No clamp: e = inf gives rcp = 0 and tanh = 1, e = 0 gives tanh = -1.
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float tanh_ex2(float x) { return fmaf(-2.0f, rcp_approx(ex2_approx(x * 2.885390081777927f) + 1.0f), 1.0f); }
// sigmoid of a number in [-1, 1] (the gate applies it to a tanh): 0.5 + f P(f^2), degree-4 minimax P, 5e-8 absolute -- FMA
// pipe work instead of two more MUFU operations per element (the epilogues are MUFU-bound: 16 per clock per SM)
__device__ __forceinline__ float sigmoid_fast(float f) {
  const float u = f * f;
  float p = fmaf(u, 1.6739570128265768e-05f, -0.00020698922162409872f);
  p = fmaf(u, p, 0.0020820044446736574f);
  p = fmaf(u, p, -0.020833170041441917f);
  p = fmaf(u, p, 0.25f);
  return fmaf(f, p, 0.5f);
}
__device__ __forceinline__ float4 ldg4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float& f4at(float4& v, int e) { return reinterpret_cast<float*>(&v)[e]; }

// a pipeline wait that never completes is a bug in this file, not a data condition: stop the kernel instead of hanging the GPU
__device__ __forceinline__ void wait_or_trap(uint32_t bar, uint32_t parity, volatile int* abort_words) {
  if (!mbar_wait(bar, parity, abort_words, 1, 4000000000LL)) __trap();
}
struct Ctl {                 // barriers and bookkeeping at the end of dynamic shared memory
  uint64_t bar_main, bar_wgrad;          // tcgen05.commit: the GEMMs / the weight-gradient GEMM of a tile have retired
  uint64_t full_main, full_wgrad;        // workers -> issuer warps: the operands are in shared memory
  uint32_t tmem_slot;
  int abort_words[2];
};

__device__ __forceinline__ uint32_t cta_setup(Ctl* ctl) {
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(smem_u32(&ctl->bar_main), 1);
    mbar_init(smem_u32(&ctl->bar_wgrad), 1);
    mbar_init(smem_u32(&ctl->full_main), 1);
    mbar_init(smem_u32(&ctl->full_wgrad), 1);
    ctl->abort_words[0] = ctl->abort_words[1] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ctl->tmem_slot)), "r"(kTmemCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return ctl->tmem_slot;
}
__device__ __forceinline__ void cta_teardown(uint32_t tmem) {
  tc_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
  }
}

// one instruction chain (called by a whole warp): nk K-steps of 8, A and B descriptors advancing by a_adv / b_adv bytes
__device__ __forceinline__ void issue_chain(uint32_t d_tmem, uint32_t a_addr, uint32_t a_lbo, uint32_t a_adv, uint32_t b_addr,
                                            uint32_t b_lbo, uint32_t b_adv, int nk, uint32_t idesc, uint32_t acc_first) {
  const uint64_t da = make_desc(a_addr, a_lbo, 128), db = make_desc(b_addr, b_lbo, 128);
  const uint64_t as = (uint64_t)(a_adv >> 4), bs = (uint64_t)(b_adv >> 4);
#pragma unroll 4
  for (int k = 0; k < nk; k++) mma_tf32_elect(d_tmem, da + k * as, db + k * bs, idesc, k > 0 ? 1u : acc_first);
}

// a chain whose A operand lives in tensor memory: K step k reads columns a_tmem + 8 k .. + 7
__device__ __forceinline__ void issue_chain_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_addr, uint32_t b_lbo, uint32_t b_adv,
                                               int nk, uint32_t idesc, uint32_t acc_first) {
  const uint64_t db = make_desc(b_addr, b_lbo, 128), bs = (uint64_t)(b_adv >> 4);
#pragma unroll 4
  for (int k = 0; k < nk; k++) mma_tf32_ts_elect(d_tmem, a_tmem + 8 * k, db + k * bs, idesc, k > 0 ? 1u : acc_first);
}

// weight operand with the hi part in rows 0..31 and the lo part in rows 32..63: value(n, k) for n, k < 32 / K
template <int K, typename F>
__device__ __forceinline__ void stage_weight(unsigned char* dst, F value) {
  if (threadIdx.x >= kWorkers) return;
  float v[K * 32 / kWorkers];
#pragma unroll
  for (int u = 0; u < K * 32 / kWorkers; u++) { const int i = threadIdx.x + u * kWorkers; v[u] = value(i & 31, i >> 5); }     // all loads in flight at once
#pragma unroll
  for (int u = 0; u < K * 32 / kWorkers; u++) {
    const int i = threadIdx.x + u * kWorkers, k = i >> 5, n = i & 31;
    float h, l;
    split_tf32(v[u], h, l);
    unsigned char* p = dst + (k >> 2) * kWCH + n * 16 + (k & 3) * 4;
    *reinterpret_cast<float*>(p) = h;
    *reinterpret_cast<float*>(p + 32 * 16) = l;
  }
}

// coalesced tile access: a thread's element i (i = 0, 1) is row (tid >> 3) + 64 i, 4-channel chunk tid & 7
// =====================================================================================================================
// forward
// =====================================================================================================================
constexpr int kFwdX = 16 * kCHS;                                   // one of X_hi / X_lo: 8 tap chunks | 8 current chunks
constexpr int kFwdSmem = 2 * kFwdX + 16 * kWCH + 8 * kWCH + 2 * 32 * 4 + (int)sizeof(Ctl);
int fwd_smem_bytes() { return kFwdSmem; }

__global__ void __launch_bounds__(kThreads, 1)
k_fwd_layer_tc(const float* __restrict__ x_l, float* __restrict__ x_next, const float* __restrict__ filt_k,
               const float* __restrict__ filt_b, const float* __restrict__ res_k, const float* __restrict__ res_b,
               const float* __restrict__ cond_next, int B, int T, int d, int P, int L, int frames) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* X_hi = smem;
  unsigned char* X_lo = X_hi + kFwdX;
  unsigned char* WfB = X_lo + kFwdX;
  unsigned char* WrB = WfB + 16 * kWCH;
  float* s_bf = reinterpret_cast<float*>(WrB + 8 * kWCH);
  float* s_br = s_bf + 32;
  Ctl* ctl = reinterpret_cast<Ctl*>(s_br + 32);
  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int row = (warp & 3) * 32 + lane, cb = ((warp >> 2) & 3) * 8;   // epilogue: this thread's row (TMEM lane) and channel base
  const int rA = tid >> 3, c4 = tid & 7;                                // coalesced access: rows rA, rA + 64, chunk c4
  // a[t][n] = sum_kk [tap | cur][t][kk] Wf[kk][n]: B(n, kk) = filt_k[kk * 32 + n]  (filt_k = [tap][cin][cout], tap 0 pairs with x[t-d])
  stage_weight<64>(WfB, [&](int n, int k) { return filt_k[k * kR + n]; });
  stage_weight<32>(WrB, [&](int n, int k) { return res_k[k * kR + n]; });
  if (tid < kR) { s_bf[tid] = filt_b[tid]; s_br[tid] = res_b[tid]; }
  const uint32_t tmem = cta_setup(ctl);
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  const uint32_t bar = smem_u32(&ctl->bar_main), full = smem_u32(&ctl->full_main);
  uint32_t phase = 0;
  const int tiles_per_b = (T + kRows - 1) / kRows, n_tiles = B * tiles_per_b;
  constexpr uint32_t kI64 = idesc_tf32(128, 64), kI32 = idesc_tf32(128, 32);
  if (warp >= 16) {
    if (warp == 16) {                     // GEMM issue: filter conv, then residual 1x1, per tile
      grid_dependency_wait();
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        wait_or_trap(full, phase, ctl->abort_words); phase ^= 1;
        tc_fence_after();
        issue_chain(tmem, smem_u32(X_hi), kCHS, 2 * kCHS, smem_u32(WfB), kWCH, 2 * kWCH, 8, kI64, 0);
        issue_chain(tmem + 64, smem_u32(X_lo), kCHS, 2 * kCHS, smem_u32(WfB), kWCH, 2 * kWCH, 8, kI32, 0);
        tc_commit_elect(bar);
        wait_or_trap(full, phase, ctl->abort_words); phase ^= 1;
        tc_fence_after();
        // residual 1x1: c = (c_hi, c_lo) is the A operand, written to tensor memory by the row threads (columns 96.., 224..)
        issue_chain_ts(tmem + 128, tmem + 96, smem_u32(WrB), kWCH, 2 * kWCH, 4, kI64, 0);
        issue_chain_ts(tmem + 192, tmem + 224, smem_u32(WrB), kWCH, 2 * kWCH, 4, kI32, 0);
        tc_commit_elect(bar);
      }
    }
    cta_teardown(tmem);
    return;
  }
  float4 pc[2], pt[2];
  auto load_tile = [&](int tile) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kRows;
    const float* xb = x_l + (size_t)b * T * kR;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int t = t0 + rA + 64 * i;
      pc[i] = make_float4(0, 0, 0, 0); pt[i] = pc[i];
      if (t < T) {
        pc[i] = ldg4(xb + (size_t)t * kR + c4 * 4);
        if (t - d >= 0) pt[i] = ldg4(xb + (size_t)(t - d) * kR + c4 * 4);
      }
    }
  };
  grid_dependency_wait();
  if ((int)blockIdx.x < n_tiles) load_tile(blockIdx.x);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kRows;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int r = rA + 64 * i;
      split_store4(X_hi + c4 * kCHS + r * 16, X_lo + c4 * kCHS + r * 16, pt[i]);
      split_store4(X_hi + (8 + c4) * kCHS + r * 16, X_lo + (8 + c4) * kCHS + r * 16, pc[i]);
    }
    fence_async_smem();
    worker_sync();
    if (tid == 0) mbar_arrive(full);
    // next layer's conditioning of this thread's row (one line per warp: a tile lies inside few latent frames) and the next
    // tile's operand rows: in flight during the GEMMs
    const int t = t0 + row;
    float4 cn[2];
#pragma unroll
    for (int j = 0; j < 2; j++)
      cn[j] = (t < T && cond_next) ? ldg4(cond_next + ((size_t)b * frames + t / P) * L * kR + cb + 4 * j) : make_float4(0, 0, 0, 0);
    if (tile + (int)gridDim.x < n_tiles) load_tile(tile + gridDim.x);
    wait_or_trap(bar, phase, ctl->abort_words); phase ^= 1;
    tc_fence_after();
    {
      float a0[8], a1[8], a2[8];
      tc_ld8(lane_base + cb, a0); tc_ld8(lane_base + 32 + cb, a1); tc_ld8(lane_base + 64 + cb, a2);
      tc_wait_ld();
      // gate: tanh, sigmoid OF THE TANH, product (ops.py:28,33,36); c goes to tensor memory as the A operand of the residual
      // GEMM (no shared-memory image, no proxy fence, and the GEMM reads no A tile from shared memory)
      float ch[8], cl[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float f = tanh_ex2((a2[i] + a1[i]) + a0[i] + s_bf[cb + i]);
        split_tf32(f * sigmoid_fast(f), ch[i], cl[i]);
      }
      tc_st8(lane_base + 96 + cb, ch);
      tc_st8(lane_base + 224 + cb, cl);
      tc_wait_st();
    }
    tc_fence_before();
    worker_sync();
    if (tid == 0) mbar_arrive(full);
    // x_l[t] back from its operand image: hi + lo is x exactly
    float4 xv[2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int chunk = 8 + (cb >> 2) + j;
      const float4 h = *reinterpret_cast<const float4*>(X_hi + chunk * kCHS + row * 16), l = *reinterpret_cast<const float4*>(X_lo + chunk * kCHS + row * 16);
      xv[j] = make_float4(h.x + l.x, h.y + l.y, h.z + l.z, h.w + l.w);
    }
    wait_or_trap(bar, phase, ctl->abort_words); phase ^= 1;
    tc_fence_after();
    {
      float r0[8], r1[8], r2[8];
      tc_ld8(lane_base + 128 + cb, r0); tc_ld8(lane_base + 160 + cb, r1); tc_ld8(lane_base + 192 + cb, r2);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 2; j++) {
        float4 v;
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int i = 4 * j + e;
          const float res = (r2[i] + r1[i]) + r0[i] + s_br[cb + i];             // residual 1x1 (ops.py:39)
          f4at(v, e) = (f4at(xv[j], e) + res) * SRWN_SQRT_HALF + f4at(cn[j], e);     // ops.py:40, next layer's conditioning (model.py:183)
        }
        *reinterpret_cast<float4*>(X_hi + ((cb >> 2) + j) * kCHS + row * 16) = v;     // staged in the (dead) tap rows for a coalesced store
      }
    }
    tc_fence_before();
    worker_sync();
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int r = rA + 64 * i, tt = t0 + r;
      if (tt < T) *reinterpret_cast<float4*>(x_next + ((size_t)b * T + tt) * kR + c4 * 4) = *reinterpret_cast<const float4*>(X_hi + c4 * kCHS + r * 16);
    }
    worker_sync();
  }
  cta_teardown(tmem);
}

// =====================================================================================================================
// gate backward
// =====================================================================================================================
constexpr int kGateX = 2 * 16 * kCHS;                       // X_hi | X_lo
constexpr int kGateG = 8 * kCHS;                            // one of G_hi / G_lo
constexpr int kGateGT = 32 * kTC64;                         // [g_hi ; g_lo]^T, and the same for [c_hi ; c_lo]^T
constexpr int kGateSmem = kGateX + 2 * kGateG + 2 * kGateGT + 16 * kWCH + 8 * kWCH + 32 * 4 + (int)sizeof(Ctl);
int gate_smem_bytes() { return kGateSmem; }

__global__ void __launch_bounds__(kThreads, 1)
k_bwd_gate_tc(const float* __restrict__ x_l, const float* __restrict__ g_in, float* __restrict__ da_out,
              const float* __restrict__ filt_k, const float* __restrict__ filt_b, const float* __restrict__ res_k,
              float* __restrict__ partial, int B, int T, int d) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* X_hi = smem;
  unsigned char* X_lo = X_hi + 16 * kCHS;
  unsigned char* G_hi = smem + kGateX;
  unsigned char* G_lo = G_hi + kGateG;
  // its own buffer, not the dead rows of X: the next tile's operand image is stored while the weight-gradient GEMM of this
  // tile still reads c^T (aliasing X gave wrong dWr as soon as a CTA walked more than one tile).  32 time chunks of 64 rows;
  // the M = 128 instruction reads 1 KB past the last chunk, into GT
  unsigned char* CT = G_lo + kGateG;
  unsigned char* GT = CT + kGateGT;
  unsigned char* WfB = GT + kGateGT;
  unsigned char* WrT = WfB + 16 * kWCH;
  float* s_bf = reinterpret_cast<float*>(WrT + 8 * kWCH);
  Ctl* ctl = reinterpret_cast<Ctl*>(s_bf + 32);
  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int row = (warp & 3) * 32 + lane, cb = ((warp >> 2) & 3) * 8;
  const int rA = tid >> 3, c4 = tid & 7;
  stage_weight<64>(WfB, [&](int n, int k) { return filt_k[k * kR + n]; });
  // dc[t][k] = sum_n dres[t][n] Wr[k][n]: B(row = k, K index = n) = res_k[k * 32 + n]
  stage_weight<32>(WrT, [&](int krow, int n) { return res_k[krow * kR + n]; });
  if (tid < kR) s_bf[tid] = filt_b[tid];
  const uint32_t tmem = cta_setup(ctl);
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  const uint32_t bar = smem_u32(&ctl->bar_main), bar_w = smem_u32(&ctl->bar_wgrad);
  const uint32_t full = smem_u32(&ctl->full_main), full_w = smem_u32(&ctl->full_wgrad);
  uint32_t phase = 0, phase_w = 0;
  const int tiles_per_b = (T + kRows - 1) / kRows, n_tiles = B * tiles_per_b;
  constexpr uint32_t kI64 = idesc_tf32(128, 64), kI32 = idesc_tf32(128, 32);
  if (warp >= 16) {
    grid_dependency_wait();
    if (warp == 16) {                     // a = [tap | cur] Wf and dc = dres Wr^T
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        wait_or_trap(full, phase, ctl->abort_words); phase ^= 1;
        tc_fence_after();
        issue_chain(tmem, smem_u32(X_hi), kCHS, 2 * kCHS, smem_u32(WfB), kWCH, 2 * kWCH, 8, kI64, 0);
        issue_chain(tmem + 64, smem_u32(X_lo), kCHS, 2 * kCHS, smem_u32(WfB), kWCH, 2 * kWCH, 8, kI32, 0);
        issue_chain(tmem + 96, smem_u32(G_hi), kCHS, 2 * kCHS, smem_u32(WrT), kWCH, 2 * kWCH, 4, kI64, 0);
        issue_chain(tmem + 160, smem_u32(G_lo), kCHS, 2 * kCHS, smem_u32(WrT), kWCH, 2 * kWCH, 4, kI32, 0);
        tc_commit_elect(bar);
      }
    } else if (warp == 17) {              // dWr[k][n] += sum_t c[t][k] dres[t][n]: [c_hi ; c_lo]^T x [g_hi ; g_lo]^T, 16 steps of 8 time steps
      uint32_t acc = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        wait_or_trap(full_w, phase_w, ctl->abort_words); phase_w ^= 1;
        tc_fence_after();
#ifdef SRWN_TUNING
        const bool stamp = blockIdx.x == 0 && (tile - (int)blockIdx.x) / (int)gridDim.x == 3 && (threadIdx.x & 31) == 0;
        if (stamp) g_tc_trace[1][12] = clock64();
#endif
        issue_chain(tmem + 192, smem_u32(CT), kTC64, 2 * kTC64, smem_u32(GT), kTC64, 2 * kTC64, 16, kI64, acc);
        tc_commit_elect(bar_w);
#ifdef SRWN_TUNING
        if (stamp) g_tc_trace[1][13] = clock64();
        if (blockIdx.x == 0 && (tile - (int)blockIdx.x) / (int)gridDim.x == 3) {      // how long the 16 instructions take to retire under load
          wait_or_trap(bar_w, phase_w ^ 1, ctl->abort_words);
          if (stamp) g_tc_trace[1][14] = clock64();
        }
#endif
        acc = 1;
      }
    }
    cta_teardown(tmem);
    return;
  }
  float gsum[8];
#pragma unroll
  for (int i = 0; i < 8; i++) gsum[i] = 0.f;
  float4 xc[2], xt[2], gg[2];
  // the next tile's rows are fetched in two portions at different points of the tile: all SMs run in step, one burst of every
  // load saturates HBM for ~2000 clocks and the LSU queue stalls the issuing warps for that long
  auto load_tile = [&](int tile, int part) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kRows;
    const float* xb = x_l + (size_t)b * T * kR;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int t = t0 + rA + 64 * i;
      if (part == 0) {
        xc[i] = make_float4(0, 0, 0, 0); xt[i] = xc[i];
        if (t < T) {
          xc[i] = ldg4(xb + (size_t)t * kR + c4 * 4);
          if (t - d >= 0) xt[i] = ldg4(xb + (size_t)(t - d) * kR + c4 * 4);
        }
      } else {
        gg[i] = t < T ? ldg4(g_in + ((size_t)b * T + t) * kR + c4 * 4) : make_float4(0, 0, 0, 0);
      }
    }
  };
  grid_dependency_wait();
  int n_done = 0;
  if ((int)blockIdx.x < n_tiles) { load_tile(blockIdx.x, 0); load_tile(blockIdx.x, 1); }
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, n_done++) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kRows;
    TC_STAMP(1, n_done, 0);
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int r = rA + 64 * i;
      split_store4(X_hi + c4 * kCHS + r * 16, X_lo + c4 * kCHS + r * 16, xt[i]);
      split_store4(X_hi + (8 + c4) * kCHS + r * 16, X_lo + (8 + c4) * kCHS + r * 16, xc[i]);
      const float4 gs = make_float4(gg[i].x * SRWN_SQRT_HALF, gg[i].y * SRWN_SQRT_HALF, gg[i].z * SRWN_SQRT_HALF, gg[i].w * SRWN_SQRT_HALF);   // dres
      split_store4(G_hi + c4 * kCHS + r * 16, G_lo + c4 * kCHS + r * 16, gs);
    }
    TC_STAMP(1, n_done, 1);
    fence_async_smem();
    worker_sync();
    if (tid == 0) mbar_arrive(full);
    TC_STAMP(1, n_done, 2);
    const bool more = tile + (int)gridDim.x < n_tiles;
    if (more) load_tile(tile + gridDim.x, 0);                                // next tile's x rows, in flight during the GEMMs
    // transposed copy of dres (this thread's row) for the weight gradient, while the GEMMs run
    if (n_done > 0) { wait_or_trap(bar_w, phase_w, ctl->abort_words); phase_w ^= 1; }      // the previous tile's dWr has read CT / GT
    TC_STAMP(1, n_done, 3);
    {
      unsigned char* gt = GT + (row >> 2) * kTC64 + (row & 3) * 4;
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const int chunk = (cb >> 2) + j;
        float4 h = *reinterpret_cast<const float4*>(G_hi + chunk * kCHS + row * 16), l = *reinterpret_cast<const float4*>(G_lo + chunk * kCHS + row * 16);
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int n = cb + 4 * j + e;
          *reinterpret_cast<float*>(gt + n * 16) = f4at(h, e);
          *reinterpret_cast<float*>(gt + (32 + n) * 16) = f4at(l, e);
          gsum[4 * j + e] += f4at(h, e) + f4at(l, e);
        }
      }
    }
    if (more) load_tile(tile + gridDim.x, 1);                                // and its g rows (this tile's are consumed)
    TC_STAMP(1, n_done, 4);
    wait_or_trap(bar, phase, ctl->abort_words); phase ^= 1;
    TC_STAMP(1, n_done, 5);
    tc_fence_after();
    {
      float a0[8], a1[8], a2[8], d0[8], d1[8], d2[8], da[8];
      tc_ld8(lane_base + cb, a0); tc_ld8(lane_base + 32 + cb, a1); tc_ld8(lane_base + 64 + cb, a2);
      tc_ld8(lane_base + 96 + cb, d0); tc_ld8(lane_base + 128 + cb, d1); tc_ld8(lane_base + 160 + cb, d2);
      tc_wait_ld();
      unsigned char* ct = CT + (row >> 2) * kTC64 + (row & 3) * 4;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float f = tanh_ex2((a2[i] + a1[i]) + a0[i] + s_bf[cb + i]);       // recomputed gate (ops.py:28,33,36)
        const float sg = sigmoid_fast(f);
        const float dc = (d2[i] + d1[i]) + d0[i];
        const float df = dc * (sg + f * sg * (1.f - sg));                        // d(f sigmoid(f)) / df
        da[i] = df * (1.f - f * f);                                              // tanh'
        float h, l;
        split_tf32(f * sg, h, l);
        *reinterpret_cast<float*>(ct + (cb + i) * 16) = h;
        *reinterpret_cast<float*>(ct + (32 + cb + i) * 16) = l;
      }
      // da staged in the (dead) dres rows for a coalesced store
#pragma unroll
      for (int j = 0; j < 2; j++)
        *reinterpret_cast<float4*>(G_hi + ((cb >> 2) + j) * kCHS + row * 16) = make_float4(da[4 * j], da[4 * j + 1], da[4 * j + 2], da[4 * j + 3]);
    }
    TC_STAMP(1, n_done, 6);
    tc_fence_before();
    fence_async_smem();
    worker_sync();
    if (tid == 0) mbar_arrive(full_w);
    TC_STAMP(1, n_done, 7);
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int r = rA + 64 * i, tt = t0 + r;
      if (tt < T) *reinterpret_cast<float4*>(da_out + ((size_t)b * T + tt) * kR + c4 * 4) = *reinterpret_cast<const float4*>(G_hi + c4 * kCHS + r * 16);
    }
    TC_STAMP(1, n_done, 8);
    worker_sync();
    TC_STAMP(1, n_done, 9);
  }
  // ---- per-CTA partial sums: dWr | dbr ----
  float* pp = partial + (size_t)blockIdx.x * (kR * kR + kR);
  float* red = reinterpret_cast<float*>(G_hi);               // [64][33] floats + [16][8]
  if (n_done > 0) {
    wait_or_trap(bar_w, phase_w, ctl->abort_words);
    tc_fence_after();
    float v0[8], v1[8];
    tc_ld8(lane_base + 192 + cb, v0); tc_ld8(lane_base + 224 + cb, v1);
    tc_wait_ld();
    if (row < 64) {
#pragma unroll
      for (int i = 0; i < 8; i++) red[row * 33 + cb + i] = v0[i] + (row < 32 ? v1[i] : 0.f);     // hi row: hi*hi + hi*lo; lo row: lo*hi
    }
  }
  float* red2 = red + 64 * 33;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    float v = gsum[i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red2[warp * 8 + i] = v;
  }
  worker_sync();
  for (int i = tid; i < kR * kR; i += kWorkers) pp[i] = n_done > 0 ? red[(i >> 5) * 33 + (i & 31)] + red[(32 + (i >> 5)) * 33 + (i & 31)] : 0.f;
  if (tid < kR) {                                            // channel tid: quarter tid >> 3 = warps 4 (tid >> 3) .. + 3
    const int w0 = 4 * (tid >> 3), e = tid & 7;
    pp[kR * kR + tid] = (red2[w0 * 8 + e] + red2[(w0 + 1) * 8 + e]) + (red2[(w0 + 2) * 8 + e] + red2[(w0 + 3) * 8 + e]);
  }
  cta_teardown(tmem);
}

// =====================================================================================================================
// conv backward
// =====================================================================================================================
constexpr int kConvDA = 2 * 16 * kCHS;                      // DA_hi | DA_lo: 8 chunks da[t] | 8 chunks da[t+d]
constexpr int kConvDAT = 32 * kTC64;                        // [da_hi ; da_lo]^T
constexpr int kConvXT = 32 * kTC128;                        // [tap_hi ; cur_hi ; tap_lo ; cur_lo]^T
constexpr int kConvXR = 16 * kCHS;                          // x rows as loaded (fp32): 8 tap chunks | 8 current chunks
constexpr int kConvSmem = kConvDA + kConvDAT + kConvXT + kConvXR + 16 * kWCH + (int)sizeof(Ctl);
int conv_smem_bytes() { return kConvSmem; }

__global__ void __launch_bounds__(kThreads, 1)
k_bwd_conv_tc(const float* __restrict__ x_l, const float* __restrict__ g_in, const float* __restrict__ da_in,
              float* __restrict__ dx_out, const float* __restrict__ filt_k, float* __restrict__ partial,
              float* __restrict__ dcond, int B, int T, int d, int P, int frames) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* DA_hi = smem;
  unsigned char* DA_lo = DA_hi + 16 * kCHS;
  unsigned char* DAT = smem + kConvDA;
  unsigned char* XT = DAT + kConvDAT;
  unsigned char* XR = XT + kConvXT;
  unsigned char* WB = XR + kConvXR;
  Ctl* ctl = reinterpret_cast<Ctl*>(WB + 16 * kWCH);
  float* red = reinterpret_cast<float*>(XR);                // [128][33] floats once the transposed copies are made
  const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int row = (warp & 3) * 32 + lane, cb = ((warp >> 2) & 3) * 8;
  const int rA = tid >> 3, c4 = tid & 7;
  // dx[t][k] = sum_n da[t][n] W1[k][n] + da[t+d][n] W0[k][n]: B(row = k, K index j) = j < 32 ? W1[k][j] : W0[k][j - 32]
  stage_weight<64>(WB, [&](int krow, int j) { return j < 32 ? filt_k[kR * kR + krow * kR + j] : filt_k[krow * kR + (j - 32)]; });
  const uint32_t tmem = cta_setup(ctl);
  const uint32_t lane_base = tmem + ((uint32_t)((warp & 3) * 32) << 16);
  const uint32_t bar = smem_u32(&ctl->bar_main), bar_w = smem_u32(&ctl->bar_wgrad);
  const uint32_t full = smem_u32(&ctl->full_main), full_w = smem_u32(&ctl->full_wgrad);
  uint32_t phase = 0, phase_w = 0;
  const int tiles_per_b = (T + kRows - 1) / kRows, n_tiles = B * tiles_per_b;
  constexpr uint32_t kI64 = idesc_tf32(128, 64), kI32 = idesc_tf32(128, 32);
  if (warp >= 16) {
    grid_dependency_wait();
    if (warp == 16) {                     // dx = [da | da(t+d)] [W1 ; W0]^T
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        wait_or_trap(full, phase, ctl->abort_words); phase ^= 1;
        tc_fence_after();
        issue_chain(tmem, smem_u32(DA_hi), kCHS, 2 * kCHS, smem_u32(WB), kWCH, 2 * kWCH, 8, kI64, 0);
        issue_chain(tmem + 64, smem_u32(DA_lo), kCHS, 2 * kCHS, smem_u32(WB), kWCH, 2 * kWCH, 8, kI32, 0);
        tc_commit_elect(bar);
      }
    } else if (warp == 17) {              // dWf[kk][n] += sum_t [tap | cur][t][kk] da[t][n]: [x_hi ; x_lo]^T (M = 128) x [da_hi ; da_lo]^T (N = 64)
      uint32_t acc = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        wait_or_trap(full_w, phase_w, ctl->abort_words); phase_w ^= 1;
        tc_fence_after();
        issue_chain(tmem + 128, smem_u32(XT), kTC128, 2 * kTC128, smem_u32(DAT), kTC64, 2 * kTC64, 16, kI64, acc);
        tc_commit_elect(bar_w);
        acc = 1;
      }
    }
    cta_teardown(tmem);
    return;
  }
  float dsum[8];
#pragma unroll
  for (int i = 0; i < 8; i++) dsum[i] = 0.f;
  float4 xc[2], xt[2], dac[2], daf[2], gq[2];
  // the next tile's rows are fetched in three portions at different points of the tile (see k_bwd_gate_tc)
  auto load_tile = [&](int tile, int part) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kRows;
    const float* xb = x_l + (size_t)b * T * kR;
    const float* db = da_in + (size_t)b * T * kR;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int t = t0 + rA + 64 * i;
      if (part == 0) {
        xc[i] = make_float4(0, 0, 0, 0); xt[i] = xc[i];
        if (t < T) {
          xc[i] = ldg4(xb + (size_t)t * kR + c4 * 4);
          if (t - d >= 0) xt[i] = ldg4(xb + (size_t)(t - d) * kR + c4 * 4);
        }
      } else if (part == 1) {
        dac[i] = make_float4(0, 0, 0, 0); daf[i] = dac[i];
        if (t < T) {
          dac[i] = ldg4(db + (size_t)t * kR + c4 * 4);
          if (t + d < T) daf[i] = ldg4(db + (size_t)(t + d) * kR + c4 * 4);
        }
      } else {
        gq[i] = t < T ? ldg4(g_in + ((size_t)b * T + t) * kR + c4 * 4) : make_float4(0, 0, 0, 0);
      }
    }
  };
  grid_dependency_wait();
  int n_done = 0;
  if ((int)blockIdx.x < n_tiles) { load_tile(blockIdx.x, 0); load_tile(blockIdx.x, 1); load_tile(blockIdx.x, 2); }
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, n_done++) {
    const int b = tile / tiles_per_b, t0 = (tile % tiles_per_b) * kRows;
    TC_STAMP(2, n_done, 0);
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int r = rA + 64 * i;
      split_store4(DA_hi + c4 * kCHS + r * 16, DA_lo + c4 * kCHS + r * 16, dac[i]);
      split_store4(DA_hi + (8 + c4) * kCHS + r * 16, DA_lo + (8 + c4) * kCHS + r * 16, daf[i]);
      *reinterpret_cast<float4*>(XR + c4 * kCHS + r * 16) = xt[i];
      *reinterpret_cast<float4*>(XR + (8 + c4) * kCHS + r * 16) = xc[i];
    }
    const float4 g0 = gq[0], g1 = gq[1];                   // this tile's rows of g, for the coalesced epilogue
    TC_STAMP(2, n_done, 1);
    fence_async_smem();
    worker_sync();
    if (tid == 0) mbar_arrive(full);
    TC_STAMP(2, n_done, 2);
    const bool more = tile + (int)gridDim.x < n_tiles;
    if (more) load_tile(tile + gridDim.x, 0);
    // transposed copies (this thread's row) for the weight gradient, while the dx GEMMs run
    if (n_done > 0) { wait_or_trap(bar_w, phase_w, ctl->abort_words); phase_w ^= 1; }      // the previous tile's dWf has read DAT / XT
    TC_STAMP(2, n_done, 3);
    {
      unsigned char* dt = DAT + (row >> 2) * kTC64 + (row & 3) * 4;
      unsigned char* xq = XT + (row >> 2) * kTC128 + (row & 3) * 4;
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const int chunk = (cb >> 2) + j;
        float4 h = *reinterpret_cast<const float4*>(DA_hi + chunk * kCHS + row * 16), l = *reinterpret_cast<const float4*>(DA_lo + chunk * kCHS + row * 16);
        float4 xth, xtl, xch, xcl;
        split4(*reinterpret_cast<const float4*>(XR + chunk * kCHS + row * 16), xth, xtl);
        split4(*reinterpret_cast<const float4*>(XR + (8 + chunk) * kCHS + row * 16), xch, xcl);
#pragma unroll
        for (int e = 0; e < 4; e++) {
          const int n = cb + 4 * j + e;
          *reinterpret_cast<float*>(dt + n * 16) = f4at(h, e);
          *reinterpret_cast<float*>(dt + (32 + n) * 16) = f4at(l, e);
          *reinterpret_cast<float*>(xq + n * 16) = f4at(xth, e);
          *reinterpret_cast<float*>(xq + (32 + n) * 16) = f4at(xch, e);
          *reinterpret_cast<float*>(xq + (64 + n) * 16) = f4at(xtl, e);
          *reinterpret_cast<float*>(xq + (96 + n) * 16) = f4at(xcl, e);
          dsum[4 * j + e] += f4at(h, e) + f4at(l, e);
        }
      }
    }
    TC_STAMP(2, n_done, 4);
    fence_async_smem();
    worker_sync();                                           // XR is free from here on: it becomes `red`
    if (tid == 0) mbar_arrive(full_w);
    if (more) load_tile(tile + gridDim.x, 1);
    TC_STAMP(2, n_done, 5);
    wait_or_trap(bar, phase, ctl->abort_words); phase ^= 1;
    TC_STAMP(2, n_done, 6);
    tc_fence_after();
    {
      float a0[8], a1[8], a2[8];
      tc_ld8(lane_base + cb, a0); tc_ld8(lane_base + 32 + cb, a1); tc_ld8(lane_base + 64 + cb, a2);
      tc_wait_ld();
#pragma unroll
      for (int i = 0; i < 8; i++) red[row * 33 + cb + i] = (a2[i] + a1[i]) + a0[i];
    }
    TC_STAMP(2, n_done, 7);
    tc_fence_before();
    if (more) load_tile(tile + gridDim.x, 2);
    worker_sync();
    TC_STAMP(2, n_done, 8);
    // coalesced: dx = g sqrt(1/2) + (da W1^T + da[t+d] W0^T), stored; and the conditioning gradient (x_l carries cond_l,
    // model.py:183): dcond_l[b][frame] += sum over the frame's rows of dx_l.  Fixed summation order and ONE atomic per
    // (latent frame, channel) and tile: with P = 128 the frame's sum is a single add onto zero, with P = 256 a commutative
    // pair, so the gradient is reproducible bit for bit.  A warp holds rows 4 warp .. + 3 (+ 64): lanes of equal chunk are
    // summed by shuffles, the 32 row groups of the tile by one warp in row order.
    float* ps = reinterpret_cast<float*>(DA_lo);                            // [32 row groups][32 channels]; free since the dx GEMM retired
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int r = rA + 64 * i, tt = t0 + r;
      const float4 gvv = i == 0 ? g0 : g1;
      const float* rp = red + r * 33 + c4 * 4;
      float4 v = make_float4(0, 0, 0, 0);
      if (tt < T) {
        v = make_float4(fmaf(gvv.x, SRWN_SQRT_HALF, rp[0]), fmaf(gvv.y, SRWN_SQRT_HALF, rp[1]), fmaf(gvv.z, SRWN_SQRT_HALF, rp[2]), fmaf(gvv.w, SRWN_SQRT_HALF, rp[3]));
        *reinterpret_cast<float4*>(dx_out + ((size_t)b * T + tt) * kR + c4 * 4) = v;
      }
      TC_STAMP(2, n_done, 13 + i);
      if (P % 4 == 0) {
#pragma unroll
        for (int o = 8; o <= 16; o <<= 1) {
          v.x += __shfl_xor_sync(0xffffffffu, v.x, o); v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
          v.z += __shfl_xor_sync(0xffffffffu, v.z, o); v.w += __shfl_xor_sync(0xffffffffu, v.w, o);
        }
        if (lane < 8) *reinterpret_cast<float4*>(ps + (16 * i + warp) * 32 + 4 * lane) = v;
      } else if (tt < T) {                                                   // a row group may straddle frames: per-element atomics
        float* dp = dcond + ((size_t)b * frames + tt / P) * kR + c4 * 4;
        atomicAdd(dp, v.x); atomicAdd(dp + 1, v.y); atomicAdd(dp + 2, v.z); atomicAdd(dp + 3, v.w);
      }
    }
    TC_STAMP(2, n_done, 9);
    worker_sync();
    TC_STAMP(2, n_done, 10);
    if (tid < 32 && P % 4 == 0) {
      const int ch = tid;
      if (P % kRows == 0) {                                                  // the whole tile is one latent frame
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < 32; q++) acc += ps[q * 32 + ch];
        if (t0 < T) atomicAdd(dcond + ((size_t)b * frames + t0 / P) * kR + ch, acc);
      } else {
        float acc = 0.f;
        int cur = -1;
        for (int q = 0; q < 32; q++) {
          const int tp = t0 + 4 * q;                                         // row group q = rows 4 q .. 4 q + 3
          if (tp >= T) break;
          const int f = tp / P;
          if (f != cur && cur >= 0) { atomicAdd(dcond + ((size_t)b * frames + cur) * kR + ch, acc); acc = 0.f; }
          cur = f;
          acc += ps[q * 32 + ch];
        }
        if (cur >= 0) atomicAdd(dcond + ((size_t)b * frames + cur) * kR + ch, acc);
      }
    }
    TC_STAMP(2, n_done, 11);
    worker_sync();
    TC_STAMP(2, n_done, 12);
  }
  // ---- per-CTA partial sums: dWf | dbf ----
  float* pp = partial + (size_t)blockIdx.x * (2 * kR * kR + kR);
  float* red2 = reinterpret_cast<float*>(DA_hi);             // [16][8]
  if (n_done > 0) {
    wait_or_trap(bar_w, phase_w, ctl->abort_words);
    tc_fence_after();
    float v0[8], v1[8];
    tc_ld8(lane_base + 128 + cb, v0); tc_ld8(lane_base + 160 + cb, v1);
    tc_wait_ld();
#pragma unroll
    for (int i = 0; i < 8; i++) red[row * 33 + cb + i] = v0[i] + (row < 64 ? v1[i] : 0.f);      // hi rows: hi*hi + hi*lo; lo rows: lo*hi
  }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    float v = dsum[i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red2[warp * 8 + i] = v;
  }
  worker_sync();
  for (int i = tid; i < 2 * kR * kR; i += kWorkers) pp[i] = n_done > 0 ? red[(i >> 5) * 33 + (i & 31)] + red[(64 + (i >> 5)) * 33 + (i & 31)] : 0.f;
  if (tid < kR) {
    const int w0 = 4 * (tid >> 3), e = tid & 7;
    pp[2 * kR * kR + tid] = (red2[w0 * 8 + e] + red2[(w0 + 1) * 8 + e]) + (red2[(w0 + 2) * 8 + e] + red2[(w0 + 3) * 8 + e]);
  }
  cta_teardown(tmem);
}

}  // namespace traintc
