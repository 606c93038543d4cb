// Fused residual-stack kernel on tcgen05 tensor cores (sm_100a), fp16 operands, fp32 accumulate.
//
// One persistent, warp-specialised CTA per SM streams a contiguous piece of the (utterance, time)
// line in chunks of NT MMA tiles of 128 rows (= TMEM lanes): 384 time steps for the teacher (NT = 3), 512 for the
// student (NT = 4, tiles_of()).  For a chunk, ALL layers run on-chip:
//   * the residual stream lives in fp32 registers of the epilogue thread that owns the row,
//   * its 16-bit image (the conv operand) lives in shared memory in the UMMA canonical K-major
//     no-swizzle layout [k-chunk][row][8 elems]; the dilated tap of layer l is the SAME buffer
//     addressed d_l rows earlier, so the "halo" costs no copy inside a chunk,
//   * rows older than the chunk (the last d_l inputs of every layer) come from a small per-CTA
//     ring in global memory (L2 resident) written by the previous chunk,
//   * the skip sum over layers accumulates in TMEM (128 fp32 columns per tile) and never leaves
//     the SM; the output head (relu, 1x1 S->S, relu, 1x1 S->4M) and the mixture-of-logistics
//     likelihood run from TMEM as the chunk's epilogue.
// Warp roles: warp 0 = loader (cp.async.bulk weights and ring -> halo rows per layer) + TMEM owner, warps 1..4 NT = NT tile
// groups of four warps (tcgen05.ld -> gate math -> operand stores; one elected lane per group issues the tile's MMAs),
// last warp (hand-off instantiation only) = publisher of the ring flags.
// Work decomposition: the (utterance, chunk) line is cut into contiguous pieces, one per TEAM of G CTAs; the members
// of a team take the piece's chunks round-robin (member j: chunks j, j+G, ...).  Chunk n+1 needs, per layer, the last
// d_l input rows of chunk n (the history ring): the team shares one ring block in global memory (L2 resident) and chunk
// n's CTA publishes "ring l of chunk n is written" through a per-(team, layer) flag, so chunk n+1's CTA runs the same
// layers about one layer behind -- a wavefront over (chunk, layer) with no recomputation inside a piece.  Only a piece
// that starts mid-utterance recomputes the receptive field (sum of dilations, rounded up to whole chunks, pruned to the
// dependency cone) with outputs discarded; that cost is shared by the G members.  Results do not depend on the
// partition or on G (tests: bit-exact under batch permutation, oracle comparisons at several B x T).
//
// Reference semantics: ops.py:6-46 (block, gate = sigmoid(tanh(.)) per ops.py:33),
// model.py:172-196 (decoder), model.py:423-452 + 479-482 (student flow), ops.py:124-175 (NLL).
#include "common.cuh"
#include "mol.cuh"
#include "umma.cuh"
#include "philox.cuh"
#include "partition.h"
#include <cuda_fp16.h>
#include <algorithm>
#include <cstdlib>

namespace fused {

constexpr int kTile = 128;
// Tiles (independent layer chains) per chunk.  Teacher: 3 -- a tile holds 128 fp32 skip-sum columns + 32 accumulator columns
// of the 512 TMEM columns.  Student: 4 -- a flow has no skip path (48 columns per tile), so what limits it is the register
// file: 17-18 warps leave 96 registers per thread (ptxas: 28 bytes of spills), and one more chain per SM hides more of the
// per-tile latency chain than the narrower register budget costs.
__host__ __device__ constexpr int tiles_of(bool teacher) { return teacher ? 3 : 4; }
__host__ __device__ constexpr int chunk_of(bool teacher) { return kTile * tiles_of(teacher); }     // time steps per chunk
constexpr int kHalo = 512;                      // largest dilation the layout supports
constexpr int kMaxLayers = 40;

// packed operand image (bytes, per layer): WF [8 kc][32 n][8] | WRS [4 kc][160 or 32 n][8]
constexpr int kWfBytes = 64 * 32 * 2;           // 4096
constexpr int kWrsTeacher = 32 * 160 * 2;       // 10240
constexpr int kWrsStudent = 32 * 32 * 2;        // 2048
constexpr int kH1Bytes = 128 * 128 * 2;         // 32768
constexpr int kH2Bytes = 128 * 32 * 2;          // 8192

struct Params {
  const uint8_t* packed;      // per-stack packed image
  const float* x_in;          // [B][T] stack input (audio / noise / previous flow output)
  const float* x_scored;      // teacher: audio whose likelihood is taken (may be null)
  const float* cb;            // [B][frames][L+1][32] fp32: folded biases + conditioning
  uint8_t* rings;             // per-team history rings
  const Seg* segs;            // [teams][kMaxSeg]
  const int* nseg;            // [teams]
  uint32_t* flags;            // [teams][kMaxLayers]: flags[l] = number of chunks of the piece whose ring l is published
  int G;                      // CTAs per team
  long long wait_limit;       // clocks a pipeline wait may spin before it raises the abort flag
  NoiseSpec noise;            // student, first flow: x_in[b][t] is the logistic draw (seed, stream, b*T + t) instead of a tensor
  float* logits_out;          // teacher, optional [B][T][O]
  float* nll_out;             // teacher, optional [B][T]
  double* nll_partial;        // teacher, optional [grid]
  float* scale_out;           // student [B][T]
  float* mean_out;            // student [B][T]
  float* x_out;               // student [B][T]
  int* err;                   // error words (pinned host memory, mapped): [0] flag [1] code [2] chunk [3] cta
#ifdef SRWN_TUNING
  long long* trace;           // optional [7 roles][kMaxLayers][12] clock64 stamps of CTA 0 (tuning aid)
  int trace_chunk;
#endif
  int T, L, P, frames, O, M;
  int ring_bytes_per_team;
  int dil[kMaxLayers];
  int ring_off[kMaxLayers];   // byte offset of layer l's ring inside a CTA's ring block
  int rsuf[kMaxLayers + 1];   // rsuf[l] = dil[l] + ... + dil[L-1]: how far back h_l is needed before the first output row
};

// ---- shared memory map ------------------------------------------------------------------
template <bool TEACHER>
struct SmemMapT {
  static constexpr int NT = tiles_of(TEACHER);
  static constexpr int rows = kHalo + NT * kTile;                 // rows per activation buffer
  static constexpr int hbuf = 0;                                  // 2 x [4][rows][16 B]
  static constexpr int hbuf_bytes = 4 * rows * 16;                // 57344 (teacher) / 65536 (student)
  static constexpr int cbuf = hbuf + 2 * hbuf_bytes;              // NT x 8 KB: scratch of the teardown's NLL reduction only
  static constexpr int cbuf_bytes = 4 * kTile * 16;               // 8192
  static constexpr int wst = cbuf + NT * cbuf_bytes;              // 2 stages
  static constexpr int wst_bytes = kWfBytes + (TEACHER ? kWrsTeacher : kWrsStudent);   // 14336 / 6144
  static constexpr int head = wst + 2 * wst_bytes;                // H1 | H2 (teacher only)
  static constexpr int bias = head + (TEACHER ? kH1Bytes + kH2Bytes : 0);   // [kMaxLayers][32] filter bias fp32
  static constexpr int hbias = bias + kMaxLayers * 32 * 4;        // skip_b_sum[128] | h1_b[128] | h2_b[32] | flow hk[64] hb[2]
  static constexpr int front = hbias + (128 + 128 + 32 + 64 + 4) * 4;   // fk[64]
  static constexpr int cbs = front + 64 * 4;                      // [NT tiles][kMaxLayers+1][32] folded bias + conditioning of the chunk
  static constexpr int bars = cbs + NT * (kMaxLayers + 1) * 32 * 4;
  static constexpr int n_bars = 40;
  static constexpr int misc = bars + n_bars * 8;                  // [0] tmem ptr, [8] abort flag + code, [16..16+4NT) ring-row counters
  static constexpr int total = misc + 64;
};
static_assert(SmemMapT<true>::total <= 232448 && SmemMapT<false>::total <= 232448, "shared memory budget");
// A3/A4 (head operands, 3 x 32 KB) overlay the two activation buffers
static_assert(3 * 16 * kTile * 16 <= 2 * SmemMapT<true>::hbuf_bytes, "head operand overlay");

// mbarrier indices for NT tiles
template <int NT>
struct BarT {
  static constexpr int D1 = 0;              // [NT] MMA -> tile group: filter-conv accumulator ready (tcgen05.commit)
  static constexpr int D2 = NT;             // [NT] MMA -> tile group: residual accumulator ready (tcgen05.commit)
  static constexpr int HD = 2 * NT;         // [NT tiles][2 layer parities] tile group -> higher tiles: input rows of a layer stored (128 arrivals)
  static constexpr int WFULL = 4 * NT;      // [2] loader -> tile groups: layer weights landed (tx bytes)
  static constexpr int WEMPTY = WFULL + 2;  // [2] MMA -> loader: all residual/skip MMAs of the layer retired (NT commits)
  static constexpr int HALO = WFULL + 4;    // [2] loader -> tile groups: halo rows of the layer landed
  static constexpr int G1 = WFULL + 6;      // [2] MMA -> loader/tile groups: all filter-conv MMAs of the layer retired (NT commits)
  static constexpr int HDD = WFULL + 8;     // [NT] MMA -> tile group: head accumulator ready
  static constexpr int TAIL = HDD + NT;     // loader -> tile groups: a pruned warm-up chunk may write the ring behind its last layer
  static constexpr int C2 = TAIL + 1;       // [NT tiles][2 layer parities] MMA -> tile groups: the residual and skip MMAs of a tile-layer retired, its TMEM
                                            // operand region is free.  Two barriers per tile: a leading tile may be two layers ahead of the one that asks, and
                                            // a single barrier's parity could not tell "retired two layers ago" from "not yet"
  static constexpr int count = C2 + 2 * NT;
};
static_assert(BarT<3>::count <= 40 && BarT<4>::count <= 40, "barrier slots");

using namespace umma;

// gate of ops.py:28,33,36 on two channels: f = tanh(a); out = f * sigmoid(f).  f lies in [-1,1], where
// sigmoid(f) = 0.5 + f*P(f^2) with a degree-2 minimax P (max error of the product 1.5e-6, far below the
// 16-bit operand rounding), so the gate costs one MUFU (tanh.approx) per channel plus packed FMA-pipe work.
__device__ __forceinline__ uint32_t gate2(f2_t a) {
  float a0, a1;
  upk(a, a0, a1);
  const f2_t f = pk(tanh_fast(a0), tanh_fast(a1));
  const f2_t s = mul2(f, f);
  f2_t t = fma2(s, pk(0.0017294071149080992f, 0.0017294071149080992f), pk(-0.020638039335608482f, -0.020638039335608482f));
  t = fma2(s, t, pk(0.2499687224626541f, 0.2499687224626541f));
  const f2_t c = fma2(f, pk(0.5f, 0.5f), mul2(s, t));
  float c0, c1;
  upk(c, c0, c1);
  return pack2(c0, c1);
}

// stores one row (32 values) as 4 x 16 B into a [kc][rows][8] operand buffer
__device__ __forceinline__ void store_row(uint8_t* buf, int rows_per_kc, int row, const float* v) {
#pragma unroll
  for (int kc = 0; kc < 4; kc++) {
    uint4 q;
    q.x = pack2(v[kc * 8 + 0], v[kc * 8 + 1]); q.y = pack2(v[kc * 8 + 2], v[kc * 8 + 3]);
    q.z = pack2(v[kc * 8 + 4], v[kc * 8 + 5]); q.w = pack2(v[kc * 8 + 6], v[kc * 8 + 7]);
    *reinterpret_cast<uint4*>(buf + ((size_t)kc * rows_per_kc + row) * 16) = q;
  }
}
// same, from 16 already packed 16-bit pairs
__device__ __forceinline__ void store_row_packed(uint8_t* buf, int rows_per_kc, int row, const uint32_t* w) {
#pragma unroll
  for (int kc = 0; kc < 4; kc++)
    *reinterpret_cast<uint4*>(buf + ((size_t)kc * rows_per_kc + row) * 16) =
        make_uint4(w[kc * 4 + 0], w[kc * 4 + 1], w[kc * 4 + 2], w[kc * 4 + 3]);
}

#ifndef SRWN_TUNING      // production builds carry no trace code (it costs ~10 % even when disabled at run time)
#define TRACE(role, layer, slot) do {} while (0)
#else
#define TRACE(role, layer, slot)                                                            \
  do {                                                                                      \
    if (tracing) p.trace[((role) * kMaxLayers + (layer)) * 12 + (slot)] = clock64();      \
  } while (0)
#endif

// ---- the kernel --------------------------------------------------------------------------
// 2 + 4 NT warps (teacher 14, student 18): warp 0 = loader + TMEM owner, warps 1..4 NT = NT tile groups of four warps, one warp per
// SMSP (row = TMEM lane = 32*(warp&3) + lane), warp 4 NT + 1 = publisher of the ring flags (off the layer chain).  Warp w sits on SMSP q = w&3 at level j = (w-1)/4 and
// belongs to tile (j+q+1)%NT, so that tile m's MMA-issuing warp is the highest warp id of SMSP m (the
// arbiter prefers high warp ids, and tcgen05 issue from a busy SMSP is what the layer chain waits on).
constexpr int kLoadWarp = 0;
// warps: loader | 4 per tile | publisher (exists only in the hand-off instantiation, G > 1)
__host__ __device__ constexpr int threads_of(bool handoff, int nt) { return (1 + 4 * nt + (handoff ? 1 : 0)) * 32; }

// ---- cross-CTA ring hand-off ------------------------------------------------------------------------
// consumer: chunk n waits until flags[l] >= n (rings of chunks 0..n-1 published), then orders its bulk loads (async proxy)
// after the acquire
// One acquire load per ring: measured faster than polling relaxed and fencing once for several rings (2.29 vs 2.56 ms
// at 32x64000, G = 7; profiles/r02d_handoff_variants.log).  The spin lives out of line: the loop bodies of three different
// warp roles share the instruction cache.
__device__ __noinline__ bool flag_spin(const uint32_t* f, uint32_t need, volatile int* abort_flag, const int* gerr, int code, long long limit) {
  const long long t0 = clock64();
  int spins = 0;
  uint32_t v;
  while (true) {
    __nanosleep(32);
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
    if (v >= need) return true;
    if (*abort_flag) return false;
    if (((++spins) & 1023) == 0 && *reinterpret_cast<const volatile int*>(gerr)) return false;   // another CTA aborted (host memory: polled rarely)
    if (clock64() - t0 > limit) {
      if (atomicCAS((int*)abort_flag, 0, 1) == 0) ((int*)abort_flag)[1] = code;
      return false;
    }
  }
}
// one acquire load, no spin: used to take the NEXT ring's flag while the loader would otherwise idle
__device__ __forceinline__ bool flag_try(const uint32_t* f, uint32_t need) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
  if (v < need) return false;
  asm volatile("fence.proxy.async;" ::: "memory");
  return true;
}
__device__ __forceinline__ bool flag_wait(const uint32_t* f, uint32_t need, volatile int* abort_flag, const int* gerr, int code, long long limit) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
  if (v < need && !flag_spin(f, need, abort_flag, gerr, code, limit)) return false;
  asm volatile("fence.proxy.async;" ::: "memory");       // the ring rows are read by bulk copies (async proxy)
  return true;
}
// producer, one thread per tile group, after the group barrier that follows the group's ring stores (generic st.global by
// up to 128 threads; the barrier orders them before this thread): count the rows in the group's shared-memory counter
// with release at CTA scope, so that the publisher's acquire -- and, through its GPU-scope release, the consumer CTA --
// observes them.  No per-thread fence or atomic sits on the layer chain.
__device__ __forceinline__ void ring_rows_done(uint32_t counter_addr, uint32_t rows) {
  asm volatile("red.release.cta.shared::cta.add.u32 [%0], %1;" ::"r"(counter_addr), "r"(rows) : "memory");
}
// rows of ring r (dilation d) that tile group m writes: chunk rows rc in [chunk - d, chunk) that fall into tile m
__device__ __forceinline__ int ring_rows_of(int d, int m, int chunk) {
  const int lo = max(chunk - d, m * kTile), hi = (m + 1) * kTile;
  return hi > lo ? hi - lo : 0;
}
__device__ __forceinline__ uint32_t ld_acquire_cta_shared(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
// producer, publisher lane: flags[l] = max(flags[l], chunks) with release at GPU scope (cumulative over the rows it acquired)
__device__ __forceinline__ void flag_publish(uint32_t* f, uint32_t chunks) {
  asm volatile("red.release.gpu.global.max.u32 [%0], %1;" ::"l"(f), "r"(chunks) : "memory");
}

// HANDOFF = false (teams of one CTA): the CTA hands its rings to itself across the chunk-end barrier; no flag, counter or
// publisher code is instantiated and the block has 13 warps.
template <bool TEACHER, bool HANDOFF>
__global__ void __launch_bounds__(threads_of(HANDOFF, tiles_of(TEACHER)), 1) k_fused(const Params p) {
  constexpr int NT = tiles_of(TEACHER), CH = NT * kTile;       // tiles and time steps per chunk
  constexpr int kThreads = threads_of(HANDOFF, NT);
  constexpr int kPubWarp = 1 + 4 * NT;
  constexpr int TCOLS = TEACHER ? 160 : 64;                    // TMEM columns per tile
  using SM = SmemMapT<TEACHER>;
  constexpr int ROWS = SM::rows;
  using BR = BarT<NT>;
  constexpr int BAR_D1 = BR::D1, BAR_D2 = BR::D2, BAR_HD = BR::HD, BAR_WFULL = BR::WFULL, BAR_WEMPTY = BR::WEMPTY, BAR_HALO = BR::HALO,
                BAR_G1 = BR::G1, BAR_HDD = BR::HDD, BAR_TAIL = BR::TAIL, BAR_C2 = BR::C2;
  (void)BAR_HDD; (void)BAR_C2; (void)kPubWarp;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t sbase = smem_u32(smem);
  volatile int* abort_flag = reinterpret_cast<volatile int*>(smem + SM::misc + 8);   // [0] flag [1] code
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM::misc);
  auto bar = [&](int i) { return sbase + SM::bars + i * 8; };
  const int L = p.L;
  constexpr int wrs_bytes = TEACHER ? kWrsTeacher : kWrsStudent;
  constexpr int layer_bytes = kWfBytes + wrs_bytes;
  constexpr int wrs_rows = TEACHER ? 160 : 32;

  // ---- one-time setup ---------------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < NT; i++) {
      mbar_init(bar(BAR_D1 + i), 1); mbar_init(bar(BAR_D2 + i), 1); mbar_init(bar(BAR_HDD + i), 1);
      mbar_init(bar(BAR_C2 + 2 * i), 1); mbar_init(bar(BAR_C2 + 2 * i + 1), 1);
      mbar_init(bar(BAR_HD + 2 * i), kTile); mbar_init(bar(BAR_HD + 2 * i + 1), kTile);
    }
    for (int i = 0; i < 2; i++) {
      mbar_init(bar(BAR_WFULL + i), 1); mbar_init(bar(BAR_WEMPTY + i), NT);
      mbar_init(bar(BAR_HALO + i), 1); mbar_init(bar(BAR_G1 + i), NT);
    }
    mbar_init(bar(BAR_TAIL), 1);
    abort_flag[0] = 0; abort_flag[1] = 0;
    for (int i = 0; i < NT; i++) reinterpret_cast<volatile uint32_t*>(smem + SM::misc + 16)[i] = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {  // resident constants: biases, front conv, head weights (plain loads; made visible below)
    const uint8_t* pk_ = p.packed;
    const size_t off_fixed = (size_t)L * layer_bytes;     // [filter bias L*32 f32][front 96 f32 -> 64 used][head...]
    const float* fbias = reinterpret_cast<const float*>(pk_ + off_fixed);
    float* s_bias = reinterpret_cast<float*>(smem + SM::bias);
    for (int i = tid; i < L * 32; i += kThreads) s_bias[i] = fbias[i];
    const float* ffront = fbias + kMaxLayers * 32;
    float* s_front = reinterpret_cast<float*>(smem + SM::front);
    for (int i = tid; i < 64; i += kThreads) s_front[i] = ffront[i];
    const float* fhb = ffront + 64;
    float* s_hb = reinterpret_cast<float*>(smem + SM::hbias);
    for (int i = tid; i < 128 + 128 + 32 + 64 + 4; i += kThreads) s_hb[i] = fhb[i];
    if (TEACHER) {
      const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(fhb + 128 + 128 + 32 + 64 + 4));
      uint4* dst = reinterpret_cast<uint4*>(smem + SM::head);
      for (int i = tid; i < (kH1Bytes + kH2Bytes) / 16; i += kThreads) dst[i] = src[i];
    }
  }
  fence_async_smem();
  if (warp == kLoadWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int G = p.G, team = (int)blockIdx.x / G, member = (int)blockIdx.x % G;
  const Seg* segs = p.segs + (size_t)team * kMaxSeg;
  const int nseg = p.nseg[team];
  uint8_t* ring = p.rings + (size_t)team * p.ring_bytes_per_team;
  uint32_t* flags = p.flags + (size_t)team * kMaxLayers;
  const uint32_t ringcnt = sbase + SM::misc + 16;   // [3] ring rows written so far by tile group m (monotonic)
  uint32_t pub_expect = 0;                              // publisher lane m: rows group m has to have written
  int seq = 0;                                          // chunk sequence number inside the piece
  int u0e = 0, u0o = 0, lay_base = 0;                 // phases of the parity-indexed / per-layer barriers used so far
  int chunk_idx = 0;                                  // chunks processed so far
  int head_idx = 0;                                   // chunks with a head phase so far
  int tail_idx = 0;                                   // pruned warm-up chunks (Lc < L) so far
  double nll_acc = 0.0;
  const bool elected = elect_one();

  for (int si = 0; si < nseg; si++) {
    const Seg sg = segs[si];
    for (int t0 = sg.t_start; t0 < sg.t_end; t0 += CH) {
      const int n = seq++;
      if (n % G != member) continue;                    // another member of the team runs this chunk
      const bool warm = TEACHER ? (t0 + CH <= sg.t_out) : false;   // student chunks always need h (cheap)
      const bool do_head = TEACHER && !warm;
      // A warm-up chunk only feeds the rings: layer l's output h_{l+1} is needed on the rsuf[l+1] rows before the first
      // output row t_out (h_{l+1}[t] reads h_l[t] and h_l[t - d_l]), so a chunk that ends `dist` rows before t_out runs
      // the layers with rsuf[l+1] > dist and nothing deeper; rows outside that cone hold garbage nobody reads.
      int Lc = L;
      if (t0 + CH <= sg.t_out) {
        const int dist = sg.t_out - (t0 + CH);
        Lc = 0;
        while (Lc < L && p.rsuf[Lc + 1] > dist) Lc++;
        if (Lc < 1) Lc = 1;
      }
#define U0(par) ((par) ? u0o : u0e)
#ifdef SRWN_TUNING
      const bool tracing_chunk = p.trace != nullptr && blockIdx.x == 0 && chunk_idx == p.trace_chunk;
#else
      constexpr bool tracing_chunk = false; (void)tracing_chunk;
#endif

      if (warp == kLoadWarp) {
        // ================= loader: weights (bulk copy) + halo rows (cp.async) per layer ============
        bool have_next = false;                                // the flag of ring l was acquired during the previous iteration
        for (int l = 0; l < Lc; l++) {
          const int s = l & 1;
          const int use = U0(s) + (l >> 1);                  // how many times stage s was used before
          [[maybe_unused]] const bool tracing = tracing_chunk && lane == 0;
          TRACE(6, l, 0);
          // halo rows of layer l: inputs at t0-d .. t0-1 (zeros before the segment start).  The halo goes first:
          // its condition (filter-conv MMAs of layer l-2 retired) holds earlier than the weight stage's.
          if (l >= 2 && !mbar_wait(bar(BAR_G1 + s), (use - 1) & 1, abort_flag, 0x1100000 | l, p.wait_limit)) break;   // G1 of layer l-2 retired
          TRACE(6, l, 2);
          // ring l of the previous chunk of the piece (written by another member of the team unless G == 1); also taken
          // at an utterance start, where the rows are not read: this chunk may overwrite the ring only after chunk n-1
          // has read it, which its publication implies
          if (HANDOFF && n > 0 && !have_next &&
              !flag_wait(flags + l, (uint32_t)n, abort_flag, p.err, 0x1200000 | l, p.wait_limit)) break;
          have_next = false;
          const int d = p.dil[l];
          const uint8_t* rl = ring + p.ring_off[l];
          const uint32_t dst0 = sbase + SM::hbuf + s * SM::hbuf_bytes;
          const int slot0 = (int)((unsigned)t0 % (unsigned)d);   // (t0 - d + i) mod d == (t0 + i) mod d
          if (t0 - d >= sg.t_start) {
            // every halo row exists: per 16-byte K chunk the ring is one or two contiguous pieces, moved by
            // bulk copies that complete on the HALO barrier (no generic-proxy stores, no fence)
            if (lane == 0) {
              mbar_expect_tx(bar(BAR_HALO + s), (uint32_t)(4 * d * 16));
              const uint32_t n1 = (uint32_t)(d - slot0) * 16, n2 = (uint32_t)slot0 * 16;
#pragma unroll
              for (int kc = 0; kc < 4; kc++) {
                const uint32_t dst = dst0 + (uint32_t)(kc * ROWS + kHalo - d) * 16;
                const uint8_t* src = rl + (size_t)kc * d * 16;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst), "l"(src + (size_t)slot0 * 16), "r"(n1), "r"(bar(BAR_HALO + s)) : "memory");
                if (n2)
                  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                               ::"r"(dst + n1), "l"(src), "r"(n2), "r"(bar(BAR_HALO + s)) : "memory");
              }
            }
            __syncwarp();
          } else {
            // segment start: rows before it are the zero padding of ops.py:9
            for (int kc = 0; kc < 4; kc++) {
              for (int i = lane; i < d; i += 32) {
                const uint32_t dst = dst0 + (uint32_t)(kc * ROWS + kHalo - d + i) * 16;
                if (t0 - d + i >= sg.t_start) {
                  int slot = slot0 + i; if (slot >= d) slot -= d;
                  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(rl + ((size_t)kc * d + slot) * 16) : "memory");
                } else {
                  asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(dst), "r"(0) : "memory");
                }
              }
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar(BAR_HALO + s));
          }
          // the acquire of the next ring's flag (an L2 round trip and a fence, about a microsecond) goes here, where the loader
          // would wait for the weight stage anyway, instead of between "buffer free" and the halo copy of the next layer
          if (HANDOFF && n > 0 && l + 1 < Lc) have_next = flag_try(flags + l + 1, (uint32_t)n);
          if (!mbar_wait(bar(BAR_WEMPTY + s), (use & 1) ^ 1, abort_flag, 0x1000000 | l, p.wait_limit)) break;
          if (lane == 0) {
            mbar_expect_tx(bar(BAR_WFULL + s), layer_bytes);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(sbase + SM::wst + s * SM::wst_bytes),
                           "l"(p.packed + (size_t)l * layer_bytes), "r"(layer_bytes), "r"(bar(BAR_WFULL + s)) : "memory");
          }
          TRACE(6, l, 1);
          TRACE(6, l, 3);
        }
        // a pruned warm-up chunk writes ring Lc behind its last layer without reading it: the write has to come after
        // chunk n-1's rows of the same ring
        if (Lc < L && !*abort_flag) {
          const bool ok = n == 0 || !HANDOFF || flag_wait(flags + Lc, (uint32_t)n, abort_flag, p.err, 0x1300000 | Lc, p.wait_limit);
          if (ok && lane == 0) mbar_arrive(bar(BAR_TAIL));
        }
      } else if (HANDOFF && warp == kPubWarp) {
        // ================= publisher: ring l of this chunk is complete -> flags[l] = n + 1 ========================
        // Rings written by this chunk: 0 (front conv) and l+1 by the residual epilogue of layer l < Lc (l+1 < L).  Lane m
        // follows tile group m: ring r is written by the rows rc >= CH - d_r, i.e. a known number of rows per group.
        const int last = Lc < L - 1 ? Lc : L - 1;
        bool ok = true;
        for (int r = 0; r <= last && ok; r++) {
          if (lane < NT) {
            const int rows = ring_rows_of(p.dil[r], lane, CH);
            if (rows) {
              pub_expect += (uint32_t)rows;
              if ((int32_t)(ld_acquire_cta_shared(ringcnt + 4 * lane) - pub_expect) < 0) {
                const long long t0 = clock64();
                while ((int32_t)(ld_acquire_cta_shared(ringcnt + 4 * lane) - pub_expect) < 0) {
                  __nanosleep(128);            // this warp has the highest id of its scheduler: a busy spin would starve the tile warps there
                  if (*abort_flag) { ok = false; break; }
                  if (clock64() - t0 > p.wait_limit) {
                    if (atomicCAS((int*)abort_flag, 0, 1) == 0) ((int*)abort_flag)[1] = 0x4000000 | (lane << 8) | r;
                    ok = false; break;
                  }
                }
              }
            }
          }
          ok = __all_sync(0xffffffffu, ok);
          if (ok && lane == 0) flag_publish(flags + r, (uint32_t)n + 1);
        }
        // rings this (warm-up) chunk did not write hold rows nobody reads: release them right away
        if (ok && lane == 0)
          for (int r = last + 1; r < L; r++) flag_publish(flags + r, (uint32_t)n + 1);
      } else {
        // ================= tile group m: MMA issue + epilogues; row = TMEM lane ====================
        // Per layer: [rows of the layer input stored] -> group barrier -> filter-conv GEMM (4 MMAs) ->
        // gate epilogue -> group barrier -> residual GEMM (2 MMAs, committed first) + skip GEMM (2 MMAs,
        // accumulating in TMEM, off the critical path) -> residual epilogue -> next layer's rows.
        // All control flow is uniform across the group (an aborted wait keeps walking the barriers).
        const int gw = warp & 3, m = (((warp - 1) >> 2) + gw + 1) % NT;
        // MMA issue is spread over SMSPs: tile m's issuer is its warp on SMSP m (tcgen05 instructions
        // serialise within an SMSP)
        const bool issuer = gw == m;
        const bool leader = issuer && elected;
        const int row = gw * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(gw * 32) << 16;
        const int t = t0 + m * kTile + row;
        const bool in_utt = t < p.T;
        int frame = (t0 + m * kTile) / p.P;
        if (frame > p.frames - 1) frame = p.frames - 1;
        const float* cb_g = p.cb + ((size_t)sg.b * p.frames + frame) * (size_t)(L + 1) * 32;
        float* cb = reinterpret_cast<float*>(smem + SM::cbs) + m * (kMaxLayers + 1) * 32;
        for (int i = row; i < (L + 1) * 32; i += kTile) cb[i] = __ldg(cb_g + i);   // one latent frame per tile
        group_sync(m);
        const float* s_bias = reinterpret_cast<const float*>(smem + SM::bias);
        const float* s_front = reinterpret_cast<const float*>(smem + SM::front);
        const int rc = m * kTile + row;                 // row inside the chunk
        f2_t h2[16];                                    // fp32 residual stream of this row, packed pairs
        float v[32];
        uint32_t w16[16];
        bool alive = true;
        [[maybe_unused]] const bool tracing = tracing_chunk && row == 0;
        constexpr uint32_t id32 = make_idesc(0, 128, 32), id128 = make_idesc(0, 128, 128);      // fp16 operands
        // descriptor low words that do not depend on the layer
        const uint32_t hb_lo0 = ((sbase + SM::hbuf) >> 4) + (uint32_t)(kHalo + m * kTile) + ((uint32_t)ROWS << 16);
        const uint32_t wb_lo0 = (sbase + SM::wst) >> 4;
        const uint32_t d_conv = tmem + m * TCOLS, d_skip = tmem + m * TCOLS + 32;
        // The gate output is the A operand of the residual (and skip) GEMM in tensor memory.  Student: the tile's unused skip
        // columns.  Teacher: 3 x 160 columns leave 32, i.e. TWO 16-column operand regions for three tiles; a region is live from
        // the gate epilogue until the tile's residual + skip MMAs retire (a few hundred clocks of the ~3000 a layer takes), and
        // the tiles run ~1000 clocks apart, so use g = 3 * (layers done) + m takes region g & 1 after waiting (almost never) for
        // use g - 2 to retire (BAR_C2 of tile (m + 1) % 3).
        uint32_t d_cop = d_skip;
        // student: a plain mbarrier arrive by a warp that does not issue, once it has seen the tile's commit barrier complete, can
        // stand in for the issuing lane's SECOND tcgen05.commit of a GEMM (same MMAs covered).  Measured per instantiation
        // (alternating runs, 8x64000 with teams of 9 / 64x64000 with one CTA per piece): for BAR_WEMPTY behind the residual
        // GEMM 0.534 -> 0.500 ms with the hand-off, +0.5 % without; for BAR_G1 behind the filter conv 0.500 -> 0.526 ms with the
        // hand-off, 3.421 -> 3.400 ms without.  Each instantiation takes the one that pays: G1 arrives late in the student
        // kernel without the hand-off, WEMPTY in the one with it.  (Teacher: neither does.)
        constexpr bool kLateG1 = !TEACHER && !HANDOFF;
        constexpr bool kLateWempty = !TEACHER && HANDOFF;

        // front: RightShift + K=2 causal conv on one channel (model.py:172-173), + bias + conditioning
        {
          // stack input at (b, tt): a tensor, or (student, first flow) the logistic noise drawn in place (student.py:104)
          auto x_at = [&](int tt) -> float {
            const size_t i = (size_t)sg.b * p.T + tt;
            if (!TEACHER && p.noise.on) return philox::logistic_at(p.noise.seed, p.noise.stream, (uint64_t)i);
            return __ldg(p.x_in + i);
          };
          const float xm1 = (t >= 1 && t - 1 < p.T) ? x_at(t - 1) : 0.f;
          const float xm2 = (t >= 2 && t - 2 < p.T) ? x_at(t - 2) : 0.f;
#pragma unroll
          for (int j = 0; j < 16; j++) {
            const float a = fmaf(xm2, s_front[2 * j], fmaf(xm1, s_front[32 + 2 * j], cb[2 * j]));
            const float b = fmaf(xm2, s_front[2 * j + 1], fmaf(xm1, s_front[32 + 2 * j + 1], cb[2 * j + 1]));
            h2[j] = pk(a, b);
            w16[j] = pack2(a, b);
          }
          alive = mbar_wait(bar(BAR_HALO + 0), U0(0) & 1, abort_flag, 0x2000000 | (m << 8), p.wait_limit);      // ring 0 was read for this chunk
          store_row_packed(smem + SM::hbuf, ROWS, kHalo + rc, w16);
          const int d0 = p.dil[0];
          fence_async_smem();
          mbar_arrive(bar(BAR_HD + 2 * m + 0));
          if (rc >= CH - d0) store_row_packed(ring + p.ring_off[0], d0, t % d0, w16);     // published at the top of layer 0
        }

        for (int l = 0; l < Lc; l++) {
          const int s = l & 1, sn = s ^ 1;
          const uint32_t ph = (lay_base + l) & 1, phs = (U0(s) + (l >> 1)) & 1;
          TRACE(m, l, 0);
          // ---- filter-conv GEMM: K = 64, steps 0,1 = tap rows (W[0], d rows earlier), 2,3 = current rows (W[1])
          const uint32_t hb_lo = hb_lo0 + (uint32_t)(s * (SM::hbuf_bytes >> 4));
          const uint32_t wb_lo = wb_lo0 + (uint32_t)(s * (SM::wst_bytes >> 4));
          const uint32_t dl = (uint32_t)p.dil[l];
          const uint32_t b1_lo = wb_lo + (32u << 16);
          const uint32_t b2_lo = wb_lo + (kWfBytes >> 4) + ((uint32_t)wrs_rows << 16);
          // the conditions the GEMM depends on are checked by different warps in parallel; the group
          // barrier then publishes them (and this tile's operand rows) to the issuing lane
          if (gw == ((m + 3) & 3)) {
            alive = mbar_wait(bar(BAR_WFULL + s), phs, abort_flag, 0x3000000 | (m << 8) | l, p.wait_limit) && alive;
            if (NT > 3 && m >= 3) alive = mbar_wait(bar(BAR_HD + 2 * (m - 3) + s), phs, abort_flag, 0x3300000 | (m << 8) | l, p.wait_limit) && alive;
          }
          if (gw == ((m + 1) & 3) && m >= 1) alive = mbar_wait(bar(BAR_HD + 2 * (m - 1) + s), phs, abort_flag, 0x3100000 | (m << 8) | l, p.wait_limit) && alive;
          if (gw == ((m + 2) & 3) && m >= 2) alive = mbar_wait(bar(BAR_HD + 2 * (m - 2) + s), phs, abort_flag, 0x3200000 | (m << 8) | l, p.wait_limit) && alive;
          group_sync(m);
          TRACE(m, l, 1);
          // ring l of this chunk (front conv / residual epilogue of layer l-1) is complete for this group: tell the publisher
          if (HANDOFF && gw == (m == 0 ? 1 : 0) && lane == 0) {       // a low row of the tile: it writes ring rows only for the largest dilations, so the release rarely waits for stores of its own
            const int rows = ring_rows_of((int)dl, m, CH);
            if (rows) ring_rows_done(ringcnt + 4 * m, (uint32_t)rows);
          }
          if (issuer) {
            tc_fence_after();
            if (leader) {
              tc_mma<0>(d_conv, desc_from_lo(hb_lo - dl), desc_from_lo(b1_lo), id32);
              tc_mma<1>(d_conv, desc_from_lo(hb_lo - dl + 2 * ROWS), desc_from_lo(b1_lo + 64), id32);
              tc_mma<1>(d_conv, desc_from_lo(hb_lo), desc_from_lo(b1_lo + 128), id32);
              tc_mma<1>(d_conv, desc_from_lo(hb_lo + 2 * ROWS), desc_from_lo(b1_lo + 192), id32);
              tc_commit(bar(BAR_D1 + m));
              if constexpr (!kLateG1) tc_commit(bar(BAR_G1 + s));               // NT arrivals (one per tile) complete the phase
            }
            __syncwarp();
          }
          TRACE(m, l, 2);
          // while the GEMM runs: poll the two conditions the next operand store depends on
          //  - activation buffer sn is free once the filter-conv MMAs of layer l-1 retired (all tiles),
          //  - ring l+1 may be overwritten once this chunk's halo of layer l+1 was read
          bool next_ok = true;
          if (l + 1 < Lc && !issuer) {
            if (l >= 1) next_ok = mbar_poll(bar(BAR_G1 + sn), (U0(sn) + ((l - 1) >> 1)) & 1);
            next_ok = mbar_poll(bar(BAR_HALO + sn), (U0(sn) + ((l + 1) >> 1)) & 1) && next_ok;
          }

          // ---- gate: tanh, sigmoid of the tanh, product (ops.py:28,33,36) ----
          alive = mbar_wait(bar(BAR_D1 + m), ph, abort_flag, 0x2100000 | (m << 8) | l, p.wait_limit) && alive;
          if (kLateG1 && gw == ((m + 2) & 3) && lane == 0) mbar_arrive(bar(BAR_G1 + s));      // the tile's filter-conv MMAs retired (D1): same signal, no second commit
          TRACE(m, l, 3);
          tc_fence_after();
          tc_ld32(d_conv + lane_addr, v);
          tc_wait_ld();
          TRACE(m, l, 4);
          {
            const ulonglong2* b2 = reinterpret_cast<const ulonglong2*>(s_bias + l * 32);
#pragma unroll
            for (int q = 0; q < 8; q++) {
              const ulonglong2 bb = b2[q];
              const f2_t d0 = pk(v[4 * q], v[4 * q + 1]), d1 = pk(v[4 * q + 2], v[4 * q + 3]);
              w16[2 * q] = gate2(add2(d0, bb.x));
              w16[2 * q + 1] = gate2(add2(d1, bb.y));
            }
          }
          // the gate output as the A operand of the residual GEMM in tensor memory: no shared-memory store, no proxy fence,
          // and the MMA reads no A tile from shared memory
          if constexpr (TEACHER) {
            const int cuse = lay_base + l, prev = m == 2 ? cuse : cuse - 1;
            d_cop = tmem + 480 + 16 * ((cuse + m) & 1);
            if (prev >= 0) alive = mbar_wait(bar(BAR_C2 + 2 * ((m + 1) % 3) + (prev & 1)), (uint32_t)((prev >> 1) & 1), abort_flag, 0x2800000 | (m << 8) | l, p.wait_limit) && alive;
            tc_fence_after();
          }
          tc_st16(d_cop + lane_addr, w16);
          tc_wait_st();
          tc_fence_before();
          TRACE(m, l, 5);
          next_ok = group_sync_and(m, next_ok);         // true: every polling warp saw both conditions
          TRACE(m, l, 6);
          if (issuer) {
            tc_fence_after();
            if (leader) {
              // residual first (it is what the layer chain waits for); the skip sum accumulates in TMEM behind it
              tc_mma_ts<0>(d_conv, d_cop, desc_from_lo(b2_lo), id32);
              tc_mma_ts<1>(d_conv, d_cop + 8, desc_from_lo(b2_lo + 2 * wrs_rows), id32);
              tc_commit(bar(BAR_D2 + m));
              if (TEACHER && !warm) {
                tc_mma_ts_dyn(d_skip, d_cop, desc_from_lo(b2_lo + 32), id128, l > 0 ? 1u : 0u);
                tc_mma_ts<1>(d_skip, d_cop + 8, desc_from_lo(b2_lo + 2 * wrs_rows + 32), id128);
              }
              if constexpr (TEACHER) tc_commit(bar(BAR_C2 + 2 * m + ((lay_base + l) & 1)));      // the operand region of this tile-layer is free
              if constexpr (!kLateWempty) tc_commit(bar(BAR_WEMPTY + s));           // NT arrivals free the weight stage
            }
            __syncwarp();
          }
          TRACE(m, l, 7);

          // ---- residual: dense = (inputs + residual) * sqrt(1/2) (ops.py:39-40), next conditioning ----
          alive = mbar_wait(bar(BAR_D2 + m), ph, abort_flag, 0x2200000 | (m << 8) | l, p.wait_limit) && alive;
          // student, hand-off instantiation: the residual MMAs are the only readers of the weight stage and they have retired
          // (D2), so a plain arrive by a warp that does not issue replaces the issuing lane's second tcgen05.commit.  Measured
          // in alternating runs: 0.534 -> 0.500 ms per flow launch at 8x64000 (teams of 9); without the hand-off (64x64000,
          // one CTA per piece) the same change is 0.5 % slower, so that instantiation keeps the commit.  The arriving warp is
          // the one after the issuer: the next (m + 2) measures the same (0.500 ms per flow at 8x64000), (m + 3) -- the warp
          // that waits for the next weight stage -- 0.533 ms.
          if (kLateWempty && gw == ((m + 1) & 3) && lane == 0) mbar_arrive(bar(BAR_WEMPTY + s));
          TRACE(m, l, 8);
          tc_fence_after();
          tc_ld32(d_conv + lane_addr, v);
          tc_wait_ld();
          {
            const ulonglong2* c2 = reinterpret_cast<const ulonglong2*>(cb + (l + 1) * 32);
            const f2_t sq = pk(SRWN_SQRT_HALF, SRWN_SQRT_HALF);
#pragma unroll
            for (int q = 0; q < 8; q++) {
              const ulonglong2 cc = c2[q];
              h2[2 * q] = fma2(add2(h2[2 * q], pk(v[4 * q], v[4 * q + 1])), sq, cc.x);
              h2[2 * q + 1] = fma2(add2(h2[2 * q + 1], pk(v[4 * q + 2], v[4 * q + 3])), sq, cc.y);
            }
          }
          TRACE(m, l, 9);
          if (l + 1 < L) {
#pragma unroll
            for (int j = 0; j < 16; j++) { float a, b; upk(h2[j], a, b); w16[j] = pack2(a, b); }
            if (l + 1 < Lc) {
              if (!next_ok) {                           // rare: the polls were too early
                if (l >= 1) alive = mbar_wait(bar(BAR_G1 + sn), (U0(sn) + ((l - 1) >> 1)) & 1, abort_flag, 0x2300000 | (m << 8) | l, p.wait_limit) && alive;
                alive = mbar_wait(bar(BAR_HALO + sn), (U0(sn) + ((l + 1) >> 1)) & 1, abort_flag, 0x2400000 | (m << 8) | l, p.wait_limit) && alive;
              }
              TRACE(m, l, 10);
              store_row_packed(smem + SM::hbuf + sn * SM::hbuf_bytes, ROWS, kHalo + rc, w16);
              tc_fence_before();
              fence_async_smem();
              mbar_arrive(bar(BAR_HD + 2 * m + sn));
            } else {
              tc_fence_before();                        // last layer of a pruned warm-up chunk: only the ring rows below
              alive = mbar_wait(bar(BAR_TAIL), tail_idx & 1, abort_flag, 0x2700000 | (m << 8) | l, p.wait_limit) && alive;
            }
            // history for the next chunk (read by the loader after the chunk-end barrier)
            const int dn = p.dil[l + 1];
            if (rc >= CH - dn) store_row_packed(ring + p.ring_off[l + 1], dn, t % dn, w16);   // published at the top of layer l+1
            TRACE(m, l, 11);
          } else {
            tc_fence_before();
          }
        }

        if (TEACHER) {
          if (do_head) {
            const float* s_hb = reinterpret_cast<const float*>(smem + SM::hbias);
            uint8_t* a3 = smem + SM::hbuf + m * (16 * kTile * 16);
            const uint32_t a3_lo = ((sbase + SM::hbuf + m * (16 * kTile * 16)) >> 4) + ((uint32_t)kTile << 16);
            // all filter-conv MMAs of the last layer retired -> both activation buffers are free
            alive = mbar_wait(bar(BAR_G1 + ((L - 1) & 1)), (U0((L - 1) & 1) + ((L - 1) >> 1)) & 1, abort_flag, 0x2500000 | (m << 8), p.wait_limit) && alive;
            // the skip accumulator is complete once this tile's last skip MMA retired (WEMPTY commit of the last layer)
            alive = mbar_wait(bar(BAR_WEMPTY + ((L - 1) & 1)), (U0((L - 1) & 1) + ((L - 1) >> 1)) & 1, abort_flag, 0x2510000 | (m << 8), p.wait_limit) && alive;
            tc_fence_after();
#pragma unroll 1
            for (int hs = 0; hs < 2; hs++) {
              // hs = 0: relu(sum of skips + summed skip biases) -> operand of the S->S conv (model.py:190-193)
              // hs = 1: relu(. + b1) -> operand of the S->4M conv (model.py:194-196)
              for (int q = 0; q < 4; q++) {
                tc_ld32(d_skip + lane_addr + q * 32, v);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 32; j++) v[j] = fmaxf(v[j] + s_hb[hs * 128 + q * 32 + j], 0.f);
                store_row(a3 + (size_t)q * 4 * kTile * 16, kTile, row, v);
              }
              tc_fence_before();
              fence_async_smem();
              group_sync(m);
              if (issuer) {
                tc_fence_after();
                if (leader && !*abort_flag) {
                  const uint32_t wlo = ((sbase + SM::head + (hs == 0 ? 0 : kH1Bytes)) >> 4) + ((uint32_t)(hs == 0 ? 128 : 32) << 16);
                  const int nrows = hs == 0 ? 128 : 32;
#pragma unroll
                  for (int j = 0; j < 8; j++)
                    tc_mma_dyn(hs == 0 ? d_skip : d_conv, desc_from_lo(a3_lo + 2 * j * kTile), desc_from_lo(wlo + 2 * j * nrows),
                               hs == 0 ? id128 : id32, j);
                  tc_commit(bar(BAR_HDD + m));
                }
                __syncwarp();
              }
              alive = mbar_wait(bar(BAR_HDD + m), (head_idx * 2 + hs) & 1, abort_flag, 0x2600000 | (m << 8) | hs, p.wait_limit) && alive;
              tc_fence_after();
            }
            tc_ld32(d_conv + lane_addr, v);
            tc_wait_ld();
            tc_fence_before();
            if (alive && in_utt && t >= sg.t_out) {
#pragma unroll
              for (int j = 0; j < 32; j++) v[j] += s_hb[256 + j];
              const size_t at = (size_t)sg.b * p.T + t;
              float nl = 0.f;
              if (p.x_scored) {                      // ops.py:124-175; M == 5 keeps the logits in registers
                const float xs = __ldg(p.x_scored + at);
                if (p.M == 5) nl = mol_nll_fixed<5>(xs, v);
                else {
                  float lg[32];
#pragma unroll
                  for (int j = 0; j < 32; j++) lg[j] = v[j];
                  nl = mol_nll_one(xs, lg, p.M);
                }
              }
              if (p.logits_out) {
                float* dst = p.logits_out + at * p.O;
                if (p.O == 20) {
#pragma unroll
                  for (int j = 0; j < 5; j++)
                    reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                } else {
#pragma unroll
                  for (int j = 0; j < 32; j++) if (j < p.O) dst[j] = v[j];
                }
              }
              if (p.x_scored) {
                if (p.nll_out) p.nll_out[at] = nl;
                nll_acc += (double)nl;
              }
            }
          }
        } else {
          // student flow head: relu -> 1x1 R->2; scale = exp(p0), mean = p1; out = x*scale + mean
          // (model.py:451-452, 479-482)
          const float* s_hb = reinterpret_cast<const float*>(smem + SM::hbias);
          const float* hk = s_hb + 288;
          float p0 = 0.f, p1 = 0.f;
#pragma unroll
          for (int j = 0; j < 16; j++) {
            float a, b;
            upk(h2[j], a, b);
            const float e0 = fmaxf(a, 0.f), e1 = fmaxf(b, 0.f);
            p0 = fmaf(e0, hk[4 * j], p0); p1 = fmaf(e0, hk[4 * j + 1], p1);
            p0 = fmaf(e1, hk[4 * j + 2], p0); p1 = fmaf(e1, hk[4 * j + 3], p1);
          }
          if (alive && in_utt && t >= sg.t_out) {
            const size_t at = (size_t)sg.b * p.T + t;
            const float sc = expf(p0 + hk[64]);
            const float mu = p1 + hk[65];
            p.scale_out[at] = sc;
            p.mean_out[at] = mu;
            const float xin = p.noise.on ? philox::logistic_at(p.noise.seed, p.noise.stream, (uint64_t)at) : __ldg(p.x_in + at);
            p.x_out[at] = fmaf(xin, sc, mu);
          }
        }
      }
      if (HANDOFF && Lc < L && warp != kLoadWarp && warp != kPubWarp) {        // pruned warm-up chunk: ring Lc was written behind the last layer
        const int gw = warp & 3, m = (((warp - 1) >> 2) + gw + 1) % NT;
        group_sync(m);
        if (gw == (m == 0 ? 1 : 0) && lane == 0) {
          const int rows = ring_rows_of(p.dil[Lc], m, CH);
          if (rows) ring_rows_done(ringcnt + 4 * m, (uint32_t)rows);
        }
      }
      if (do_head) head_idx++;
      if (Lc < L) tail_idx++;
      chunk_idx++;
      u0e += (Lc + 1) >> 1; u0o += Lc >> 1; lay_base += Lc;
      tc_fence_before();
      asm volatile("fence.proxy.async;" ::: "memory");   // ring rows (generic stores) -> next chunk's bulk loads
      __syncthreads();          // chunk boundary: every role is quiescent, buffers and rings are consistent
      tc_fence_after();
      if (*abort_flag) break;
    }
    if (*abort_flag) break;
  }

  // ---- teardown ------------------------------------------------------------------------------
  if (TEACHER && p.nll_partial) {
    double* s_red = reinterpret_cast<double*>(smem + SM::cbuf);     // reuse (everything is quiescent)
    for (int s = 16; s >= 1; s >>= 1) nll_acc += __shfl_xor_sync(0xffffffffu, nll_acc, s);
    if (lane == 0) s_red[warp] = nll_acc;
    __syncthreads();
    if (tid == 0) {
      double tot = 0;
      for (int w = 1; w <= 4 * NT; w++) tot += s_red[w];   // tile-group warps only
      p.nll_partial[blockIdx.x] = tot;
    }
  }
  if (tid == 0 && *abort_flag) {     // pinned host memory, read by the next API call (no atomics over the bus: any aborting CTA may win)
    volatile int* e = p.err;
    e[1] = abort_flag[1]; e[2] = chunk_idx; e[3] = blockIdx.x;
    __threadfence_system();
    e[0] = 1;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kLoadWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
  }
}

// sums the per-CTA partial log-likelihoods in a fixed order (deterministic for a given partition)
// (one warp: lane i adds partials i, i + 32, ... in ascending order, then a fixed shuffle tree -- the loads of a single
// thread walking all partials were a 9 us dependent chain)
__global__ void k_sum_partials(const double* __restrict__ part, int n, float* __restrict__ out) {
  double tot = 0;
  for (int i = threadIdx.x; i < n; i += 32) tot += part[i];
  for (int s = 16; s >= 1; s >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, s);
  if (threadIdx.x == 0) *out = (float)tot;
}

// cb[b][frame][0] = front bias + cond_0; cb[..][l+1] = sqrt(1/2)*res_bias_l + cond_{l+1} (0 past the last layer)
__global__ void k_fold_bias(const float* __restrict__ cond, const float* __restrict__ front_b,
                            const float* __restrict__ res_b, float* __restrict__ cb, int L) {
  const int bf = blockIdx.x;
  for (int o = threadIdx.x; o < (L + 1) * 32; o += blockDim.x) {
    const int i = o / 32, j = o % 32;
    float v = i < L ? cond[((size_t)bf * L + i) * 32 + j] : 0.f;
    v += i == 0 ? front_b[j] : SRWN_SQRT_HALF * res_b[(i - 1) * 32 + j];
    cb[(size_t)bf * (L + 1) * 32 + o] = v;
  }
}


// conditioning 1x1 (model.py:180/431) and the bias folding above in one pass, kCondRows latent frames per CTA so that the
// conditioning weights are read once per kCondRows frames:
// cb[bf][l] = enc[bf] @ Wc_l + bc_l + (l == 0 ? front_b : sqrt(1/2) res_b[l-1]);  cb[bf][L] = sqrt(1/2) res_b[L-1]
// 16 frames per CTA of 256 threads, two CTAs per SM: one computes while the other stores (a 512-thread CTA with 32 frames
// runs its FMA phase and its 127 KB of stores one after the other: 14.07 -> 14.00 ms per student step at 64x64000)
constexpr int kCondRows = 16;
constexpr int kCondRowsPerThread = 16;
constexpr int kCondThreads = 256 * (kCondRows / kCondRowsPerThread);     // 248 of every 256 threads own a (layer, 4-channel) group
static_assert(kCondRows % kCondRowsPerThread == 0 && kCondRows >= kCondRowsPerThread, "kCondRows is a multiple of 16");
// Register-blocked: a thread owns 4 consecutive output channels of one (layer, frame-half) for kCondRows / 2 frames, so one
// 16-byte weight load and one broadcast 16-byte read of the encodings feed 16 FMAs each (the first version issued one
// shared-memory read per FMA and was bound by that pipe).  The sum over the conditioning channels runs in ascending
// order from the folded bias, as before: results are bit-identical.  The student's flows (stacks) are folded by one launch.
__global__ void __launch_bounds__(kCondThreads, 512 / kCondThreads)
k_cond_fold(const float* __restrict__ enc, const float* __restrict__ cond_k, const float* __restrict__ cond_b,
            const float* __restrict__ front_b, const float* __restrict__ res_b, float* __restrict__ cb,
            int BF, int L, int C, size_t w_stride, size_t cb_stride) {
  constexpr int RH = kCondRowsPerThread;
  {                                                   // blockIdx.y = stack (student flow): same layout, `w_stride` floats further
    const size_t wo = (size_t)blockIdx.y * w_stride;
    cond_k += wo; cond_b += wo; front_b += wo; res_b += wo; cb += (size_t)blockIdx.y * cb_stride;
  }
  __shared__ __align__(16) float s_enc[kCondRows][kMaxCond];
  const int bf0 = blockIdx.x * kCondRows;
  for (int i = threadIdx.x; i < kCondRows * kMaxCond; i += blockDim.x) {
    const int r = i / kMaxCond, c = i % kMaxCond;
    s_enc[r][c] = (bf0 + r < BF && c < C) ? enc[(size_t)(bf0 + r) * C + c] : 0.f;
  }
  __syncthreads();
  const int half = threadIdx.x / 256, r0 = half * RH;
  for (int g = threadIdx.x % 256; g < (L + 1) * 8; g += 256) {
    const int l = g / 8, j = (g % 8) * 4, o = l * 32 + j;
    float4 base;
    {
      const float4 cbv = l < L ? *reinterpret_cast<const float4*>(cond_b + l * 32 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (l == 0) {
        const float4 f = *reinterpret_cast<const float4*>(front_b + j);
        base = make_float4(cbv.x + f.x, cbv.y + f.y, cbv.z + f.z, cbv.w + f.w);
      } else {
        const float4 rb = *reinterpret_cast<const float4*>(res_b + (l - 1) * 32 + j);
        base = make_float4(cbv.x + SRWN_SQRT_HALF * rb.x, cbv.y + SRWN_SQRT_HALF * rb.y, cbv.z + SRWN_SQRT_HALF * rb.z, cbv.w + SRWN_SQRT_HALF * rb.w);
      }
    }
    float4 acc[RH];
#pragma unroll
    for (int r = 0; r < RH; r++) acc[r] = base;
    if (l < L) {
      const float* wk = cond_k + (size_t)l * C * 32 + j;
      const int C4 = C & ~3;
      for (int c = 0; c < C4; c += 4) {
        float4 w[4];
#pragma unroll
        for (int k = 0; k < 4; k++) w[k] = __ldg(reinterpret_cast<const float4*>(wk + (size_t)(c + k) * 32));
#pragma unroll
        for (int r = 0; r < RH; r++) {
          const float4 e = *reinterpret_cast<const float4*>(&s_enc[r0 + r][c]);
          const float ev[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
          for (int k = 0; k < 4; k++) {
            acc[r].x = fmaf(ev[k], w[k].x, acc[r].x); acc[r].y = fmaf(ev[k], w[k].y, acc[r].y);
            acc[r].z = fmaf(ev[k], w[k].z, acc[r].z); acc[r].w = fmaf(ev[k], w[k].w, acc[r].w);
          }
        }
      }
      for (int c = C4; c < C; c++) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(wk + (size_t)c * 32));
#pragma unroll
        for (int r = 0; r < RH; r++) {
          const float e = s_enc[r0 + r][c];
          acc[r].x = fmaf(e, w.x, acc[r].x); acc[r].y = fmaf(e, w.y, acc[r].y);
          acc[r].z = fmaf(e, w.z, acc[r].z); acc[r].w = fmaf(e, w.w, acc[r].w);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < RH; r++)
      if (bf0 + r0 + r < BF) *reinterpret_cast<float4*>(cb + (size_t)(bf0 + r0 + r) * (L + 1) * 32 + o) = acc[r];
  }
}

}  // namespace fused

using namespace fused;

// ---- host side ---------------------------------------------------------------------------------
static size_t stack_image_bytes(const srwn_ctx* c) {
  const bool teacher = c->cfg.kind == SRWN_TEACHER;
  const size_t layer_bytes = kWfBytes + (teacher ? kWrsTeacher : kWrsStudent);
  size_t n = (size_t)c->cfg.n_layers * layer_bytes;
  n += (size_t)(kMaxLayers * 32 + 64 + 128 + 128 + 32 + 64 + 4) * 4;
  if (teacher) n += kH1Bytes + kH2Bytes;
  return (n + 255) & ~(size_t)255;
}

bool fused_supported(const srwn_ctx* c) {
  if (c->cfg.n_layers > kMaxLayers || c->cfg.pool_stride % kTile != 0) return false;
  for (int d : c->dilations) if (d > kHalo) return false;
  if (c->cfg.kind == SRWN_TEACHER && 4 * c->cfg.num_mixtures > 32) return false;
  return true;
}

int fused_check_config(const srwn_ctx* c) {
  if (fused_supported(c)) return SRWN_OK;
  return srwn_fail(SRWN_ERR_UNSUPPORTED, "the fused 16-bit kernel needs at most %d layers, dilations <= %d and pool_stride %% %d == 0",
                   kMaxLayers, kHalo, kTile);
}

// one fused launch gives every utterance a segment of its own: at most sm_count teams of kMaxSeg segments (partition.h)
int fused_check_batch(const srwn_ctx* c, int B) {
  if (B > fused_max_batch(c->sm_count))
    return srwn_fail(SRWN_ERR_UNSUPPORTED, "the fused 16-bit kernel takes at most %lld utterances per call (%d per SM on %d SMs), "
                     "got B = %d", fused_max_batch(c->sm_count), kMaxSeg, c->sm_count, B);
  return SRWN_OK;
}

size_t fused_packed_bytes(const srwn_ctx* c) {
  return fused_supported(c) ? (size_t)c->n_stacks * stack_image_bytes(c) : 0;
}

static uint16_t to_bits(float f) {
  __half h = __float2half_rn(f);
  return *reinterpret_cast<uint16_t*>(&h);
}

// element (n, k) of a K-major operand with `rows` N-rows: [k/8][n][k%8]
static inline size_t kmajor_idx(int n, int k, int rows) { return ((size_t)(k / 8) * rows + n) * 8 + (k % 8); }

int fused_pack_weights(srwn_ctx* c, cudaStream_t st) {
  if (!fused_supported(c) || !c->d_packed) return SRWN_OK;
  const bool teacher = c->cfg.kind == SRWN_TEACHER;
  const int L = c->cfg.n_layers, O = 4 * c->cfg.num_mixtures;
  const size_t img = stack_image_bytes(c);
  const size_t layer_bytes = kWfBytes + (teacher ? kWrsTeacher : kWrsStudent);
  const int wrs_rows = teacher ? 160 : 32;
  std::vector<uint8_t> host((size_t)c->n_stacks * img, 0);
  const float* W = srwn_host_weights(c);
  const StackOffsets& o = c->off;
  for (int s = 0; s < c->n_stacks; s++) {
    const float* w = W + (size_t)s * c->stack_floats;
    uint8_t* base = host.data() + (size_t)s * img;
    for (int l = 0; l < L; l++) {
      uint16_t* wf = reinterpret_cast<uint16_t*>(base + (size_t)l * layer_bytes);
      uint16_t* wrs = reinterpret_cast<uint16_t*>(base + (size_t)l * layer_bytes + kWfBytes);
      const float* fk = w + o.filt_k + (size_t)l * 2 * kR * kR;      // [2][Cin][Cout]
      for (int k = 0; k < 64; k++)
        for (int n = 0; n < 32; n++) wf[kmajor_idx(n, k, 32)] = to_bits(fk[(size_t)k * kR + n]);
      const float* rk = w + o.res_k + (size_t)l * kR * kR;          // [Cin][Cout]
      for (int k = 0; k < 32; k++)
        for (int n = 0; n < 32; n++) wrs[kmajor_idx(n, k, wrs_rows)] = to_bits(rk[(size_t)k * kR + n]);
      if (teacher) {
        const float* sk = w + o.skip_k + (size_t)l * kR * kS;       // [Cin][S]
        for (int k = 0; k < 32; k++)
          for (int n = 0; n < kS; n++) wrs[kmajor_idx(32 + n, k, wrs_rows)] = to_bits(sk[(size_t)k * kS + n]);
      }
    }
    float* fx = reinterpret_cast<float*>(base + (size_t)L * layer_bytes);
    for (int l = 0; l < L; l++)
      for (int j = 0; j < 32; j++) fx[l * 32 + j] = w[o.filt_b + (size_t)l * kR + j];
    float* ffront = fx + kMaxLayers * 32;
    for (int j = 0; j < 64; j++) ffront[j] = w[o.front_k + j];       // [2][R]
    float* fhb = ffront + 64;
    if (teacher) {
      for (int j = 0; j < 128; j++) { fhb[j] = w[o.skip_b_sum + j]; fhb[128 + j] = w[o.head1_b + j]; }
      for (int j = 0; j < 32; j++) fhb[256 + j] = j < O ? w[o.head2_b + j] : 0.f;
      uint16_t* h1 = reinterpret_cast<uint16_t*>(fhb + 128 + 128 + 32 + 64 + 4);
      uint16_t* h2 = h1 + 128 * 128;
      for (int k = 0; k < 128; k++) {
        for (int n = 0; n < 128; n++) h1[kmajor_idx(n, k, 128)] = to_bits(w[o.head1_k + (size_t)k * kS + n]);
        for (int n = 0; n < 32; n++) h2[kmajor_idx(n, k, 32)] = to_bits(n < O ? w[o.head2_k + (size_t)k * O + n] : 0.f);
      }
    } else {
      for (int j = 0; j < 64; j++) fhb[288 + j] = w[o.head1_k + j];  // [R][2]
      fhb[288 + 64] = w[o.head1_b + 0]; fhb[288 + 65] = w[o.head1_b + 1];
    }
  }
  SRWN_CUDA(cudaMemcpyAsync(c->d_packed, host.data(), host.size(), cudaMemcpyHostToDevice, st));
  SRWN_CUDA(cudaStreamSynchronize(st));
  return SRWN_OK;
}

struct FusedWs {
  float* cb; uint8_t* rings; uint32_t* flags; double* partial;
#ifdef SRWN_TUNING
  long long* trace;
#endif
  float *scales, *means;
  size_t bytes;
};

static FusedWs carve_fused(const srwn_ctx* c, int B, int T, void* ws, size_t cap) {
  WsCarver w(ws, cap);
  FusedWs r{};
  const size_t frames = T / c->cfg.pool_stride, L = c->cfg.n_layers, n = (size_t)B * T;
  const int grid = c->sm_count > 0 ? c->sm_count : 148;
  const size_t nst = c->cfg.kind == SRWN_STUDENT ? (size_t)c->cfg.num_flows : 1;   // stacks folded / flagged up front
  r.cb = w.take<float>((size_t)B * frames * (L + 1) * 32 * nst);
  r.rings = w.take<uint8_t>((size_t)grid * ((size_t)c->sum_dilation * 64 + 256));     // one block per team, at most `grid` teams
  r.flags = w.take<uint32_t>((size_t)grid * kMaxLayers * nst);
  r.partial = w.take<double>(grid);
#ifdef SRWN_TUNING
  r.trace = w.take<long long>(7 * kMaxLayers * 12);
#endif
  if (c->cfg.kind == SRWN_STUDENT) {
    r.scales = w.take<float>(n * c->cfg.num_flows);
    r.means = w.take<float>(n * c->cfg.num_flows);
  }
  r.bytes = w.used;
  return r;
}

// device copy of the partition: segs [grid][kMaxSeg] | nseg [grid]  (allocated at srwn_create)
size_t fused_partition_bytes(const srwn_ctx* c) {
  const size_t grid = c->sm_count > 0 ? c->sm_count : 148;
  return grid * kMaxSeg * sizeof(Seg) + grid * sizeof(int);
}

size_t fused_workspace_bytes(const srwn_ctx* c, int B, int T) {
  return carve_fused(c, B, T, nullptr, 0).bytes;
}

template <bool TEACHER>
static int launch_fused(srwn_ctx* c, const Params& p, int grid, cudaStream_t st) {
  const bool handoff = p.G > 1;
  auto kern = handoff ? k_fused<TEACHER, true> : k_fused<TEACHER, false>;
  SRWN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemMapT<TEACHER>::total));
  // the members of a team wait on one another's ring flags: the launch must be co-resident (grid <= SM count, one CTA
  // per SM), which a cooperative launch guarantees or refuses
  Params pl = p;
  void* args[] = {&pl};
  SRWN_CUDA(cudaLaunchCooperativeKernel((const void*)kern, dim3(grid), dim3(threads_of(handoff, tiles_of(TEACHER))), args, SmemMapT<TEACHER>::total, st));
  SRWN_LAUNCH_CHECK();
  return SRWN_OK;
}

static int prepare(srwn_ctx* c, int stack, const float* enc, int B, int T, int out0, const FusedWs& w, Params* p,
                   int* grid, bool first, cudaStream_t st) {
  const int L = c->cfg.n_layers, P = c->cfg.pool_stride, frames = T / P;
  int rc = sticky_error(c);
  if (rc) return rc;
  // conditioning of every stack and the ring flags of every launch are prepared by the first call of a sequence (the
  // student's flows then launch back to back)
  const int nst = c->cfg.kind == SRWN_STUDENT ? c->cfg.num_flows : 1;
  const size_t cb_stride = (size_t)B * frames * (L + 1) * 32, flag_stride = (size_t)c->sm_count * kMaxLayers;
  if (first) {
    const float* s0 = stack_w(c, 0);
    k_cond_fold<<<dim3((B * frames + kCondRows - 1) / kCondRows, nst), kCondThreads, 0, st>>>(
        enc, s0 + c->off.cond_k, s0 + c->off.cond_b, s0 + c->off.front_b, s0 + c->off.res_b, w.cb, B * frames, L,
        c->cfg.cond_channels, c->stack_floats, cb_stride);
    SRWN_LAUNCH_CHECK();
    SRWN_CUDA(cudaMemsetAsync(w.flags, 0, flag_stride * nst * sizeof(uint32_t), st));
  }
  const size_t seg_bytes = (size_t)c->sm_count * kMaxSeg * sizeof(Seg), n_bytes = (size_t)c->sm_count * sizeof(int);
  if (first && (c->part_B != B || c->part_T != T || c->part_out0 != out0 || c->part_team_req != c->team_size)) {
    // the work partition depends on (B, T, out0) and the team size only: built once, kept on the device next to the handle.
    // The staging vector belongs to the handle (a copy from pageable memory returns once the bytes are staged).
    const bool teacher = c->cfg.kind == SRWN_TEACHER;
    Partition part = make_partition(B, T, out0, chunk_of(teacher), teacher ? 1.10 : 1.04, c->dilations, c->sm_count, c->team_size);
    if (part.teams == 0) return srwn_fail(SRWN_ERR_UNSUPPORTED, "no work partition holds B = %d utterances", B);   // fused_check_batch
    c->part_host.assign(seg_bytes + n_bytes, 0);
    memcpy(c->part_host.data(), part.segs.data(), std::min(seg_bytes, part.segs.size() * sizeof(Seg)));
    memcpy(c->part_host.data() + seg_bytes, part.nseg.data(), std::min(n_bytes, part.nseg.size() * sizeof(int)));
    SRWN_CUDA(cudaMemcpyAsync(c->d_part, c->part_host.data(), c->part_host.size(), cudaMemcpyHostToDevice, st));
    c->part_B = B; c->part_T = T; c->part_out0 = out0; c->part_team_req = c->team_size;
    c->part_teams = part.teams; c->part_G = part.G;
  }
  *grid = c->part_teams * c->part_G;
  memset(p, 0, sizeof(*p));
  const size_t img = stack_image_bytes(c);
  p->packed = (const uint8_t*)c->d_packed + (size_t)stack * img;
  p->cb = w.cb + (size_t)stack * cb_stride; p->rings = w.rings; p->flags = w.flags + (size_t)stack * flag_stride; p->err = c->h_err; p->G = c->part_G;
  p->wait_limit = c->wait_limit_clocks;
  p->segs = reinterpret_cast<const Seg*>(c->d_part);
  p->nseg = reinterpret_cast<const int*>(reinterpret_cast<const uint8_t*>(c->d_part) + seg_bytes);
  p->T = T; p->L = L; p->P = P; p->frames = frames;
  p->O = 4 * c->cfg.num_mixtures; p->M = c->cfg.num_mixtures;
  p->ring_bytes_per_team = c->sum_dilation * 64 + 256;
  int off = 0;
  for (int l = 0; l < L; l++) { p->dil[l] = c->dilations[l]; p->ring_off[l] = off; off += c->dilations[l] * 64; }
  p->rsuf[L] = 0;
  for (int l = L - 1; l >= 0; l--) p->rsuf[l] = p->rsuf[l + 1] + c->dilations[l];
#ifdef SRWN_TUNING
  p->trace = getenv("SRWN_TRACE") ? w.trace : nullptr;
  p->trace_chunk = getenv("SRWN_TRACE") ? atoi(getenv("SRWN_TRACE")) : 0;
#endif
  return SRWN_OK;
}

int run_teacher_fused(srwn_ctx* c, const float* x_in, const float* enc, const float* x_scored,
                      float* nll_out, float* nll_sum, float* logits_out, int B, int T,
                      void* ws, size_t ws_bytes, cudaStream_t st) {
  FusedWs w = carve_fused(c, B, T, ws, ws_bytes);
  int rc = check_workspace(ws, ws_bytes, w.bytes);
  if (rc) return rc;
  Params p;
  int grid = 0;
  rc = prepare(c, 0, enc, B, T, 0, w, &p, &grid, true, st);
  if (rc) return rc;
  p.x_in = x_in; p.x_scored = x_scored; p.logits_out = logits_out; p.nll_out = nll_out;
  p.nll_partial = (x_scored && nll_sum) ? w.partial : nullptr;
  {
    ProfScope prof(c, st, "k_fused<teacher,fp16>", 1);
    rc = launch_fused<true>(c, p, grid, st);
    if (rc) return rc;
  }
  if (p.nll_partial) {
    k_sum_partials<<<1, 32, 0, st>>>(w.partial, grid, nll_sum);
    SRWN_LAUNCH_CHECK();
  }
  return SRWN_OK;
}

int run_student_flows_fused(srwn_ctx* c, float* const* x, NoiseSpec noise, const float* enc, int B, int T, int t_out,
                            void* ws, size_t ws_bytes, const float** scales, const float** means, cudaStream_t st) {
  FusedWs w = carve_fused(c, B, T, ws, ws_bytes);
  if (int rc = check_workspace(ws, ws_bytes, w.bytes)) return rc;
  const size_t n = (size_t)B * T;
  const int F = c->cfg.num_flows;
  int grid = 0;
  for (int f = 0; f < F; f++) {                     // model.py:509-513: flows are strictly sequential
    Params p;
    int rc = prepare(c, f, enc, B, T, t_out, w, &p, &grid, f == 0, st);
    if (rc) return rc;
    p.x_in = x[f]; p.scale_out = w.scales + (size_t)f * n; p.mean_out = w.means + (size_t)f * n; p.x_out = x[f + 1];
    if (f == 0) p.noise = noise;                    // later flows read the previous flow's output
    ProfScope prof(c, st, "k_fused<student,fp16>", 1);
    rc = launch_fused<false>(c, p, grid, st);
    if (rc) return rc;
  }
  *scales = w.scales; *means = w.means;
  return SRWN_OK;
}

// partition chosen for the last fused call (tests, bench records): teams x CTAs per team
void fused_last_partition(const srwn_ctx* c, int* teams, int* G) { *teams = c->part_teams; *G = c->part_G; }

#ifdef SRWN_TUNING
// tuning aid: copies the clock64 trace of CTA 0 (see SRWN_TRACE) to the host
extern "C" int srwn_debug_read_trace(srwn_handle_t h, int32_t B, int32_t T, void* ws, size_t ws_bytes,
                                     long long* out, int32_t count) {
  FusedWs w = carve_fused(h, B, T, ws, ws_bytes);
  if (count > 7 * kMaxLayers * 12) count = 7 * kMaxLayers * 12;
  SRWN_CUDA(cudaDeviceSynchronize());
  SRWN_CUDA(cudaMemcpy(out, w.trace, sizeof(long long) * count, cudaMemcpyDeviceToHost));
  return SRWN_OK;
}

// ---- tuning aid: cost of back-to-back tcgen05.mma dispatches (one CTA, garbage operands) ------------
// Test c: warps listed in `mask` each issue CNT MMAs of width N (descriptors precomputed, fully unrolled)
// into their own TMEM columns and commit; out[c] = {max issue clocks, max issue+complete clocks}.
namespace fused {
template <int N, int CNT>
__device__ __forceinline__ void bench_issue(uint32_t tmem_col, uint32_t a_lo, uint32_t b_lo, uint32_t mbar_addr) {
  constexpr uint32_t idesc = make_idesc(0, 128, N);
#pragma unroll
  for (int i = 0; i < CNT; i++) {
    if (i == 0) tc_mma<0>(tmem_col, desc_from_lo(a_lo), desc_from_lo(b_lo), idesc);
    else tc_mma<1>(tmem_col, desc_from_lo(a_lo + (i & 3) * 256), desc_from_lo(b_lo + (i & 3) * 64), idesc);
  }
  tc_commit(mbar_addr);
}

__global__ void __launch_bounds__(416, 1) k_mma_bench(long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t mbar[16];
  __shared__ long long s_t[16][2];
  const uint32_t sbase = smem_u32(smem);
  const int warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 65536 / 4; i += 416) reinterpret_cast<uint32_t*>(smem)[i] = 0x3c003c00u;  // fp16 ones
  if (threadIdx.x == 0) {
    for (int i = 0; i < 16; i++) mbar_init(smem_u32(&mbar[i]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fence_async_smem();
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const bool leader = elect_one();
  const uint32_t a_lo = (sbase >> 4) + (128u << 16), b_lo = ((sbase + 32768) >> 4) + (32u << 16);
  uint32_t phase = 0;
  // tests: {warp mask, shape}: shape 0 = 4 x N32, 1 = 16 x N32, 2 = 2 x N160, 3 = 8 x N128
  const unsigned masks[12] = {0x1, 0x1, 0x1, 0x1, 0x7, 0x7, 0x111, 0x111, 0x7, 0x111, 0x1111, 0xF};
  const int shapes[12] = {0, 1, 2, 3, 0, 1, 0, 1, 2, 2, 1, 1};
  for (int c = 0; c < 12; c++) {
    for (int rep = 0; rep < 3; rep++) {
      __syncthreads();
      const bool mine = (masks[c] >> warp) & 1;
      long long t0 = clock64(), t1 = t0, t2 = t0;
      if (mine) {
        const uint32_t col = tmem + (warp % 3) * 160;
        const uint32_t mb = smem_u32(&mbar[warp]);
        if (leader) {
          if (shapes[c] == 0) bench_issue<32, 4>(col, a_lo, b_lo, mb);
          else if (shapes[c] == 1) bench_issue<32, 16>(col, a_lo, b_lo, mb);
          else if (shapes[c] == 2) bench_issue<160, 2>(col, a_lo, b_lo, mb);
          else bench_issue<128, 8>(col, a_lo, b_lo, mb);
        }
        __syncwarp();
        t1 = clock64();
        while (!mbar_test(mb, phase)) {}
        t2 = clock64();
      }
      if (mine && leader) { s_t[warp][0] = t1 - t0; s_t[warp][1] = t2 - t0; }
      __syncthreads();
      if (threadIdx.x == 0 && rep == 2) {
        long long a = 0, b = 0;
        for (int w = 0; w < 13; w++) if ((masks[c] >> w) & 1) { a = max(a, s_t[w][0]); b = max(b, s_t[w][1]); }
        out[c * 2] = a; out[c * 2 + 1] = b;
      }
      if (mine) phase ^= 1;   // this warp's barrier completed one phase
      __syncthreads();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
  }
}
}  // namespace fused

extern "C" int srwn_debug_mma_bench(long long* host_out24) {
  long long* d = nullptr;
  SRWN_CUDA(cudaMalloc(&d, 24 * sizeof(long long)));
  SRWN_CUDA(cudaFuncSetAttribute(fused::k_mma_bench, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
  fused::k_mma_bench<<<1, 416, 65536>>>(d);
  SRWN_CUDA(cudaDeviceSynchronize());
  SRWN_CUDA(cudaMemcpy(host_out24, d, 24 * sizeof(long long), cudaMemcpyDeviceToHost));
  cudaFree(d);
  return SRWN_OK;
}
#endif  // SRWN_TUNING
