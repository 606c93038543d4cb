// Parallel prefill of a generation state (srwn_generate_state_prefill): the state that srwn_teacher_generate_resume
// leaves after forcing n known samples, computed over time in parallel instead of step by step.
//
// With every x known there is no sequential dependency.  Let E = t0 + n and D_l = d_l + ... + d_{L-1}.  The state after
// E holds h_l (layer l's input) over [E - d_l, E); h_{l+1}[t] needs h_l[t] and h_l[t - d_l]; so layer l is needed over
// [E - D_l, E) only, and layer 0 needs x over [E - D_0 - 2, E - 1].  The result depends on the last D_0 + 2 samples
// and, where that window reaches before t0, on the state itself: taps before t0 read the state's queues (which hold
// h_l over [t0 - d_l, t0)) and x before t0 its x history.  Work and memory are therefore flat in n once n passes the
// window.
//
// One launch per layer, parallel over (utterance, position) rows; the fp32 residual stream of the window lives in two
// workspace buffers (layer l's input, layer l+1's output).  After layer l, its last d_l inputs go to the queue slots
// (t0 + i) mod d_l in the layout of the step kernel; that copy waits for the layer's launch because the layer's taps
// before t0 read the same slots.
//
// Each precision reproduces its step kernel's arithmetic per row, so the state is byte for byte the one the step
// kernel leaves:
//   * fp16 (k_ar_mma): mma.sync m16n8k16 on the same fragments, the filter conv as a tap chain and a current chain,
//     (acc + acc2) + b, gate(), the residual conv from zero, fmaf(h + r, sqrt(1/2), cb[l+1]) on an fp32 stream, the
//     front as fmaf(x[t-2], fk0, fmaf(x[t-1], fk1, cb0)) with cb from k_cond + fused::k_fold_bias.  Time steps fill
//     all 16 rows of each MMA (the step kernel uses 8); this rests on a row's result depending only on that row's
//     operands, which the GPU tests check by equality.
//   * fp32 (k_ar_generate): the FFMA sums in the step kernel's order.
#include "common.cuh"
#include "gen_state.cuh"
#include "ar_mma.cuh"
#include <algorithm>

namespace prefill {

constexpr int kThreads = 256;

// Rows of the window: buffer row r is position i = base + r of the call (i < 0 lies before t0).  The fp16 buffers keep
// a lane's eight channels together: float q*8 + k of a row is channel 8*(k/2) + 2q + (k%2), i.e. n-tile k/2 of the
// lane (g, q) fragment, so a row is read and written as two 16-byte vectors per lane.
struct Layer {
  const float* hin;          // [Bp][Wr][32] h_l over rows [0, Wr)
  float* hout;               // [Bp][Wr][32] h_{l+1} over rows [r0, Wr)
  const void* queues;        // state queues: taps before t0
  const long long* t0;
  const uint8_t* chain;      // fp16: fragment image of layer l (ar_mma_pack_weights)
  const float* w;            // fp32: stack weights
  StackOffsets off;
  const float* cond;         // fp32: [B][NF][L][32] (k_cond); fp16: [B][NF][L+1][32] folded (k_fold_bias)
  int B, Bp, Wr, base, r0, l, L, d, qoff, sum_d, P, fb, NF;
};

// ---- fp16: one warp per tile of 16 consecutive positions of one utterance ------------------------------------------
__global__ void __launch_bounds__(kThreads) k_prefill_mma(const Layer p) {
  using namespace armma;
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int warp = (blockIdx.x * kThreads + threadIdx.x) >> 5, nwarps = (gridDim.x * kThreads) >> 5;
  uint4 wft[4], wfc[4], wr[4];
  float fb[8];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    wft[j] = *reinterpret_cast<const uint4*>(p.chain + (2 * j) * kFragBytes + lane * 16);
    wfc[j] = *reinterpret_cast<const uint4*>(p.chain + (2 * j + 1) * kFragBytes + lane * 16);
    wr[j] = *reinterpret_cast<const uint4*>(p.chain + kChainWr + j * kFragBytes + lane * 16);
    fb[2 * j] = reinterpret_cast<const float*>(p.chain + kChainBias)[8 * j + 2 * q];
    fb[2 * j + 1] = reinterpret_cast<const float*>(p.chain + kChainBias)[8 * j + 2 * q + 1];
  }
  const int rows = p.Wr - p.r0, tpb = (rows + 15) / 16;
  for (int tile = warp; tile < p.Bp * tpb; tile += nwarps) {
    const int b = tile / tpb, rt = p.r0 + (tile % tpb) * 16;
    float cur[2][8];                                  // rows g, g+8: channels of n-tiles 0..3 (pairs)
    uint32_t tap[2][4];                               // their taps, fp16 pairs by n-tile
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int r = min(rt + g + 8 * h, p.Wr - 1);   // rows past the window repeat the last one and are not stored
      const float4* src = reinterpret_cast<const float4*>(p.hin + ((size_t)b * p.Wr + r) * 32 + q * 8);
      const float4 v0 = src[0], v1 = src[1];
      cur[h][0] = v0.x; cur[h][1] = v0.y; cur[h][2] = v0.z; cur[h][3] = v0.w;
      cur[h][4] = v1.x; cur[h][5] = v1.y; cur[h][6] = v1.z; cur[h][7] = v1.w;
      const int i = p.base + r;
      if (i - p.d >= 0) {
        const float4* ts = reinterpret_cast<const float4*>(p.hin + ((size_t)b * p.Wr + r - p.d) * 32 + q * 8);
        const float4 t0v = ts[0], t1v = ts[1];
        tap[h][0] = pack_h2(t0v.x, t0v.y); tap[h][1] = pack_h2(t0v.z, t0v.w);
        tap[h][2] = pack_h2(t1v.x, t1v.y); tap[h][3] = pack_h2(t1v.z, t1v.w);
      } else {                                        // before t0: the state's slot
        gen_f16_unpack(*reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(p.queues) +
                                                       gen_f16_offset(b, q, p.sum_d, p.qoff, gen_slot(p.t0, i, p.d))),
                       tap[h]);
      }
    }
    uint32_t hA[2][4];
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
      for (int j = 0; j < 4; j++) hA[h][j] = pack_h2(cur[h][2 * j], cur[h][2 * j + 1]);
    // filter conv, n-tile j: taps (k-tile 0, then 1) in acc, current (k-tile 0, then 1) in acc2
    float acc[4][4], acc2[4][4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
      for (int e = 0; e < 4; e++) { acc[j][e] = 0.f; acc2[j][e] = 0.f; }
      mma8q(acc2[j], hA[0][0], hA[1][0], hA[0][1], hA[1][1], wfc[j].x, wfc[j].y);
      mma8q(acc[j], tap[0][0], tap[1][0], tap[0][1], tap[1][1], wft[j].x, wft[j].y);
      mma8q(acc2[j], hA[0][2], hA[1][2], hA[0][3], hA[1][3], wfc[j].z, wfc[j].w);
      mma8q(acc[j], tap[0][2], tap[1][2], tap[0][3], tap[1][3], wft[j].z, wft[j].w);
    }
    uint32_t cA[2][4];                                // gate output, fp16 pairs by n-tile
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
      for (int h = 0; h < 2; h++)
        cA[h][j] = pack_h2(gate(acc[j][2 * h] + acc2[j][2 * h] + fb[2 * j]),
                           gate(acc[j][2 * h + 1] + acc2[j][2 * h + 1] + fb[2 * j + 1]));
    // residual conv (k-tile 0, then 1, from zero) and the fp32 stream update with the next layer's folded term
    float rr[4][4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
      for (int e = 0; e < 4; e++) rr[j][e] = 0.f;
      mma8q(rr[j], cA[0][0], cA[1][0], cA[0][1], cA[1][1], wr[j].x, wr[j].y);
      mma8q(rr[j], cA[0][2], cA[1][2], cA[0][3], cA[1][3], wr[j].z, wr[j].w);
    }
    const int bc = min(b, p.B - 1);                   // padding rows of the last group carry the last utterance's terms
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int r = rt + g + 8 * h;
      if (r >= p.Wr) continue;
      const int i = p.base + r;
      const float* cbf = p.cond + (((size_t)bc * p.NF + (i / p.P - p.fb)) * (p.L + 1) + p.l + 1) * 32 + 2 * q;
      float o[8];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const float2 cb = *reinterpret_cast<const float2*>(cbf + 8 * j);
        o[2 * j] = fmaf(cur[h][2 * j] + rr[j][2 * h], SRWN_SQRT_HALF, cb.x);
        o[2 * j + 1] = fmaf(cur[h][2 * j + 1] + rr[j][2 * h + 1], SRWN_SQRT_HALF, cb.y);
      }
      float4* dst = reinterpret_cast<float4*>(p.hout + ((size_t)b * p.Wr + r) * 32 + q * 8);
      dst[0] = make_float4(o[0], o[1], o[2], o[3]);
      dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
  }
}

// ---- fp32: one warp per row, lane = output channel -------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_prefill_f32(const Layer p) {
  __shared__ float s_in[kThreads / 32][2][kR], s_c[kThreads / 32][kR];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * kThreads + threadIdx.x) >> 5, nwarps = (gridDim.x * kThreads) >> 5;
  const float* W = p.w;
  const StackOffsets& o = p.off;
  float wf[2 * kR], wr[kR];
#pragma unroll
  for (int k = 0; k < 2 * kR; k++) wf[k] = W[o.filt_k + (size_t)p.l * 2 * kR * kR + (size_t)k * kR + lane];
#pragma unroll
  for (int k = 0; k < kR; k++) wr[k] = W[o.res_k + (size_t)p.l * kR * kR + (size_t)k * kR + lane];
  const float bf = W[o.filt_b + p.l * kR + lane], br = W[o.res_b + p.l * kR + lane];
  const int rows = p.Wr - p.r0;
  for (int row = warp; row < p.B * rows; row += nwarps) {
    const int b = row / rows, r = p.r0 + row % rows, i = p.base + r;
    const float cur = p.hin[((size_t)b * p.Wr + r) * kR + lane];
    const float tap = i - p.d >= 0 ? p.hin[((size_t)b * p.Wr + r - p.d) * kR + lane]
                                   : static_cast<const float*>(p.queues)[gen_f32_row(b, p.sum_d, p.qoff, gen_slot(p.t0, i, p.d)) * kR + lane];
    __syncwarp();
    s_in[wib][0][lane] = tap;
    s_in[wib][1][lane] = cur;
    __syncwarp();
    float f = bf;
#pragma unroll
    for (int kq = 0; kq < 8; kq++) {
      const float* a = &s_in[wib][kq >> 2][(kq & 3) * 8];
      float acc = 0.f;
#pragma unroll
      for (int kk = 0; kk < 8; kk++) acc = fmaf(a[kk], wf[kq * 8 + kk], acc);
      f += acc;
    }
    f = tanhf(f);
    s_c[wib][lane] = f * (1.0f / (1.0f + expf(-f)));
    __syncwarp();
    float acc = br;
#pragma unroll
    for (int k = 0; k < kR; k++) acc = fmaf(s_c[wib][k], wr[k], acc);
    const float c1 = p.cond[(((size_t)b * p.NF + (i / p.P - p.fb)) * p.L + p.l + 1) * kR + lane];
    p.hout[((size_t)b * p.Wr + r) * kR + lane] = __fadd_rn(__fmul_rn(__fadd_rn(cur, acc), SRWN_SQRT_HALF), c1);
  }
}

// ---- front (layer-0 input) over the whole window, reading x before t0 from the x history -----------------------------
template <bool FP16>
__global__ void k_prefill_front(const float* __restrict__ x, const float* __restrict__ xhist, const float* __restrict__ fk,
                                const float* __restrict__ fbias, const float* __restrict__ cond, float* __restrict__ h,
                                int B, int Bp, int n, int Wr, int base, int P, int fb, int NF, int L) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)Bp * Wr * kR) return;
  const int k = (int)(idx % kR), r = (int)((idx / kR) % Wr), b = (int)(idx / ((int64_t)kR * Wr));
  const int c = FP16 ? 8 * ((k & 7) >> 1) + 2 * (k >> 3) + (k & 1) : k;       // channel of float k of the row
  const int i = base + r;
  auto xat = [&](int t) {                            // x at position t of the call; padding utterances are silent
    if (b >= B) return 0.f;
    return t >= 0 ? x[(size_t)b * n + t] : xhist[2 * b + (-1 - t)];
  };
  const float xm1 = xat(i - 1), xm2 = xat(i - 2);
  const int bc = min(b, B - 1), f = i / P - fb;
  float v;
  if (FP16) {
    v = fmaf(xm2, fk[c], fmaf(xm1, fk[kR + c], cond[((size_t)bc * NF + f) * (L + 1) * kR + c]));
  } else {
    v = fmaf(xm2, fk[c], fmaf(xm1, fk[kR + c], fbias[c]));
    v = __fadd_rn(v, cond[((size_t)bc * NF + f) * L * kR + c]);
  }
  h[idx] = v;
}

// ---- the last d_l inputs of layer l -> its queue slots (t0 + i) mod d_l ------------------------------------------------
__global__ void k_prefill_commit_mma(const float* __restrict__ h, uint8_t* __restrict__ queues, const long long* t0,
                                     int Bp, int Wr, int base, int r0, int d, int qoff, int sum_d) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int rows = Wr - r0;
  if (idx >= (int64_t)Bp * rows * 4) return;
  const int q = (int)(idx & 3), r = r0 + (int)((idx >> 2) % rows), b = (int)((idx >> 2) / rows);
  const float4* src = reinterpret_cast<const float4*>(h + ((size_t)b * Wr + r) * kR + q * 8);
  const float4 v0 = src[0], v1 = src[1];
  const uint32_t w[4] = {armma::pack_h2(v0.x, v0.y), armma::pack_h2(v0.z, v0.w), armma::pack_h2(v1.x, v1.y),
                         armma::pack_h2(v1.z, v1.w)};
  *reinterpret_cast<uint4*>(queues + gen_f16_offset(b, q, sum_d, qoff, gen_slot(t0, base + r, d))) = gen_f16_pack(w);
}

__global__ void k_prefill_commit_f32(const float* __restrict__ h, float* __restrict__ queues, const long long* t0,
                                     int B, int Wr, int base, int r0, int d, int qoff, int sum_d) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int rows = Wr - r0;
  if (idx >= (int64_t)B * rows * kR) return;
  const int c = (int)(idx % kR), r = r0 + (int)((idx / kR) % rows), b = (int)(idx / ((int64_t)kR * rows));
  queues[gen_f32_row(b, sum_d, qoff, gen_slot(t0, base + r, d)) * kR + c] = h[((size_t)b * Wr + r) * kR + c];
}

// x history after the prefill: x[E-1], x[E-2]
__global__ void k_prefill_xhist(const float* __restrict__ x, float* __restrict__ xhist, int B, int n) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float xm2 = n >= 2 ? x[(size_t)b * n + n - 2] : xhist[2 * b];
  xhist[2 * b] = x[(size_t)b * n + n - 1];
  xhist[2 * b + 1] = xm2;
}

// the latent frames of the window, [B][NF][C], out of the call's [B][n/P][C]
__global__ void k_prefill_gather_enc(const float* __restrict__ enc, float* __restrict__ out, int B, int frames, int fb,
                                     int NF, int C) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)B * NF * C) return;
  const int ch = (int)(idx % C), f = (int)((idx / C) % NF), b = (int)(idx / ((int64_t)C * NF));
  out[idx] = enc[((size_t)b * frames + fb + f) * C + ch];
}

}  // namespace prefill

// ---- host -------------------------------------------------------------------------------------------
namespace {
struct PrefillWs { float* h[2]; float* enc; float* cond; float* cb; size_t bytes; };

// Sized by B and the window min(n, sum(d) + 2) only: a prime of any length runs in the same memory.
PrefillWs carve_prefill(const srwn_ctx* c, int B, int n, int precision, void* ws) {
  WsCarver w(ws, 0);
  PrefillWs r{};
  const int nw = std::min(n, c->sum_dilation + 2), P = c->cfg.pool_stride, L = c->cfg.n_layers;
  const size_t Bp = precision == SRWN_FP16 ? (size_t)(B + 7) / 8 * 8 : (size_t)B;
  const size_t frames = (size_t)(nw + P - 1) / P;   // the window ends on a frame boundary (n % P == 0)
  r.h[0] = w.take<float>(Bp * nw * kR);
  r.h[1] = w.take<float>(Bp * nw * kR);
  r.enc = w.take<float>((size_t)B * frames * c->cfg.cond_channels);
  r.cond = w.take<float>((size_t)B * frames * L * kR);
  if (precision == SRWN_FP16) r.cb = w.take<float>((size_t)B * frames * (L + 1) * kR);
  r.bytes = w.used;
  return r;
}

unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }
}  // namespace

size_t prefill_workspace_bytes(const srwn_ctx* c, int B, int n, int precision) {
  return carve_prefill(c, B, n, precision, nullptr).bytes;
}

int run_prefill(srwn_ctx* c, const GenState& s, const float* x, const float* enc, int B, int n, int precision, void* ws,
                size_t ws_bytes, cudaStream_t st) {
  const bool fp16 = precision == SRWN_FP16;
  const PrefillWs w = carve_prefill(c, B, n, precision, ws);
  if (int rc = check_workspace(ws, ws_bytes, w.bytes)) return rc;
  const int L = c->cfg.n_layers, P = c->cfg.pool_stride, C = c->cfg.cond_channels, sum_d = c->sum_dilation;
  const int Bp = fp16 ? (B + 7) / 8 * 8 : B;
  std::vector<int> D(L + 1, 0), qoff(L, 0);           // D[l] = d_l + ... + d_{L-1}
  for (int l = L - 1; l >= 0; l--) D[l] = D[l + 1] + c->dilations[l];
  for (int l = 1; l < L; l++) qoff[l] = qoff[l - 1] + c->dilations[l - 1];
  const int Wr = std::min(n, D[0]), base = n - Wr;   // rows of the window: positions base .. n-1
  const int fb = base / P, NF = n / P - fb;
  const float* sw = stack_w(c, 0);

  prefill::k_prefill_gather_enc<<<blocks_for((int64_t)B * NF * C, 256), 256, 0, st>>>(enc, w.enc, B, n / P, fb, NF, C);
  SRWN_LAUNCH_CHECK();
  k_cond<<<B * NF, 256, 0, st>>>(w.enc, sw + c->off.cond_k, sw + c->off.cond_b, w.cond, B * NF, L, C);
  SRWN_LAUNCH_CHECK();
  if (fp16) {
    fused::k_fold_bias<<<B * NF, 256, 0, st>>>(w.cond, sw + c->off.front_b, sw + c->off.res_b, w.cb, L);
    SRWN_LAUNCH_CHECK();
  }
  {
    const int64_t nt = (int64_t)Bp * Wr * kR;
    if (fp16)
      prefill::k_prefill_front<true><<<blocks_for(nt, 256), 256, 0, st>>>(x, s.xhist, sw + c->off.front_k, nullptr, w.cb, w.h[0],
                                                                          B, Bp, n, Wr, base, P, fb, NF, L);
    else
      prefill::k_prefill_front<false><<<blocks_for(nt, 256), 256, 0, st>>>(x, s.xhist, sw + c->off.front_k, sw + c->off.front_b,
                                                                           w.cond, w.h[0], B, Bp, n, Wr, base, P, fb, NF, L);
    SRWN_LAUNCH_CHECK();
  }
  const uint8_t* img = static_cast<const uint8_t*>(c->d_ar_packed);
  for (int l = 0; l < L; l++) {
    const float* hin = w.h[l & 1];
    if (l + 1 < L) {                                  // h_{l+1} over [n - D_{l+1}, n); the last layer's output is unused
      prefill::Layer p;
      p.hin = hin; p.hout = w.h[(l + 1) & 1]; p.queues = s.queues; p.t0 = s.t0;
      p.chain = fp16 ? img + (size_t)l * armma::kChainLayerBytes : nullptr;
      p.w = sw; p.off = c->off; p.cond = fp16 ? w.cb : w.cond;
      p.B = B; p.Bp = Bp; p.Wr = Wr; p.base = base; p.r0 = std::max(0, n - D[l + 1]) - base; p.l = l; p.L = L;
      p.d = c->dilations[l]; p.qoff = qoff[l]; p.sum_d = sum_d; p.P = P; p.fb = fb; p.NF = NF;
      const int rows = Wr - p.r0;
      const int64_t warps = fp16 ? (int64_t)Bp * ((rows + 15) / 16) : (int64_t)B * rows;
      const unsigned grid = (unsigned)std::min<int64_t>((warps + 7) / 8, (int64_t)c->sm_count * 8);
      if (fp16) prefill::k_prefill_mma<<<grid, prefill::kThreads, 0, st>>>(p);
      else prefill::k_prefill_f32<<<grid, prefill::kThreads, 0, st>>>(p);
      SRWN_LAUNCH_CHECK();
    }
    // layer l's inputs at [n - d_l, n) -> queue slots; after the launch above, whose taps before t0 read those slots
    const int r0 = std::max(0, n - c->dilations[l]) - base;
    if (fp16)
      prefill::k_prefill_commit_mma<<<blocks_for((int64_t)Bp * (Wr - r0) * 4, 256), 256, 0, st>>>(
          hin, static_cast<uint8_t*>(s.queues), s.t0, Bp, Wr, base, r0, c->dilations[l], qoff[l], sum_d);
    else
      prefill::k_prefill_commit_f32<<<blocks_for((int64_t)B * (Wr - r0) * kR, 256), 256, 0, st>>>(
          hin, static_cast<float*>(s.queues), s.t0, B, Wr, base, r0, c->dilations[l], qoff[l], sum_d);
    SRWN_LAUNCH_CHECK();
  }
  prefill::k_prefill_xhist<<<blocks_for(B, 128), 128, 0, st>>>(x, s.xhist, B, n);
  SRWN_LAUNCH_CHECK();
  return run_gen_state_advance(s.t0, n, st);
}
