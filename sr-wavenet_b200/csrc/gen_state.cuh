// The generation state (srwn_generate_state_*): one format, read and written by the step kernels (ar_generate.cu,
// ar_mma.cu) and the parallel prefill (ar_prefill.cu).  The prefill must leave exactly the bytes the step kernels leave,
// so every queue access goes through the helpers below.
//
// Buffer: header (t0, signature) | x history [B][2] fp32 at byte 256 | dilation queues of the precision:
//   * fp32: [B][sum_d][32] floats, row (b, qoff_l + slot) holds layer l's input at one position;
//   * fp16: groups of 8 utterances (one k_ar_mma CTA), [B/8][sum_d] slots of 512 bytes; utterance u of a group and
//     lane quad q own the 16 bytes at (4u + q) * 16: the fp16 pairs of channels 8j + 2q, 8j + 2q + 1 for n-tiles j in
//     the order {0, 2, 1, 3}, which is the A-fragment quad of the filter conv's k-tile 0 (ar_mma.cuh: mma8q).
// Layer l's input at position t lives in slot t mod d_l of its d_l slots.
//
// The position t0 of a state is always a multiple of pool_stride P: reset sets 0, a resume call needs T % P == 0 and a
// prefill n % P == 0.  Two states therefore agree on latent-frame boundaries and differ only in each layer's queue phase
// t0 mod d_l; srwn_generate_state_splice relies on this when it moves an utterance from one state into another.
#pragma once
#include "common.cuh"

constexpr int kGenGroup = 8;          // fp16 queues: utterances per group
constexpr int kGenSlotBytes = 512;    // fp16 queues: one slot of a group
static_assert(kGenGroup == 8, "gen_f16_offset splits the utterance index with shifts");

size_t gen_queue_bytes(const srwn_ctx* c, int B, int precision);
// Checks the arguments of a call on `state` (the C entry points' order: handle, B, precision, then check_bt(B, T)), then
// that the state was last reset on h for B and precision, without touching the device; fills *s with the state's parts.
int gen_state_open(const srwn_ctx* h, void* state, int B, int T, int precision, GenState* s);
void gen_state_forget(const srwn_ctx* h);    // srwn_destroy: h's states (generation and synthesis) are no longer valid
// host registry of state owners: the handle and signature a state buffer was last reset with
void state_owner_record(const srwn_ctx* h, const void* state, const int32_t* sig, int n);
int state_owner_check(const srwn_ctx* h, const void* state, const int32_t* sig, int n, const char* reset_fn);
int run_gen_state_advance(long long* t0, int T, cudaStream_t st);

// fp32 queues: row of layer l (queue offset qoff), slot `slot`, utterance b
__device__ __forceinline__ size_t gen_f32_row(int b, int sum_d, int qoff, int slot) {
  return (size_t)b * sum_d + qoff + slot;
}
// fp16 queues: byte offset of (utterance b, lane quad q) in slot `slot` of layer l
__device__ __forceinline__ size_t gen_f16_offset(int b, int q, int sum_d, int qoff, int slot) {
  return ((size_t)(b >> 3) * sum_d + qoff + slot) * kGenSlotBytes + ((b & 7) * 4 + q) * 16;
}
// a lane's 16 bytes of an fp16 slot from / to its four words in n-tile order
__device__ __forceinline__ uint4 gen_f16_pack(const uint32_t (&w)[4]) { return make_uint4(w[0], w[2], w[1], w[3]); }
__device__ __forceinline__ void gen_f16_unpack(const uint4 s, uint32_t (&w)[4]) { w[0] = s.x; w[1] = s.z; w[2] = s.y; w[3] = s.w; }
// slot of position *t0 + i of a layer of dilation d, also for i < 0 (before t0)
__device__ __forceinline__ int gen_slot(const long long* t0, int i, int d) {
  const long long t = *t0 + i;
  return (int)(((t % d) + d) % d);
}
