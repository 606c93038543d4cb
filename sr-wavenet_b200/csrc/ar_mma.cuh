// Device arithmetic shared by the tensor-core generation kernel (ar_mma.cu) and the parallel prefill (ar_prefill.cu).
// The prefill reproduces the generation kernel's state bit for bit, so both must evaluate a layer with these exact
// functions: keep them in one place.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>
#include "gen_state.cuh"

namespace armma {

constexpr int kU = kGenGroup;                         // utterances per CTA: one group of the fp16 queues
constexpr int kSlotBytes = kGenSlotBytes;             // queue slot / gate output of one layer: [lane][4 x b32]
// A layer's chain image (ar_mma_pack_weights): filter-conv B fragment pairs 2j (taps) and 2j + 1 (current) of n-tile j |
// residual-conv B fragment pairs j | filter bias (32 fp32).  A fragment pair is 32 lanes x 16 bytes.
constexpr int kFragBytes = 512;
constexpr int kChainWr = 8 * kFragBytes, kChainBias = kChainWr + 4 * kFragBytes;
constexpr int kChainLayerBytes = kChainBias + 32 * 4;

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
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
}  // namespace armma
