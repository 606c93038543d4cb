// Student layer kernels on tcgen05 (kind::tf32, 3xTF32 split): the forward for the fp32-grade stack (stack_f32.cu),
// the two backward kernels for the distillation step (train_f32.cu).
#pragma once
#include "common.cuh"

namespace traintc {

constexpr int kThreads = 576;      // 16 worker warps + 2 issuing warps
int fwd_smem_bytes();
int gate_smem_bytes();
int conv_smem_bytes();

// x_{l+1} = (x_l + c Wr + br) sqrt(1/2) + cond_{l+1}   (ops.py:23-46 without the skip output, model.py:415-454)
__global__ void k_fwd_layer_tc(const float* __restrict__ x_l, float* __restrict__ x_next, const float* __restrict__ filt_k,
                               const float* __restrict__ filt_b, const float* __restrict__ res_k, const float* __restrict__ res_b,
                               const float* __restrict__ cond_next, int B, int T, int d, int P, int L, int frames);
// g = dL/dx_{l+1} -> da = dL/da (pre-activation of the filter conv); partial[cta] = dWr [32][32] | dbr [32]
__global__ void k_bwd_gate_tc(const float* __restrict__ x_l, const float* __restrict__ g_in, float* __restrict__ da_out,
                              const float* __restrict__ filt_k, const float* __restrict__ filt_b, const float* __restrict__ res_k,
                              float* __restrict__ partial, int B, int T, int d);
// dx_l = g sqrt(1/2) + da W1^T + da[t+d] W0^T; partial[cta] = dWf [64][32] | dbf [32]; dcond[b][t/P] += dx_l[t]
__global__ void k_bwd_conv_tc(const float* __restrict__ x_l, const float* __restrict__ g_in, const float* __restrict__ da_in,
                              float* __restrict__ dx_out, const float* __restrict__ filt_k, float* __restrict__ partial,
                              float* __restrict__ dcond, int B, int T, int d, int P, int frames);

}  // namespace traintc
