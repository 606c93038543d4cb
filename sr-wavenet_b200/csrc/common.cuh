// Shared declarations for libsrwn.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stddef.h>
#include <string>
#include <vector>
#include "../../include/srwn.h"

#define SRWN_SQRT_HALF 0.7071067811865476f   // literal at ops.py:40

// Kernels are specialised for the hyper-parameters teacher.py:55-62 / student.py:70-73 use.
constexpr int kR = 32;    // dilation_channels
constexpr int kS = 128;   // skip_channels
constexpr int kK = 2;     // filter_width
constexpr int kMaxCond = 64;
constexpr int kMaxLogit = 32;  // 4*M padded

// ---- error plumbing ---------------------------------------------------------------
int srwn_fail(int code, const char* fmt, ...);
void srwn_count_launch(int n = 1);

#define SRWN_CUDA(expr)                                                              \
  do {                                                                               \
    cudaError_t _e = (expr);                                                         \
    if (_e != cudaSuccess)                                                           \
      return srwn_fail(SRWN_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                \
                       cudaGetErrorString(_e), __FILE__, __LINE__);                  \
  } while (0)

#define SRWN_LAUNCH_CHECK()                                                          \
  do {                                                                               \
    srwn_count_launch();                                                             \
    cudaError_t _e = cudaGetLastError();                                             \
    if (_e != cudaSuccess)                                                           \
      return srwn_fail(SRWN_ERR_CUDA, "kernel launch failed: %s (%s:%d)",            \
                       cudaGetErrorString(_e), __FILE__, __LINE__);                  \
  } while (0)

// ---- device weight arena ----------------------------------------------------------
// One "stack" = one decoder (teacher) or one flow (student).  All fp32, TF layout
// ([Cin][Cout] row-major for 1x1 kernels, [K][Cin][Cout] for the dilated convs).
struct StackOffsets {
  size_t front_k, front_b;            // [2][R], [R]            causal_conv (model.py:173/424)
  size_t cond_k, cond_b;              // [L][C][R], [L][R]      model.py:180/431
  size_t filt_k, filt_b;              // [L][2][R][R], [L][R]   ops.py:27
  size_t res_k, res_b;                // [L][R][R], [L][R]      ops.py:39
  size_t skip_k, skip_b;              // [L][R][S], [L][S]      ops.py:44 (teacher only)
  size_t head1_k, head1_b;            // teacher [S][S],[S]     model.py:193 ; student [R][2],[2] model.py:452
  size_t head2_k, head2_b;            // teacher [S][4M],[4M]   model.py:196
  size_t skip_b_sum;                  // [S] sum over layers of skip_b (derived at commit)
  size_t end;
};

struct srwn_ctx {
  srwn_config_t cfg;
  std::vector<int32_t> dilations;
  int n_stacks;                       // 1 (teacher) or num_flows
  StackOffsets off;                   // offsets (in floats) inside one stack
  size_t stack_floats;
  float* d_weights;                   // n_stacks * stack_floats
  std::vector<uint8_t> is_set;        // per (stack, variable)
  int32_t* d_dilations;
  int sum_dilation;                   // sum of dilations (queue rows per utterance)
  int32_t* d_queue_off;               // [L] prefix sums of dilations
  bool committed;
  bool device_dirty;                  // device weights changed by srwn_adam_step: host mirror and packed images are stale
  int device;
  int sm_count;
  // packed fp16 operand images of the fused kernel, one per stack (built at commit)
  void* d_packed;
  size_t packed_bytes;
  void* d_part;                       // work partition of the fused kernel for (part_B, part_T, team size): segs | nseg (allocated at create)
  int part_B, part_T, part_team_req, part_teams, part_G;
  std::vector<uint8_t> part_host;     // host staging of d_part
  int team_size;                      // srwn_set_team_size: CTAs per team of the fused kernel, 0 = chosen per (B, T)
  long long wait_limit_clocks;        // srwn_set_wait_limit: how long a fused-kernel pipeline wait may spin before aborting
  int* h_err;                         // pinned, mapped: abort words of the fused kernel [flag, code, chunk, cta]
  void* d_ar_packed;                  // fragment-ordered fp16 weights of the tensor-core generation kernel (built at commit)
  // optional timing of the dominant kernel(s) of the last call (srwn_set_profiling)
  int profiling;
  cudaEvent_t prof_ev[2];
  int prof_launches;
  const char* prof_name;
};

// brackets the dominant kernel launches of a call with CUDA events on the launch stream; name == nullptr times nothing
struct ProfScope {
  srwn_ctx* c; cudaStream_t st; bool on;
  ProfScope(srwn_ctx* c_, cudaStream_t st_, const char* name, int launches) : c(c_), st(st_), on(c_->profiling && name) {
    if (on) { c->prof_name = name; c->prof_launches = launches; cudaEventRecord(c->prof_ev[0], st); }
  }
  ~ProfScope() { if (on) cudaEventRecord(c->prof_ev[1], st); }
};

// ---- programmatic dependent launch (PDL) of the layer kernels -----------------------------------------
// A layer kernel launched with launch_dependent may start (and stage its weights) while the previous kernel on the stream
// drains; everything the previous launch wrote is visible after grid_dependency_wait (a no-op in a plain launch).  The
// trigger right after it lets the NEXT launch's CTAs take the SM slots this grid frees as its CTAs exit (all of this
// grid's CTAs are resident from the start, so nothing of it can be starved).
__device__ __forceinline__ void grid_dependency_wait() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <typename... KArgs, typename... Args>
cudaError_t launch_dependent(void (*kern)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

inline const float* stack_w(const srwn_ctx* c, int stack) {
  return c->d_weights + (size_t)stack * c->stack_floats;
}

// ---- workspace carving ------------------------------------------------------------
struct WsCarver {
  uint8_t* base; size_t used; size_t cap;
  __host__ WsCarver(void* p, size_t cap_) : base((uint8_t*)p), used(0), cap(cap_) {}
  template <typename T> __host__ T* take(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
    T* r = (T*)(base ? base + used : nullptr);
    used += bytes;
    return r;
  }
};

// on-device noise (philox.cuh): element i of (seed, stream); `on` = 0 means the caller supplied the tensor
struct NoiseSpec { unsigned long long seed, stream; int on; };

// The parts of a generation state (gen_state.cuh) a generation kernel reads and writes.
struct GenState {
  long long* t0;              // position of step 0 of the call; advanced by T after the kernel
  float* xhist;               // [B][2]: x[t0-1], x[t0-2]
  void* queues;               // dilation queues in the precision's layout (gen_state.cuh)
};

// ---- kernels and entry points implemented across translation units ------------------
// api.cu
int check_bt(const srwn_ctx* c, int B, int T);
const float* srwn_host_weights(srwn_ctx* c);
// stack_f32.cu
__global__ void k_cond(const float* __restrict__ enc, const float* __restrict__ cond_k,
                       const float* __restrict__ cond_b, float* __restrict__ cond,
                       int frames_total, int L, int C);
__global__ void k_front(const float* __restrict__ x, const float* __restrict__ fk,
                        const float* __restrict__ fb, const float* __restrict__ cond,
                        float* __restrict__ hc, int T, int P, int L, int frames);
// h1 == nullptr keeps every layer input: h0 is then [L+1][B][T][R] (the training forward, not profiled)
int run_stack_f32(srwn_ctx* c, int stack, const float* xin, const float* enc, int B, int T,
                  float* h0, float* h1, float* skip, float* cond, float** h_final,
                  cudaStream_t st);
int run_teacher_head_f32(srwn_ctx* c, const float* skip, float* logits, int B, int T,
                         cudaStream_t st);
int run_flow_head_f32(srwn_ctx* c, int stack, const float* h, const float* xin, float* scale,
                      float* mean, float* xout, int B, int T, cudaStream_t st);
int run_flow_compose(const float* z, NoiseSpec noise, float* z_out, const float* scales, const float* means, int F,
                     float* out, float* s_tot, float* mu_tot, int64_t n, cudaStream_t st);
// random.cu
int run_random_fill(float* out, int64_t n, uint64_t seed, uint64_t stream, int logistic, float lo, float hi, cudaStream_t st);
// mol.cu
int run_mol_loss(const float* x, const float* l, float* nll_out, float* nll_sum,
                 int B, int T, int M, cudaStream_t st);
int run_mol_sample(const float* l, const float* u1, const float* u2, float* out,
                   int32_t* idx_out, int B, int T, int M, cudaStream_t st);
// ar_generate.cu
size_t ar_workspace_bytes(const srwn_ctx* c, int B, int T);
// rs == null: one call from silence; otherwise resume from (and advance) the caller's state.  For t < n_prefix, x[t]
// is x_prefix [B][n_prefix] instead of a draw (resumed calls only).
int run_ar_generate(srwn_ctx* c, const float* enc, const float* u1, const float* u2,
                    float* x_out, float* logits_out, int B, int T, void* ws, size_t ws_bytes,
                    cudaStream_t st, const GenState* rs, const float* x_prefix, int n_prefix);
// train_f32.cu
size_t train_workspace_bytes(const srwn_ctx* c, int B, int T);
int run_student_forward_train(srwn_ctx* c, const float* z, const float* enc, float* out, float* s_tot,
                              float* mu_tot, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st);
int run_student_backward(srwn_ctx* c, const float* z, const float* enc, const float* d_pre, const float* d_s_extra,
                         float* grads, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st);
int run_mol_nll_grad(const float* x, const float* l, float* dx, float* nll, int B, int T, int M, cudaStream_t st);
int run_distill_finish(const double* sums, const double* power, float alpha, float beta, float inv_norm, float* out2, cudaStream_t st);
int run_clip_by_global_norm(float* grads, int64_t n, float clip, float* scratch1, cudaStream_t st);
int run_axpy(float* y, const float* x, float a, int64_t n, cudaStream_t st);
int run_entropy(const float* s_tot, double* per_example, int B, int T, cudaStream_t st);
int run_adam(srwn_ctx* c, const float* grads, float* m, float* v, float* scratch1, float clip, float lr, float b1, float b2,
             float eps, int step, cudaStream_t st);
// ar_mma.cu
bool ar_mma_supported(const srwn_ctx* c);
int ar_mma_pack_weights(srwn_ctx* c, cudaStream_t st);
size_t ar_mma_workspace_bytes(const srwn_ctx* c, int B, int T);
int run_ar_mma(srwn_ctx* c, const float* enc, const float* u1, const float* u2, float* x_out,
               float* logits_out, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st, const GenState* rs,
               const float* x_prefix, int n_prefix);
int ar_mma_check_error(const srwn_ctx* c, int B, int T, void* ws, size_t ws_bytes, cudaStream_t st);
// ar_prefill.cu: the state srwn_teacher_generate_resume leaves after forcing x [B][n], computed in parallel
size_t prefill_workspace_bytes(const srwn_ctx* c, int B, int n, int precision);
int run_prefill(srwn_ctx* c, const GenState& s, const float* x, const float* enc, int B, int n, int precision, void* ws,
                size_t ws_bytes, cudaStream_t st);
// fused.cu
namespace fused {
__global__ void k_fold_bias(const float* __restrict__ cond, const float* __restrict__ front_b,
                            const float* __restrict__ res_b, float* __restrict__ cb, int L);
}
bool fused_supported(const srwn_ctx* c);
size_t fused_packed_bytes(const srwn_ctx* c);
int fused_pack_weights(srwn_ctx* c, cudaStream_t st);
size_t fused_workspace_bytes(const srwn_ctx* c, int op, int B, int T);
int run_teacher_fused(srwn_ctx* c, const float* x_in, const float* enc,
                      const float* x_scored, float* nll_out, float* nll_sum,
                      float* logits_out, int B, int T, void* ws, size_t ws_bytes,
                      cudaStream_t st);
int run_student_fused(srwn_ctx* c, const float* z, NoiseSpec noise, float* z_out, const float* enc, float* out,
                      float* s_tot, float* mu_tot, float* x_last, int B, int T,
                      void* ws, size_t ws_bytes, cudaStream_t st);
int fused_check_error(void* ws, size_t ws_bytes, const srwn_ctx* c, int B, int T, cudaStream_t st);
size_t fused_partition_bytes(const srwn_ctx* c);
void fused_last_partition(const srwn_ctx* c, int* teams, int* G);
