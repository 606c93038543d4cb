/*
 * srwn.h -- C ABI of the B200-native SR-WaveNet hot path (libsrwn.so).
 *
 * The reference (tachitachi/SR-WaveNet) has no FFI: its boundary is the Python API of
 * ops.py / model.py, every call ending in one tf.Session.run.  Each entry point below
 * replaces one such graph evaluation; the reference interface it stands in for is cited
 * as file:line (relative to the reference tree).  The Python shim in
 * sr-wavenet_b200/{ops,model}.py keeps the reference's names and argument meaning and
 * calls these functions through ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - every function returns an int status (SRWN_OK == 0); srwn_last_error() gives the
 *     message of the last failure on the calling thread.
 *   - all tensor pointers are DEVICE pointers owned by the caller, dense, fp32,
 *     channels-last [B, T, C] exactly like the reference's tensors, unless a parameter
 *     is documented as host memory.
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it.
 *   - no hidden allocation after srwn_create/srwn_commit_weights: scratch memory is a
 *     caller-owned workspace sized by srwn_workspace_bytes().
 *   - a handle is not thread-safe; use one handle per GPU / per host thread.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails
 *     with SRWN_ERR_CUDA.
 */
#ifndef SRWN_H_
#define SRWN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRWN_ABI_VERSION 7

enum srwn_status {
  SRWN_OK = 0,
  SRWN_ERR_INVALID = 1,      /* bad argument / shape */
  SRWN_ERR_CUDA = 2,         /* CUDA runtime error (message has the cudaError string) */
  SRWN_ERR_WEIGHTS = 3,      /* unknown / missing / mis-shaped variable */
  SRWN_ERR_UNSUPPORTED = 4,  /* configuration outside what the kernels are built for */
  SRWN_ERR_WORKSPACE = 5     /* workspace too small */
};

enum srwn_kind {
  SRWN_TEACHER = 0,          /* WaveNetAutoEncoder decoder stack, model.py:158-200 */
  SRWN_STUDENT = 1           /* ParallelWaveNet IAF flows,        model.py:415-535 */
};

enum srwn_precision {
  SRWN_FP32 = 0,             /* fp32 FFMA path, parity <= 1e-4 relative */
  SRWN_BF16 = 1,             /* reserved, refused with SRWN_ERR_UNSUPPORTED: bf16 operands miss the 2e-2 logit bound on the
                                30-layer stack (measured 2.5e-2); the 16-bit tensor-core path is SRWN_FP16 */
  SRWN_FP16 = 2              /* same kernel with fp16 MMA operands (8x smaller operand rounding) */
};

enum srwn_op {               /* argument of srwn_workspace_bytes */
  SRWN_OP_TEACHER_LOGITS = 0,
  SRWN_OP_TEACHER_NLL = 1,
  SRWN_OP_TEACHER_GENERATE = 2,
  SRWN_OP_STUDENT_FORWARD = 3,
  SRWN_OP_STUDENT_TRAIN = 4,   /* workspace of srwn_student_forward_train + srwn_student_backward */
  SRWN_OP_TEACHER_PREFILL = 5, /* workspace of srwn_generate_state_prefill (T = its n) */
  SRWN_OP_STUDENT_STREAM = 6   /* workspace of srwn_student_forward_resume (T = its S) */
};

/* Constructor arguments of WaveNetAutoEncoder (model.py:76-77) / ParallelWaveNet
 * (model.py:291-292) that shape the hot path.  `dilations` is the plain list the
 * reference passes (teacher.py:55-57); it is copied. */
typedef struct srwn_config {
  int32_t kind;               /* enum srwn_kind */
  int32_t n_layers;           /* len(dilations) */
  const int32_t* dilations;   /* host pointer, n_layers entries */
  int32_t filter_width;       /* model.py:76 filter_width (kernels are built for 2) */
  int32_t dilation_channels;  /* R, residual channels (32) */
  int32_t skip_channels;      /* S (teacher.py:62 -> 128) */
  int32_t cond_channels;      /* latent_channels + condition_size: width of `encoding` */
  int32_t pool_stride;        /* P: T == P * encoding frames (model.py:183) */
  int32_t num_mixtures;       /* M, teacher only: logits have 4*M channels */
  int32_t num_flows;          /* student only (student.py:71 -> 4) */
} srwn_config_t;

typedef struct srwn_ctx* srwn_handle_t;

/* ---- lifetime ------------------------------------------------------------------- */
int srwn_abi_version(void);
const char* srwn_last_error(void);

/* Replaces graph construction in WaveNetAutoEncoder.__init__/createDecoder
 * (model.py:76-135,158-200) or ParallelWaveNet.__init__/createNetwork
 * (model.py:291-314,489-535).  Allocates the device weight arena on the current device. */
int srwn_create(const srwn_config_t* cfg, srwn_handle_t* out);
int srwn_destroy(srwn_handle_t h);

/* Replaces tf.train.Saver.restore / variable assignment (model.py:217-228,540-555).
 * `name` is the TF variable name (e.g. "WaveNetAutoEncoder/Decoder/conv1d_3/kernel",
 * "ParallelWaveNet/Flow2/Flow2/dilated_conv_7_filter/dilated_conv_7_Kernel"); `data` is
 * HOST fp32 in TF layout ([K,Cin,Cout] kernels).  Dead variables of the reference graph
 * (the `_gate` convs ops.py:31-33; the student's skip convs model.py:438-454) are
 * accepted and ignored.  Returns SRWN_ERR_WEIGHTS for unknown names or wrong shapes. */
int srwn_set_weight(srwn_handle_t h, const char* name, const float* data,
                    const int64_t* shape, int32_t ndim);
/* Reads a variable back (tf.train.Saver.save, model.py:230-239). `data` is HOST memory
 * with room for `count` floats. */
int srwn_get_weight(srwn_handle_t h, const char* name, float* data, int64_t count);
/* Checks that every live variable was set and builds the packed operand images the
 * kernels read (fp16 UMMA layouts, summed skip bias). Must follow any srwn_set_weight. */
int srwn_commit_weights(srwn_handle_t h, void* stream);

/* Synchronises `stream` and reports whether the last fused-kernel call that used this workspace
 * aborted (a bounded on-device pipeline wait expired; outputs are then invalid). */
int srwn_check_async_error(srwn_handle_t h, int32_t op, int32_t B, int32_t T, int32_t precision,
                           void* workspace, size_t workspace_bytes, void* stream);
/* The abort words only (pinned host memory), without synchronising any stream: for callers that keep several launches in
 * flight and have already waited on an event for the launch they ask about.  Does not clear the error. */
int srwn_peek_async_error(srwn_handle_t h);
/* Synchronises `stream` and reports (then clears) the abort words of the fused-kernel calls issued on this handle so far
 * (a bounded on-device pipeline wait expired; the outputs of that call are invalid).  The words live in pinned host
 * memory: once a launch has aborted, every later call on the handle is refused with SRWN_ERR_CUDA until this function
 * has been called, so a caller that keeps its results on the device cannot consume them unnoticed for long. */
/* Fused tensor-core kernel: CTAs per team (teams walk contiguous pieces of the (utterance, chunk) line as a wavefront
 * over chunks and layers, handing the per-layer history rings from CTA to CTA).  0 (default) = chosen per (B, T).
 * Results do not depend on it.  srwn_last_partition reports the choice of the last fused call. */
int srwn_set_team_size(srwn_handle_t h, int32_t ctas_per_team);
/* How many SM clocks a pipeline wait inside the fused kernel may spin before the launch aborts (default 1e9, about half a
 * second; every wait is bounded so that a lost signal surfaces as SRWN_ERR_CUDA instead of a hung GPU). */
int srwn_set_wait_limit(srwn_handle_t h, int64_t clocks);
int srwn_last_partition(srwn_handle_t h, int32_t* teams, int32_t* ctas_per_team);
/* 1 if `op` (enum srwn_op) is built for `precision` with this handle's configuration, else 0. */
int srwn_supports(srwn_handle_t h, int32_t op, int32_t precision);
int srwn_workspace_bytes(srwn_handle_t h, int32_t op, int32_t B, int32_t T,
                         int32_t precision, size_t* bytes);

/* ---- teacher (model.py:158-200) ------------------------------------------------- */
/* get_logits(inputs, encoding) (model.py:279-285): x [B,T] teacher-forcing audio,
 * enc [B,T/P,C] -> logits [B,T,4M]. */
int srwn_teacher_logits(srwn_handle_t h, const float* x, const float* enc, float* logits,
                        int32_t B, int32_t T, int32_t precision,
                        void* workspace, size_t workspace_bytes, void* stream);
/* loss_encoding (model.py:114-115): decoder teacher-forced on x_in, mixture-of-logistics
 * negative log-likelihood of x_scored (the reference scores the same audio; distillation
 * scores the student's output against logits of the real audio, model.py:374).
 * nll_out [B,T] (ops.py:175, sum_all=False) and/or nll_sum [1] (ops.py:172); either
 * may be NULL.  logits_out [B,T,4M] optional (NULL to skip the store). */
int srwn_teacher_nll(srwn_handle_t h, const float* x_in, const float* enc,
                     const float* x_scored, float* nll_out, float* nll_sum,
                     float* logits_out, int32_t B, int32_t T, int32_t precision,
                     void* workspace, size_t workspace_bytes, void* stream);
/* The autoregressive loop of teacher.py:153-170 restated with per-layer dilation
 * queues: x[t] = clip(MoL_sample(logits_t)), logits_t from x[<t] and enc[t/P].
 * u1 [B,T,M], u2 [B,T] are the uniforms of ops.py:187,196 (injected for parity).
 * x_out [B,T]; logits_out [B,T,4M] optional.
 * precision: SRWN_FP32 = fp32 FFMA kernel (parity grade); SRWN_FP16 = tensor-core kernel
 * (mma.sync, fp16 operands and queue state, fp32 accumulate and residual stream). */
int srwn_teacher_generate(srwn_handle_t h, const float* enc, const float* u1,
                          const float* u2, float* x_out, float* logits_out,
                          int32_t B, int32_t T, int32_t precision,
                          void* workspace, size_t workspace_bytes, void* stream);
/* Resumable generation: the same recurrence continued across calls through a caller-owned DEVICE state (streaming,
 * long outputs in bounded memory, priming with real audio: step by step through x_prefix, or in one parallel pass
 * through srwn_generate_state_prefill).
 * srwn_generate_state_bytes: size of the state of B utterances for `precision` (SRWN_FP32 or SRWN_FP16); it does not
 *   depend on T.  It holds the dilation queues in the layout of the precision's kernel (fp16: ceil(B/8) * sum(d) * 512
 *   bytes; fp32: B * sum(d) * 32 floats), x[t-1] and x[t-2] of each utterance, the position t0 of the next step and a
 *   signature (B, precision, layers, sum(d), pool_stride).  Its first 8 bytes are t0, an int64.
 * srwn_generate_state_reset: zero queues and x history, t0 = 0 (the zero padding of ops.py:9).  A state is used only on
 *   the handle, B and precision it was last reset for; any other call is refused with SRWN_ERR_INVALID.
 * srwn_teacher_generate_resume: steps t0 .. t0+T-1, t0 read from the state on the device (no host synchronisation);
 *   the state then holds t0+T.  enc [B,T/P,C] are the frames of THIS call, u1 [B,T,M] and u2 [B,T] its uniforms.
 *   x_prefix [B,n_prefix] (0 <= n_prefix <= T; NULL when 0): for the first n_prefix steps x[t] is the given sample
 *   instead of a draw (teacher forcing through the queues: priming); logits are still computed and x_out holds the
 *   forced values.  Workspace: srwn_workspace_bytes(SRWN_OP_TEACHER_GENERATE, B, T) with this call's T.  With the same
 *   uniforms, generating T1 + T2 samples in two calls gives bit for bit what one call over T1 + T2 gives. */
int srwn_generate_state_bytes(srwn_handle_t h, int32_t B, int32_t precision, size_t* bytes);
int srwn_generate_state_reset(srwn_handle_t h, void* state, int32_t B, int32_t precision, void* stream);
int srwn_teacher_generate_resume(srwn_handle_t h, void* state, const float* enc, const float* u1,
                                 const float* u2, const float* x_prefix, int32_t n_prefix, float* x_out,
                                 float* logits_out, int32_t B, int32_t T, int32_t precision,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* srwn_generate_state_prefill: primes a state with n known samples in one parallel pass.  x [B,n] are the samples of
 *   positions t0 .. t0+n-1 and enc [B,n/P,C] their frames (the convention of a resume call); t0 is read on the device.
 *   Afterwards the state is byte for byte the state srwn_teacher_generate_resume leaves after a call of T = n with
 *   x_prefix = x (both precisions, any t0), and holds t0+n.  No audio and no logits are produced (srwn_teacher_nll scores
 *   a prime).  Only the last sum(d) + 2 samples reach the state, so the cost and the workspace
 *   (srwn_workspace_bytes(SRWN_OP_TEACHER_PREFILL, B, n)) depend on B and min(n, sum(d) + 2) only.  Refused: n <= 0 or
 *   n % pool_stride != 0, a null x, enc or state, a state not reset on this handle for this B and precision, a student
 *   handle, fp16 where the tensor-core generation kernel does not cover the configuration, a small workspace. */
int srwn_generate_state_prefill(srwn_handle_t h, void* state, const float* x, const float* enc, int32_t n, int32_t B,
                                int32_t precision, void* workspace, size_t workspace_bytes, void* stream);
/* srwn_generate_state_splice: for each i < n, utterance src_rows[i] of `src` (src_B utterances) replaces utterance
 *   dst_rows[i] of `dst` (dst_B utterances); both states were reset on h for their B and this precision.  The row arrays
 *   are HOST memory.  A state's position t0 is always a multiple of pool_stride (reset sets 0, resume and prefill advance
 *   by multiples of it), so two states agree on latent-frame boundaries; the splice copies each layer's d queue entries,
 *   rotated from src's phase t0 mod d to dst's (both t0 read on the device: no synchronisation), and the x history.
 *   dst's t0, its other utterances and all of src stay unchanged.  Generating on dst then continues each spliced
 *   utterance bit for bit as generating on src would (with the same frames and uniforms): continuous batching refills
 *   the slot of a finished utterance with a freshly primed one.  No workspace; n == 0 does nothing.  Refused with
 *   SRWN_ERR_INVALID before any work: a null state, a state not reset on this handle for its B and precision,
 *   src == dst, n < 0, a row out of range, a destination row named twice, a student handle; SRWN_ERR_UNSUPPORTED as
 *   srwn_generate_state_bytes for the precision. */
int srwn_generate_state_splice(srwn_handle_t h, void* dst, int32_t dst_B, const int32_t* dst_rows,
                               const void* src, int32_t src_B, const int32_t* src_rows, int32_t n,
                               int32_t precision, void* stream);

/* ---- student (model.py:415-535) ------------------------------------------------- */
/* generate(sess, inputs, encoding) (model.py:570-576): z [B,T] logistic noise ->
 * out [B,T] = clip(z*s_tot + mu_tot, -1, 1) (model.py:535); s_tot, mu_tot [B,T]
 * (model.py:517-533) and x_last [B,T] (chained flow output) are optional outputs. */
int srwn_student_forward(srwn_handle_t h, const float* z, const float* enc, float* out,
                         float* s_tot, float* mu_tot, float* x_last,
                         int32_t B, int32_t T, int32_t precision,
                         void* workspace, size_t workspace_bytes, void* stream);
/* generate(sess, noise, encoding) (model.py:570-576) with the logistic noise of student.py:104 / :172 drawn ON THE DEVICE:
 * z[b,t] = log u - log(1-u), u = Philox4x32-10(seed; stream_id; b*T + t) in (0,1).  With SRWN_FP16 the fused flow kernel
 * evaluates the draw in place (front conv taps, affine head, composition): no noise tensor is read.  z_out (optional)
 * receives the draws, so srwn_student_forward(z_out, ...) reproduces the call.  srwn_random_logistic fills the same
 * values; srwn_random_uniform serves the mixture sampler's uniforms (ops.py:187, 196). */
int srwn_student_sample(srwn_handle_t h, uint64_t seed, uint64_t stream_id, const float* enc, float* out,
                        float* s_tot, float* mu_tot, float* x_last, float* z_out, int32_t B, int32_t T,
                        int32_t precision, void* workspace, size_t workspace_bytes, void* stream);
/* Synthesis in chunks: the same flows continued across calls through a caller-owned DEVICE state (audio while the
 * encoding is still arriving, clips longer than one call's workspace).
 * srwn_student_state_bytes: size of the state of B utterances for `precision` (SRWN_FP32 or SRWN_FP16; it does not depend
 *   on the clip length).  It holds, per flow, the last H samples of that flow's input (z for flow 0, flow f-1's output
 *   after), the last H/P frames of `enc`, the position t0 and a signature (B, precision, flows, layers, sum(d), P, C); its
 *   first 8 bytes are t0, an int64.  H = (filter_width - 1) * sum(d) + filter_width rounded up to a multiple of
 *   pool_stride P: the rows one output sample of a flow depends on.
 * srwn_student_state_reset: zero histories, t0 = 0.  A state is used only on the handle, B and precision it was last
 *   reset for.
 * srwn_student_forward_resume: the S samples t0 .. t0+S-1 (S > 0 and t0 multiples of P).  z [B,S] their noise, or NULL
 *   to draw it on the device (element b*S + s of Philox stream (seed, stream_id), as srwn_student_sample; z_out [B,S],
 *   optional, receives the draws); enc [B,S/P,C] their frames; out, and optionally s_tot, mu_tot, x_last, as
 *   srwn_student_forward, each [B,S].  The host passes t0 (it sets how many carried rows the call recomputes:
 *   min(t0, H)); the state holds t0 as well, and a call whose t0 disagrees raises the handle's abort words on the device
 *   (no synchronisation): the outputs of that call are invalid, the state is left as it was, later calls are refused
 *   with SRWN_ERR_CUDA until srwn_check_async_error(SRWN_OP_STUDENT_STREAM, ...) reports it.  Afterwards the state holds
 *   t0+S.  Workspace: srwn_workspace_bytes(SRWN_OP_STUDENT_STREAM, B, S).  With injected noise, any split of a clip into
 *   such calls gives bit for bit the out, s_tot, mu_tot and x_last of one srwn_student_forward over the clip, in both
 *   precisions.  Refused with SRWN_ERR_INVALID before any work: a null state, enc or out, a teacher handle, S <= 0 or
 *   S % P != 0, t0 < 0 or t0 % P != 0, a state not reset on this handle for this B and precision; SRWN_BF16 with
 *   SRWN_ERR_UNSUPPORTED. */
int srwn_student_state_bytes(srwn_handle_t h, int32_t B, int32_t precision, size_t* bytes);
int srwn_student_state_reset(srwn_handle_t h, void* state, int32_t B, int32_t precision, void* stream);
int srwn_student_forward_resume(srwn_handle_t h, void* state, int64_t t0, const float* z, uint64_t seed, uint64_t stream_id,
                                const float* enc, float* out, float* s_tot, float* mu_tot, float* x_last, float* z_out,
                                int32_t B, int32_t S, int32_t precision, void* workspace, size_t workspace_bytes,
                                void* stream);
int srwn_random_logistic(float* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream);
int srwn_random_uniform(float* out, int64_t n, uint64_t seed, uint64_t stream_id, float lo, float hi, void* stream);

/* ---- student distillation step (model.py:356-401, student.py:107 train_fast) ------------------
 * The reference builds one graph: student forward, loss (teacher cross-entropy of the student's
 * samples - alpha * entropy + gamma * spectral power loss) / B, gradients, clip_by_global_norm(1),
 * Adam.  Here the device side is four calls; the host glue (model.py mirror) supplies the loss
 * gradients between them and the NCCL all-reduce of `grads` across ranks before srwn_adam_step:
 *   1. srwn_student_forward_train: fp32 forward that keeps every layer input in `workspace`
 *      (size: srwn_workspace_bytes(op = SRWN_OP_STUDENT_TRAIN)); out/s_tot/mu_tot [B,T].
 *   2. caller: d_pre = dLoss/d(z*s_tot + mu_tot) [B,T] (zero where model.py:535 clips) and
 *      d_s_extra = dLoss/ds_tot from terms that use s_tot directly (the entropy, model.py:356).
 *      srwn_mol_loss_grad gives d(-log p)/dx of ops.py:124-175 for fixed logits.
 *   3. srwn_student_backward: gradients of every student variable into `grads`, a flat fp32
 *      buffer of srwn_param_count() elements laid out like the weight arena
 *      (srwn_weight_offset(name) locates a variable); same workspace as step 1.
 *   4. srwn_adam_step: tf.clip_by_global_norm(clip) + tf.train.AdamOptimizer update of the
 *      device weights (m, v: caller-owned fp32 state of srwn_param_count() elements, zeroed at
 *      start; step counts from 1; scratch: 1 float).  Call srwn_commit_weights afterwards before
 *      using the 16-bit paths (their packed operand images are rebuilt from the device weights). */
int srwn_param_count(srwn_handle_t h, int64_t* count);
int srwn_weight_offset(srwn_handle_t h, const char* name, int64_t* offset, int64_t* count);
int srwn_student_forward_train(srwn_handle_t h, const float* z, const float* enc, float* out,
                               float* s_tot, float* mu_tot, int32_t B, int32_t T,
                               void* workspace, size_t workspace_bytes, void* stream);
int srwn_student_backward(srwn_handle_t h, const float* z, const float* enc, const float* d_pre,
                          const float* d_s_extra, float* grads, int32_t B, int32_t T,
                          void* workspace, size_t workspace_bytes, void* stream);
int srwn_mol_loss_grad(const float* x, const float* l, float* dx, float* nll_out,
                       int32_t B, int32_t T, int32_t M, void* stream);
/* The whole device weight arena (layout of srwn_weight_offset; count = srwn_param_count) copied to (to_handle = 0) or from
 * (to_handle = 1) a DEVICE buffer: data-parallel replicas broadcast rank 0's weights through it before the first step. */
int srwn_weights_flat(srwn_handle_t h, float* buffer, int64_t count, int32_t to_handle, void* stream);
/* {loss, power_loss} of model.py:378-379 as fp32 device values: out2[0] = (beta*sums[0] - alpha*sums[1] + *power) * inv_norm,
 * out2[1] = *power (sums from srwn_distill_loss_grad, power from srwn_stft_power_loss). */
int srwn_distill_finish(const double* sums, const double* power, float alpha, float beta, float inv_norm,
                        float* out2, void* stream);
/* tf.clip_by_global_norm(grads, clip_norm) in place (model.py:385; ParallelWaveNet.train clips per example, model.py:603-632).
 * scratch: one device float. */
int srwn_clip_by_global_norm(float* grads, int64_t n, float clip_norm, float* scratch, void* stream);
/* y += a * x (host-side averaging of per-example gradients in model.py:621, kept on the device). */
int srwn_axpy(float* y, const float* x, float a, int64_t n, void* stream);
/* per_example[b] = sum_t (log s_tot[b,t] + 2): the entropy term of model.py:356 per example (getEntropy, model.py:578-600). */
int srwn_entropy(const float* s_tot, double* per_example, int32_t B, int32_t T, void* stream);
int srwn_adam_step(srwn_handle_t h, const float* grads, float* m, float* v, float* scratch,
                   float clip_norm, float lr, float beta1, float beta2, float eps, int32_t step,
                   void* stream);

/* ---- spectral power loss and loss glue of the distillation step (model.py:356-379; SURVEY.md 8(f)-2) ----
 * srwn_stft_power: s(x) = mean over frames of |tf.contrib.signal.stft(x, frame_length, frame_step)|^2
 *   (model.py:360-367: periodic Hann window, fft_length = frame_length (a power of two), no padding,
 *   F = 1 + (T - frame_length) / frame_step frames); x [B,T] -> power [B, frame_length/2 + 1].
 * srwn_stft_power_loss: loss[0] (device double) = gamma * sum (s(truth) - s(out))^2 (model.py:369-371) and,
 *   when d_out != NULL, d_out [B,T] = dLoss/d out.  T < frame_length is an error (the reference's
 *   mean over zero frames is NaN).  Workspace: srwn_stft_workspace_bytes.
 * srwn_distill_loss_grad: the elementwise rest of model.py:356-379 / :535 for given per-sample
 *   cross-entropy terms: d_pre = (beta * d_ce + d_pow) * [-1 <= z*s_tot + mu_tot <= 1] * inv_norm,
 *   d_s = -alpha * inv_norm / s_tot, sums[0] = sum nll, sums[1] = sum(log s_tot + 2) (the entropy,
 *   model.py:356).  `sums` is a device buffer of SRWN_DISTILL_SUMS_LEN doubles (partials after the
 *   first two); nll and d_pow may be NULL.  All sums are taken in a fixed order. */
#define SRWN_DISTILL_SUMS_LEN 1024
int srwn_stft_workspace_bytes(int32_t B, int32_t T, int32_t frame_length, int32_t frame_step,
                              size_t* bytes);
int srwn_stft_power(const float* x, float* power, int32_t B, int32_t T, int32_t frame_length,
                    int32_t frame_step, void* workspace, size_t workspace_bytes, void* stream);
int srwn_stft_power_loss(const float* truth, const float* out, float gamma, double* loss,
                         float* d_out, int32_t B, int32_t T, int32_t frame_length,
                         int32_t frame_step, void* workspace, size_t workspace_bytes, void* stream);
int srwn_distill_loss_grad(const float* z, const float* s_tot, const float* mu_tot,
                           const float* nll, const float* d_ce, const float* d_pow, float alpha,
                           float beta, float inv_norm, float* d_pre, float* d_s, double* sums,
                           int32_t B, int32_t T, void* stream);

/* ---- teacher encoder (model.py:137-155; SURVEY.md 8(f)-1, the row next to the hot path) ---------
 * A separate handle: the encoder shares no variable with the decoder.  createEncoder stacks
 * ResidualDilationLayerNC (ops.py:48-57): relu -> K=2 conv with SAME padding (looks one step AHEAD,
 * `dilation_rate` is ignored) -> relu -> 1x1 "residual" (no skip connection) and 1x1 skip; the skips
 * are summed, reduced to `latent_channels` by a 1x1 conv and average-pooled by `pool_stride`. */
typedef struct srwn_encoder_config {
  int32_t n_layers;           /* len(dilations): layers after nc_conv (model.py:144) */
  int32_t filter_width;       /* kernels are built for 2 */
  int32_t encoder_channels;   /* model.py:76 encoder_channels (128) */
  int32_t skip_channels;      /* teacher.py:62 -> 128 */
  int32_t latent_channels;    /* teacher.py:44 -> 32 */
  int32_t pool_stride;        /* teacher.py:38 -> 128 */
} srwn_encoder_config_t;
typedef struct srwn_encoder* srwn_encoder_t;

int srwn_encoder_create(const srwn_encoder_config_t* cfg, srwn_encoder_t* out);
int srwn_encoder_destroy(srwn_encoder_t e);
/* TF variable names under "WaveNetAutoEncoder/Encoder/": "<layer>_NC/conv1d/{kernel,bias}" with
 * <layer> = nc_conv | dilated_conv_<i>, "conv1d[_<n>]/{kernel,bias}" with n = 2j residual / 2j+1
 * skip of layer j (0 = nc_conv, whose skip is dead: model.py:141) and n = 2(n_layers+1) the latent
 * conv.  HOST fp32, TF layout. */
int srwn_encoder_set_weight(srwn_encoder_t e, const char* name, const float* data,
                            const int64_t* shape, int32_t ndim);
int srwn_encoder_commit(srwn_encoder_t e, void* stream);
int srwn_encoder_supports(srwn_encoder_t e, int32_t precision);
int srwn_encoder_workspace_bytes(srwn_encoder_t e, int32_t B, int32_t T, int32_t precision,
                                 size_t* bytes);
/* encode(inputs) (model.py:250-255): x [B,T] audio -> encoding [B, T/pool_stride, latent].
 * SRWN_FP32: FFMA kernels (parity grade).  SRWN_FP16 / SRWN_BF16: tcgen05 kernels, one launch per
 * layer, 16-bit activations between layers (needs encoder_channels = 128, T % 128 == 0,
 * pool_stride % 128 == 0). */
int srwn_teacher_encode(srwn_encoder_t e, const float* x, float* encoding, int32_t B, int32_t T,
                        int32_t precision, void* workspace, size_t workspace_bytes, void* stream);
int srwn_encoder_check_async_error(srwn_encoder_t e, int32_t B, int32_t T, int32_t precision,
                                   void* workspace, size_t workspace_bytes, void* stream);
int srwn_encoder_set_profiling(srwn_encoder_t e, int32_t enable);
int srwn_encoder_last_ms(srwn_encoder_t e, float* ms);

/* ---- stateless ops (ops.py) ----------------------------------------------------- */
/* _DilatedCausalConv1d / DilatedCausalConv1d (ops.py:6-20): x [B,T,Cin],
 * filters [K,Cin,Cout], bias [Cout] or NULL -> y [B,T,Cout]. */
int srwn_dilated_causal_conv1d(const float* x, const float* filters, const float* bias,
                               float* y, int32_t B, int32_t T, int32_t Cin, int32_t Cout,
                               int32_t K, int32_t dilation, void* stream);
/* ResidualDilationLayer (ops.py:23-46): x [B,T,R] -> dense [B,T,R], skip [B,T,S]
 * (skip_k/skip_b/skip may be NULL). Gate = sigmoid(tanh(filter_conv)) as in ops.py:33. */
int srwn_residual_dilation_layer(const float* x, const float* filt_k, const float* filt_b,
                                 const float* res_k, const float* res_b,
                                 const float* skip_k, const float* skip_b,
                                 float* dense, float* skip, int32_t B, int32_t T,
                                 int32_t R, int32_t S, int32_t K, int32_t dilation,
                                 void* stream);
/* tf.layers.conv1d(padding='SAME', strides=1) of the non-causal layers (ResidualDilationLayerNC, ops.py:48-57): x [B,T,Cin],
 * filters [K,Cin,Cout], bias [Cout] or NULL -> y [B,T,Cout]; (K-1)/2 taps reach back, the rest forward (TensorFlow's padding).
 * flags: bit 0 = relu on the input, bit 1 = relu on the output. */
int srwn_conv1d_same(const float* x, const float* filters, const float* bias, float* y, int32_t B, int32_t T,
                     int32_t Cin, int32_t Cout, int32_t K, int32_t flags, void* stream);
/* log_prob_from_logits (reduce = 0: y [rows,C]) and log_sum_exp (reduce = 1: y [rows]) over the last axis (ops.py:111-122). */
int srwn_log_softmax(const float* x, float* y, int64_t rows, int32_t C, int32_t reduce, void* stream);
/* RightShift (ops.py:78-80). */
int srwn_right_shift(const float* x, float* y, int32_t B, int32_t T, int32_t C,
                     int32_t shift, void* stream);
/* ResizeEmbeddingNearestNeighbor (ops.py:64-74): x [B,L,C] -> y [B,out_size,C]. */
int srwn_resize_nearest(const float* x, float* y, int32_t B, int32_t L, int32_t C,
                        int32_t out_size, void* stream);
/* Pieces of the classification / embedding heads WaveNet (model.py:8-72) and SiameseWaveNet (model.py:660-798), which
 * reuse the residual block: in-place relu (model.py:48,51), tf.nn.pool(AVG, VALID) over `window` time steps
 * (model.py:55, 711: x [B,T,C] -> y [B,T-window+1,C]), softmax over the channels (model.py:57) and the Euclidean
 * distance of two embeddings sqrt(1e-8 + sum (a-b)^2) (model.py:735: a, b [B,D] -> d [B]). */
int srwn_relu(float* x, int64_t n, void* stream);
int srwn_avg_pool_time(const float* x, float* y, int32_t B, int32_t T, int32_t C, int32_t window, void* stream);
int srwn_softmax(const float* x, float* y, int64_t rows, int32_t C, void* stream);
int srwn_pair_distance(const float* a, const float* b, float* d, int32_t B, int32_t D, void* stream);
/* discretized_mix_logistic_loss (ops.py:124-175): x [B,T], l [B,T,4M];
 * nll_out [B,T] and/or nll_sum [1] (either may be NULL). */
int srwn_mol_loss(const float* x, const float* l, float* nll_out, float* nll_sum,
                  int32_t B, int32_t T, int32_t M, void* stream);
/* sample_from_discretized_mix_logistic (ops.py:178-201) with injected uniforms:
 * l [B,T,4M], u1 [B,T,M], u2 [B,T] -> out [B,T]; idx_out [B,T] int32 (the Gumbel-argmax
 * mixture index of ops.py:187) optional. */
int srwn_mol_sample(const float* l, const float* u1, const float* u2, float* out,
                    int32_t* idx_out, int32_t B, int32_t T, int32_t M, void* stream);

/* Optional timing of the dominant kernel(s) of the last call on this handle: when enabled, the
 * library brackets them with CUDA events on the launch stream.  srwn_last_kernel_ms waits for
 * the closing event and returns the elapsed time of those `launches` back-to-back launches and
 * the kernel's name (static string).  Used by bench.py's roofline. */
int srwn_set_profiling(srwn_handle_t h, int32_t enable);
int srwn_last_kernel_ms(srwn_handle_t h, float* ms, int32_t* launches, const char** name);

/* Number of kernels this library launched on behalf of the calling process since load
 * (bench.py's gpu_launches). */
int64_t srwn_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SRWN_H_ */
