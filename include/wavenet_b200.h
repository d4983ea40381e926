/* wavenet_b200.h — C ABI of libwavenet_b200.so
 *
 * B200-native (sm_100a) implementation of the WaveNet residual-stack training pass of
 * jirsat/wavenets.  The reference has NO native ABI (pure Python on TensorFlow/Keras); each
 * entry point below names the reference Python interface it stands in for (file:line under
 * the reference repo).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative wn_status; wn_last_error() gives text.
 *     The Python shim maps WN_ERR_VALUE -> ValueError and WN_ERR_UNSUPPORTED ->
 *     NotImplementedError (reference: model.py:52-70,250,307,500,549; layers.py:133,148,162,175).
 *   - tensors are channels-last, row-major, exactly as the reference's (B,T,C) tensors.
 *   - "dev" pointers are CUDA device pointers on the handle's device; "host" pointers are
 *     ordinary host memory.  `stream` is a cudaStream_t passed as void* (NULL = legacy default).
 *   - no CPU fallback: wn_create fails with WN_ERR_CUDA when no sm_100 device is usable.
 *   - no global state besides the handle (and a thread-local error string).
 */
#ifndef WAVENET_B200_H_
#define WAVENET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wn_handle wn_handle;

enum wn_status {
  WN_OK = 0,
  WN_ERR_VALUE = -1,        /* invalid hyper-parameter / shape  -> ValueError            */
  WN_ERR_UNSUPPORTED = -2,  /* valid in the reference API but not built -> NotImplemented */
  WN_ERR_CUDA = -3,         /* CUDA runtime / driver failure                              */
  WN_ERR_STATE = -4         /* call order problem (e.g. backward before forward)          */
};

enum wn_activation { WN_ACT_LINEAR = 0, WN_ACT_RELU = 1, WN_ACT_LEAKY_RELU = 2, WN_ACT_TANH = 3, WN_ACT_SIGMOID = 4 };
enum wn_sampling { WN_CATEGORICAL = 0, WN_LOGISTIC = 1, WN_GAUSSIAN = 2 };
enum wn_precision {
  WN_FP32 = 0,   /* fp32 storage + FFMA accumulate: the <=1e-4 parity tier                */
  WN_BF16 = 1    /* bf16 storage, tcgen05/TMEM fp32 accumulate: the throughput tier        */
};

#define WN_MAX_LIST 8
#define WN_MAX_DILATIONS 512

/* Mirrors WaveNet.__init__ kwargs (reference model.py:14-34) plus what Keras infers at build
 * time (cond_in) and what the device workspace needs (max_batch/max_time). */
typedef struct wn_config {
  int32_t kernel_size;                 /* model.py:15; layers.py:10 `kernel`                   */
  int32_t channels;                    /* R                                                     */
  int32_t blocks;
  int32_t layers_per_block;
  int32_t activation;                  /* wn_activation; pre-stack + head hidden layers         */
  int32_t conditioning;                /* 0 None, 1 'global' ('local' is broken upstream)        */
  int32_t n_mapping;                   /* len(mapping_layers)                                   */
  int32_t mapping_layers[WN_MAX_LIST];
  int32_t mapping_activation;          /* wn_activation                                         */
  int32_t cond_in;                     /* width of the conditioning input (one-hot depth)       */
  int32_t dilation_bound;
  int32_t num_mixtures;                /* 0 = None                                              */
  int32_t sampling_function;           /* wn_sampling                                           */
  int32_t bits;
  int32_t skip_channels;               /* 0 = None (skip aliases conv1 output, layers.py:216-219)*/
  int32_t dilation_channels;           /* 0 = None (= channels, layers.py:49-50)                */
  int32_t use_residual;
  int32_t use_skip;
  int32_t n_final;                     /* len(final_layers_channels)                            */
  int32_t final_layers_channels[WN_MAX_LIST];
  float   l2_reg_factor;
  float   dropout;                     /* layers.py:109-112: inverted dropout on each block's conv branch, training passes only */
  /* explicit per-conv dilations (blocks*layers_per_block entries) — used by the bare
   * WaveNetLayer mirror (layers.py:10-20 `dilation_rate`); 0 => model.py:79-81 schedule.      */
  int32_t n_dilations;
  int32_t dilations[WN_MAX_DILATIONS];
  int32_t has_input_conv;              /* 1 for WaveNet (model.py:84-88); 0 for a bare layer     */
  int32_t has_head;                    /* 1 for WaveNet (model.py:105-119); 0 for a bare layer   */
  int32_t precision;                   /* wn_precision                                          */
  int32_t max_batch;                   /* workspace is sized for (max_batch, max_time)          */
  int32_t max_time;
  int32_t device;                      /* CUDA device ordinal                                   */
} wn_config;

/* ---- lifetime (replaces WaveNet.__init__ + build, model.py:14-155,171-211) ------------- */
int wn_create(const wn_config* cfg, wn_handle** out);
void wn_destroy(wn_handle* h);
const char* wn_last_error(void);

/* ---- static facts ------------------------------------------------------------------------ */
/* model.py:79-81,93-94,122: dilation of conv j of block b, and the receptive field */
int wn_receptive_field(const wn_handle* h);
int wn_dilation(const wn_handle* h, int block, int j);

/* ---- parameters: Keras `trainable_variables` order and layouts (SURVEY 8b) --------------- */
int wn_num_params(const wn_handle* h);
int64_t wn_param_count(const wn_handle* h);               /* total scalar count (flat length) */
/* name: e.g. "block3/dil0/kernel"; shape: up to 3 dims (K,Cin,Cout)/(in,out)/(C); offset into flat buffers */
int wn_param_info(const wn_handle* h, int i, char* name, int name_len, int32_t* shape, int32_t* ndim, int64_t* offset);
float* wn_params_dev(wn_handle* h);                        /* flat fp32 master weights (device) */
float* wn_grads_dev(wn_handle* h);                         /* flat fp32 gradients (device)      */
int wn_set_param(wn_handle* h, int i, const float* host);  /* Keras layout, fp32 */
int wn_get_param(wn_handle* h, int i, float* host);
int wn_get_grad(wn_handle* h, int i, float* host);
/* call after writing wn_params_dev() directly (e.g. an optimizer step): re-packs the
 * kernel-side weight copies (transposes, gate interleave, bf16). */
int wn_params_changed(wn_handle* h, void* stream);

/* ---- device input pipeline (SURVEY 8f-3): preprocess_dataset (utils.py:22-85) and inverse_mu_law (callbacks.py:126-131)
 * speech (n_samples) int16 (scaled by 2^-15, utils.py:52-55) or fp32 -> optional mu-law (utils.py:35) ->
 * frames (wn_num_frames, T+1) with hop T (utils.py:36-38); valid[f] = 1 iff the frame is finite and inside [-1,1]
 * (utils.py:58-70).  wn_one_hot = tf.one_hot (utils.py:47). */
int64_t wn_num_frames(int64_t n_samples, int T);
int wn_preprocess_frames(const void* speech_dev, int is_int16, int64_t n_samples, int T, int apply_mulaw, float* frames_dev, int32_t* valid_dev,
                         void* stream);
int wn_inverse_mu_law(const float* y_dev, float* x_dev, int64_t n, void* stream);
int wn_one_hot(const int32_t* ids_dev, int n, int depth, float* out_dev, void* stream);

/* ---- sampling + MSE metric (SURVEY 8f-2): WaveNet.sample_waveform (model.py:393-503) and the compiled
 *      MeanSquaredError between y_true and the sampled waveform inside train_step/test_step (model.py:338-346).
 *      deterministic != 0: argmax bin / mean of the heaviest mixture component (bit-comparable with the reference);
 *      otherwise a Philox draw per (b,t) keyed by `seed` — TF's stateless RNG stream (seed (4,2), identical for every
 *      batch row, model.py:408,428,437) cannot be reproduced, so stochastic parity is statistical.
 *      out (B,T) fp32 in [-1,1]. */
int wn_sample_waveform(wn_handle* h, const float* pred_dev, int B, int T, int deterministic, uint64_t seed, float* out_dev, void* stream);
int wn_sample_last_step(wn_handle* h, const float* frames_dev, int deterministic, uint64_t seed, float* out_dev, float* mse_dev /* 2 floats or NULL */,
                        void* stream);

/* ---- autoregressive generation (SURVEY 8f-4): WaveNet.generate (model.py:258-307) with the per-layer single-step form
 *      of WaveNetLayer.generate (layers.py:226-290): every dilated conv keeps the history of its input, one new sample costs
 *      one K-tap matrix-vector product per conv (fp32, master weights).  prime (B, n_prime) fp32 = the reference's `sample`
 *      window (n_prime = receptive field there); out (B, length): out[b][i] = sample n_prime + i, drawn like
 *      wn_sample_waveform (deterministic: argmax / heaviest-component mean, what `_generation` does, model.py:255).
 *      teacher (B, length) or NULL: forced continuation, for checking the step against WaveNet.call; pred (B, length, Cout)
 *      or NULL receives the predictive distribution of every generated position. */
int wn_generate(wn_handle* h, const float* prime_dev, int n_prime, const float* cond_dev, int B, int length, int deterministic, uint64_t seed,
                float* out_dev, float* pred_dev, const float* teacher_dev, void* stream);

/* ---- optimizer (SURVEY 8f-1): train.py:225-226 `tf.keras.optimizers.Adam(learning_rate=lr, clipnorm=1.0)` applied by
 *      model.py:336 `optimizer.apply_gradients`.  Keras 3 semantics: every variable's gradient is clipped to L2 norm
 *      <= clipnorm (tf.clip_by_norm) on each replica BEFORE the cross-replica sum; then
 *      m += (g-m)(1-b1); v += (g^2-v)(1-b2); w -= lr*sqrt(1-b2^t)/(1-b1^t) * m/(sqrt(v)+eps).
 *      Call order per step: wn_train_step -> wn_clip_grads -> [all-reduce of wn_grads_dev()] -> wn_adam_step. */
int wn_adam_init(wn_handle* h, float lr, float beta1, float beta2, float eps, float clipnorm /* 0 = off */);
int wn_clip_grads(wn_handle* h, void* stream);
int wn_adam_step(wn_handle* h, float lr /* < 0: keep */, void* stream);   /* also re-packs the kernel-side weights */
int wn_adam_state(wn_handle* h, float** m_dev, float** v_dev, float** grad_norms_dev, int64_t* step);
/* copies Adam's moments (flat fp32 device buffers of wn_param_count() floats, e.g. another handle's wn_adam_state) and the
 * step counter into this handle: a model rebuilt for a larger (batch, time) workspace keeps training where it was, like a
 * Keras optimizer whose slots outlive a re-traced train_step (model.py:211,336). */
int wn_adam_restore(wn_handle* h, const float* m_dev, const float* v_dev, int64_t step);

/* ---- dropout (layers.py:109-112,195-196; Keras Dropout on the block input of the conv branch) --------
 * Training passes draw keep-masks with a counter-based Philox-4x32-10 keyed by (seed, step): TF's RNG
 * stream cannot be reproduced, so parity runs inject the masks instead.
 * keep_host: [blocks][B*T*channels] bytes (1 = keep), NULL returns to Philox masks. */
int wn_set_dropout_masks(wn_handle* h, const uint8_t* keep_host, int B, int T);
int wn_set_dropout_seed(wn_handle* h, uint64_t seed);

/* ---- target quantiser (model.py:151-155,320: Keras Discretization) ----------------------- */
/* idx[i] = #{k in 1..2^bits-1 : -1 + k*2^(1-bits) <= x[i]}, bit-exact, comparison based */
int wn_quantize(const float* x_dev, int64_t* idx_dev, int64_t n, int bits, void* stream);

/* ---- WaveNet.call (model.py:213-239): x (B,T) fp32, cond (B,cond_in) fp32 or NULL ->
 *      out (B,T,2^bits) softmax probabilities or (B,T,3M) mixture parameters, fp32 -------- */
int wn_forward(wn_handle* h, const float* x_dev, const float* cond_dev, int B, int T, float* out_dev, void* stream);
/* the same with Keras' `training` argument (model.py:213, layers.py:178,195-196): training != 0 applies the block dropout
 * (fresh Philox masks, or the masks injected with wn_set_dropout_masks) exactly as the forward half of wn_train_step does. */
int wn_forward_ex(wn_handle* h, const float* x_dev, const float* cond_dev, int B, int T, int training, float* out_dev, void* stream);

/* ---- WaveNet.loss_fn(target, pred) (model.py:505-551) on MATERIALISED predictions ------------------------------------
 * pred (B,T,Cout) fp32 = a WaveNet.call output (softmax probabilities, or [weights | means | log-scales] mixture
 * parameters); out (B,T) fp32 per-position losses, NOT reduced (the caller applies tf.nn.compute_average_loss, model.py:328).
 * categorical: target_is_int64 != 0: (B,T) int64 class indices (prepare_target's output), else (B,T) fp32 samples that are
 *   quantised on the fly; Keras 3 sparse_categorical_crossentropy on probabilities: clip to [1e-7, 1-1e-7], log, softmax
 *   cross entropy on those logits.  mixtures: (B,T) fp32 samples (model.py:155: the target is the waveform itself). */
int wn_loss_fn(wn_handle* h, const void* target_dev, int target_is_int64, const float* pred_dev, int B, int T, float* out_dev, void* stream);

/* ---- WaveNet.train_step up to the gradients (model.py:309-335) and test_step (:362-381) ---
 * frames (B,T+1) fp32 in [-1,1]; loss_dev points at TWO floats, the reference's two metrics
 * (model.py:340-344): loss_dev[0] = sum_{b,t} l / (B*n_replicas)  ('loss', compute_average_loss),
 * loss_dev[1] = l2_reg_factor * sum(kernel^2) / n_replicas ('reg_loss', 0 when l2_reg_factor == 0);
 * the gradients are those of their sum (model.py:334-335) and land in wn_grads_dev() (overwritten). */
int wn_train_step(wn_handle* h, const float* frames_dev, const float* cond_dev, int B, int T,
                  int n_replicas, float* loss_dev, void* stream);
int wn_test_step(wn_handle* h, const float* frames_dev, const float* cond_dev, int B, int T,
                 int n_replicas, float* loss_dev, void* stream);
/* same with HOST buffers: H2D of frames/cond, step, D2H of the two loss floats, stream sync. */
int wn_train_step_host(wn_handle* h, const float* frames_host, const float* cond_host, int B, int T,
                       int n_replicas, float* loss_host);

/* ---- data parallelism: tf.distribute.MirroredStrategy (train.py:203) = one replica per GPU, gradients SUM-reduced inside
 *      optimizer.apply_gradients (model.py:336; the loss is already divided by the global batch, model.py:328).  One
 *      process per GPU here; the replicas' handles share an NCCL communicator (NCCL is dlopen'ed: libnccl.so.2 already in
 *      the process, else the system one, else $WN_NCCL_LIB).  Rank 0 draws the 128-byte id, every rank passes it (sent by
 *      whatever channel the host has: torch.distributed, MPI, a file) to wn_comm_init together with its rank.
 *      wn_comm_attach takes an ncclComm_t the caller already owns (e.g. TensorFlow's or torch's) instead.
 *      wn_allreduce_grads: ncclAllReduce(SUM, fp32) in place over wn_grads_dev() on `stream`; a no-op for one replica.
 *      wn_comm_fuse_allreduce(on): wn_train_step(n_replicas > 1) enqueues that all-reduce itself behind the backward pass,
 *      inside the captured step graph (use when nothing — e.g. per-replica clipnorm — must run between the two). */
int wn_nccl_unique_id(uint8_t* id128);
int wn_comm_init(wn_handle* h, const uint8_t* id128, int nranks, int rank);
int wn_comm_attach(wn_handle* h, void* nccl_comm /* ncclComm_t or NULL to detach */, int nranks, int rank);
int wn_comm_fuse_allreduce(wn_handle* h, int on);
int wn_allreduce_grads(wn_handle* h, void* stream);
const char* wn_nccl_info(void);   /* "NCCL <version> from <path>" or "unavailable: ..." */

/* ---- WaveNetLayer.call (layers.py:178-224) and its adjoint, block granularity -------------
 * x (B,T,R) fp32; cond (B,Cc) fp32 time-constant conditioning or NULL;
 * x_out (B,T,R), skip (B,T,S or R) fp32.  Backward takes d x_out / d skip (either may be NULL
 * = zero) and returns dx (B,T,R) and dcond (B,Cc) (may be NULL); parameter gradients of that
 * block are written into wn_grads_dev(). */
int wn_layer_forward(wn_handle* h, int block, const float* x_dev, const float* cond_dev, int B, int T,
                     float* x_out_dev, float* skip_dev, void* stream);
/* WaveNetLayer.call(inputs, training) (layers.py:178,192-196): training != 0 applies the block's inverted dropout to the
 * conv branch (the residual keeps the un-masked input); the keep-mask is the injected one (wn_set_dropout_masks) or a fresh
 * Philox draw for this block, and wn_layer_backward of the block uses the same mask. */
int wn_layer_forward_ex(wn_handle* h, int block, const float* x_dev, const float* cond_dev, int B, int T, int training,
                        float* x_out_dev, float* skip_dev, void* stream);
/* WaveNetLayer.call with a conditioning SEQUENCE (layers.py:115-120,203-204): cond (B,T,cond_in) fp32, one vector per
 * time step (local conditioning), added to the gated conv's pre-activation as conv_cond(cond) at every t; the dropout
 * mask (training != 0) applies to x only.  The block must have conditioning and the handle no head (has_head = 0).  Any
 * cond_in and every kernel_size work on both tiers.  The sequence buffer must stay valid until the block's wn_layer_backward.
 * WN_ERR_VALUE: NULL sequence or a block without conditioning; WN_ERR_UNSUPPORTED: a model handle. */
int wn_layer_forward_seq(wn_handle* h, int block, const float* x_dev, const float* cond_dev /* (B,T,cond_in) fp32 */, int B, int T,
                         int training, float* x_out_dev, float* skip_dev, void* stream);
/* Adjoint of the block's last forward (WN_ERR_STATE before any): dcond_dev receives (B,T,cond_in) when that forward was
 * wn_layer_forward_seq, (B,cond_in) otherwise. */
int wn_layer_backward(wn_handle* h, int block, const float* dx_out_dev, const float* dskip_dev,
                      float* dx_dev, float* dcond_dev, void* stream);

/* ---- kernel-level test hooks (bf16 tier; no reference counterpart) -------------------------
 * The two tcgen05 mainloops without a model around them, for tests against a plain fp32 matmul:
 *   conv_gemm: out[(b,t), n] = sum_s A[(b, t+shifts[s]), 0:K] . W[n, s*K : (s+1)*K]   (rows outside [0,T) are zero)
 *   wgrad    : out[s*K + c, n] = sum_{b,t} A[(b, t+shifts[s]), c] * G[(b,t), n]
 * A (B,T,lda) bf16, W [N16][nseg*K] bf16, G (B,T,ldg) bf16, out fp32.  Synchronous. */
/* an intermediate tensor of the last step as fp32 on the host (rows = B*T of that step); returns the row width.
 * name: "h0", "z"(l), "g"(l), "xout"(l), "skipsum", "hact"(i), "logits", "dlogits", "dskip", "dz"(l), "dx"(l),
 * "act"(16 l + j: output of pre-stack conv j of block l) */
int wn_debug_tensor(wn_handle* h, const char* name, int index, float* out_host, int64_t capacity);
int wn_debug_conv_gemm(const void* a_bf16_dev, int lda, int B, int T, int nseg, const int* shifts, int K,
                       const void* w_bf16_dev, int N, int N16, int tile, float* out_dev, void* stream);
int wn_debug_wgrad(const void* a_bf16_dev, int lda, const void* g_bf16_dev, int ldg, int B, int T, int nseg,
                   const int* shifts, int K, int N, float* out_dev, void* stream);

/* micro-benchmark of one mainloop: `reps` back-to-back launches, CUDA-event timed (ms per launch).
 * which: 0 conv GEMM (W = g_or_w [N][nseg*K], bf16 out (B,T,ldo)), 1 wgrad + split reduction, 2 wgrad kernel alone */
int wn_debug_bench(int which, int reps, const void* a_bf16_dev, int lda, const void* g_or_w_bf16_dev, int ldg, int B, int T,
                   int nseg, const int* shifts, int K, int N, void* out_dev, int ldo, float* ms_out);

/* ---- introspection for benchmarks --------------------------------------------------------- */
/* number of kernel launches issued by the last wn_train_step / wn_forward on this handle */
int64_t wn_last_launch_count(const wn_handle* h);
/* accumulate CUDA-event time of one kernel class over subsequent steps: tag 0 = off,
 * 1 = dilated-conv GEMMs (fwd+dgrad+wgrad), 2 = all GEMMs, 3 = loss/head reductions */
int wn_fused_forward_blocks(const wn_handle* h);  /* blocks of the last forward that ran as one fused gate+conv1 launch */
/* 256x256 weight-gradient tiles (conv1, conv_skip, gated conv, head; tape.gradient of model.py:335) that the last training
 * step computed in the grouped launch behind the dgrad chain; 0 = per-block launches. side_launches (may be null): how many
 * of the launches ran beside the chain on the SMs it leaves idle */
int wn_grouped_wgrad_tiles(const wn_handle* h, int* side_launches);
/* the same plus the number of 256x256 fp32 partial tiles (tiles x row splits) the finish launch reads (its HBM traffic) */
int wn_grouped_wgrad_info(const wn_handle* h, int* tiles, int* partial_tiles, int* side_launches);
/* layers of the last forward (block loop of WaveNet.call, model.py:229-234) that ran inside the ONE persistent stack launch;
 * 0 = one launch (or more) per block */
int wn_stack_forward_layers(const wn_handle* h);
/* blocks whose backward chain (gate adjoint + dgrad: the autodiff of layers.py:199-224) ran inside the ONE persistent
 * stack-backward launch of the last training step; 0 = two launches per block */
int wn_stack_backward_layers(const wn_handle* h);
/* Gradient slices the last training step all-reduced EARLY, on its communication stream, beside the kernels of the next
 * weight-gradient bucket (0: one all-reduce behind the backward pass).  With a communicator that reduces inside the step
 * (wn_comm_fuse_allreduce) and the persistent stack-backward launch, the grouped weight-gradient launch runs in WN_AR_BUCKETS
 * (default 2) groups of blocks; only the last group's slice (+ head, input conv, mapping) is reduced after the pass.
 * Replaces: the overlap of gradient reduction with backprop that tf.distribute.MirroredStrategy gets from per-variable
 * all-reduces (train.py:203, model.py:336). */
int wn_allreduce_buckets(const wn_handle* h);
int wn_profile_begin(wn_handle* h, int tag);
int wn_profile_end(wn_handle* h, double* ms, int64_t* launches);
/* per-launch record of the last wn_profile_end: returns the number of timed launches; fills duration (ms) and a
 * short label of launch i: the phase ("input_conv_fwd", "cond_fwd", "skip_sum", "head_fwd", "loss", "loss_finalize",
 * "head_bwd", "wgrad_group_finish", "input_conv_bwd", "cond_bwd") or, inside the block loop, the kernel ("stack_fwd",
 * "block_fwd", "gate", "bias_act_res", "gate_bwd", "dgrad", "wgrad_dilated", "wgrad_1x1", "wgrad_group", "misc") */
int wn_profile_get(wn_handle* h, int i, double* ms, char* label, int label_len);
const char* wn_build_info(void);

#ifdef __cplusplus
}
#endif
#endif  /* WAVENET_B200_H_ */
