// wn_api.cu — host orchestration + C ABI of libwavenet_b200.so  (see include/wavenet_b200.h)
//
// Path (reference file:line): WaveNet.train_step model.py:309-335 -> WaveNet.call :213-239 ->
// WaveNetLayer.call layers.py:178-224, its adjoint, and the loss model.py:505-551.
//
// Every contraction of the pass is one of two kernels (gemm_simt.cuh / gemm_tc.cuh):
//   conv_gemm : shifted-row GEMM with a fused epilogue (forward convs, dgrads, 1x1s, skip sum)
//   wgrad     : time-contraction GEMM (weight gradients), deterministic split reduction
// plus the HBM-bound kernels of kernels_misc.cuh.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/wavenet_b200.h"
#include "common.cuh"
#include "epilogues.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "gemm_tc_block.cuh"
#include "gemm_tc_wgroup.cuh"
#include "gemm_tc_stack.cuh"
#include "gemm_tc_stack_bwd.cuh"
#include "kernels_misc.cuh"
#include "generate.cuh"
#include "nccl_dl.cuh"

// ============================================================================ errors
static thread_local char g_err[512] = "";
static void set_err(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* wn_last_error(void) { return g_err; }
extern "C" const char* wn_build_info(void) {
  return "libwavenet_b200 sm_100a; fp32 FFMA tier + bf16 tcgen05/TMEM/TMA tier; built " __DATE__ " " __TIME__;
}

#define CK(expr)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (expr);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      set_err("CUDA error %s (%s) at %s:%d", cudaGetErrorName(e_), cudaGetErrorString(e_), __FILE__, __LINE__); \
      return WN_ERR_CUDA;                                                                 \
    }                                                                                     \
  } while (0)
#define RET(expr)              \
  do {                         \
    int r_ = (expr);           \
    if (r_ != WN_OK) return r_; \
  } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline int rup(int a, int b) { return (a + b - 1) / b * b; }

// ============================================================================ model description
struct ParamInfo {
  std::string name;
  int shape[3];
  int ndim;
  long long offset, count;
};

struct ConvP {           // one Conv1D of the reference (dilated K-tap or 1x1)
  int K = 1, cin = 0, cout = 0, dil = 1;
  int w_idx = -1, b_idx = -1;
  bool gate = false;     // gated conv: forward weight columns tile-interleaved [filter|gate]
  // fp32 tier packed copies
  float* Wf = nullptr; int Npad = 0;      // [K*cin][Npad]      forward
  float* Wb = nullptr; int Cpad = 0;      // [K*cout][Cpad]     dgrad (block k = W[k]^T)
  // bf16 tier packed copies (K-major "B operand" matrices, see gemm_tc.cuh)
  bf16* Wf16 = nullptr; int Kf16 = 0;     // [Npad16][K*cin]    forward:  row n, contraction contiguous
  bf16* Wb16 = nullptr; int Kb16 = 0;     // [Cpad16][K*cout]   dgrad
  int N16 = 0, C16 = 0, tileN16 = 0;
};

struct BlockP {
  std::vector<ConvP> stack;   // dilated stack, last one gated (layers.py:64-88)
  ConvP conv1;                // layers.py:92-96
  bool has_skip = false;
  ConvP conv_skip;            // layers.py:98-104
  bool has_cond = false;
  int cw_idx = -1, cb_idx = -1;  // conv_cond kernel/bias (layers.py:117-120)
  // dg GEMM weights [Wr^T ; Ws^T] : fp32 [(R+S)][Dpad] ; bf16 [Dpad16][(R+S)]
  float* Wdg = nullptr; int Dpad = 0;
  bf16* Wdg16 = nullptr;
  // bf16 tier: conv1 with the residual folded into the contraction, B operand [R16][D + R] = [Wr^T | I]:
  // x_out = [g | x] . [Wr ; I] + b  (the x . I products are exact in the fp32 accumulator).  Takes the residual
  // read out of the epilogue, whose TMA input ring was the long pole of this kernel (3 k cycles per tile).
  bf16* Wres16 = nullptr;
  // layer handles with conditioning: a conditioning SEQUENCE (B,T,Cc) enters the gated conv's contraction as one more
  // segment (shift 0), so its weights follow the taps in the same packed operand
  float* Wfc = nullptr;                   // fp32 [K*cin + Cc][Npad]: gated conv rows, then Wc rows (same interleaved columns)
  float* Wct = nullptr; int Ccpad = 0;    // fp32 [2D][Ccpad]: Wc^T, operand of d cond = dz Wc^T
  bf16* Wfc16 = nullptr; int Kfc16 = 0;   // bf16 [N16][K*cin + Ccs]: gated conv, then Wc zero-padded to Ccs columns
  bf16* Wct16 = nullptr; int Cc16 = 0, tileCc16 = 0;   // bf16 [Cc16][2D]: Wc, B operand of d cond
};

struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0;
  bool dry = true;
  void* take(size_t bytes) {
    off = (off + 255) & ~(size_t)255;
    void* p = dry ? nullptr : base + off;
    off += bytes;
    return p;
  }
};

struct wn_handle {
  wn_config cfg;
  int R, D, S, Sp /*skip-sum width*/, K, L, Cc, Cout;
  bool alias_skip;
  std::vector<int> dil;  // flattened
  int rf;
  std::vector<ParamInfo> params;
  long long n_scalars = 0;
  float* d_params = nullptr;
  float* d_grads = nullptr;
  // network
  ConvP input_conv;
  std::vector<BlockP> blocks;
  std::vector<ConvP> head;
  std::vector<int> map_w, map_b, map_width;
  float* Wskip = nullptr; int Spad = 0;   // fp32 [L*D][Spad]
  bf16* Wskip16 = nullptr;                // bf16 [Spad16][L*D]
  float* bskip_sum = nullptr;             // [Sp]
  int* d_bskip_offsets = nullptr;
  int* d_cond_offsets = nullptr;          // [2L]: offsets of conv_cond kernel / bias of every block in the flat buffers
  // packed pool
  Arena pack, ws;
  int maxB, maxT;
  // workspace (void*: element type depends on precision)
  void* h0 = nullptr;
  std::vector<std::vector<void*>> acts;   // [block][j] pre-stack outputs (B,T,D)
  std::vector<void*> zbuf, xout;          // per block
  void* G_all = nullptr;                  // [L][B*T][D]  (sized with maxB*maxT rows per slab)
  void* skipsum = nullptr;
  std::vector<void*> hact;                // head hidden activations
  float* logits = nullptr; int ldl = 0;   // fp32 [rows][ldl]
  void* dlogits = nullptr; int ldd = 0;
  void *dhA = nullptr, *dhB = nullptr;    // head backward ping-pong (width max head)
  void* dskip = nullptr;
  void *dxA = nullptr, *dxB = nullptr, *dotmp = nullptr;
  void *dcatA = nullptr, *dcatB = nullptr;   // bf16 tier: [d x_out (R) | d skip (S)] side by side, ping-pong
  void* dz = nullptr;
  void *dpA = nullptr, *dpB = nullptr;    // pre-stack backward ping-pong (B,T,D)
  float* colpart = nullptr; int col_chunks = 0;
  float* wg_partial = nullptr; long long wg_partial_elems = 0;
  float* cs_partial = nullptr;            // [splits*slots][max N] column-sum partials of the tcgen05 wgrad
  float* wg_partial_side = nullptr; float* cs_partial_side = nullptr;   // same, for wgrads issued on the side stream
  void* dz2 = nullptr;                    // second dz buffer (side-stream wgrad of block l reads dz while block l-1 writes)
  float* loss_partial = nullptr; int loss_parts_cap = 0;
  float* cond_act[WN_MAX_LIST + 1] = {};  // mapping activations (B, width)
  float* cond_dact = nullptr;             // scratch (B, max width)
  float* cond_dact2 = nullptr;
  float* cb = nullptr;                    // [L][B][2D]
  float* dcb = nullptr;                   // [L][B][2D]
  float* dcond = nullptr;                 // (B,Cc)
  float* l2_sum = nullptr;
  // dropout (layers.py:195-196): keep-masks [L][maxB*maxT*R] bytes, dropped block inputs, raw dgrad scratch
  uint8_t* drop_mask = nullptr;
  std::vector<void*> xdrop;
  void* ddrop = nullptr;
  unsigned long long* d_drop_ctr = nullptr;
  unsigned long long drop_seed = 0x243F6A8885A308D3ull;
  bool drop_injected = false;   // masks were supplied by wn_set_dropout_masks: do not redraw
  int drop_B = 0, drop_T = 0;   // ... packed for this (B, T), row b*T + t of every slab
  bool drop_active = false;     // the pass being enqueued is a training pass with dropout > 0
  // optimizer state (wn_adam_*): allocated on first use
  float* opt_m = nullptr; float* opt_v = nullptr;
  OptChunk* opt_chunks = nullptr; int opt_n_chunks = 0;
  int* opt_var_first = nullptr;
  float* opt_partial = nullptr; float* opt_scale = nullptr; float* opt_norms = nullptr;
  float opt_lr = 1e-3f, opt_b1 = 0.9f, opt_b2 = 0.999f, opt_eps = 1e-7f, opt_clipnorm = 0.f;
  long long opt_t = 0;
  void* layer_in = nullptr;
  float* d_loss = nullptr;                // for the host-buffer entry point
  float* d_frames = nullptr; float* d_cond_in = nullptr;
  float* pin_frames = nullptr; float* pin_cond = nullptr; float* pin_loss = nullptr;
  cudaStream_t own_stream = nullptr;
  // state
  int lastB = 0, lastT = 0;
  // the last wn_forward_ex, which wn_backward differentiates: valid until the activations, the weights or the dropout masks change
  bool fwd_valid = false;
  struct FwdRecord { int B = 0, T = 0; bool training = false; const float* x = nullptr; int ldx = 0; const float* cond = nullptr; } fwd;
  bool layer_fwd_valid[WN_MAX_DILATIONS] = {};
  bool layer_drop[WN_MAX_DILATIONS] = {};     // wn_layer_forward_ex ran block l with dropout active (its adjoint must too)
  // conditioning sequences of the layer API (wn_layer_forward_seq); buffers exist on layer handles with conditioning only
  int Ccs = 0;                            // stored width of a sequence: Cc (fp32), Cc rounded up to 32 (bf16)
  std::vector<void*> cseq;                // bf16: [block] zero-padded copy of the last sequence (rows, Ccs)
  float* cseq_bias = nullptr;             // [L][2D] gated-conv bias + conv_cond bias
  float* cseq_dw = nullptr;               // bf16: [Ccs][2D] weight gradient of the padded contraction (first Cc rows = d Wc)
  const void* layer_cseq[WN_MAX_DILATIONS] = {};   // sequence (in T, width Ccs) of block l's last forward; null: time-constant
  const void* cond_seq = nullptr;         // the sequence of the block being enqueued (null: time-constant or no conditioning)
  const float* last_cond = nullptr;
  long long launches = 0;
  // profiling
  int prof_tag = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
  std::vector<const char*> prof_labels;   // what was launched in each timed slot
  const char* cur_label = "misc";
  const char* outer_label = nullptr;      // set by OuterLabel: names a whole phase (skip sum, head, loss, ...) for the per-launch records
  std::vector<float> prof_ms;             // per-slot durations of the last wn_profile_end
  std::vector<const char*> prof_last_labels;
  size_t prof_used = 0;
  long long prof_launches = 0;
  TmapCache tmaps;
  // CUDA graphs of whole steps, keyed by the call's arguments (buffers are fixed at create time)
  struct StepGraph { const float* frames; const float* cond; int B, T, nrep; float* loss; bool train; int seen; long long launches; cudaGraphExec_t exec; };
  std::vector<StepGraph> graphs;
  int use_graphs = 1;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
  // backward on two streams: the weight-gradient kernels of a block run beside its dgrad chain
  cudaStream_t side_stream = nullptr;
  std::vector<cudaEvent_t> ev_blk_in, ev_blk_dz, ev_blk_done;
  int stack_fwd_layers = 0;   // layers of the last forward inside the stack launch
  int use_stack_fwd = 1;    // WN_TC_STACK_FWD=0: one fused launch per block instead of one for the whole stack (gemm_tc_stack.cuh)
  std::vector<TcStackPlan> stack_plans;
  // backward chain (gate adjoint + dgrad of every block) as one persistent launch (gemm_tc_stack_bwd.cuh); WN_TC_STACK_BWD=0: per-block launches
  int use_stack_bwd = 1, stack_bwd_layers = 0;
  std::vector<TcStackBwdPlan> stack_bwd_plans;
  int fused_fwd_launches = 0;  // fused block-forward launches of the last step (0: separate gate / conv1 kernels)
  // grouped weight gradients (gemm_tc_wgroup.cuh): d z and d x_out of EVERY block are kept (no ping-pong) and all block
  // weight gradients run as one launch behind the dgrad chain.  WN_TC_GROUP_WGRAD=0 switches back to per-block launches.
  int use_group_wgrad = 0;
  void* dz_all = nullptr;     // [L][rows][2D]
  void* dx_all = nullptr;     // [L][rows][R]: d x_out of block l
  void* do_all = nullptr;     // [L][rows][R]: d x_out + d skip of block l (skip_channels=None with use_skip: skip = conv1 output)
  std::vector<std::vector<void*>> dp_keep;   // [block][j]: gradient wrt the output of pre-stack conv j (B,T,D)
  struct WgPlan { int B, T; bool drop; bool sb; int nb; TcWgGroupPlan plan; void release() { plan.release(); } };
  std::vector<WgPlan> wg_plans;
  std::vector<TcWgJobDesc> wg_jobs;   // collected by block_backward while a pass is enqueued
  int wg_last_tiles = 0, wg_last_side = 0;   // grouped tiles / side launches of the last backward pass
  int wg_last_partials = 0;                  // fp32 partial tiles (tiles x row splits) its finish launch reads
  int wg_side_every = 5;              // every n-th block hands its weight gradients to a side launch (WN_TC_GROUP_SIDE_EVERY, 0 = off)
  cudaEvent_t ev_wg_side = nullptr;
  int wg_force_split = 0, wg_pair_tiles = 1;   // WN_TC_GROUP_SPLIT=n / WN_TC_GROUP_NH2=0: A/B switches
  // every weight re-pack as one launch: job table recorded on the first wn_params_changed (buffers never move)
  // autoregressive generation state (wn_generate): histories of every dilated conv's input, scratch, step graphs
  struct Gen {
    int B = 0, cap = 0;
    float* audio = nullptr; std::vector<std::vector<float*>> hist; float* z = nullptr; float* skipsum = nullptr;
    std::vector<float*> hbuf; float* logits = nullptr; float* sampled = nullptr; int* t_dev = nullptr;
    std::vector<float*> wcat, bcat;          // per block [D][R+S] = [Wr | Ws], [R+S]: conv1 and conv_skip as one product
    std::vector<void*> allocs;
  } gen;
  std::vector<PackJob> pack_jobs;
  PackJob* d_pack_jobs = nullptr; long long pack_blocks = 0; bool pack_ready = false;
  // data parallelism (train.py:203): NCCL communicator of the replicas; the gradient all-reduce is the only collective
  wn_ncclComm_t comm = nullptr; bool comm_owned = false; int comm_nranks = 1, comm_rank = 0;
  int ar_in_step = 0;       // wn_train_step enqueues the all-reduce itself, behind the backward pass (inside the step graph)
  // bucketed all-reduce (SURVEY.md 8e "overlap by launching per-bucket all-reduces"): with the stack-backward launch every filter
  // gradient comes out of the grouped weight-gradient launch at the end of the pass; that launch runs bucket by bucket (blocks
  // L-1 .. 0 in ar_buckets groups), and the gradients of a finished bucket are all-reduced on comm_stream while the next bucket
  // is computed.  Only the last bucket's all-reduce (+ head, input conv, mapping) stays exposed.
  int ar_buckets = 2;       // WN_AR_BUCKETS
  int ar_first_pct = 70;    // WN_AR_FIRST: share of the blocks in the first of two buckets
  bool ar_now = false;      // the step being enqueued all-reduces its gradients
  long long ar_early_lo = -1, ar_early_hi = -1;   // scalars [lo, hi) of the flat buffer already all-reduced by model_backward
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t ev_bucket[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_comm_done = nullptr;
  int last_ar_buckets = 0;        // gradient slices the last training step all-reduced EARLY (beside the next bucket's kernels)
};

enum { CLS_DILATED = 1, CLS_GEMM = 2, CLS_LOSS = 3, CLS_MISC = 4 };

struct LaunchScope {
  wn_handle* h; cudaStream_t st; bool timed = false; size_t slot = 0;
  LaunchScope(wn_handle* h_, cudaStream_t st_, int cls) : h(h_), st(st_) {
    h->launches++;
    const int t = h->prof_tag;
    if (t && ((t == 1 && cls == CLS_DILATED) || (t == 2 && (cls == CLS_DILATED || cls == CLS_GEMM)) || (t == 3 && cls == CLS_LOSS) ||
              (t == 4))) {
      if (h->prof_used == h->prof_events.size()) {
        cudaEvent_t a, b;
        cudaEventCreate(&a); cudaEventCreate(&b);
        h->prof_events.push_back({a, b});
      }
      slot = h->prof_used++;
      if (h->prof_labels.size() <= slot) h->prof_labels.resize(slot + 1);
      h->prof_labels[slot] = h->outer_label ? h->outer_label : h->cur_label;
      cudaEventRecord(h->prof_events[slot].first, st);
      timed = true;
      h->prof_launches++;
    }
  }
  ~LaunchScope() {
    if (timed) cudaEventRecord(h->prof_events[slot].second, st);
  }
};

// names every launch issued while it lives (wins over the per-kernel labels): bench.py groups the timed launches by it
struct OuterLabel {
  wn_handle* h; const char* prev;
  OuterLabel(wn_handle* h_, const char* l) : h(h_), prev(h_->outer_label) { h->outer_label = l; }
  ~OuterLabel() { h->outer_label = prev; }
};

// names the launches of one kernel kind (when no OuterLabel is set)
struct LaunchLabel {
  wn_handle* h;
  LaunchLabel(wn_handle* h_, const char* l) : h(h_) { h->cur_label = l; }
  ~LaunchLabel() { h->cur_label = "misc"; }
};

// captured step graphs bake in the launch sequence and the plans' tables: anything that changes either drops them
static void drop_graphs(wn_handle* h) {
  for (auto& g : h->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  h->graphs.clear();
}

// Plans of the persistent launches are built per shape on first use and kept, at most 4 of a kind.  Building allocates and
// copies synchronously, so nothing is built while st is being captured: *out stays null then, and when the kernel does not take
// the shape (the build returns -100).
template <class Plan, class Build>
static int new_plan(wn_handle* h, cudaStream_t st, std::vector<Plan>& plans, const Plan& fresh, const char* what, Build build, Plan** out) {
  *out = nullptr;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cs);
  if (cs != cudaStreamCaptureStatusNone) return WN_OK;
  if (plans.size() >= 4) {
    CK(cudaDeviceSynchronize());
    drop_graphs(h);
    for (auto& q : plans) q.release();
    plans.clear();
  }
  plans.push_back(fresh);
  const int r = build(plans.back());
  if (r == 0) { *out = &plans.back(); return WN_OK; }
  plans.pop_back();
  if (r == -100) return WN_OK;
  set_err("%s plan failed (%d): %s", what, r, tc_last_error());
  return WN_ERR_CUDA;
}

// the kept plan whose key matches (at most one does), else a new one
template <class Plan, class Match, class Build>
static int plan_for(wn_handle* h, cudaStream_t st, std::vector<Plan>& plans, Match match, const char* what, Build build, Plan** out) {
  for (auto& q : plans) if (match(q)) { *out = &q; return WN_OK; }
  return new_plan(h, st, plans, Plan{}, what, build, out);
}
// the persistent launches return -100 for a shape they do not take: nothing ran, so the launch is not counted.  *ran: it ran
template <class Launch>
static int launch_persistent(wn_handle* h, cudaStream_t st, const char* label, const char* what, Launch launch, bool* ran) {
  LaunchLabel lab(h, label);
  LaunchScope ls(h, st, CLS_DILATED);
  const int r = launch();
  *ran = r == 0;
  if (r == -100) h->launches--;
  else if (r != 0) { set_err("%s launch failed (%d): %s", what, r, tc_last_error()); return WN_ERR_CUDA; }
  return WN_OK;
}
// a persistent stack launch is free of deadlock only while a layer has more 256-row tiles than the GPU has CTA pairs (DESIGN.md §5)
static bool more_tiles_than_pairs(int B, int Tn) { return B * cdiv(Tn, 256) > tc_num_sms() / 2; }

// ============================================================================ build
static int add_param(wn_handle* h, const std::string& name, std::initializer_list<int> shape) {
  ParamInfo p;
  p.name = name;
  p.ndim = (int)shape.size();
  p.count = 1;
  int i = 0;
  for (int s : shape) { p.shape[i++] = s; p.count *= s; }
  for (; i < 3; ++i) p.shape[i] = 1;
  p.offset = h->n_scalars;
  // keep every tensor 16-byte aligned in the flat buffers
  h->n_scalars += (p.count + 3) / 4 * 4;
  h->params.push_back(p);
  return (int)h->params.size() - 1;
}

static int validate_config(const wn_config& c) {
  // reference model.py:52-70
  if (c.conditioning != 0 && c.conditioning != 1) { set_err("Conditioning must be 'global', 'local' or None."); return c.conditioning == 2 ? WN_ERR_UNSUPPORTED : WN_ERR_VALUE; }
  if (c.kernel_size < 2) { set_err("Kernel size must be at least 2."); return WN_ERR_VALUE; }
  if (c.dilation_bound < 1) { set_err("dilation bound must be power of kernel_size."); return WN_ERR_VALUE; }
  {
    long long v = 1; bool ok = false;
    for (int i = 0; i < 40 && v <= c.dilation_bound; ++i) { if (v == c.dilation_bound) { ok = true; break; } v *= c.kernel_size; }
    if (!ok && c.n_dilations == 0) { set_err("dilation bound must be power of kernel_size."); return WN_ERR_VALUE; }
  }
  if (c.layers_per_block < 1) { set_err("Layers per block must be at least 1."); return WN_ERR_VALUE; }
  if (c.blocks < 1) { set_err("Blocks must be at least 1."); return WN_ERR_VALUE; }
  if (c.num_mixtures < 0) { set_err("Number of mixtures must be at least 1 or None."); return WN_ERR_VALUE; }
  if (c.dropout < 0 || c.dropout > 1) { set_err("Dropout must be between 0 and 1."); return WN_ERR_VALUE; }
  if (c.sampling_function < 0 || c.sampling_function > 2) { set_err("Sampling function must be categorical, logistic or gaussian."); return WN_ERR_VALUE; }
  if (c.sampling_function == WN_CATEGORICAL && c.num_mixtures != 0) { set_err("Categorical sampling cannot be used with mixtures."); return WN_ERR_VALUE; }
  if (c.has_head && c.sampling_function != WN_CATEGORICAL && c.num_mixtures == 0) { set_err("mixture sampling needs num_mixtures"); return WN_ERR_VALUE; }
  if (c.channels < 1 || c.max_batch < 1 || c.max_time < 1) { set_err("channels / max_batch / max_time must be positive"); return WN_ERR_VALUE; }
  if (c.kernel_size > WN_MAX_TAPS) { set_err("kernel_size > %d not built", WN_MAX_TAPS); return WN_ERR_UNSUPPORTED; }
  if (c.num_mixtures > WN_MAX_MIX) { set_err("num_mixtures > %d not built", WN_MAX_MIX); return WN_ERR_UNSUPPORTED; }
  if (c.blocks * c.layers_per_block > WN_MAX_DILATIONS) { set_err("too many dilated convs"); return WN_ERR_UNSUPPORTED; }
  if (c.n_mapping < 0 || c.n_mapping > WN_MAX_LIST || c.n_final < 0 || c.n_final > WN_MAX_LIST) { set_err("list too long"); return WN_ERR_VALUE; }
  if (c.has_head && c.sampling_function == WN_CATEGORICAL && (c.bits < 1 || c.bits > 16)) { set_err("bits must be in 1..16"); return WN_ERR_VALUE; }
  if (c.conditioning && c.cond_in < 1) { set_err("conditioning needs cond_in >= 1"); return WN_ERR_VALUE; }
  if (c.precision != WN_FP32 && c.precision != WN_BF16) { set_err("unknown precision"); return WN_ERR_VALUE; }
  return WN_OK;
}

static ConvP make_conv(wn_handle* h, const std::string& pfx, int K, int cin, int cout, int dil, bool gate) {
  ConvP c;
  c.K = K; c.cin = cin; c.cout = cout; c.dil = dil; c.gate = gate;
  c.w_idx = add_param(h, pfx + "/kernel", {K, cin, cout});
  c.b_idx = add_param(h, pfx + "/bias", {cout});
  return c;
}

template <class T> static size_t esz() { return sizeof(T); }

// lays out (dry==true: only measures) every packed weight copy and workspace buffer
static void layout_buffers(wn_handle* h) {
  const bool bf = h->cfg.precision == WN_BF16;
  const size_t es = bf ? 2 : 4;
  Arena& P = h->pack;
  auto lay_conv = [&](ConvP& c) {
    if (!bf) {
      c.Npad = rup(c.cout, 64);
      c.Wf = (float*)P.take((size_t)c.K * c.cin * c.Npad * 4);
      c.Cpad = rup(c.cin, 64);
      c.Wb = (float*)P.take((size_t)c.K * c.cout * c.Cpad * 4);
    } else {
      tc_pick_tile(c.cout, c.gate, &c.N16, &c.tileN16);
      c.Kf16 = c.K * c.cin;
      c.Wf16 = (bf16*)P.take((size_t)c.N16 * c.Kf16 * 2);
      int tn;
      tc_pick_tile(c.cin, false, &c.C16, &tn);
      c.Kb16 = c.K * c.cout;
      c.Wb16 = (bf16*)P.take((size_t)c.C16 * rup(c.Kb16, 64) * 2);
    }
  };
  if (h->cfg.has_input_conv) { /* input conv is elementwise: uses the flat params directly */ }
  for (auto& b : h->blocks) {
    for (auto& c : b.stack) lay_conv(c);
    lay_conv(b.conv1);
    if (b.has_skip) lay_conv(b.conv_skip);
    const int rs = h->R + (b.has_skip ? h->S : 0);
    if (!bf) {
      b.Dpad = rup(h->D, 64);
      b.Wdg = (float*)P.take((size_t)rs * b.Dpad * 4);
    } else {
      int n16, tn;
      tc_pick_tile(h->D, false, &n16, &tn);
      b.Dpad = n16;
      b.Wdg16 = (bf16*)P.take((size_t)n16 * rup(rs, 64) * 2);
      if (h->cfg.use_residual) b.Wres16 = (bf16*)P.take((size_t)b.conv1.N16 * (h->D + h->R) * 2);
    }
    if (b.has_cond && h->Ccs > 0) {
      const ConvP& c = b.stack.back();
      if (!bf) {
        b.Wfc = (float*)P.take((size_t)(c.K * c.cin + h->Cc) * c.Npad * 4);
        b.Ccpad = rup(h->Cc, 64);
        b.Wct = (float*)P.take((size_t)c.cout * b.Ccpad * 4);
      } else {
        b.Kfc16 = c.K * c.cin + h->Ccs;
        b.Wfc16 = (bf16*)P.take((size_t)c.N16 * b.Kfc16 * 2);
        tc_pick_tile(h->Cc, false, &b.Cc16, &b.tileCc16);
        b.Wct16 = (bf16*)P.take((size_t)b.Cc16 * c.cout * 2);
      }
    }
  }
  for (auto& c : h->head) lay_conv(c);
  if (!bf) {
    h->Spad = rup(h->Sp, 64);
    h->Wskip = (float*)P.take((size_t)h->L * h->D * h->Spad * 4);
  } else {
    int tn;
    tc_pick_tile(h->Sp, false, &h->Spad, &tn);
    h->Wskip16 = (bf16*)P.take((size_t)h->Spad * h->L * h->D * 2);
  }
  h->bskip_sum = (float*)P.take((size_t)h->Sp * 4);
  h->d_bskip_offsets = (int*)P.take((size_t)h->L * 4 * 2);
  h->d_cond_offsets = (int*)P.take((size_t)h->L * 4 * 2);

  Arena& W = h->ws;
  const size_t rows = (size_t)h->maxB * h->maxT;
  const int R = h->R, D = h->D, Sp = h->Sp, L = h->L;
  h->h0 = W.take(rows * R * es);
  h->acts.assign(L, {});
  h->zbuf.assign(L, nullptr);
  h->xout.assign(L, nullptr);
  for (int l = 0; l < L; ++l) {
    const int depth = (int)h->blocks[l].stack.size();
    h->acts[l].assign(depth - 1 > 0 ? depth - 1 : 0, nullptr);
    for (int j = 0; j + 1 < depth; ++j) h->acts[l][j] = W.take(rows * D * es);
    h->zbuf[l] = W.take(rows * 2 * D * es);
    h->xout[l] = W.take(rows * R * es);
  }
  h->G_all = W.take((size_t)L * rows * D * es);
  h->skipsum = W.take(rows * Sp * es);
  int maxhead = Sp > R ? Sp : R;
  h->hact.assign(h->head.size() > 0 ? h->head.size() - 1 : 0, nullptr);
  for (size_t i = 0; i + 1 < h->head.size(); ++i) {
    h->hact[i] = W.take(rows * h->head[i].cout * es);
    if (h->head[i].cout > maxhead) maxhead = h->head[i].cout;
  }
  if (h->cfg.has_head) {
    h->ldl = h->Cout;
    h->logits = (float*)W.take(rows * h->ldl * 4);
    h->ldd = bf ? rup(h->Cout, 64) : h->Cout;
    h->dlogits = W.take(rows * h->ldd * es);
    h->dhA = W.take(rows * maxhead * es);
    h->dhB = W.take(rows * maxhead * es);
  }
  h->dskip = W.take(rows * Sp * es);
  h->dxA = W.take(rows * R * es);
  h->dxB = W.take(rows * R * es);
  h->dotmp = W.take(rows * R * es);
  if (h->use_group_wgrad) {
    h->dz_all = W.take((size_t)L * rows * 2 * D * es);
    h->dx_all = W.take((size_t)L * rows * R * es);
    if (h->alias_skip && h->cfg.use_skip) h->do_all = W.take((size_t)L * rows * R * es);
    h->dp_keep.assign(L, {});
    for (int l = 0; l < L; ++l) {
      const int depth = (int)h->blocks[l].stack.size();
      for (int j = 0; j + 1 < depth; ++j) h->dp_keep[l].push_back(W.take(rows * D * es));
    }
  } else if (bf && !h->alias_skip && h->cfg.use_skip) {
    h->dcatA = W.take(rows * (size_t)(R + h->S) * es);
    h->dcatB = W.take(rows * (size_t)(R + h->S) * es);
  }
  h->dz = W.take(rows * 2 * D * es);
  h->dz2 = W.take(rows * 2 * D * es);
  h->dpA = W.take(rows * D * es);
  h->dpB = W.take(rows * D * es);
  // reductions
  h->col_chunks = cdiv(h->maxT, 64);   // input-conv wgrad partials use 64-row chunks; column sums 256-row chunks
  int nmax = 2 * D;
  if (R > nmax) nmax = R;
  if (Sp > nmax) nmax = Sp;
  for (auto& c : h->head) if (c.cout > nmax) nmax = c.cout;
  const int kin = (h->K + 1);
  size_t colpart_elems = (size_t)h->maxB * h->col_chunks * (nmax > kin * R ? nmax : kin * R);
  h->colpart = (float*)W.take(colpart_elems * 4);
  // wgrad partials: nsplit * ktot * N, largest contraction
  long long maxkn = 0;
  auto upd = [&](long long k, long long n) { if ((k + 1) * n > maxkn) maxkn = (k + 1) * n; };      // (+ 1: the fp32 tier's column-sum row)
  for (auto& b : h->blocks) {
    for (auto& c : b.stack) upd((long long)c.K * c.cin, c.cout);
    upd(D, R);
    if (b.has_skip) upd(D, h->S);
    if (b.has_cond && h->Ccs > 0) upd(h->Ccs, 2 * D);
  }
  for (auto& c : h->head) upd(c.cin, c.cout);
  h->wg_partial_elems = maxkn * WN_MAX_WGRAD_SPLITS;
  h->wg_partial = (float*)W.take((size_t)h->wg_partial_elems * 4);
  h->wg_partial_side = (float*)W.take((size_t)h->wg_partial_elems * 4);
  if (bf) {
    int max_mt = 1;
    auto mt = [&](int K, int cin) { const int m = K * cdiv(cin, 128); if (m > max_mt) max_mt = m; };
    for (auto& b : h->blocks) { for (auto& c : b.stack) mt(c.K, c.cin); mt(1, D); }
    if (h->Ccs > 0) mt(1, h->Ccs);
    for (auto& c : h->head) mt(1, c.cin);
    h->cs_partial = (float*)W.take((size_t)tc_wgrad_cs_rows(h->maxB, h->maxT, max_mt) * (size_t)rup(nmax, 4) * 4);
    h->cs_partial_side = (float*)W.take((size_t)tc_wgrad_cs_rows(h->maxB, h->maxT, max_mt) * (size_t)rup(nmax, 4) * 4);
  }
  h->loss_parts_cap = cdiv((long long)rows, 8) + 8;
  h->loss_partial = (float*)W.take((size_t)h->loss_parts_cap * 4);
  int maxw = h->cfg.cond_in;
  for (int i = 0; i < h->cfg.n_mapping; ++i) if (h->cfg.mapping_layers[i] > maxw) maxw = h->cfg.mapping_layers[i];
  if (h->cfg.conditioning) {
    for (int i = 0; i < h->cfg.n_mapping; ++i) h->cond_act[i] = (float*)W.take((size_t)h->maxB * h->cfg.mapping_layers[i] * 4);
    h->cond_dact = (float*)W.take((size_t)h->maxB * maxw * 4);
    h->cond_dact2 = (float*)W.take((size_t)h->maxB * maxw * 4);
    h->cb = (float*)W.take((size_t)L * h->maxB * 2 * D * 4);
    h->dcb = (float*)W.take((size_t)L * h->maxB * 2 * D * 4);
    h->dcond = (float*)W.take((size_t)h->maxB * (h->Cc > 0 ? h->Cc : 1) * 4);
  }
  if (h->Ccs > 0) {
    h->cseq.assign(L, nullptr);
    if (bf) {
      for (int l = 0; l < L; ++l) h->cseq[l] = W.take(rows * h->Ccs * 2);
      h->cseq_dw = (float*)W.take((size_t)h->Ccs * 2 * D * 4);
    }
    h->cseq_bias = (float*)W.take((size_t)L * 2 * D * 4);
  }
  h->l2_sum = (float*)W.take(16);
  if (h->cfg.dropout > 0.f) {
    h->drop_mask = (uint8_t*)W.take((size_t)L * rows * R);
    h->xdrop.assign(L, nullptr);
    for (int l = 0; l < L; ++l) h->xdrop[l] = W.take(rows * R * es);
    h->ddrop = W.take(rows * R * es);
    h->d_drop_ctr = (unsigned long long*)W.take(16);
  }
  h->d_loss = (float*)W.take(16);
  h->layer_in = W.take(rows * R * es);
  h->d_frames = (float*)W.take((size_t)h->maxB * (h->maxT + 1) * 4);
  h->d_cond_in = (float*)W.take((size_t)h->maxB * (h->cfg.cond_in > 0 ? h->cfg.cond_in : 1) * 4);
}

extern "C" int wn_create(const wn_config* cfg, wn_handle** out) {
  if (!cfg || !out) { set_err("null argument"); return WN_ERR_VALUE; }
  *out = nullptr;
  RET(validate_config(*cfg));
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_err("no CUDA device: libwavenet_b200 has no CPU fallback");
    return WN_ERR_CUDA;
  }
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) {
    set_err("device %d is sm_%d%d; libwavenet_b200 is built for sm_100a only", cfg->device, prop.major, prop.minor);
    return WN_ERR_CUDA;
  }
  wn_handle* h = new wn_handle();
  h->cfg = *cfg;
  const wn_config& c = h->cfg;
  h->K = c.kernel_size;
  h->R = c.channels;
  h->D = c.dilation_channels > 0 ? c.dilation_channels : c.channels;
  h->S = c.skip_channels;
  h->alias_skip = c.skip_channels == 0;
  h->Sp = h->alias_skip ? h->R : h->S;
  h->L = c.blocks;
  h->Cout = c.num_mixtures > 0 ? 3 * c.num_mixtures : (1 << c.bits);
  h->Cc = 0;
  if (c.conditioning) h->Cc = c.n_mapping > 0 ? c.mapping_layers[c.n_mapping - 1] : c.cond_in;
  // layer handles (no head) may be called with a conditioning sequence: model handles allocate nothing for it
  if (c.conditioning && !c.has_head) h->Ccs = c.precision == WN_BF16 ? rup(h->Cc, 32) : h->Cc;
  h->maxB = c.max_batch;
  h->maxT = c.max_time;
  // dilation schedule (model.py:79-81) unless given explicitly (bare WaveNetLayer)
  const int nconv = c.blocks * c.layers_per_block;
  if (c.n_dilations > 0) {
    if (c.n_dilations != nconv) { set_err("n_dilations must equal blocks*layers_per_block"); delete h; return WN_ERR_VALUE; }
    h->dil.assign(c.dilations, c.dilations + nconv);
  } else {
    int max_power = (int)(log((double)c.dilation_bound) / log((double)c.kernel_size));
    // guard against floating error exactly like int(math.log(bound, k)) for exact powers
    { long long v = 1; int pw = 0; while (v < c.dilation_bound) { v *= c.kernel_size; ++pw; } max_power = pw; }
    if (max_power < 1) { set_err("dilation bound must be power of kernel_size."); delete h; return WN_ERR_VALUE; }
    for (int i = 0; i < nconv; ++i) {
      long long d = 1;
      for (int p = 0; p < i % max_power; ++p) d *= c.kernel_size;
      h->dil.push_back((int)d);
    }
  }
  long long sumd = 0;
  for (int d : h->dil) sumd += d;
  h->rf = (int)(1 + sumd * (c.kernel_size - 1) + 1);  // model.py:122

  // ---- parameters in Keras tracking order
  if (c.has_input_conv) h->input_conv = make_conv(h, "causal", h->K, 1, h->R, 1, false);
  h->blocks.resize(h->L);
  for (int b = 0; b < h->L; ++b) {
    BlockP& bl = h->blocks[b];
    char pfx[64];
    int cin = h->R;
    for (int j = 0; j < c.layers_per_block; ++j) {
      const bool last = j == c.layers_per_block - 1;
      snprintf(pfx, sizeof(pfx), "block%d/dil%d", b, j);
      bl.stack.push_back(make_conv(h, pfx, h->K, cin, last ? 2 * h->D : h->D, h->dil[b * c.layers_per_block + j], last));
      cin = h->D;
    }
    snprintf(pfx, sizeof(pfx), "block%d/conv1", b);
    bl.conv1 = make_conv(h, pfx, 1, h->D, h->R, 1, false);
    bl.has_skip = !h->alias_skip;
    if (bl.has_skip) {
      snprintf(pfx, sizeof(pfx), "block%d/conv_skip", b);
      bl.conv_skip = make_conv(h, pfx, 1, h->D, h->S, 1, false);
    }
    bl.has_cond = c.conditioning != 0;
    if (bl.has_cond) {
      snprintf(pfx, sizeof(pfx), "block%d/conv_cond", b);
      bl.cw_idx = add_param(h, std::string(pfx) + "/kernel", {1, h->Cc, 2 * h->D});
      bl.cb_idx = add_param(h, std::string(pfx) + "/bias", {2 * h->D});
    }
  }
  if (c.has_head) {
    int cin = c.use_skip ? h->Sp : h->R;
    for (int i = 0; i <= c.n_final; ++i) {
      char pfx[32];
      snprintf(pfx, sizeof(pfx), "final%d", i);
      const int ch = i < c.n_final ? c.final_layers_channels[i] : h->Cout;
      h->head.push_back(make_conv(h, pfx, 1, cin, ch, 1, false));
      cin = ch;
    }
  }
  if (c.conditioning && c.has_head) {
    int cin = c.cond_in;
    for (int i = 0; i < c.n_mapping; ++i) {
      char pfx[32];
      snprintf(pfx, sizeof(pfx), "mapping%d", i);
      h->map_w.push_back(add_param(h, std::string(pfx) + "/kernel", {cin, c.mapping_layers[i]}));
      h->map_b.push_back(add_param(h, std::string(pfx) + "/bias", {c.mapping_layers[i]}));
      h->map_width.push_back(c.mapping_layers[i]);
      cin = c.mapping_layers[i];
    }
  }
  if (c.precision == WN_BF16) {
    int r = tc_check_config(h->R, h->D, h->Sp, c.kernel_size);
    if (r != 0) {
      set_err("bf16/tcgen05 tier needs channels, dilation_channels and skip_channels to be multiples of 32 (got R=%d D=%d S=%d); use precision=fp32", h->R, h->D, h->Sp);
      delete h;
      return WN_ERR_UNSUPPORTED;
    }
    for (auto& hc : h->head)
      if (hc.cin % 32 != 0) { set_err("bf16 tier needs head widths that are multiples of 32"); delete h; return WN_ERR_UNSUPPORTED; }
  }

  // ---- grouped weight gradients: bf16 tier, separate skip projection (or none), widths in whole 256-channel pair tiles
  if (c.precision == WN_BF16) {
    const char* e = getenv("WN_TC_GROUP_WGRAD");
    bool ok = !(e && e[0] == '0') && h->R % 256 == 0 && h->D % 256 == 0 && h->K <= TC_MAX_TAPS;
    for (auto& b : h->blocks) if (b.has_skip && h->S % 256 != 0) ok = false;
    if (ok) {
      // d z, d x_out (and d x_out + d skip when the skip aliases conv1, and the pre-stack gradients of multi-dilation
      // blocks) of every block stay resident
      size_t free_b = 0, total_b = 0;
      cudaMemGetInfo(&free_b, &total_b);
      double per_row = 0.0;
      for (auto& b : h->blocks) per_row += 2.0 * h->D + h->R + ((h->alias_skip && c.use_skip) ? h->R : 0) + ((double)b.stack.size() - 1.0) * h->D;
      const double extra = per_row * h->maxB * h->maxT * 2.0;
      if (extra > 0.25 * (double)free_b) ok = false;
    }
    h->use_group_wgrad = ok ? 1 : 0;
    { const char* s = getenv("WN_TC_GROUP_SPLIT"); if (s) h->wg_force_split = atoi(s); }
    { const char* s = getenv("WN_TC_GROUP_NH2"); if (s && s[0] == '0') h->wg_pair_tiles = 0; }
    { const char* s = getenv("WN_TC_GROUP_SIDE_EVERY"); if (s) h->wg_side_every = atoi(s); }
  }
  // ---- allocate
  h->pack.dry = true; h->ws.dry = true;
  layout_buffers(h);
  const size_t pack_bytes = h->pack.off + 256, ws_bytes = h->ws.off + 256;
  h->pack = Arena(); h->ws = Arena();
  cudaError_t e;
  if ((e = cudaMalloc(&h->d_params, (size_t)h->n_scalars * 4 + 64)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_grads, (size_t)h->n_scalars * 4 + 64)) != cudaSuccess ||
      (e = cudaMalloc(&h->pack.base, pack_bytes)) != cudaSuccess || (e = cudaMalloc(&h->ws.base, ws_bytes)) != cudaSuccess) {
    set_err("cudaMalloc failed (%s): params %lld scalars, packed %zu B, workspace %zu B", cudaGetErrorString(e), h->n_scalars, pack_bytes, ws_bytes);
    wn_destroy(h);
    return WN_ERR_CUDA;
  }
  h->pack.cap = pack_bytes; h->ws.cap = ws_bytes;
  h->pack.dry = false; h->ws.dry = false;
  layout_buffers(h);
  cudaMemset(h->d_params, 0, (size_t)h->n_scalars * 4);
  cudaMemset(h->d_grads, 0, (size_t)h->n_scalars * 4);
  cudaMemset(h->pack.base, 0, pack_bytes);
  cudaMemset(h->ws.base, 0, ws_bytes);
  cudaMallocHost(&h->pin_frames, (size_t)h->maxB * (h->maxT + 1) * 4);
  cudaMallocHost(&h->pin_cond, (size_t)h->maxB * (c.cond_in > 0 ? c.cond_in : 1) * 4);
  cudaMallocHost(&h->pin_loss, 16);
  cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming);
  { const char* e = getenv("WN_CUDA_GRAPH"); if (e && e[0] == '0') h->use_graphs = 0; }
  { const char* e = getenv("WN_TC_STACK_FWD"); if (e && e[0] == '0') h->use_stack_fwd = 0; }
  { const char* e = getenv("WN_TC_STACK_BWD"); if (e && e[0] == '0') h->use_stack_bwd = 0; }
  cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&h->ev_wg_side, cudaEventDisableTiming);
  {
    // highest priority: the blocks of an early bucket's all-reduce must be scheduled as soon as CTAs of the running weight-gradient
    // launch retire, not behind the CTAs that launch still has pending (measured at 8 GPUs: without it the overlap won 0.02 ms)
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&h->comm_stream, cudaStreamNonBlocking, hi) != cudaSuccess) {
      cudaGetLastError();
      cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking);
    }
  }
  for (int i = 0; i < 8; ++i) cudaEventCreateWithFlags(&h->ev_bucket[i], cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->ev_comm_done, cudaEventDisableTiming);
  { const char* e = getenv("WN_AR_FIRST"); if (e) { h->ar_first_pct = atoi(e); if (h->ar_first_pct < 10) h->ar_first_pct = 10; if (h->ar_first_pct > 90) h->ar_first_pct = 90; } }
  { const char* e = getenv("WN_AR_BUCKETS"); if (e) { h->ar_buckets = atoi(e); if (h->ar_buckets < 1) h->ar_buckets = 1; if (h->ar_buckets > 8) h->ar_buckets = 8; } }
  for (int i = 0; i < h->L; ++i) {
    cudaEvent_t a, b2, c2;
    cudaEventCreateWithFlags(&a, cudaEventDisableTiming); cudaEventCreateWithFlags(&b2, cudaEventDisableTiming); cudaEventCreateWithFlags(&c2, cudaEventDisableTiming);
    h->ev_blk_in.push_back(a); h->ev_blk_dz.push_back(b2); h->ev_blk_done.push_back(c2);
  }
  // offsets of the per-block skip biases (or conv1 biases when aliased) for bskip_sum
  {
    std::vector<int> offs;
    for (auto& b : h->blocks) offs.push_back((int)h->params[b.has_skip ? b.conv_skip.b_idx : b.conv1.b_idx].offset);
    cudaMemcpy(h->d_bskip_offsets, offs.data(), offs.size() * 4, cudaMemcpyHostToDevice);
    if (c.conditioning) {
      std::vector<int> co;
      for (auto& b : h->blocks) { co.push_back((int)h->params[b.cw_idx].offset); co.push_back((int)h->params[b.cb_idx].offset); }
      cudaMemcpy(h->d_cond_offsets, co.data(), co.size() * 4, cudaMemcpyHostToDevice);
    }
  }
  if (c.precision == WN_BF16) {
    int r = tc_init();
    if (r != 0) { set_err("cannot resolve cuTensorMapEncodeTiled from the driver"); wn_destroy(h); return WN_ERR_CUDA; }
  }
  CK(cudaDeviceSynchronize());
  int r = wn_params_changed(h, nullptr);
  if (r != WN_OK) { wn_destroy(h); return r; }
  *out = h;
  return WN_OK;
}

extern "C" void wn_destroy(wn_handle* h) {
  if (!h) return;
  cudaDeviceSynchronize();
  if (h->comm && h->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  for (auto& p : h->prof_events) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  drop_graphs(h);
  for (auto e : h->ev_blk_in) cudaEventDestroy(e);
  for (auto e : h->ev_blk_dz) cudaEventDestroy(e);
  for (auto e : h->ev_blk_done) cudaEventDestroy(e);
  if (h->side_stream) cudaStreamDestroy(h->side_stream);
  if (h->ev_wg_side) cudaEventDestroy(h->ev_wg_side);
  if (h->comm_stream) cudaStreamDestroy(h->comm_stream);
  for (int i = 0; i < 8; ++i) if (h->ev_bucket[i]) cudaEventDestroy(h->ev_bucket[i]);
  if (h->ev_comm_done) cudaEventDestroy(h->ev_comm_done);
  if (h->ev_in) cudaEventDestroy(h->ev_in);
  if (h->ev_out) cudaEventDestroy(h->ev_out);
  for (void* a : h->gen.allocs) cudaFree(a);
  for (auto& wp : h->wg_plans) wp.release();
  for (auto& sp : h->stack_plans) sp.release();
  for (auto& sp : h->stack_bwd_plans) sp.release();
  cudaFree(h->d_pack_jobs);
  cudaFree(h->opt_m); cudaFree(h->opt_v); cudaFree(h->opt_chunks); cudaFree(h->opt_var_first);
  cudaFree(h->opt_partial); cudaFree(h->opt_scale); cudaFree(h->opt_norms);
  cudaFree(h->d_params); cudaFree(h->d_grads); cudaFree(h->pack.base); cudaFree(h->ws.base);
  cudaFreeHost(h->pin_frames); cudaFreeHost(h->pin_cond); cudaFreeHost(h->pin_loss);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

extern "C" int wn_receptive_field(const wn_handle* h) { return h ? h->rf : WN_ERR_VALUE; }
extern "C" int wn_dilation(const wn_handle* h, int block, int j) {
  if (!h || block < 0 || block >= h->L || j < 0 || j >= h->cfg.layers_per_block) { set_err("bad block/conv index"); return WN_ERR_VALUE; }
  return h->dil[block * h->cfg.layers_per_block + j];
}
extern "C" int wn_num_params(const wn_handle* h) { return h ? (int)h->params.size() : WN_ERR_VALUE; }
extern "C" int64_t wn_param_count(const wn_handle* h) { return h ? h->n_scalars : WN_ERR_VALUE; }
extern "C" int wn_param_info(const wn_handle* h, int i, char* name, int name_len, int32_t* shape, int32_t* ndim, int64_t* offset) {
  if (!h || i < 0 || i >= (int)h->params.size()) { set_err("bad param index"); return WN_ERR_VALUE; }
  const ParamInfo& p = h->params[i];
  if (name && name_len > 0) { strncpy(name, p.name.c_str(), name_len - 1); name[name_len - 1] = 0; }
  if (shape) for (int k = 0; k < 3; ++k) shape[k] = p.shape[k];
  if (ndim) *ndim = p.ndim;
  if (offset) *offset = p.offset;
  return WN_OK;
}
extern "C" float* wn_params_dev(wn_handle* h) { return h ? h->d_params : nullptr; }
extern "C" float* wn_grads_dev(wn_handle* h) { return h ? h->d_grads : nullptr; }
extern "C" int wn_set_param(wn_handle* h, int i, const float* host) {
  if (!h || i < 0 || i >= (int)h->params.size() || !host) { set_err("bad param index"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpy(h->d_params + h->params[i].offset, host, h->params[i].count * 4, cudaMemcpyHostToDevice));
  h->fwd_valid = false;
  return WN_OK;  // caller must call wn_params_changed() after the last wn_set_param
}
extern "C" int wn_get_param(wn_handle* h, int i, float* host) {
  if (!h || i < 0 || i >= (int)h->params.size() || !host) { set_err("bad param index"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpy(host, h->d_params + h->params[i].offset, h->params[i].count * 4, cudaMemcpyDeviceToHost));
  return WN_OK;
}
extern "C" int wn_get_grad(wn_handle* h, int i, float* host) {
  if (!h || i < 0 || i >= (int)h->params.size() || !host) { set_err("bad param index"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaMemcpy(host, h->d_grads + h->params[i].offset, h->params[i].count * 4, cudaMemcpyDeviceToHost));
  return WN_OK;
}

// ============================================================================ weight packing
__global__ void bias_table_sum(const float* __restrict__ params, const int* __restrict__ offsets, int L, int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int l = 0; l < L; ++l) s += params[offsets[l] + i];
  out[i] = s;
}

static void pack_emit(wn_handle* h, const float* src, int rows, int cols, void* dst, int dst_ld, int mode, int tile, int D, int dst_cols, long long total) {
  if (total <= 0) return;
  PackJob j{src, dst, rows, cols, dst_ld, mode, tile, D, dst_cols, h->pack_blocks, total};
  h->pack_jobs.push_back(j);
  h->pack_blocks += (total + 255) / 256;
}
template <class TO>
static void pack_launch(wn_handle* h, cudaStream_t st, const float* src, int rows, int cols, TO* dst, int dst_ld, int mode, int tile, int D,
                        int dst_cols) {
  (void)st;
  pack_emit(h, src, rows, cols, dst, dst_ld, mode, tile, D, dst_cols, mode == 2 ? (long long)rows * dst_cols : (long long)rows * cols);
}

extern "C" int wn_params_changed(wn_handle* h, void* stream) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const bool bf = h->cfg.precision == WN_BF16;
  const float* P = h->d_params;
  auto run_jobs = [&]() -> int {
    if (bf) pack_all_kernel<bf16><<<(unsigned)h->pack_blocks, 256, 0, st>>>(h->d_pack_jobs, (int)h->pack_jobs.size());
    else pack_all_kernel<float><<<(unsigned)h->pack_blocks, 256, 0, st>>>(h->d_pack_jobs, (int)h->pack_jobs.size());
    bias_table_sum<<<cdiv(h->Sp, 128), 128, 0, st>>>(P, h->d_bskip_offsets, h->L, h->Sp, h->bskip_sum);
    h->launches += 2;
    CK(cudaGetLastError());
    h->fwd_valid = false;
    return WN_OK;
  };
  if (h->pack_ready) return run_jobs();
  auto W = [&](const ConvP& c) { return P + h->params[c.w_idx].offset; };
  auto pack_conv = [&](ConvP& c) {
    const int ktot = c.K * c.cin;
    if (!bf) {
      // forward [ktot][Npad]
      if (c.gate) pack_launch<float>(h, st, W(c), ktot, c.cout, c.Wf, c.Npad, 2, 64, c.cout / 2, c.Npad);
      else pack_launch<float>(h, st, W(c), ktot, c.cout, c.Wf, c.Npad, 0, 0, 0, 0);
      // dgrad: block k = W[k]^T  -> [cout][Cpad]
      for (int k = 0; k < c.K; ++k)
        pack_launch<float>(h, st, W(c) + (size_t)k * c.cin * c.cout, c.cin, c.cout, c.Wb + (size_t)k * c.cout * c.Cpad, c.Cpad, 1, 0, 0, 0);
    } else {
      // forward B operand [N16][ktot]: row n = (permuted) output column, contraction contiguous
      if (c.gate) {
        // transpose of the interleaved matrix: do it via a temporary-free two-step: pack mode 2 into
        // the dgrad scratch is not possible (sizes differ), so use the dedicated kernel
        pack_emit(h, W(c), ktot, c.cout, c.Wf16, c.Kf16, 3, c.tileN16, c.cout / 2, c.N16, (long long)c.N16 * ktot);
      } else {
        pack_launch<bf16>(h, st, W(c), ktot, c.cout, c.Wf16, c.Kf16, 1, 0, 0, 0);
      }
      // dgrad B operand [C16][K*cout]: row = input channel, contraction index (k, cout)
      for (int k = 0; k < c.K; ++k)
        pack_launch<bf16>(h, st, W(c) + (size_t)k * c.cin * c.cout, c.cin, c.cout, c.Wb16 + (size_t)k * c.cout, rup(c.Kb16, 64), 0, 0, 0, 0);
    }
  };
  for (int l = 0; l < h->L; ++l) {
    BlockP& b = h->blocks[l];
    for (auto& c : b.stack) pack_conv(c);
    pack_conv(b.conv1);
    if (b.has_skip) pack_conv(b.conv_skip);
    const int rs = h->R + (b.has_skip ? h->S : 0);
    const ConvP& sk = b.has_skip ? b.conv_skip : b.conv1;
    if (!bf) {
      pack_launch<float>(h, st, W(b.conv1), h->D, h->R, b.Wdg, b.Dpad, 1, 0, 0, 0);
      if (b.has_skip) pack_launch<float>(h, st, W(b.conv_skip), h->D, h->S, b.Wdg + (size_t)h->R * b.Dpad, b.Dpad, 1, 0, 0, 0);
      pack_launch<float>(h, st, W(sk), h->D, h->Sp, h->Wskip + (size_t)l * h->D * h->Spad, h->Spad, 0, 0, 0, 0);
    } else {
      // dg B operand [Dpad16][rs]: row = channel of g, contraction over (R | S)
      pack_launch<bf16>(h, st, W(b.conv1), h->D, h->R, b.Wdg16, rup(rs, 64), 0, 0, 0, 0);
      if (b.has_skip) pack_launch<bf16>(h, st, W(b.conv_skip), h->D, h->S, b.Wdg16 + h->R, rup(rs, 64), 0, 0, 0, 0);
      // skip-sum B operand [Spad16][L*D]: row = skip channel, contraction over (l, d)
      pack_launch<bf16>(h, st, W(sk), h->D, h->Sp, h->Wskip16 + (size_t)l * h->D, h->L * h->D, 1, 0, 0, 0);
      if (b.Wres16) {
        pack_launch<bf16>(h, st, W(b.conv1), h->D, h->R, b.Wres16, h->D + h->R, 1, 0, 0, 0);
        pack_emit(h, nullptr, 0, 0, b.Wres16 + h->D, h->D + h->R, 4, 0, 0, 0, h->R);
      }
    }
    if (b.Wfc || b.Wfc16) {
      // conditioning-sequence operands: [gated conv taps ; Wc] with the gated conv's column order, and Wc for d cond
      const ConvP& c = b.stack.back();
      const int ktot = c.K * c.cin, Cc = h->Cc;
      const float* Wc = P + h->params[b.cw_idx].offset;
      if (!bf) {
        pack_launch<float>(h, st, W(c), ktot, c.cout, b.Wfc, c.Npad, 2, 64, c.cout / 2, c.Npad);
        pack_launch<float>(h, st, Wc, Cc, c.cout, b.Wfc + (size_t)ktot * c.Npad, c.Npad, 2, 64, c.cout / 2, c.Npad);
        pack_launch<float>(h, st, Wc, Cc, c.cout, b.Wct, b.Ccpad, 1, 0, 0, 0);
      } else {
        pack_emit(h, W(c), ktot, c.cout, b.Wfc16, b.Kfc16, 3, c.tileN16, c.cout / 2, c.N16, (long long)c.N16 * ktot);
        pack_emit(h, Wc, Cc, c.cout, b.Wfc16 + ktot, b.Kfc16, 3, c.tileN16, c.cout / 2, c.N16, (long long)c.N16 * Cc);
        pack_launch<bf16>(h, st, Wc, Cc, c.cout, b.Wct16, c.cout, 0, 0, 0, 0);
      }
    }
  }
  for (auto& c : h->head) pack_conv(c);
  CK(cudaMalloc(&h->d_pack_jobs, h->pack_jobs.size() * sizeof(PackJob)));
  CK(cudaMemcpy(h->d_pack_jobs, h->pack_jobs.data(), h->pack_jobs.size() * sizeof(PackJob), cudaMemcpyHostToDevice));
  h->pack_ready = true;
  return run_jobs();
}

// ============================================================================ GEMM dispatch
struct SegH { const void* A; int lda; int shift; int K; };
struct GemmH {
  int B, T, N;
  int nseg; SegH seg[WN_MAX_SEG];
  int n_outer = 1; long long outer_stride = 0;
  const float* W32 = nullptr; int Npad = 0;     // fp32: [ktot][Npad]
  const bf16* W16 = nullptr; int ktot16 = 0; int N16 = 0; int tile16 = 0;  // bf16: [N16][ktot16]
  int l2_a = 0, l2_in[2] = {0, 0}, l2_out[3] = {0, 0, 0};   // bf16 tier: L2 policy codes (TC_L2_*), see tc_common.cuh
  int l2_seg[WN_MAX_SEG] = {-1, -1, -1, -1, -1};            // per-segment override of l2_a
};

// bf16 tier: map the generic epilogue description onto the TMA-staged tcgen05 kernel (tc_epilogues.cuh);
// the fp32-output head GEMM (logits) and shapes the half-panel maps cannot express use the direct-store kernel.
static inline bool tc_io_ok(const void* p, int ld, int n) { return ((uintptr_t)p & 15) == 0 && ld % 8 == 0 && n % 16 == 0; }

template <class Epi>
static int tc_dispatch(wn_handle* h, cudaStream_t st, const TcGemmDesc& d, const typename Epi::Params& ep) { return tc_conv_gemm<Epi>(h->tmaps, st, d, ep); }
template <>
int tc_dispatch<EpiBiasActRes<bf16, bf16, true>>(wn_handle* h, cudaStream_t st, const TcGemmDesc& d, const EpiBiasActRes<bf16, bf16, true>::Params& ep) {
  if (!tc_io_ok(ep.out, ep.ldo, ep.N) || (ep.res && !tc_io_ok(ep.res, ep.ldr, ep.N))) return tc_conv_gemm<EpiBiasActRes<bf16, bf16, true>>(h->tmaps, st, d, ep);
  TcEpiBiasActRes<true>::Params q{ep.bias, ep.cbias, ep.ldcb, ep.act, ep.N};
  TcEpiIo in[2] = {{ep.res, ep.ldr, ep.N, 0}, {nullptr, 0, 0, 0}};
  TcEpiIo out[3] = {{ep.out, ep.ldo, ep.N, 0}, {}, {}};
  return tc_conv_gemm_staged<TcEpiBiasActRes<true>>(h->tmaps, st, d, q, in, ep.res ? 1u : 0u, out);
}
template <>
int tc_dispatch<EpiGate<bf16, true>>(wn_handle* h, cudaStream_t st, const TcGemmDesc& d, const EpiGate<bf16, true>::Params& ep) {
  TcEpiGate<true>::Params q{ep.bias, ep.cbias, ep.D};
  TcEpiIo out[3] = {{ep.z, 2 * ep.D, ep.D, 0}, {ep.z + ep.D, 2 * ep.D, ep.D, 0}, {ep.g, ep.ldg, ep.D, 0}};
  return tc_conv_gemm_staged<TcEpiGate<true>>(h->tmaps, st, d, q, nullptr, 0u, out);
}
template <>
int tc_dispatch<EpiGateBwd<bf16, true>>(wn_handle* h, cudaStream_t st, const TcGemmDesc& d, const EpiGateBwd<bf16, true>::Params& ep) {
  TcEpiGateBwd<true>::Params q{ep.D};
  TcEpiIo in[2] = {{ep.z, 2 * ep.D, ep.D, 0}, {ep.z + ep.D, 2 * ep.D, ep.D, 0}};
  TcEpiIo out[3] = {{ep.dz, 2 * ep.D, ep.D, 0}, {ep.dz + ep.D, 2 * ep.D, ep.D, 0}, {}};
  return tc_conv_gemm_staged<TcEpiGateBwd<true>>(h->tmaps, st, d, q, in, 3u, out);
}
template <>
int tc_dispatch<EpiActBwd<bf16, bf16>>(wn_handle* h, cudaStream_t st, const TcGemmDesc& d, const EpiActBwd<bf16, bf16>::Params& ep) {
  const bool use_y = ep.y && ep.act != ACT_LINEAR;
  if (!tc_io_ok(ep.out, ep.ldo, ep.N) || (ep.add && !tc_io_ok(ep.add, ep.lda, ep.N)) || (use_y && !tc_io_ok(ep.y, ep.ldy, ep.N)))
    return tc_conv_gemm<EpiActBwd<bf16, bf16>>(h->tmaps, st, d, ep);
  TcEpiActBwd::Params q{ep.act};
  TcEpiIo in[2] = {{ep.add, ep.lda, ep.N, 0}, {ep.y, ep.ldy, ep.N, 0}};
  TcEpiIo out[3] = {{ep.out, ep.ldo, ep.N, 0}, {}, {}};
  return tc_conv_gemm_staged<TcEpiActBwd>(h->tmaps, st, d, q, in, (ep.add ? 1u : 0u) | (use_y ? 2u : 0u), out);
}

template <class T, class Epi>
static int run_conv_gemm(wn_handle* h, cudaStream_t st, int cls, const GemmH& g, const typename Epi::Params& ep) {
  LaunchLabel lab(h, Epi::kLabel);
  LaunchScope ls(h, st, cls);
  if constexpr (sizeof(T) == 4) {
    ConvGemmArgsF a;
    a.B = g.B; a.T = g.T; a.Npad = g.Npad; a.nseg = g.nseg; a.n_outer = g.n_outer; a.a_outer_stride = g.outer_stride; a.W = g.W32;
    for (int s = 0; s < g.nseg; ++s) a.seg[s] = SegF{(const float*)g.seg[s].A, g.seg[s].lda, g.seg[s].shift, g.seg[s].K};
    dim3 grid(g.B * cdiv(g.T, 64), g.Npad / 64);
    conv_gemm_simt<Epi><<<grid, 256, 0, st>>>(a, ep);
    return WN_OK;
  } else {
    TcGemmDesc d;
    d.B = g.B; d.T = g.T; d.nseg = g.nseg; d.n_outer = g.n_outer; d.outer_stride = g.outer_stride;
    for (int s = 0; s < g.nseg; ++s) d.seg[s] = TcSeg{(const bf16*)g.seg[s].A, g.seg[s].lda, g.seg[s].shift, g.seg[s].K};
    d.W = g.W16; d.ktot = g.ktot16; d.N16 = g.N16; d.tileN = g.tile16;
    d.l2_a = g.l2_a;
    for (int s = 0; s < g.nseg && s < TC_MAX_SEG; ++s) d.l2_seg[s] = g.l2_seg[s];
    for (int k = 0; k < 2; ++k) d.l2_in[k] = g.l2_in[k];
    for (int k = 0; k < 3; ++k) d.l2_out[k] = g.l2_out[k];
    int r = tc_dispatch<Epi>(h, st, d, ep);
    if (r != 0) { set_err("tcgen05 conv_gemm launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
    return WN_OK;
  }
}

struct WgradH {
  int B, T, N; const void* G; int ldg;
  int nseg; SegH seg[WN_MAX_SEG];
  float* dst;          // [ktot][N] Keras layout in the flat grad buffer
  const float* w; float l2coef;  // optional L2 term: dst += l2coef * w
  // column sums of G ride along: bias gradient [N] and (conditioning) per-batch sums [B][ldpb]
  float* bias_dst = nullptr; float* per_batch = nullptr; int ldpb = 0;
  // bf16 tier only: columns [N0, N) belong to a second variable (conv1 | conv_skip in one launch)
  int N0 = 0; float* dst1 = nullptr; const float* w1 = nullptr; float* bias1 = nullptr;
  bool side = false;   // issued on the side stream: uses the side copies of the partial buffers
  int l2_a = 0, l2_g = 0;   // bf16 tier: L2 policy codes of the two operands
};

template <class T>
static void run_colsum(wn_handle* h, cudaStream_t st, const void* G, int ldg, int B, int Tn, int N, float* per_batch, int ldpb, float* total);

template <class T>
static int run_wgrad(wn_handle* h, cudaStream_t st, int cls, const WgradH& g) {
  LaunchLabel lab(h, cls == CLS_DILATED ? "wgrad_dilated" : "wgrad_1x1");
  int ktot = 0;
  for (int s = 0; s < g.nseg; ++s) ktot += g.seg[s].K;
  int nsplit = 1;
  if constexpr (sizeof(T) == 4) {
    int ktiles = 0;
    for (int s = 0; s < g.nseg; ++s) ktiles += cdiv(g.seg[s].K, 64);
    const int ntiles = cdiv(g.N, 64);
    const int chunks = g.B * cdiv(g.T, 16);
    nsplit = 296 * 2 / (ktiles * ntiles);
    if (nsplit < 1) nsplit = 1;
    if (nsplit > WN_MAX_WGRAD_SPLITS) nsplit = WN_MAX_WGRAD_SPLITS;
    if (nsplit > chunks) nsplit = chunks;
    const int cps = cdiv(chunks, nsplit);
    nsplit = cdiv(chunks, cps);
    WgradArgsF a;
    a.B = g.B; a.T = g.T; a.N = g.N; a.G = (const float*)g.G; a.ldg = g.ldg; a.nseg = g.nseg; a.ktot = ktot;
    for (int s = 0; s < g.nseg; ++s) a.seg[s] = SegF{(const float*)g.seg[s].A, g.seg[s].lda, g.seg[s].shift, g.seg[s].K};
    a.partial = h->wg_partial; a.chunks_per_split = cps;
    // bias gradient = column sums of G: they ride along as row ktot of the partials (per-batch sums, i.e. conditioned gated convs,
    // keep the separate column-sum launches)
    const bool cs_row = g.bias_dst != nullptr && g.per_batch == nullptr;
    a.cs_row = cs_row ? 1 : 0;
    {
      LaunchScope ls(h, st, cls);
      wgrad_simt<<<dim3(ktiles, ntiles, nsplit), 256, 0, st>>>(a);
    }
    if (cs_row) {
      LaunchScope ls(h, st, cls);
      const long long n = (long long)ktot * g.N;
      reduce_parts2<<<cdiv(n + g.N, 256), 256, 0, st>>>(h->wg_partial, nsplit, n + g.N, g.dst, n, g.bias_dst, g.N, g.l2coef != 0.f ? g.w : nullptr, g.l2coef);
      return WN_OK;
    }
    if (g.bias_dst || g.per_batch) run_colsum<T>(h, st, g.G, g.ldg, g.B, g.T, g.N, g.per_batch, g.ldpb, g.bias_dst);
  } else {
    TcWgradDesc d;
    d.B = g.B; d.T = g.T; d.N = g.N; d.G = (const bf16*)g.G; d.ldg = g.ldg; d.nseg = g.nseg; d.ktot = ktot;
    for (int s = 0; s < g.nseg; ++s) d.seg[s] = TcSeg{(const bf16*)g.seg[s].A, g.seg[s].lda, g.seg[s].shift, g.seg[s].K};
    d.l2_a = g.l2_a; d.l2_g = g.l2_g;
    float* const wgp = g.side ? h->wg_partial_side : h->wg_partial;
    float* const csp = g.side ? h->cs_partial_side : h->cs_partial;
    d.partial = wgp;
    const bool want_cs = g.bias_dst || g.per_batch || g.bias1;
    d.cs_partial = want_cs ? csp : nullptr;
    TcWgradPlan plan{};
    {
      LaunchScope ls(h, st, cls);
      int r = tc_wgrad(h->tmaps, st, d, &plan);
      if (r != 0) { set_err("tcgen05 wgrad launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
    }
    TcWgradFinish f{};
    f.partial = wgp; f.nsplit = plan.nsplit; f.ktot = ktot; f.N = g.N; f.N0 = g.dst1 ? g.N0 : g.N;
    f.dst0 = g.dst; f.dst1 = g.dst1; f.l2coef = g.l2coef;
    f.w0 = g.l2coef != 0.f ? g.w : nullptr; f.w1 = g.l2coef != 0.f ? g.w1 : nullptr;
    f.cs = csp; f.slots = plan.slots; f.cps = plan.chunks_per_split; f.chunks_t = plan.chunks_t; f.B = g.B; f.mtiles = plan.mtiles;
    f.bias0 = g.bias_dst; f.bias1 = g.bias1; f.per_batch = g.per_batch; f.ldpb = g.ldpb;
    f.wblocks = cdiv((long long)ktot * g.N, 256);
    const int nblocks = f.wblocks + (want_cs ? cdiv(g.N, 32) : 0);
    // one finish per weight gradient: one finish launch for both wgrads of a block measured SLOWER on C2 (7.48 vs 7.38 ms/step:
    // the deferred partials fall out of L2 before the merged finish reads them)
    LaunchScope ls(h, st, cls);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(nblocks); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 1);
    CK(cudaLaunchKernelEx(&cfg, tc_wgrad_finish, f));
    return WN_OK;
  }
  {
    LaunchScope ls(h, st, cls);
    const long long n = (long long)ktot * g.N;
    reduce_parts<<<cdiv(n, 256), 256, 0, st>>>(h->wg_partial, nsplit, n, g.dst, n, g.l2coef != 0.f ? g.w : nullptr, g.l2coef);
  }
  return WN_OK;
}

// column sums of G (B,T,N) -> total[N] and/or per_batch[B][ldpb]
template <class T>
static void run_colsum(wn_handle* h, cudaStream_t st, const void* G, int ldg, int B, int Tn, int N, float* per_batch, int ldpb, float* total) {
  const int chunks = cdiv(Tn, 256);
  {
    LaunchScope ls(h, st, CLS_MISC);
    colsum_stage1<T><<<dim3(cdiv(N, 32), chunks, B), 256, 0, st>>>((const T*)G, ldg, h->colpart, Tn, N, 256);
  }
  {
    LaunchScope ls(h, st, CLS_MISC);
    colsum_stage2<<<cdiv(N, 32), 256, 0, st>>>(h->colpart, B, chunks, N, per_batch, ldpb, total);
  }
}

// ============================================================================ forward pieces
static inline float* P_(wn_handle* h, int idx) { return h->d_params + h->params[idx].offset; }
static inline float* G_(wn_handle* h, int idx) { return h->d_grads + h->params[idx].offset; }

template <class T> static inline bool vec_ok(int ld) { return (ld * (int)sizeof(T)) % 16 == 0; }

static void fill_w(GemmH& g, const ConvP& c, bool dgrad) {
  if (!dgrad) { g.W32 = c.Wf; g.Npad = c.Npad; g.W16 = c.Wf16; g.ktot16 = c.Kf16; g.N16 = c.N16; g.tile16 = c.tileN16; }
  else { g.W32 = c.Wb; g.Npad = c.Cpad; g.W16 = c.Wb16; g.ktot16 = rup(c.Kb16, 64); g.N16 = c.C16; g.tile16 = 0; }
}

// conditioning: mapping MLP (model.py:141-148,222) and the per-block time-constant bias
// cb[l][b][:] = cond[b] @ Wc_l + bc_l  (layers.py:203-204 with cond constant in time)
// one single-block launch each way for the conditioning MLP while it is as small as it really is (above 2^20 MACs: per layer)
static bool mapping_args(wn_handle* h, const float* cond_in, int B, float l2coef, MapArgs* a) {
  const int nl = (int)h->map_w.size();
  if (nl < 1 || nl > WN_MAX_LIST) return false;
  long long macs = 0;
  int k = h->cfg.cond_in;
  for (int i = 0; i < nl; ++i) { macs += (long long)B * k * h->map_width[i]; k = h->map_width[i]; }
  if (macs > (1 << 20)) return false;
  a->n_layers = nl; a->B = B; a->cond_in = h->cfg.cond_in; a->act = h->cfg.mapping_activation; a->l2coef = l2coef; a->x0 = cond_in;
  for (int i = 0; i < nl; ++i) {
    a->width[i] = h->map_width[i];
    a->W[i] = P_(h, h->map_w[i]); a->bias[i] = P_(h, h->map_b[i]);
    a->gW[i] = G_(h, h->map_w[i]); a->gb[i] = G_(h, h->map_b[i]);
    a->actv[i] = h->cond_act[i];
  }
  a->d0 = h->dcond; a->d1 = h->cond_dact; a->d2 = h->cond_dact2;
  return true;
}
// the mapping MLP's output (cond_in itself without mapping layers)
static const float* cond_forward(wn_handle* h, cudaStream_t st, const float* cond_in, int B) {
  MapArgs ma;
  if (mapping_args(h, cond_in, B, 0.f, &ma)) {
    LaunchScope ls(h, st, CLS_MISC);
    mapping_fwd_fused<<<1, 256, 0, st>>>(ma);
    return h->cond_act[ma.n_layers - 1];
  }
  const float* cur = cond_in;
  int width = h->cfg.cond_in;
  for (size_t i = 0; i < h->map_w.size(); ++i) {
    LaunchScope ls(h, st, CLS_MISC);
    const int n = h->map_width[i];
    dense_small_fwd<<<cdiv(B * n, 128), 128, 0, st>>>(cur, width, P_(h, h->map_w[i]), P_(h, h->map_b[i]), h->cond_act[i], n, B, width, n,
                                                    h->cfg.mapping_activation);
    cur = h->cond_act[i];
    width = n;
  }
  return cur;
}
static void cond_bias_block(wn_handle* h, cudaStream_t st, int l, const float* cond, int B) {
  const BlockP& b = h->blocks[l];
  LaunchScope ls(h, st, CLS_MISC);
  const int n = 2 * h->D;
  dense_small_fwd<<<cdiv(B * n, 128), 128, 0, st>>>(cond, h->Cc, P_(h, b.cw_idx), P_(h, b.cb_idx), h->cb + (size_t)l * h->maxB * n, n, B, h->Cc, n,
                                                  ACT_LINEAR);
}
// ---- conditioning of the whole model: the mapping MLP, then cb of every block; h->last_cond: the mapped conditioning (null without)
static void model_cond_forward(wn_handle* h, cudaStream_t st, const float* cond_in, int B) {
  h->last_cond = nullptr;
  if (!h->cfg.conditioning) return;
  OuterLabel ol(h, "cond_fwd");
  h->last_cond = cond_forward(h, st, cond_in, B);
  LaunchScope ls(h, st, CLS_MISC);
  const int n = 2 * h->D;
  cond_bias_all<<<dim3(cdiv(B * n, 128), h->L), 128, 0, st>>>(h->last_cond, h->Cc, h->d_params, h->d_cond_offsets, h->cb, (long long)h->maxB * n, B, n);
}

// the conv part of a fused-kernel desc (gemm_tc_block.cuh, gemm_tc_stack.cuh): conv cv over A (row width lda), writing xout
static TcBlockDesc conv_desc(wn_handle* h, const ConvP& cv, const void* A, int lda, void* xout, int B, int Tn) {
  TcBlockDesc d{};
  d.B = B; d.T = Tn; d.nseg = cv.K; d.Cin = cv.cin; d.D = h->D; d.R = h->R; d.has_res = 1;
  for (int k = 0; k < cv.K; ++k) d.shift[k] = -(cv.K - 1 - k) * cv.dil;
  d.A = (const bf16*)A; d.lda = lda; d.xout = (bf16*)xout;
  d.W1 = cv.Wf16; d.k1 = cv.Kf16; d.bias_g = P_(h, cv.b_idx);
  return d;
}
// block l's gated conv over A + gate + conv1 + residual x_in as one fused-kernel desc
static TcBlockDesc block_desc(wn_handle* h, int l, const void* A, int lda, const void* x_in, bool has_cb, int B, int Tn) {
  const BlockP& b = h->blocks[l];
  TcBlockDesc d = conv_desc(h, b.stack.back(), A, lda, h->xout[l], B, Tn);
  d.X = (const bf16*)x_in; d.ldx = h->R; d.W2 = b.Wres16;
  d.z = (bf16*)h->zbuf[l]; d.g = (bf16*)h->G_all + (size_t)l * h->maxB * h->maxT * h->D;
  d.cbias = has_cb ? h->cb + (size_t)l * h->maxB * 2 * h->D : nullptr;
  d.bias_r = P_(h, b.conv1.b_idx);
  return d;
}

// training-mode dropout on block l's conv branch only: xdrop[l]; the residual still reads x_in (layers.py:192-196)
template <class T>
static const void* dropout_conv_input(wn_handle* h, cudaStream_t st, int l, const void* x_in, int B, int Tn) {
  LaunchScope ls(h, st, CLS_MISC);
  const long long n = (long long)B * Tn * h->R;
  dropout_apply<T><<<cdiv(n, 256), 256, 0, st>>>((const T*)x_in, h->drop_mask + (size_t)l * h->maxB * h->maxT * h->R, (T*)h->xdrop[l], n,
                                                1.0f / (1.0f - h->cfg.dropout));
  return h->xdrop[l];
}

// WaveNetLayer.call for block l (layers.py:178-224); x_in (B,T,R) in T
template <class T>
static int block_forward(wn_handle* h, cudaStream_t st, int l, const void* x_in, bool has_cb, int B, int Tn) {
  BlockP& b = h->blocks[l];
  const int depth = (int)b.stack.size();
  const size_t rows_cap = (size_t)h->maxB * h->maxT;
  const void* cur = h->drop_active ? dropout_conv_input<T>(h, st, l, x_in, B, Tn) : x_in;
  int curw = h->R;
  for (int j = 0; j < depth; ++j) {
    const ConvP& c = b.stack[j];
    GemmH g;
    g.B = B; g.T = Tn; g.N = c.cout; g.nseg = c.K;
    for (int k = 0; k < c.K; ++k) g.seg[k] = SegH{cur, curw, -(c.K - 1 - k) * c.dil, c.cin};
    fill_w(g, c, false);
    if (j < depth - 1) {
      typename EpiBiasActRes<T, T, sizeof(T) == 2>::Params ep{};
      ep.out = (T*)h->acts[l][j]; ep.ldo = h->D; ep.bias = P_(h, c.b_idx); ep.cbias = nullptr; ep.ldcb = 0;
      ep.act = h->cfg.activation; ep.res = nullptr; ep.ldr = 0; ep.N = c.cout; ep.vec = vec_ok<T>(h->D);
      g.l2_out[0] = TC_L2_LAST;   // the next conv of the stack reads it right away
      RET((run_conv_gemm<T, EpiBiasActRes<T, T, sizeof(T) == 2>>(h, st, CLS_DILATED, g, ep)));
      cur = h->acts[l][j];
      curw = h->D;
    } else {
      if constexpr (sizeof(T) == 2) {
        // bf16 tier: gated conv + gate + conv1 (+ residual) as ONE kernel when the shapes allow (gemm_tc_block.cuh)
        if (b.Wres16 && h->cfg.use_residual && c.K <= TC_MAX_TAPS && !h->cond_seq) {
          const TcBlockDesc d = block_desc(h, l, cur, curw, x_in, has_cb, B, Tn);
          bool ran;
          RET(launch_persistent(h, st, "block_fwd", "fused block forward", [&] { return c.tileN16 == 256 ? tc_block_fwd(h->tmaps, st, d) : -100; }, &ran));
          if (ran) { h->fused_fwd_launches++; return WN_OK; }      // else: the separate kernels below
        }
      }
      typename EpiGate<T, sizeof(T) == 2>::Params ep{};
      ep.z = (T*)h->zbuf[l];
      ep.g = (T*)h->G_all + (size_t)l * rows_cap * h->D;
      ep.ldg = h->D; ep.bias = P_(h, c.b_idx);
      ep.cbias = has_cb ? h->cb + (size_t)l * h->maxB * 2 * h->D : nullptr;
      ep.D = h->D; ep.vec = vec_ok<T>(h->D);
      if (h->cond_seq) {
        // conditioning sequence: conv_cond is one more segment of the contraction (layers.py:203-204), bc joins the bias
        g.seg[g.nseg++] = SegH{h->cond_seq, h->Ccs, 0, h->Ccs};
        g.W32 = b.Wfc; g.W16 = b.Wfc16; g.ktot16 = b.Kfc16;
        ep.bias = h->cseq_bias + (size_t)l * 2 * h->D;
      }
      // z is not needed before the backward pass (streaming store); g feeds conv1 next; x_in is conv1's residual
      g.l2_a = depth == 1 ? TC_L2_LAST : TC_L2_NORMAL;
      g.l2_out[0] = g.l2_out[1] = TC_L2_FIRST; g.l2_out[2] = TC_L2_LAST;
      RET((run_conv_gemm<T, EpiGate<T, sizeof(T) == 2>>(h, st, CLS_DILATED, g, ep)));
    }
  }
  // conv1 (+ residual)
  {
    const ConvP& c = b.conv1;
    GemmH g;
    g.B = B; g.T = Tn; g.N = h->R; g.nseg = 1;
    g.seg[0] = SegH{(const T*)h->G_all + (size_t)l * rows_cap * h->D, h->D, 0, h->D};
    fill_w(g, c, false);
    typename EpiBiasActRes<T, T, sizeof(T) == 2>::Params ep{};
    ep.out = (T*)h->xout[l]; ep.ldo = h->R; ep.bias = P_(h, c.b_idx); ep.act = ACT_LINEAR;
    ep.res = h->cfg.use_residual ? (const T*)x_in : nullptr; ep.ldr = h->R; ep.N = h->R; ep.vec = vec_ok<T>(h->R);
    if (sizeof(T) == 2 && b.Wres16) {
      // residual through the contraction: second segment x_in against the identity block of [Wr^T | I]
      g.nseg = 2;
      g.seg[1] = SegH{x_in, h->R, 0, h->R};
      g.W16 = b.Wres16; g.ktot16 = h->D + h->R;
      ep.res = nullptr;
    }
    // g and x_in are next used a whole pass later; x_out is the next block's operand
    g.l2_a = TC_L2_FIRST; g.l2_in[0] = TC_L2_FIRST; g.l2_out[0] = TC_L2_LAST;
    RET((run_conv_gemm<T, EpiBiasActRes<T, T, sizeof(T) == 2>>(h, st, CLS_GEMM, g, ep)));
  }
  return WN_OK;
}

// skip of blocks [l0, l0+nl): out = sum_l g_l @ Ws_l + sum_l bs_l  (model.py:236; Ws := Wr when aliased)
template <class T, class TO>
static int skip_gemm(wn_handle* h, cudaStream_t st, int l0, int nl, TO* out, int ldo, const float* bias, int B, int Tn) {
  const size_t rows_cap = (size_t)h->maxB * h->maxT;
  GemmH g;
  g.B = B; g.T = Tn; g.N = h->Sp; g.nseg = 1;
  g.seg[0] = SegH{(const T*)h->G_all + (size_t)l0 * rows_cap * h->D, h->D, 0, h->D};
  g.n_outer = nl; g.outer_stride = (long long)rows_cap * h->D;
  g.W32 = h->Wskip ? h->Wskip + (size_t)l0 * h->D * h->Spad : nullptr; g.Npad = h->Spad;
  g.W16 = h->Wskip16 ? h->Wskip16 + (size_t)l0 * h->D : nullptr; g.ktot16 = h->L * h->D; g.N16 = h->Spad; g.tile16 = 0;
  typename EpiBiasActRes<T, TO, sizeof(T) == 2>::Params ep{};
  ep.out = out; ep.ldo = ldo; ep.bias = bias; ep.act = ACT_LINEAR; ep.N = h->Sp; ep.vec = vec_ok<TO>(ldo);
  g.l2_a = TC_L2_FIRST; g.l2_out[0] = TC_L2_LAST;
  return run_conv_gemm<T, EpiBiasActRes<T, TO, sizeof(T) == 2>>(h, st, CLS_GEMM, g, ep);
}

// ---- input conv (model.py:84-88) into h0.  HBM-bound, small CTAs
template <class T>
static void input_conv_forward(wn_handle* h, cudaStream_t st, const float* x, int ldx, int B, int Tn) {
  OuterLabel ol(h, "input_conv_fwd");
  LaunchScope ls(h, st, CLS_MISC);
  const long long total = (long long)B * Tn * h->R;
  if (h->R % 8 == 0 && h->R / 8 <= 256)
    input_conv_fwd_rows<T><<<cdiv((long long)B * Tn, ICF_ROWS), 256, 0, st>>>(x, ldx, P_(h, h->input_conv.w_idx), P_(h, h->input_conv.b_idx), (T*)h->h0, B, Tn, h->R, h->K);
  else if (h->R % 8 == 0)
    input_conv_fwd_vec8<T><<<cdiv(total / 8, 256), 256, 0, st>>>(x, ldx, P_(h, h->input_conv.w_idx), P_(h, h->input_conv.b_idx), (T*)h->h0, B, Tn, h->R, h->K);
  else
    input_conv_fwd<T><<<cdiv(total, 256), 256, 0, st>>>(x, ldx, P_(h, h->input_conv.w_idx), P_(h, h->input_conv.b_idx), (T*)h->h0, B, Tn, h->R, h->K);
}

// The whole residual stack runs as ONE persistent launch (gemm_tc_stack.cuh) when every block takes the fused forward and a
// layer has more 256-row tiles than the GPU has CTA pairs.  Multi-dilation blocks (layers.py:64-88): every conv in front of the
// gated conv is a PLAIN layer of the same launch (its output is kept for the backward pass, as before).
static bool stack_forward_ok(wn_handle* h, int B, int Tn) {
  bool ok = h->use_stack_fwd && h->cfg.use_residual && h->L >= 2 && h->D == h->R && (h->D == 256 || h->D == 128) && more_tiles_than_pairs(B, Tn);
  for (auto& b : h->blocks) {
    if (!ok) break;
    const ConvP& cv = b.stack.back();
    ok = b.Wres16 != nullptr && cv.tileN16 == 256 && cv.K <= TC_MAX_TAPS && cv.cin % 64 == 0;
    for (size_t j = 0; ok && j + 1 < b.stack.size(); ++j) {
      const ConvP& pc = b.stack[j];
      // plain layers run as one 256-wide tile per m tile: D = 256 only; all convs share K and the input width
      ok = h->D == 256 && pc.cout == h->D && pc.cin == cv.cin && pc.K == cv.K && pc.Wf16 != nullptr && pc.N16 == 256 && b.stack.size() <= 16;
    }
  }
  return ok;
}

// ---- every block's convs, gate, conv1 and residual as one persistent launch; *stacked: it ran (else the per-block loop runs them)
static int stack_forward(wn_handle* h, cudaStream_t st, int B, int Tn, bool* stacked) {
  const wn_config& c = h->cfg;
  const bool has_cb = c.conditioning != 0;
  // one desc per CONV: the plain convs of block l, then its gated conv + tail
  std::vector<TcBlockDesc> descs;
  for (int l = 0; l < h->L; ++l) {
    const BlockP& b = h->blocks[l];
    const void* x_in = l > 0 ? h->xout[l - 1] : h->h0;
    // training-mode dropout without leaving the launch: the conv branch of block l reads xdrop[l] = keep_l * x / (1 - rate),
    // written by the OUT epilogue of block l-1 next to x_out (block 0: by dropout_conv_input on h0 below); the residual reads x
    const void* cur = h->drop_active ? (const void*)h->xdrop[l] : x_in;
    int lda = h->R;
    for (size_t j = 0; j + 1 < b.stack.size(); ++j) {
      TcBlockDesc d = conv_desc(h, b.stack[j], cur, lda, h->acts[l][j], B, Tn);
      d.plain = 1; d.act = c.activation;
      descs.push_back(d);
      cur = h->acts[l][j];
      lda = h->D;
    }
    TcBlockDesc d = block_desc(h, l, cur, lda, x_in, has_cb, B, Tn);
    if (h->drop_active && l + 1 < h->L) { d.mask_next = h->drop_mask + (size_t)(l + 1) * h->maxB * h->maxT * h->R; d.xdrop_next = (bf16*)h->xdrop[l + 1]; }
    descs.push_back(d);
  }
  if (h->drop_active) for (TcBlockDesc& d : descs) d.drop_scale = 1.0f / (1.0f - c.dropout);
  TcStackPlan* sp = nullptr;
  RET(plan_for(h, st, h->stack_plans, [&](const TcStackPlan& q) { return q.B == B && q.T == Tn && q.cb == has_cb && q.drop == (h->drop_active && h->L > 1); },
               "stack forward", [&](TcStackPlan& p) { return tc_stack_build(h->tmaps, descs, &p); }, &sp));
  if (!sp) return WN_OK;
  // block 0's masked input from the input conv's output (every later block's comes out of the launch itself)
  if (h->drop_active) dropout_conv_input<bf16>(h, st, 0, h->h0, B, Tn);
  RET(launch_persistent(h, st, "stack_fwd", "stack forward", [&] { return tc_stack_launch(st, *sp, descs[0]); }, stacked));
  if (*stacked) { h->fused_fwd_launches = h->L; h->stack_fwd_layers = h->L; }
  return WN_OK;
}

// ---- skip sum and head convs on the last block's output, into the logits
template <class T>
static int head_forward(wn_handle* h, cudaStream_t st, int B, int Tn) {
  const wn_config& c = h->cfg;
  const void* head_in = h->xout[h->L - 1];
  int head_w = h->R;
  if (c.use_skip) {
    OuterLabel ol(h, "skip_sum");
    RET((skip_gemm<T, T>(h, st, 0, h->L, (T*)h->skipsum, h->Sp, h->bskip_sum, B, Tn)));
    head_in = h->skipsum;
    head_w = h->Sp;
  }
  OuterLabel ol_head(h, "head_fwd");
  for (size_t i = 0; i < h->head.size(); ++i) {
    const ConvP& hc = h->head[i];
    GemmH g;
    g.B = B; g.T = Tn; g.N = hc.cout; g.nseg = 1;
    g.seg[0] = SegH{head_in, head_w, 0, hc.cin};
    fill_w(g, hc, false);
    if (i + 1 < h->head.size()) {
      typename EpiBiasActRes<T, T, sizeof(T) == 2>::Params ep{};
      ep.out = (T*)h->hact[i]; ep.ldo = hc.cout; ep.bias = P_(h, hc.b_idx); ep.act = c.activation; ep.N = hc.cout; ep.vec = vec_ok<T>(hc.cout);
      RET((run_conv_gemm<T, EpiBiasActRes<T, T, sizeof(T) == 2>>(h, st, CLS_GEMM, g, ep)));
      head_in = h->hact[i];
      head_w = hc.cout;
    } else {
      typename EpiBiasActRes<T, float, sizeof(T) == 2>::Params ep{};
      ep.out = h->logits; ep.ldo = h->ldl; ep.bias = P_(h, hc.b_idx); ep.act = ACT_LINEAR; ep.N = hc.cout; ep.vec = vec_ok<float>(h->ldl);
      RET((run_conv_gemm<T, EpiBiasActRes<T, float, sizeof(T) == 2>>(h, st, CLS_GEMM, g, ep)));
    }
  }
  return WN_OK;
}

// WaveNet.call up to the logits (model.py:213-239).  x (B,T) fp32 with row stride ldx.
template <class T>
static int model_forward(wn_handle* h, cudaStream_t st, const float* x, int ldx, const float* cond_in, int B, int Tn) {
  h->fused_fwd_launches = 0; h->stack_fwd_layers = 0;
  model_cond_forward(h, st, cond_in, B);
  input_conv_forward<T>(h, st, x, ldx, B, Tn);
  bool stacked = false;
  if constexpr (sizeof(T) == 2) {
    if (stack_forward_ok(h, B, Tn)) RET(stack_forward(h, st, B, Tn, &stacked));
  }
  for (int l = 0; !stacked && l < h->L; ++l) RET(block_forward<T>(h, st, l, l > 0 ? h->xout[l - 1] : h->h0, h->cfg.conditioning != 0, B, Tn));
  return head_forward<T>(h, st, B, Tn);
}

// loss (model.py:505-551) on the logits; optionally dlogits and probabilities
template <class T>
static int loss_forward(wn_handle* h, cudaStream_t st, const float* frames, int B, int Tn, float scale, bool want_grad, float* probs, float* loss_out) {
  const wn_config& c = h->cfg;
  const long long rows = (long long)B * Tn;
  int nparts;
  {
    OuterLabel ol(h, "loss");
    LaunchScope ls(h, st, CLS_LOSS);
    if (c.sampling_function == WN_CATEGORICAL) {
      nparts = cdiv(rows, 8);
      if (h->Cout == 256 && h->ldl == 256 && h->ldd % 4 == 0)
        softmax_ce_reg_kernel<T, 2><<<nparts, 256, 0, st>>>(h->logits, frames, Tn, rows, c.bits, scale, want_grad ? (T*)h->dlogits : nullptr, h->ldd, probs,
                                                           loss_out ? h->loss_partial : nullptr);
      else
        softmax_ce_kernel<T><<<nparts, 256, 0, st>>>(h->logits, h->Cout, frames, Tn, rows, c.bits, scale, want_grad ? (T*)h->dlogits : nullptr, h->ldd,
                                                    probs, loss_out ? h->loss_partial : nullptr);
    } else {
      mixture_loss_launch<T>(st, &nparts, h->logits, h->ldl, c.num_mixtures, frames, Tn, rows, c.bits, c.sampling_function == WN_GAUSSIAN ? 2 : 1, scale,
                             want_grad ? (T*)h->dlogits : nullptr, h->ldd, loss_out ? h->loss_partial : nullptr, Tn + 1, 1, nullptr);
    }
  }
  if (loss_out) {
    float l2coef = 0.f;
    if (c.l2_reg_factor > 0.f) {
      // model.py:331-334: reg * sum(kernel^2), scaled by 1/replicas (folded into `scale`*B)
      cudaMemsetAsync(h->l2_sum, 0, 4, st);
      for (auto& p : h->params) {
        if (p.name.size() < 6 || p.name.compare(p.name.size() - 6, 6, "kernel") != 0) continue;
        LaunchScope ls(h, st, CLS_MISC);
        sumsq_accum<<<1, 1024, 0, st>>>(h->d_params + p.offset, p.count, h->l2_sum);
      }
      l2coef = c.l2_reg_factor * scale * (float)B;   // reg / n_replicas
    }
    OuterLabel ol(h, "loss_finalize");
    LaunchScope ls(h, st, CLS_LOSS);
    loss_finalize<<<1, 1024, 0, st>>>(h->loss_partial, nparts, scale, l2coef != 0.f ? h->l2_sum : nullptr, l2coef, loss_out);
  }
  return WN_OK;
}

// ============================================================================ backward pieces
// adjoint of block_forward.  dxout / dskip may be null (zero).  Writes dx_in (if non-null) and
// this block's parameter gradients.  dcb row l gets per-batch sums of dz when conditioned.
// Two-stream schedule of one block's backward: the dgrad chain (gate adjoint -> dgrad) is the critical path on
// the main stream; the weight-gradient kernels only consume, so they run on a side stream and fill the SMs the
// persistent GEMMs leave idle in their last partial wave.  Events order producer -> consumer and protect the
// ping-pong buffers (dz, d x_out) from being overwritten while a side kernel still reads them.
// a conv whose output nothing reads (conv1 of the last block under use_skip, conv_skip without use_skip): the data term
// of its gradients is zero, the L2 term (model.py:331-334) is not
static void unused_conv_grads(wn_handle* h, cudaStream_t st, int w_idx, int b_idx, float l2coef) {
  const long long cnt = h->params[w_idx].count;
  if (l2coef != 0.f) {
    LaunchScope ls(h, st, CLS_MISC);
    reduce_parts<<<cdiv(cnt, 256), 256, 0, st>>>(G_(h, w_idx), 0, 0, G_(h, w_idx), cnt, P_(h, w_idx), l2coef);
  } else {
    cudaMemsetAsync(G_(h, w_idx), 0, cnt * 4, st);
  }
  cudaMemsetAsync(G_(h, b_idx), 0, h->params[b_idx].count * 4, st);
}

struct BwdSide {
  cudaStream_t side;
  cudaEvent_t ev_in;     // recorded on MAIN by the caller: this block's upstream gradients are complete
  cudaEvent_t ev_dz;     // recorded on MAIN here: dz of this block is complete
  cudaEvent_t ev_done;   // recorded on SIDE here: all side work of this block is complete
  cudaEvent_t wait_dz;   // MAIN waits before writing dz      (side work of block l+2 read the same buffer), may be null
  cudaEvent_t wait_dx;   // MAIN waits before writing dx_in   (side work of block l+1 read that buffer), may be null
};

// how block_backward runs one block of a backward pass (the default: alone, on one stream)
struct BlockBwdMode {
  void* dz = nullptr;                // gate-adjoint output (null: h->dz)
  const BwdSide* side = nullptr;     // two-stream schedule: the block's events
  // the weight gradients of conv1, conv_skip and the dilated stack are not launched here; their operands stay in per-block
  // buffers and the problems are appended to h->wg_jobs for the grouped launch (gemm_tc_wgroup.cuh)
  bool grouped = false;
  // the gate adjoint and the dgrad of this block run inside the persistent stack-backward launch (gemm_tc_stack_bwd.cuh):
  // only the weight-gradient problems are collected here
  bool in_stack = false;
  // false: no weight gradient of the block is launched, collected or written; a conditioned block's per-batch sums of d z
  // (which its gated conv's weight gradient would produce) are column sums of their own
  bool param_grads = true;
  int side_group = -1, bucket = 0;   // grouped: side launch (-1: the final launch) and all-reduce bucket of the problems
};

// grouped weight-gradient problem of conv cv: dW = A^T G over its taps (tap k reads A shifted by -(K-1-k)*dil), the bias
// gradient from the column sums of G, the L2 term when the model has one
static TcWgJobDesc wg_job(wn_handle* h, const ConvP& cv, const void* A, int lda, const void* G, int ldg, int group, int bucket) {
  TcWgJobDesc j{};
  j.A = (const bf16*)A; j.lda = lda; j.cin = cv.cin; j.ntaps = cv.K;
  for (int k = 0; k < cv.K; ++k) j.shift[k] = -(cv.K - 1 - k) * cv.dil;
  j.G = (const bf16*)G; j.ldg = ldg; j.N = cv.cout;
  j.dst = G_(h, cv.w_idx); j.w = h->cfg.l2_reg_factor > 0.f ? P_(h, cv.w_idx) : nullptr; j.bias = G_(h, cv.b_idx);
  j.group = group; j.bucket = bucket;
  return j;
}
// the same product as one per-block launch (run_wgrad)
static WgradH wgrad_of(wn_handle* h, const ConvP& cv, const void* A, int lda, const void* G, int ldg, int B, int Tn, float l2coef) {
  WgradH w{};
  w.B = B; w.T = Tn; w.N = cv.cout; w.G = G; w.ldg = ldg; w.nseg = cv.K;
  for (int k = 0; k < cv.K; ++k) w.seg[k] = SegH{A, lda, -(cv.K - 1 - k) * cv.dil, cv.cin};
  w.dst = G_(h, cv.w_idx); w.w = P_(h, cv.w_idx); w.l2coef = l2coef; w.bias_dst = G_(h, cv.b_idx);
  return w;
}

template <class T>
static int block_backward(wn_handle* h, cudaStream_t st, int l, const void* x_in, const void* dxout, int ldxo, const void* dskip, int ldsk,
                          void* dx_in, int ldxi, int B, int Tn, float l2coef, const BlockBwdMode& m) {
  BlockP& b = h->blocks[l];
  void* const dzbuf = m.dz ? m.dz : h->dz;
  const BwdSide* const sd = m.side;
  const bool group = m.grouped, skip_chain = m.in_stack;
  const int depth = (int)b.stack.size();
  const size_t rows_cap = (size_t)h->maxB * h->maxT;
  const long long nR = (long long)B * Tn * h->R;
  const T* g_l = (const T*)h->G_all + (size_t)l * rows_cap * h->D;
  const int R = h->R, D = h->D, S = h->S;
  // bf16 tier: d x_out and d skip live side by side in one (rows, R+S) buffer -> conv1 and conv_skip
  // share one wgrad launch (g is read once) and the dg GEMM reads a single K = R+S segment
  const bool cat = sizeof(T) == 2 && b.has_skip && dxout && dskip && ldxo == ldsk && (const T*)dskip == (const T*)dxout + R;
  // ---- d o  (gradient wrt conv1 output)
  const void* d_o = dxout;
  int ld_o = ldxo;
  // (inside the stack-backward launch the sum d x_out + d skip is never materialised: both DG segments meet the same Wr^T columns,
  // and conv1's weight gradient is two products accumulated by the grouped launch's finish)
  const bool alias_split = h->alias_skip && skip_chain && dxout && dskip;
  if (h->alias_skip && !alias_split) {
    if (dxout && dskip) {
      LaunchScope ls(h, st, CLS_MISC);
      // (grouped weight gradients read d_o at the end of the pass: one buffer per block instead of the shared scratch)
      void* const d_o_buf = group && h->do_all ? (void*)((T*)h->do_all + (size_t)l * rows_cap * R) : h->dotmp;
      add2_kernel<T><<<cdiv(nR, 256), 256, 0, st>>>((const T*)dxout, (const T*)dskip, (T*)d_o_buf, nR);
      d_o = d_o_buf;
      ld_o = R;
    } else if (dskip) {
      d_o = dskip;
      ld_o = ldsk;
    }
  }
  // ---- conv1 / conv_skip weight + bias grads (side stream unless they read the shared d_o scratch)
  const bool side1 = sd != nullptr && d_o != h->dotmp;
  cudaStream_t s1 = side1 ? sd->side : st;
  if (side1) CK(cudaStreamWaitEvent(sd->side, sd->ev_in, 0));
  if (!m.param_grads) {
    // (input gradients only: conv1 / conv_skip contribute their dgrads below, through Wdg)
  } else if (group) {
    if constexpr (sizeof(T) == 2) {
      if (d_o) {
        TcWgJobDesc j = wg_job(h, b.conv1, g_l, D, d_o, ld_o, m.side_group, m.bucket);
        if (alias_split) j.bias_add_G = (const bf16*)dskip;
        h->wg_jobs.push_back(j);
        if (alias_split) {
          TcWgJobDesc j2 = j;
          j2.G = (const bf16*)dskip; j2.ldg = ldsk; j2.w = nullptr; j2.bias = nullptr; j2.bias_add_G = nullptr; j2.acc_prev = true;
          h->wg_jobs.push_back(j2);
        }
      } else {
        unused_conv_grads(h, st, b.conv1.w_idx, b.conv1.b_idx, l2coef);
      }
      if (b.has_skip) {
        if (dskip) {
          h->wg_jobs.push_back(wg_job(h, b.conv_skip, g_l, D, dskip, ldsk, m.side_group, m.bucket));
        } else {
          unused_conv_grads(h, st, b.conv_skip.w_idx, b.conv_skip.b_idx, l2coef);
        }
      }
    }
  } else if (cat) {
    WgradH w{};
    w.B = B; w.T = Tn; w.N = R + S; w.G = dxout; w.ldg = ldxo; w.nseg = 1; w.seg[0] = SegH{g_l, D, 0, D};
    w.dst = G_(h, b.conv1.w_idx); w.w = P_(h, b.conv1.w_idx); w.l2coef = l2coef; w.bias_dst = G_(h, b.conv1.b_idx);
    w.N0 = R; w.dst1 = G_(h, b.conv_skip.w_idx); w.w1 = P_(h, b.conv_skip.w_idx); w.bias1 = G_(h, b.conv_skip.b_idx);
    w.side = side1;
    w.l2_a = TC_L2_FIRST;   // last use of g_l
    RET(run_wgrad<T>(h, s1, CLS_GEMM, w));
  } else if (d_o) {
    WgradH w = wgrad_of(h, b.conv1, g_l, D, d_o, ld_o, B, Tn, l2coef);
    w.side = side1;
    RET(run_wgrad<T>(h, s1, CLS_GEMM, w));
  } else {
    unused_conv_grads(h, st, b.conv1.w_idx, b.conv1.b_idx, l2coef);
  }
  if (m.param_grads && b.has_skip && !cat && !group) {
    if (dskip) {
      WgradH w = wgrad_of(h, b.conv_skip, g_l, D, dskip, ldsk, B, Tn, l2coef);
      w.side = side1;
      RET(run_wgrad<T>(h, s1, CLS_GEMM, w));
    } else {
      unused_conv_grads(h, st, b.conv_skip.w_idx, b.conv_skip.b_idx, l2coef);
    }
  }
  // ---- dz = gate'(z) * (d_o Wr^T + dskip Ws^T)
  if (!skip_chain) {
    GemmH g;
    g.B = B; g.T = Tn; g.N = D; g.nseg = 0;
    int koff = 0;
    const bool use_o = d_o != nullptr;
    const bool use_s = b.has_skip && dskip != nullptr;
    if (!use_o && !use_s) { set_err("block_backward: no upstream gradient"); return WN_ERR_STATE; }
    if (cat) {
      g.seg[g.nseg++] = SegH{dxout, ldxo, 0, R + S};
    } else {
      if (use_o) g.seg[g.nseg++] = SegH{d_o, ld_o, 0, R};
      else koff = R;
      if (use_s) {
        g.seg[g.nseg++] = SegH{dskip, ldsk, 0, S};
      }
    }
    const int rs = R + (b.has_skip ? S : 0);
    g.W32 = b.Wdg ? b.Wdg + (size_t)koff * b.Dpad : nullptr; g.Npad = b.Dpad;
    g.W16 = b.Wdg16 ? b.Wdg16 + koff : nullptr; g.ktot16 = rup(rs, 64); g.N16 = b.Dpad; g.tile16 = 0;
    typename EpiGateBwd<T, sizeof(T) == 2>::Params ep{};
    ep.z = (const T*)h->zbuf[l]; ep.dz = (T*)dzbuf; ep.D = D; ep.vec = vec_ok<T>(D);
    // last use of z; dz is read next by the dgrad and the weight-gradient kernels
    g.l2_in[0] = g.l2_in[1] = TC_L2_FIRST; g.l2_out[0] = g.l2_out[1] = TC_L2_LAST;
    if (sd && sd->wait_dz) CK(cudaStreamWaitEvent(st, sd->wait_dz, 0));
    RET((run_conv_gemm<T, EpiGateBwd<T, sizeof(T) == 2>>(h, st, CLS_GEMM, g, ep)));
    if (sd) CK(cudaEventRecord(sd->ev_dz, st));
  }
  // ---- walk the dilated stack downwards
  const void* dcur = dzbuf;
  int dcw = 2 * D;
  for (int j = depth - 1; j >= 0; --j) {
    const ConvP& c = b.stack[j];
    const void* a_in = j == 0 ? (h->drop_active ? (const void*)h->xdrop[l] : x_in) : h->acts[l][j - 1];
    const int a_w = j == 0 ? R : D;
    // weight grad: rows (k, cin) <- taps of a_in shifted by -(K-1-k)*d ; the bias grad (and the
    // conditioning per-batch sums for the gated conv) are the column sums of the same G
    if (!m.param_grads) {
      // (grouped: d z of every block is kept, and model_backward sums them all in one launch behind the chain)
      if (!group && j == depth - 1 && b.has_cond) run_colsum<T>(h, st, dcur, dcw, B, Tn, c.cout, h->dcb + (size_t)l * h->maxB * 2 * D, 2 * D, nullptr);
    } else if (group) {
      if constexpr (sizeof(T) == 2) {
        TcWgJobDesc jd = wg_job(h, c, a_in, a_w, dcur, dcw, m.side_group, m.bucket);
        if (j == depth - 1 && b.has_cond) { jd.per_batch = h->dcb + (size_t)l * h->maxB * 2 * D; jd.ldpb = 2 * D; }
        h->wg_jobs.push_back(jd);
      }
    } else {
      WgradH w = wgrad_of(h, c, a_in, a_w, dcur, dcw, B, Tn, l2coef);
      if (j == depth - 1 && b.has_cond && !h->cond_seq) { w.per_batch = h->dcb + (size_t)l * h->maxB * 2 * D; w.ldpb = 2 * D; }
      // the gated conv's wgrad reads dz and forward activations only: side stream
      const bool side2 = sd != nullptr && j == depth - 1;
      if (side2) CK(cudaStreamWaitEvent(sd->side, sd->ev_dz, 0));
      w.side = side2;
      w.l2_a = TC_L2_FIRST;   // last use of this forward activation
      RET(run_wgrad<T>(h, side2 ? sd->side : st, CLS_DILATED, w));
    }
    // dgrad
    if (skip_chain && j > 0) {
      // the chain runs inside the stack-backward launch: the gradient wrt the output of conv j - 1 lands in its kept buffer
      dcur = h->dp_keep[l][j - 1];
      dcw = D;
    }
    const bool need = (j > 0 || dx_in != nullptr) && !skip_chain;
    if (need) {
      GemmH g;
      g.B = B; g.T = Tn; g.N = c.cin; g.nseg = c.K;
      for (int k = 0; k < c.K; ++k) g.seg[k] = SegH{dcur, dcw, +(c.K - 1 - k) * c.dil, c.cout};
      fill_w(g, c, true);
      typename EpiActBwd<T, T>::Params ep{};
      ep.N = c.cin;
      if (j > 0) {
        void* dst = group ? h->dp_keep[l][j - 1] : ((dcur == h->dpA) ? h->dpB : h->dpA);
        ep.out = (T*)dst; ep.ldo = D; ep.add = nullptr; ep.y = (const T*)h->acts[l][j - 1]; ep.ldy = D; ep.act = h->cfg.activation;
        ep.vec = vec_ok<T>(D);
        g.l2_in[1] = TC_L2_FIRST; g.l2_out[0] = TC_L2_LAST;
        RET((run_conv_gemm<T, EpiActBwd<T, T>>(h, st, CLS_DILATED, g, ep)));
        dcur = dst;
        dcw = D;
      } else if (h->drop_active) {
        // d(conv branch input) first, then dx = keep/(1-p) * that + residual gradient
        ep.out = (T*)h->ddrop; ep.ldo = R; ep.add = nullptr; ep.y = nullptr; ep.act = ACT_LINEAR; ep.vec = vec_ok<T>(R);
        RET((run_conv_gemm<T, EpiActBwd<T, T>>(h, st, CLS_DILATED, g, ep)));
        if (sd && sd->wait_dx) CK(cudaStreamWaitEvent(st, sd->wait_dx, 0));
        LaunchScope ls(h, st, CLS_MISC);
        dropout_bwd<T><<<cdiv(nR, 256), 256, 0, st>>>((const T*)h->ddrop, h->drop_mask + (size_t)l * rows_cap * R,
                                                     (h->cfg.use_residual && dxout) ? (const T*)dxout : nullptr, ldxo, (T*)dx_in, ldxi,
                                                     (long long)B * Tn, R, 1.0f / (1.0f - h->cfg.dropout));
      } else {
        ep.out = (T*)dx_in; ep.ldo = ldxi;
        ep.add = (h->cfg.use_residual && dxout) ? (const T*)dxout : nullptr; ep.lda = ldxo;
        ep.y = nullptr; ep.act = ACT_LINEAR; ep.vec = vec_ok<T>(R);
        g.l2_in[0] = TC_L2_FIRST; g.l2_out[0] = TC_L2_LAST;   // d x_out is dead after this; dx feeds the next block's kernels
        if (sd && sd->wait_dx) CK(cudaStreamWaitEvent(st, sd->wait_dx, 0));
        RET((run_conv_gemm<T, EpiActBwd<T, T>>(h, st, CLS_DILATED, g, ep)));
      }
    }
  }
  if (sd) CK(cudaEventRecord(sd->ev_done, sd->side));
  return WN_OK;
}

// conditioning adjoint: dWc_l, dbc_l from dcb; dcond = sum_l dcb_l Wc_l^T; then the mapping MLP
// (param_grads == false, whole model only: the dgrads alone, the mapping MLP's result in the buffers of its per-layer chain)
static int cond_backward(wn_handle* h, cudaStream_t st, const float* cond_in, const float* cond, int B, int l0, int nl, bool run_mapping, float* dcond_out,
                         float l2coef, bool skip_wgrad = false, bool param_grads = true) {
  const int n = 2 * h->D;
  if (l0 == 0 && nl == h->L) {
    if (!skip_wgrad && param_grads) {
      LaunchScope ls(h, st, CLS_MISC);
      cond_wgrad_all<<<dim3(cdiv((h->Cc + 1) * n, 128), h->L), 128, 0, st>>>(cond, h->Cc, h->dcb, (long long)h->maxB * n, h->d_params, h->d_grads,
                                                                          h->d_cond_offsets, B, n, l2coef, 0);
    }
    {
      LaunchScope ls(h, st, CLS_MISC);
      cond_dgrad_all<<<B * h->Cc, 256, 0, st>>>(h->dcb, (long long)h->maxB * n, h->d_params, h->d_cond_offsets, dcond_out, h->L, B, h->Cc, n);
    }
  } else
  for (int l = l0; l < l0 + nl; ++l) {
    const BlockP& b = h->blocks[l];
    const float* d = h->dcb + (size_t)l * h->maxB * n;
    {
      LaunchScope ls(h, st, CLS_MISC);
      dense_small_wgrad<<<cdiv((h->Cc + 1) * n, 128), 128, 0, st>>>(cond, h->Cc, d, n, G_(h, b.cw_idx), G_(h, b.cb_idx), B, h->Cc, n);
    }
    if (l2coef != 0.f) {
      LaunchScope ls(h, st, CLS_MISC);
      const long long cnt = h->params[b.cw_idx].count;
      reduce_parts<<<cdiv(cnt, 256), 256, 0, st>>>(G_(h, b.cw_idx), 1, 0, G_(h, b.cw_idx), cnt, P_(h, b.cw_idx), l2coef);
    }
    {
      LaunchScope ls(h, st, CLS_MISC);
      dense_small_dgrad<<<cdiv(B * h->Cc, 4), 128, 0, st>>>(d, n, P_(h, b.cw_idx), dcond_out, h->Cc, B, h->Cc, n, l != l0);
    }
  }
  if (!run_mapping) return WN_OK;
  MapArgs ma;
  if (param_grads && dcond_out == h->dcond && mapping_args(h, cond_in, B, l2coef, &ma)) {
    LaunchScope ls(h, st, CLS_MISC);
    mapping_bwd_fused<<<1, 256, 0, st>>>(ma);
    return WN_OK;
  }
  float* dcur = dcond_out;
  for (int i = (int)h->map_w.size() - 1; i >= 0; --i) {
    const int nn = h->map_width[i];
    const int kin = i > 0 ? h->map_width[i - 1] : h->cfg.cond_in;
    const float* inp = i > 0 ? h->cond_act[i - 1] : cond_in;
    {
      LaunchScope ls(h, st, CLS_MISC);
      dense_small_actgrad<<<cdiv(B * nn, 128), 128, 0, st>>>(dcur, h->cond_act[i], B * nn, h->cfg.mapping_activation);
    }
    if (param_grads) {
      LaunchScope ls(h, st, CLS_MISC);
      dense_small_wgrad<<<cdiv((kin + 1) * nn, 128), 128, 0, st>>>(inp, kin, dcur, nn, G_(h, h->map_w[i]), G_(h, h->map_b[i]), B, kin, nn);
    }
    if (param_grads && l2coef != 0.f) {
      LaunchScope ls(h, st, CLS_MISC);
      const long long cnt = h->params[h->map_w[i]].count;
      reduce_parts<<<cdiv(cnt, 256), 256, 0, st>>>(G_(h, h->map_w[i]), 1, 0, G_(h, h->map_w[i]), cnt, P_(h, h->map_w[i]), l2coef);
    }
    if (i > 0) {
      float* dn = (dcur == h->cond_dact) ? h->cond_dact2 : h->cond_dact;
      LaunchScope ls(h, st, CLS_MISC);
      dense_small_dgrad<<<cdiv(B * kin, 4), 128, 0, st>>>(dcur, nn, P_(h, h->map_w[i]), dn, kin, B, kin, nn, 0);
      dcur = dn;
    }
  }
  return WN_OK;
}

// per-block events of the two-stream backward (see BwdSide); records "upstream gradients ready" on the main stream
static const BwdSide* side_setup(wn_handle* h, cudaStream_t st, int l, bool on, BwdSide* sd) {
  if (!on) return nullptr;
  sd->side = h->side_stream;
  sd->ev_in = h->ev_blk_in[l]; sd->ev_dz = h->ev_blk_dz[l]; sd->ev_done = h->ev_blk_done[l];
  sd->wait_dz = l + 2 < h->L ? h->ev_blk_done[l + 2] : nullptr;
  sd->wait_dx = l + 1 < h->L ? h->ev_blk_done[l + 1] : nullptr;
  cudaEventRecord(sd->ev_in, st);
  return sd;
}

// ============================================================================ backward pass
// The schedule of a backward pass, decided once per pass from the handle and the shape:
//   fp32 tier                          per-block chain on one stream
//   bf16, not grouped                  per-block chain, weight gradients on the side stream (use_side); with a separate skip,
//                                      d x_out and d skip side by side in ping-pong buffers (cat)
//   bf16, grouped (R, D, S multiples   per-block chain, every block's weight gradients in one grouped launch behind it; those of
//   of 256)                            every n-th block in side launches beside the chain (side_pairs)
//   bf16, grouped, stack backward (sb) the chain as one persistent launch, then the grouped launch, bucket by bucket (nb) when the
//                                      step all-reduces its gradients
// Without parameter gradients (wn_backward_ex with param_grads == 0) the same chain runs on the same buffers, alone: no weight-
// gradient launch of any kind, no side stream, no side launches (the persistent chain kernels keep their full grids).
struct BwdSchedule {
  bool param_grads = true; // the parameter gradients are computed (false: input gradients only)
  bool group = false;      // grouped weight gradients (gemm_tc_wgroup.cuh)
  bool use_side = false;   // per-block weight gradients on the side stream
  bool cat = false;        // [d x_out | d skip] ping-pong buffers
  bool sb = false;         // stack backward (gemm_tc_stack_bwd.cuh)
  int side_pairs = 0;      // CTA pairs the chain leaves to the side launches (0: none)
  int nb = 1;              // all-reduce buckets of the grouped launch
  TcWgGroupPlan* wplan = nullptr;   // grouped plan of this shape, once built
  bool side_now = false;   // the side launches run in this pass
  // side launch that takes the weight gradients of block l (-1: the final grouped launch)
  int side_group(const wn_handle* h, int l) const {
    return (side_pairs > 0 && (h->L - 1 - l) % h->wg_side_every == 0) ? (h->L - 1 - l) / h->wg_side_every : -1;
  }
  // two buckets: the first (last blocks, reduced beside the second bucket's kernels) takes ar_first_pct of the blocks — what stays
  // exposed behind the pass is the second bucket's slice, so it is the smaller one; more buckets: equal groups
  int bucket(const wn_handle* h, int l) const {
    if (nb <= 1) return 0;
    if (nb == 2) return (h->L - 1 - l) * 100 < h->L * h->ar_first_pct ? 0 : 1;
    return ((h->L - 1 - l) * nb) / h->L;
  }
};

template <class T>
static BwdSchedule bwd_schedule(wn_handle* h, int B, int Tn, bool param_grads) {
  BwdSchedule s;
  s.param_grads = param_grads;
  // (bf16 tier only: the fp32 tier's wgrad / column-sum scratch buffers are not duplicated for a second stream)
  if constexpr (sizeof(T) == 2) {
    s.group = h->use_group_wgrad != 0;
    s.use_side = param_grads && h->prof_tag == 0 && h->side_stream != nullptr && !s.group;
    s.cat = h->dcatA != nullptr;
    // Backward chain as ONE persistent launch (gemm_tc_stack_bwd.cuh): D = R = 256, d z / d x_out
    // of every block kept (grouped weight gradients), more 256-row tiles per layer than CTA pairs.  It takes every SM for the
    // whole chain, so the weight gradients all run in the one grouped launch behind it (no side launches).
    s.sb = s.group && !s.cat && h->use_stack_bwd && h->L >= 2 && h->D == h->R && h->D == 256 &&
           h->K <= TC_MAX_TAPS && more_tiles_than_pairs(B, Tn);
    for (auto& b : h->blocks) {
      if (!s.sb) break;
      // multi-dilation blocks (plain conv layers of the launch): all convs 256 wide
      s.sb = b.stack[0].cin % 64 == 0 && (!b.has_skip || h->S % 64 == 0) && b.stack.size() <= 16 &&
             (b.stack.size() == 1 || (h->D == 256 && h->dp_keep.size() == (size_t)h->L));
      for (size_t j = 0; s.sb && j + 1 < b.stack.size(); ++j) s.sb = b.stack[j].cout == h->D && b.stack[j].Wb16 != nullptr && b.stack[j].K == h->K;
    }
  }
  // Side launches: the persistent chain kernels need ceil(tiles / pairs) rounds; the same rounds fit on fewer CTA pairs
  // (256 tiles: 4 rounds on 74 or on 64 pairs), and the pairs left over run the weight gradients of every n-th block
  // beside the chain.  The plan (unit ranges per side group) exists from the second call on; the first call launches
  // every group at the end.
  if (param_grads && s.group && !s.sb && h->side_stream != nullptr && h->wg_side_every > 0 && more_tiles_than_pairs(B, Tn)) {
    const int pairs = tc_num_sms() / 2, tiles = B * cdiv(Tn, 256), rounds = cdiv(tiles, pairs);
    s.side_pairs = pairs - cdiv(tiles, rounds);
    if (s.side_pairs < 6) s.side_pairs = 0;
  }
  // bucketed all-reduce: only with the stack-backward launch (every SM busy until the chain ends, all filter gradients in the
  // final grouped launch) and a communicator that reduces inside this step
  s.nb = (param_grads && s.group && s.sb && h->ar_now && h->prof_tag == 0 && h->comm_stream != nullptr) ? std::min(std::min(h->ar_buckets, h->L), 8) : 1;
  if (s.group) for (auto& wp : h->wg_plans) if (wp.B == B && wp.T == Tn && wp.drop == h->drop_active && wp.sb == s.sb && wp.nb == s.nb) s.wplan = &wp.plan;
  s.side_now = s.wplan != nullptr && s.side_pairs > 0 && h->prof_tag == 0 && !s.wplan->side.empty();
  return s;
}

// grouped weight gradients keep d z and d x_out of every block: block l's slab of dz_all / dx_all
template <class T>
static void* dz_slab(wn_handle* h, int l) { return (T*)h->dz_all + (size_t)l * h->maxB * h->maxT * 2 * h->D; }
template <class T>
static void* dx_slab(wn_handle* h, int l) { return (T*)h->dx_all + (size_t)l * h->maxB * h->maxT * h->R; }

// ---- head, last conv first: its input gradient lands where the chain reads d x_out or d skip
template <class T>
static int head_backward(wn_handle* h, cudaStream_t st, const BwdSchedule& s, int B, int Tn, float l2coef) {
  const wn_config& c = h->cfg;
  const void* dcur = h->dlogits;
  int dw = h->ldd;
  for (int i = (int)h->head.size() - 1; i >= 0; --i) {
    OuterLabel ol_head(h, "head_bwd");
    const ConvP& hc = h->head[i];
    const void* a_in;
    int a_w;
    if (i > 0) { a_in = h->hact[i - 1]; a_w = h->head[i - 1].cout; }
    else if (c.use_skip) { a_in = h->skipsum; a_w = h->Sp; }
    else { a_in = h->xout[h->L - 1]; a_w = h->R; }
    // (the head's d-activation buffers dlogits / dhA / dhB stay intact until the end of the pass when the head has <= 3 convs)
    bool head_grouped = false;
    if constexpr (sizeof(T) == 2) {
      if (s.param_grads && s.group && h->head.size() <= 3 && tc_wgrad_group_ok(hc.cin, hc.cout) && a_w == hc.cin) {
        h->wg_jobs.push_back(wg_job(h, hc, a_in, a_w, dcur, dw, -1, s.nb - 1));      // (the head's gradients travel with the last bucket)
        head_grouped = true;
      }
    }
    if (s.param_grads && !head_grouped) RET(run_wgrad<T>(h, st, CLS_GEMM, wgrad_of(h, hc, a_in, a_w, dcur, dw, B, Tn, l2coef)));
    GemmH g;
    g.B = B; g.T = Tn; g.N = hc.cin; g.nseg = 1;
    g.seg[0] = SegH{dcur, dw, 0, (sizeof(T) == 2 && i + 1 == (int)h->head.size()) ? h->ldd : hc.cout};
    fill_w(g, hc, true);
    typename EpiActBwd<T, T>::Params ep{};
    ep.N = hc.cin; ep.add = nullptr;
    void* dst;
    if (i > 0) {
      dst = (dcur == h->dhA) ? h->dhB : h->dhA;
      ep.out = (T*)dst; ep.ldo = hc.cin; ep.y = (const T*)h->hact[i - 1]; ep.ldy = hc.cin; ep.act = c.activation; ep.vec = vec_ok<T>(hc.cin);
    } else if (s.cat) {
      const int ldc = h->R + h->S;
      dst = (T*)h->dcatA + h->R;
      ep.out = (T*)dst; ep.ldo = ldc; ep.y = nullptr; ep.act = ACT_LINEAR; ep.vec = vec_ok<T>(ldc);
    } else {
      dst = c.use_skip ? h->dskip : (s.group ? dx_slab<T>(h, h->L - 1) : h->dxA);
      ep.out = (T*)dst; ep.ldo = hc.cin; ep.y = nullptr; ep.act = ACT_LINEAR; ep.vec = vec_ok<T>(hc.cin);
    }
    RET((run_conv_gemm<T, EpiActBwd<T, T>>(h, st, CLS_GEMM, g, ep)));
    dcur = dst;
    dw = hc.cin;
  }
  return WN_OK;
}

// ---- per-block chain on [d x_out | d skip] ping-pong buffers (row width R + S); *dxout: d x_out of block 0
template <class T>
static int cat_chain(wn_handle* h, cudaStream_t st, const BwdSchedule& s, int B, int Tn, float l2coef, const void** dxout) {
  const int ldc = h->R + h->S;
  // d skip is the same for every block (model.py:236): keep a copy beside each d x_out ping-pong buffer
  CK(cudaMemcpy2DAsync((T*)h->dcatB + h->R, (size_t)ldc * sizeof(T), (const T*)h->dcatA + h->R, (size_t)ldc * sizeof(T), (size_t)h->S * sizeof(T),
                       (size_t)B * Tn, cudaMemcpyDeviceToDevice, st));
  const void* cur = nullptr;          // buffer holding d x_out of the block being processed
  void* nxt = h->dcatB;
  for (int l = h->L - 1; l >= 0; --l) {
    const void* x_in = l > 0 ? h->xout[l - 1] : h->h0;
    const void* dsk = cur ? (const void*)((const T*)cur + h->R) : (const void*)((const T*)h->dcatA + h->R);
    BwdSide sd;
    BlockBwdMode m;
    m.side = side_setup(h, st, l, s.use_side, &sd);
    m.dz = (l & 1) ? h->dz2 : h->dz;
    m.param_grads = s.param_grads;
    RET(block_backward<T>(h, st, l, x_in, cur, ldc, dsk, ldc, nxt, ldc, B, Tn, l2coef, m));
    cur = nxt;
    nxt = (nxt == h->dcatB) ? h->dcatA : h->dcatB;
  }
  *dxout = cur;
  return WN_OK;
}

// ---- gate adjoint and dgrads of every block as one persistent launch; *stacked: it ran (else the per-block chain runs them)
static int stack_backward(wn_handle* h, cudaStream_t st, int B, int Tn, const void* dxout, const void* dskip, bool* stacked) {
  const wn_config& c = h->cfg;
  const size_t rows_cap = (size_t)h->maxB * h->maxT;
  // one desc per CONV in forward order: the plain convs of block l, then its gated conv
  std::vector<TcStackBwdDesc> bdescs;
  int conv_index = 0;
  for (int l = 0; l < h->L; ++l) {
    BlockP& b = h->blocks[l];
    const int depth = (int)b.stack.size();
    const bf16* blk_dxo = l == h->L - 1 ? (const bf16*)dxout : (const bf16*)dx_slab<bf16>(h, l);      // d x_out of this block (or null)
    bf16* blk_dx = (bf16*)(l > 0 ? dx_slab<bf16>(h, l - 1) : h->dxA);                                   // gradient wrt the block input
    const int next_first = conv_index + depth;      // desc that writes blk_dxo (first conv of block l + 1), if any
    const bool dxo_in_launch = blk_dxo != nullptr && l < h->L - 1;
    for (int j = 0; j < depth; ++j, ++conv_index) {
      const ConvP& cv = b.stack[j];
      TcStackBwdDesc d{};
      const bool alias = h->alias_skip && dskip != nullptr;      // skip = conv1's output: d skip joins d x_out in front of Wr^T
      d.B = B; d.T = Tn; d.nseg = cv.K; d.D = h->D; d.R = h->R; d.S = dskip ? (alias ? h->R : h->S) : 0;
      for (int k = 0; k < cv.K; ++k) d.shift[k] = (cv.K - 1 - k) * cv.dil;
      d.Wb = cv.Wb16; d.k_b = rup(cv.Kb16, 64);
      d.drop_scale = h->drop_active ? 1.0f / (1.0f - c.dropout) : 0.f;
      d.ein_layer = -1;
      // what this conv's tile writes: the gradient wrt its input
      d.dx = j == 0 ? blk_dx : (bf16*)h->dp_keep[l][j - 1];
      if (j == 0) {
        // first conv of the block: the block input is not activated; the residual gradient joins here
        if (c.use_residual && blk_dxo) { d.out_mode = 1; d.ein = blk_dxo; d.ein_layer = dxo_in_launch ? next_first : -1; }
        if (h->drop_active) d.mask = h->drop_mask + (size_t)l * rows_cap * h->R;
      } else {
        d.out_mode = 2; d.act = c.activation; d.ein = (const bf16*)h->acts[l][j - 1];
      }
      if (j < depth - 1) {
        d.plain = 1; d.gin = (const bf16*)h->dp_keep[l][j];
      } else {
        d.dxo = blk_dxo;
        d.dskip = ((b.has_skip || alias) && dskip) ? (const bf16*)dskip : nullptr; d.lds = h->Sp;
        d.alias = alias ? 1 : 0;
        d.z = (const bf16*)h->zbuf[l]; d.dz = (bf16*)dz_slab<bf16>(h, l);
        const int rs = h->R + (b.has_skip ? h->S : 0), koff = (d.dxo || alias) ? 0 : h->R;
        d.Wdg = b.Wdg16 + koff; d.k_dg = rup(rs, 64);
        d.has_res = (c.use_residual && depth == 1) ? 1 : 0;
      }
      bdescs.push_back(d);
    }
  }
  TcStackBwdPlan* sp = nullptr;
  RET(plan_for(h, st, h->stack_bwd_plans, [&](const TcStackBwdPlan& q) { return q.B == B && q.T == Tn && q.drop == h->drop_active; },
               "stack backward", [&](TcStackBwdPlan& p) { return tc_stack_bwd_build(h->tmaps, bdescs, &p); }, &sp));
  if (!sp) return WN_OK;
  RET(launch_persistent(h, st, "stack_bwd", "stack backward", [&] { return tc_stack_bwd_launch(st, *sp, bdescs[0]); }, stacked));
  if (*stacked) h->stack_bwd_layers = h->L;
  return WN_OK;
}

// ---- per-block chain, behind the stack-backward launch when it ran (the blocks then only collect their weight-gradient
// problems); with side launches, a side group's weight gradients start as soon as its block is done.  *dxout: d x_out of block 0
template <class T>
static int block_chain(wn_handle* h, cudaStream_t st, const BwdSchedule& s, int B, int Tn, float l2coef, const void** dxout_out) {
  const wn_config& c = h->cfg;
  const void* dskip = c.use_skip ? h->dskip : nullptr;
  const void* dxout = c.use_skip ? nullptr : (s.group ? dx_slab<T>(h, h->L - 1) : h->dxA);
  bool stacked = false;
  if constexpr (sizeof(T) == 2) {
    if (s.sb) RET(stack_backward(h, st, B, Tn, dxout, dskip, &stacked));
  }
  for (int l = h->L - 1; l >= 0; --l) {
    const void* x_in = l > 0 ? h->xout[l - 1] : h->h0;
    // grouped weight gradients: d x_out and d z of every block keep their own buffers until the grouped launch
    void* dx_in = s.group ? (l > 0 ? dx_slab<T>(h, l - 1) : h->dxA) : ((dxout == h->dxA) ? h->dxB : h->dxA);
    BwdSide sd;
    BlockBwdMode m;
    m.side = side_setup(h, st, l, s.use_side, &sd);
    m.dz = s.group ? dz_slab<T>(h, l) : ((l & 1) ? h->dz2 : h->dz);
    m.grouped = s.group; m.in_stack = stacked; m.param_grads = s.param_grads;
    m.side_group = s.side_group(h, l); m.bucket = s.bucket(h, l);
    RET(block_backward<T>(h, st, l, x_in, dxout, h->R, dskip, h->Sp, dx_in, h->R, B, Tn, l2coef, m));
    if constexpr (sizeof(T) == 2) {
      const int g = m.side_group;
      if (s.side_now && g >= 0 && g < (int)s.wplan->side.size() && s.wplan->side[g].second > 0) {
        // d z_l and d x_out_l are complete behind this block's kernels: its weight gradients start on the side stream
        CK(cudaEventRecord(h->ev_blk_dz[l], st));
        CK(cudaStreamWaitEvent(h->side_stream, h->ev_blk_dz[l], 0));
        LaunchLabel lab(h, "wgrad_group");
        LaunchScope ls(h, h->side_stream, CLS_DILATED);
        int r = tc_wgrad_group_launch(h->side_stream, *s.wplan, s.wplan->side[g].first, s.wplan->side[g].second);
        if (r != 0) { set_err("grouped wgrad side launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
        h->wg_last_side++;
      }
    }
    dxout = dx_in;
  }
  *dxout_out = dxout;
  return WN_OK;
}

// ---- input conv (model.py:84-88): dW[k][c], db[c].  HBM-bound, small CTAs
template <class T>
static void input_conv_backward(wn_handle* h, cudaStream_t s_, const float* x, int ldx, const void* dxout, int ld_dx, int B, int Tn, float l2coef) {
  OuterLabel ol(h, "input_conv_bwd");
  const bool wide = h->R % 2 == 0 && h->R / 2 <= 256 && ld_dx % 2 == 0;
  const int chunks = cdiv(Tn, 64);
  const int nparts = wide ? cdiv((long long)B * Tn, ICB_ROWS) : B * chunks;
  {
    LaunchScope ls(h, s_, CLS_MISC);
    if (wide)
      input_conv_bwd_stage1_wide<T><<<nparts, 256, 0, s_>>>(x, ldx, (const T*)dxout, ld_dx, h->colpart, B, Tn, h->R, h->K);
    else
      input_conv_bwd_stage1<T><<<dim3(cdiv(h->R, 64), chunks, B), 64, 0, s_>>>(x, ldx, (const T*)dxout, ld_dx, h->colpart, B, Tn, h->R, h->K, 64);
  }
  const long long kr = (long long)h->K * h->R;
  {
    LaunchScope ls(h, s_, CLS_MISC);
    reduce_parts_tall<<<cdiv(kr, 32), 256, 0, s_>>>(h->colpart, nparts, (long long)(h->K + 1) * h->R, G_(h, h->input_conv.w_idx), kr,
                                                 l2coef != 0.f ? P_(h, h->input_conv.w_idx) : nullptr, l2coef);
  }
  {
    LaunchScope ls(h, s_, CLS_MISC);
    reduce_parts_tall<<<cdiv(h->R, 32), 256, 0, s_>>>(h->colpart + kr, nparts, (long long)(h->K + 1) * h->R, G_(h, h->input_conv.b_idx), h->R, nullptr, 0.f);
  }
}

// ---- input conv dgrad: dx (B,T) fp32 = d loss / d x from the final d h0 (row stride ld_dx: R, or R + S in the cat layout)
template <class T>
static void input_conv_dgrad_run(wn_handle* h, cudaStream_t st, const void* dh0, int ld_dx, float* dx, int B, int Tn) {
  OuterLabel ol(h, "input_dgrad");
  LaunchScope ls(h, st, CLS_MISC);
  constexpr int V = 16 / sizeof(T);
  const bool vec = (h->R * sizeof(T)) % 16 == 0 && (ld_dx * sizeof(T)) % 16 == 0 && ((uintptr_t)dh0 & 15) == 0;
  const dim3 grid(cdiv(Tn, ICD_ROWS), B);
  if (vec)
    input_conv_dgrad<T, V><<<grid, 256, 0, st>>>((const T*)dh0, ld_dx, P_(h, h->input_conv.w_idx), dx, Tn, h->R, h->K);
  else
    input_conv_dgrad<T, 1><<<grid, 256, 0, st>>>((const T*)dh0, ld_dx, P_(h, h->input_conv.w_idx), dx, Tn, h->R, h->K);
}

// ---- every block's conv1 / conv_skip / gated-conv weight gradients in ONE launch (+ one finish), or bucket by bucket with the
// early all-reduce; *cond_done: the bucket launches also wrote the conditioning filter gradients
static int grouped_wgrad(wn_handle* h, cudaStream_t st, const BwdSchedule& s, int B, int Tn, float l2coef, bool* cond_done) {
  const TcWgGroupPlan* plan = s.wplan;
  if (!plan) {
    wn_handle::WgPlan* wp = nullptr;
    RET(new_plan(h, st, h->wg_plans, wn_handle::WgPlan{B, Tn, h->drop_active, s.sb, s.nb, TcWgGroupPlan{}}, "grouped wgrad", [&](wn_handle::WgPlan& p) {
      return tc_wgrad_group_build(h->tmaps, h->wg_jobs, B, Tn, h->wg_force_split, h->wg_pair_tiles != 0, s.side_pairs, &p.plan);
    }, &wp));
    if (!wp) { set_err("grouped wgrad: no plan for (%d, %d) while capturing", B, Tn); return WN_ERR_STATE; }
    plan = &wp->plan;
  }
  LaunchLabel lab(h, "wgrad_group");
  h->wg_last_tiles = plan->ntiles; h->wg_last_partials = plan->npartial;
  if (s.nb > 1 && (int)plan->buckets.size() == s.nb && !s.side_now) {
    // ---- bucket by bucket: launch, finish, (conditioning filter gradients of the bucket's blocks,) all-reduce on comm_stream
    auto block_off = [&](int l) -> long long {
      if (l < h->L) return h->params[h->blocks[l].stack[0].w_idx].offset;
      if (!h->head.empty()) return h->params[h->head[0].w_idx].offset;
      if (!h->map_w.empty()) return h->params[h->map_w[0]].offset;
      return h->n_scalars;
    };
    for (int k = 0; k < s.nb; ++k) {
      const TcWgGroupPlan::Bucket& bk = plan->buckets[k];
      {
        LaunchScope ls(h, st, CLS_DILATED);
        int r = tc_wgrad_group_launch(st, *plan, bk.unit0, bk.nunits);
        if (r != 0) { set_err("grouped wgrad launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
      }
      {
        OuterLabel ol(h, "wgrad_group_finish");
        LaunchScope ls(h, st, CLS_DILATED);
        int r = tc_wgrad_group_finish_launch(st, *plan, l2coef, k);
        if (r != 0) { set_err("grouped wgrad finish failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
      }
      // blocks of this bucket: l_hi .. l_lo (descending walk: bucket 0 holds the last blocks)
      int l_lo = h->L, l_hi = -1;
      for (int l = 0; l < h->L; ++l) if (s.bucket(h, l) == k) { if (l < l_lo) l_lo = l; if (l > l_hi) l_hi = l; }
      if (h->cfg.conditioning && l_hi >= l_lo) {
        OuterLabel ol(h, "cond_bwd");
        LaunchScope ls(h, st, CLS_MISC);
        const int n = 2 * h->D;
        cond_wgrad_all<<<dim3(cdiv((h->Cc + 1) * n, 128), l_hi - l_lo + 1), 128, 0, st>>>(h->last_cond, h->Cc, h->dcb, (long long)h->maxB * n, h->d_params,
                                                                                     h->d_grads, h->d_cond_offsets, B, n, l2coef, l_lo);
      }
      if (k + 1 < s.nb && l_hi >= l_lo) {
        // every gradient of blocks l_lo .. l_hi is final: reduce that slice of the flat buffer beside the next bucket's kernels
        const long long lo = block_off(l_lo), hi = block_off(l_hi + 1);
        CK(cudaEventRecord(h->ev_bucket[k], st));
        CK(cudaStreamWaitEvent(h->comm_stream, h->ev_bucket[k], 0));
        h->launches++;
        const int r = g_nccl.AllReduce(h->d_grads + lo, h->d_grads + lo, (size_t)(hi - lo), WN_NCCL_FLOAT32, WN_NCCL_SUM, h->comm, h->comm_stream);
        if (r != 0) { set_err("ncclAllReduce (bucket %d) failed (%d): %s", k, r, nccl_errstr(r)); return WN_ERR_CUDA; }
        h->last_ar_buckets++;
        if (h->ar_early_lo < 0 || lo < h->ar_early_lo) h->ar_early_lo = lo;
        if (hi > h->ar_early_hi) h->ar_early_hi = hi;
      }
    }
    *cond_done = h->cfg.conditioning != 0;
    return WN_OK;
  }
  {
    LaunchScope ls(h, st, CLS_DILATED);
    // without side launches (first call of a shape, profiling passes, WN_TC_GROUP_SIDE_EVERY=0) the side groups' units, which
    // follow the final group's in the table, run in the same launch
    int r = tc_wgrad_group_launch(st, *plan, 0, s.side_now ? plan->final_units : plan->nunits);
    if (r != 0) { set_err("grouped wgrad launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
  }
  if (s.side_now) {
    // the side launches of this pass must be complete before the finish reads their partial tiles
    CK(cudaEventRecord(h->ev_wg_side, h->side_stream));
    CK(cudaStreamWaitEvent(st, h->ev_wg_side, 0));
  }
  OuterLabel ol(h, "wgrad_group_finish");
  LaunchScope ls(h, st, CLS_DILATED);
  int r = tc_wgrad_group_finish_launch(st, *plan, l2coef);
  if (r != 0) { set_err("grouped wgrad finish failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
  return WN_OK;
}

// dx (or null): d loss / d x of the input signal.  param_grads == false: no parameter gradient is computed or written
template <class T>
static int model_backward(wn_handle* h, cudaStream_t st, const float* x, int ldx, const float* cond_in, int B, int Tn, float l2coef,
                          float* dx = nullptr, bool param_grads = true) {
  const BwdSchedule s = bwd_schedule<T>(h, B, Tn, param_grads);
  h->wg_jobs.clear();
  h->wg_last_tiles = 0; h->wg_last_side = 0;
  h->stack_bwd_layers = 0;
  h->ar_early_lo = h->ar_early_hi = -1;
  h->last_ar_buckets = 0;
  const void* dxout;
  {
    // with side launches, the persistent kernels of the head and the chain leave CTA pairs free for them
    TcBalanceScope balance(s.side_now);
    RET(head_backward<T>(h, st, s, B, Tn, l2coef));
    if (s.cat) RET(cat_chain<T>(h, st, s, B, Tn, l2coef, &dxout));
    else RET(block_chain<T>(h, st, s, B, Tn, l2coef, &dxout));
  }
  const int ld_dx = s.cat ? h->R + h->S : h->R;
  if (dx) input_conv_dgrad_run<T>(h, st, dxout, ld_dx, dx, B, Tn);
  if (!s.param_grads) {
    if (!h->cfg.conditioning) return WN_OK;
    OuterLabel ol(h, "cond_bwd");
    if (s.group) {
      // the per-batch sums of every block's kept d z (the per-block chain took them block by block)
      const int n = 2 * h->D;
      LaunchScope ls(h, st, CLS_MISC);
      colsum_per_batch_slabs<T><<<dim3(cdiv(n, 64), B, h->L), 256, 0, st>>>((const T*)h->dz_all, (long long)h->maxB * h->maxT * n, n, Tn, n, h->dcb,
                                                                          (long long)h->maxB * n, n);
    }
    // d cond from the per-batch sums, through the mapping MLP's dgrads
    return cond_backward(h, st, cond_in, h->last_cond, B, 0, h->L, true, h->dcond, 0.f, false, false);
  }
  // The input conv's gradients run on the side stream beside the final grouped weight-gradient launch (their CTAs fit next to
  // the tensor kernel's on the same SMs) with side launches, and behind the stack-backward launch: d h0 is final there too.
  const bool grouped = s.group && !h->wg_jobs.empty();
  const bool icb_side = !s.side_now && h->stack_bwd_layers > 0 && h->side_stream != nullptr && h->prof_tag == 0 && grouped;
  if (s.side_now || icb_side) {
    CK(cudaEventRecord(h->ev_blk_in[0], st));
    CK(cudaStreamWaitEvent(h->side_stream, h->ev_blk_in[0], 0));
    input_conv_backward<T>(h, h->side_stream, x, ldx, dxout, ld_dx, B, Tn, l2coef);
    if (!grouped) { CK(cudaEventRecord(h->ev_wg_side, h->side_stream)); CK(cudaStreamWaitEvent(st, h->ev_wg_side, 0)); }
  }
  bool cond_wgrad_done = false;
  if constexpr (sizeof(T) == 2) {
    if (grouped) RET(grouped_wgrad(h, st, s, B, Tn, l2coef, &cond_wgrad_done));
  }
  if (icb_side) {
    // join: the input conv's gradients are part of what the all-reduce behind this pass (and the caller) reads
    CK(cudaEventRecord(h->ev_wg_side, h->side_stream));
    CK(cudaStreamWaitEvent(st, h->ev_wg_side, 0));
  }
  // join: every side-stream wgrad (and its finish kernel) is complete before anything below reads the gradients
  if (s.use_side) CK(cudaStreamWaitEvent(st, h->ev_blk_done[0], 0));
  if (!s.side_now && !icb_side) input_conv_backward<T>(h, st, x, ldx, dxout, ld_dx, B, Tn, l2coef);
  if (h->cfg.conditioning) { OuterLabel ol(h, "cond_bwd"); RET(cond_backward(h, st, cond_in, h->last_cond, B, 0, h->L, true, h->dcond, l2coef, cond_wgrad_done)); }
  return WN_OK;
}

// ============================================================================ public entry points
static int check_bt(wn_handle* h, int B, int T) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (B < 1 || T < 1 || B > h->maxB || T > h->maxT) {
    set_err("batch/time (%d,%d) outside the workspace built for (%d,%d)", B, T, h->maxB, h->maxT);
    return WN_ERR_VALUE;
  }
  return WN_OK;
}

// ============================================================================ generation (model.py:241-307; layers.py:226-290)
static int gen_alloc(wn_handle* h, int B, int cap) {
  wn_handle::Gen& G = h->gen;
  if (G.B >= B && G.cap >= cap) return WN_OK;
  for (void* a : G.allocs) cudaFree(a);
  G.allocs.clear();
  auto take = [&](size_t bytes) -> void* { void* p = nullptr; if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr; cudaMemset(p, 0, bytes); G.allocs.push_back(p); return p; };
  G.B = B; G.cap = cap;
  const size_t rows = (size_t)B * cap;
  G.audio = (float*)take(rows * 4);
  G.hist.assign(h->L + 1, {});
  bool ok = G.audio != nullptr;
  for (int l = 0; l <= h->L && ok; ++l) {
    const int depth = l < h->L ? (int)h->blocks[l].stack.size() : 1;
    G.hist[l].assign(depth, nullptr);
    for (int j = 0; j < depth && ok; ++j) { G.hist[l][j] = (float*)take(rows * (j == 0 ? h->R : h->D) * 4); ok = G.hist[l][j] != nullptr; }
  }
  G.z = (float*)take((size_t)B * 2 * h->D * 4);
  G.skipsum = (float*)take((size_t)B * h->Sp * 4);
  G.hbuf.assign(h->head.size(), nullptr);
  for (size_t i = 0; i + 1 < h->head.size() && ok; ++i) { G.hbuf[i] = (float*)take((size_t)B * h->head[i].cout * 4); ok = G.hbuf[i] != nullptr; }
  G.logits = (float*)take((size_t)B * h->Cout * 4);
  G.sampled = (float*)take((size_t)B * 4);
  G.t_dev = (int*)take(16);
  G.wcat.assign(h->L, nullptr); G.bcat.assign(h->L, nullptr);
  for (int l = 0; l < h->L && ok; ++l) {
    if (!(h->cfg.use_skip && h->blocks[l].has_skip)) continue;
    G.wcat[l] = (float*)take((size_t)h->D * (h->R + h->S) * 4);
    G.bcat[l] = (float*)take((size_t)(h->R + h->S) * 4);
    ok = G.wcat[l] && G.bcat[l];
  }
  if (!ok || !G.z || !G.skipsum || !G.logits || !G.sampled || !G.t_dev) { set_err("generation workspace allocation failed"); G.B = G.cap = 0; return WN_ERR_CUDA; }
  return WN_OK;
}

static void gen_dense(cudaStream_t st, const GenVec& v, int B, const int* t_dev) {
  const size_t smem = (size_t)GEN_ROWS * v.K * v.Cin * 4;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) { cudaFuncSetAttribute(gen_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024); }
  gen_dense_kernel<<<dim3(cdiv(v.N, 32), cdiv(B, GEN_ROWS)), 256, smem, st>>>(v, B, t_dev);
}

// one time step of the whole network on the histories; t is read from device memory
static int gen_step(wn_handle* h, cudaStream_t st, int B, bool has_cb, bool sample, int deterministic, uint64_t seed, float* pred, long long pred_bstride,
                    int t0, bool write_audio) {
  wn_handle::Gen& G = h->gen;
  const int cap = G.cap, R = h->R, D = h->D;
  const int* t = G.t_dev;
  if (h->cfg.use_skip) gen_zero_kernel<<<cdiv(B * h->Sp, 256), 256, 0, st>>>(G.skipsum, B * h->Sp);
  gen_input_conv_kernel<<<cdiv(B * R, 128), 128, 0, st>>>(G.audio, cap, P_(h, h->input_conv.w_idx), P_(h, h->input_conv.b_idx), G.hist[0][0], R, h->K, B, t);
  for (int l = 0; l < h->L; ++l) {
    const BlockP& b = h->blocks[l];
    const int depth = (int)b.stack.size();
    for (int j = 0; j < depth; ++j) {
      const ConvP& c = b.stack[j];
      GenVec v{};
      v.in = G.hist[l][j]; v.in_bstride = (long long)cap * c.cin; v.in_tstride = c.cin; v.Cin = c.cin; v.K = c.K; v.dil = c.dil;
      v.W = P_(h, c.w_idx); v.bias = P_(h, c.b_idx); v.N = c.cout;
      if (j < depth - 1) {
        v.act = h->cfg.activation;
        v.out = G.hist[l][j + 1]; v.out_bstride = (long long)cap * D; v.out_tstride = D;
      } else {
        v.act = ACT_LINEAR;
        if (has_cb) { v.cbias = h->cb + (size_t)l * h->maxB * 2 * D; v.ldcb = 2 * D; }
        v.out = G.z; v.out_bstride = 2 * D; v.out_tstride = 0;
      }
      gen_dense(st, v, B, t);
    }
    {
      GenVec v{};   // conv1 (+ residual) [| conv_skip -> running skip sum, model.py:236] on the gate of z
      v.in = G.z; v.in_bstride = 2 * D; v.in_tstride = 0; v.Cin = D; v.K = 1; v.dil = 1; v.in_gate = 1;
      v.act = ACT_LINEAR;
      v.out = G.hist[l + 1][0]; v.out_bstride = (long long)cap * R; v.out_tstride = R;
      if (h->cfg.use_residual) { v.res = G.hist[l][0]; v.res_bstride = (long long)cap * R; v.res_tstride = R; v.res_cols = R; }
      if (G.wcat[l]) {
        v.W = G.wcat[l]; v.bias = G.bcat[l]; v.N = R + h->S;
        v.acc = G.skipsum; v.acc_ld = h->Sp; v.acc_col0 = R;
      } else {
        v.W = P_(h, b.conv1.w_idx); v.bias = P_(h, b.conv1.b_idx); v.N = R;
        if (h->cfg.use_skip && h->alias_skip) { v.acc = G.skipsum; v.acc_ld = h->Sp; v.acc_col0 = -1; }
      }
      gen_dense(st, v, B, t);
    }
  }
  // head (model.py:105-119,237-238)
  const float* hin = h->cfg.use_skip ? G.skipsum : G.hist[h->L][0];
  long long hin_b = h->cfg.use_skip ? h->Sp : (long long)cap * R;
  int hin_t = h->cfg.use_skip ? 0 : R;
  for (size_t i = 0; i < h->head.size(); ++i) {
    const ConvP& hc = h->head[i];
    const bool last = i + 1 == h->head.size();
    GenVec v{};
    v.in = hin; v.in_bstride = hin_b; v.in_tstride = hin_t; v.Cin = hc.cin; v.K = 1; v.dil = 1;
    v.W = P_(h, hc.w_idx); v.bias = P_(h, hc.b_idx); v.N = hc.cout; v.act = last ? ACT_LINEAR : h->cfg.activation;
    v.out = last ? G.logits : G.hbuf[i]; v.out_bstride = hc.cout; v.out_tstride = 0;
    gen_dense(st, v, B, t);
    hin = v.out; hin_b = hc.cout; hin_t = 0;
  }
  const wn_config& c = h->cfg;
  if (pred) gen_pred_kernel<<<B, 256, 0, st>>>(G.logits, h->Cout, c.sampling_function == WN_CATEGORICAL ? 1 : 0, pred, pred_bstride, t0, t);
  if (sample) {
    const int kind = c.sampling_function == WN_CATEGORICAL ? 0 : (c.sampling_function == WN_GAUSSIAN ? 2 : 1);
    sample_kernel<<<cdiv(B, 8), 256, 0, st>>>(G.logits, h->Cout, h->Cout, c.num_mixtures, kind, 1, c.bits, deterministic, seed, nullptr, 1, B, G.sampled, nullptr, t);
  }
  gen_advance_kernel<<<1, 64, 0, st>>>(G.audio, cap, G.sampled, B, write_audio ? 1 : 0, G.t_dev);
  CK(cudaGetLastError());
  return WN_OK;
}

// prime (B, n_prime) -> out (B, length): out[b][i] = sample n_prime + i.  teacher (B, length) or NULL: forced continuation (the
// predictions, not the samples, are then the result: pred (B, length, Cout)).
extern "C" int wn_generate(wn_handle* h, const float* prime_dev, int n_prime, const float* cond_dev, int B, int length, int deterministic, uint64_t seed,
                           float* out_dev, float* pred_dev, const float* teacher_dev, void* stream) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (!h->cfg.has_head || !h->cfg.has_input_conv) { set_err("wn_generate needs a full model handle"); return WN_ERR_STATE; }
  if (h->cfg.conditioning && !cond_dev) { set_err("Conditioning must be provided."); return WN_ERR_VALUE; }
  if (!prime_dev || n_prime < 1 || B < 1 || B > 64 || B > h->maxB || length < 1 || (!out_dev && !pred_dev)) { set_err("bad generate arguments (1 <= batch <= min(64, max_batch))"); return WN_ERR_VALUE; }
  if ((size_t)GEN_ROWS * h->K * (h->R > h->D ? h->R : h->D) * 4 > 160 * 1024) { set_err("generation: K * channels too large for the step kernel"); return WN_ERR_UNSUPPORTED; }
  CK(cudaSetDevice(h->cfg.device));
  h->fwd_valid = false;       // (the conditioning MLP's activations and the conditioning biases are overwritten)
  cudaStream_t user = (cudaStream_t)stream, st = h->own_stream;
  const int cap = n_prime + length + 1;
  RET(gen_alloc(h, B, cap));
  wn_handle::Gen& G = h->gen;
  CK(cudaEventRecord(h->ev_in, user)); CK(cudaStreamWaitEvent(st, h->ev_in, 0));
  // state: zero histories are the causal padding (nothing before the prime is ever needed at the last position, model.py:122)
  CK(cudaMemsetAsync(G.audio, 0, (size_t)G.B * G.cap * 4, st));
  for (auto& hl : G.hist) for (float* p : hl) if (p) CK(cudaMemsetAsync(p, 0, (size_t)G.B * G.cap * 4 * ((p == hl[0]) ? h->R : h->D), st));
  CK(cudaMemsetAsync(G.t_dev, 0, 4, st));
  CK(cudaMemcpy2DAsync(G.audio, (size_t)G.cap * 4, prime_dev, (size_t)n_prime * 4, (size_t)n_prime * 4, B, cudaMemcpyDeviceToDevice, st));
  if (teacher_dev) CK(cudaMemcpy2DAsync(G.audio + n_prime, (size_t)G.cap * 4, teacher_dev, (size_t)length * 4, (size_t)length * 4, B, cudaMemcpyDeviceToDevice, st));
  bool has_cb = false;
  if (h->cfg.conditioning) {
    const float* cond = cond_forward(h, st, cond_dev, B);
    const int n = 2 * h->D;
    cond_bias_all<<<dim3(cdiv(B * n, 128), h->L), 128, 0, st>>>(cond, h->Cc, h->d_params, h->d_cond_offsets, h->cb, (long long)h->maxB * n, B, n);
    has_cb = true;
  }
  for (int l = 0; l < h->L; ++l) {
    if (!G.wcat[l]) continue;
    const BlockP& b = h->blocks[l];
    const size_t ld = (size_t)(h->R + h->S) * 4;
    CK(cudaMemcpy2DAsync(G.wcat[l], ld, P_(h, b.conv1.w_idx), (size_t)h->R * 4, (size_t)h->R * 4, h->D, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpy2DAsync(G.wcat[l] + h->R, ld, P_(h, b.conv_skip.w_idx), (size_t)h->S * 4, (size_t)h->S * 4, h->D, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(G.bcat[l], P_(h, b.conv1.b_idx), (size_t)h->R * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(G.bcat[l] + h->R, P_(h, b.conv_skip.b_idx), (size_t)h->S * 4, cudaMemcpyDeviceToDevice, st));
  }
  // two graphs: a teacher-forced step (priming: histories only) and a generation step
  auto capture = [&](bool sample, float* pred, bool write_audio, cudaGraphExec_t* exec) -> int {
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int r = gen_step(h, st, B, has_cb, sample, deterministic, seed, pred, (long long)length * h->Cout, n_prime - 1, write_audio);
    cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (r != WN_OK || e != cudaSuccess || !graph) { if (graph) cudaGraphDestroy(graph); set_err("generation: graph capture failed"); return WN_ERR_CUDA; }
    e = cudaGraphInstantiate(exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { set_err("generation: graph instantiation failed"); return WN_ERR_CUDA; }
    return WN_OK;
  };
  cudaGraphExec_t g_prime = nullptr, g_gen = nullptr;
  if (n_prime > 1) RET(capture(false, nullptr, false, &g_prime));
  RET(capture(!teacher_dev, pred_dev, !teacher_dev, &g_gen));
  for (int t = 0; t + 1 < n_prime; ++t) CK(cudaGraphLaunch(g_prime, st));
  for (int i = 0; i < length; ++i) CK(cudaGraphLaunch(g_gen, st));
  if (out_dev) CK(cudaMemcpy2DAsync(out_dev, (size_t)length * 4, G.audio + n_prime, (size_t)G.cap * 4, (size_t)length * 4, B, cudaMemcpyDeviceToDevice, st));
  CK(cudaEventRecord(h->ev_out, st)); CK(cudaStreamWaitEvent(user, h->ev_out, 0));
  CK(cudaStreamSynchronize(st));
  if (g_prime) cudaGraphExecDestroy(g_prime);
  cudaGraphExecDestroy(g_gen);
  return WN_OK;
}

// The entry points without a handle launch on the device that owns their buffers (a caller whose current device is another GPU
// would otherwise get an invalid-argument launch failure).
static int use_device_of(const void* dev_ptr) {
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, dev_ptr) != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
    cudaGetLastError();
    set_err("argument is not a device pointer");
    return WN_ERR_VALUE;
  }
  CK(cudaSetDevice(at.device));
  return WN_OK;
}

// ============================================================================ device input pipeline (utils.py:31-70)
extern "C" int64_t wn_num_frames(int64_t n_samples, int T) {
  if (T < 1 || n_samples < (int64_t)T + 1) return 0;
  return 1 + (n_samples - (T + 1)) / T;
}
extern "C" int wn_preprocess_frames(const void* speech_dev, int is_int16, int64_t n_samples, int T, int apply_mulaw, float* frames_dev, int32_t* valid_dev,
                                    void* stream) {
  const int64_t nf = wn_num_frames(n_samples, T);
  if (nf == 0) return WN_OK;      /* shorter than one frame: nothing to emit */
  if (!speech_dev || !frames_dev || !valid_dev || nf > 65535) { set_err("bad preprocess arguments (at most 65535 frames per call)"); return WN_ERR_VALUE; }
  RET(use_device_of(frames_dev));
  cudaStream_t st = (cudaStream_t)stream;
  fill_int_kernel<<<cdiv(nf, 256), 256, 0, st>>>(valid_dev, (int)nf, 1);
  const dim3 grid(cdiv(T + 1, 256) < 64 ? cdiv(T + 1, 256) : 64, (unsigned)nf);
  if (is_int16) preprocess_frames_kernel<short><<<grid, 256, 0, st>>>((const short*)speech_dev, 1.0f / 32768.0f, T, (int)nf, apply_mulaw, frames_dev, valid_dev);
  else preprocess_frames_kernel<float><<<grid, 256, 0, st>>>((const float*)speech_dev, 1.0f, T, (int)nf, apply_mulaw, frames_dev, valid_dev);
  CK(cudaGetLastError());
  return WN_OK;
}
extern "C" int wn_inverse_mu_law(const float* y_dev, float* x_dev, int64_t n, void* stream) {
  if (n == 0) return WN_OK;
  if (!y_dev || !x_dev || n < 0) { set_err("bad inverse_mu_law arguments"); return WN_ERR_VALUE; }
  RET(use_device_of(x_dev));
  inverse_mu_law_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(y_dev, x_dev, n);
  CK(cudaGetLastError());
  return WN_OK;
}
extern "C" int wn_one_hot(const int32_t* ids_dev, int n, int depth, float* out_dev, void* stream) {
  if (n == 0) return WN_OK;
  if (!ids_dev || !out_dev || n < 0 || depth < 1) { set_err("bad one_hot arguments"); return WN_ERR_VALUE; }
  RET(use_device_of(out_dev));
  one_hot_kernel<<<cdiv((long long)n * depth, 256), 256, 0, (cudaStream_t)stream>>>(ids_dev, n, depth, out_dev);
  CK(cudaGetLastError());
  return WN_OK;
}

// ============================================================================ sampling + MSE metric (model.py:338-346,393-503)
static int sample_common(wn_handle* h, const float* pred, int ld, int is_logits, const float* frames, int B, int T, int deterministic, uint64_t seed,
                         float* out_dev, float* mse_dev, cudaStream_t st) {
  const wn_config& c = h->cfg;
  const long long rows = (long long)B * T;
  const int kind = c.sampling_function == WN_CATEGORICAL ? 0 : (c.sampling_function == WN_GAUSSIAN ? 2 : 1);
  const int nparts = cdiv(rows, 8);
  if (mse_dev && nparts > h->loss_parts_cap) { set_err("sample: workspace too small"); return WN_ERR_STATE; }
  sample_kernel<<<nparts, 256, 0, st>>>(pred, ld, h->Cout, c.num_mixtures, kind, is_logits, c.bits, deterministic, seed, frames, T, rows, out_dev,
                                       mse_dev ? h->loss_partial : nullptr);
  if (mse_dev) loss_finalize<<<1, 1024, 0, st>>>(h->loss_partial, nparts, 1.0f / (float)rows, nullptr, 0.f, mse_dev);
  CK(cudaGetLastError());
  return WN_OK;
}
// sample_waveform(pred) for a caller-held WaveNet.call output (probabilities or mixture parameters), (B,T,Cout) fp32
extern "C" int wn_sample_waveform(wn_handle* h, const float* pred_dev, int B, int T, int deterministic, uint64_t seed, float* out_dev, void* stream) {
  RET(check_bt(h, B, T));
  if (!pred_dev || !out_dev || !h->cfg.has_head) { set_err("bad sample arguments"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  return sample_common(h, pred_dev, h->Cout, 0, nullptr, B, T, deterministic, seed, out_dev, nullptr, (cudaStream_t)stream);
}
// the same on the predictions of the LAST train/test step (kept on the device as logits), plus the MSE metric against
// y_true = frames[:,1:] (model.py:338-346): mse_dev[0] = mean over (b,t) of (y - sample)^2; mse_dev needs 2 floats
extern "C" int wn_sample_last_step(wn_handle* h, const float* frames_dev, int deterministic, uint64_t seed, float* out_dev, float* mse_dev, void* stream) {
  if (!h || !h->cfg.has_head || h->lastB < 1) { set_err("no train/test step to sample from"); return WN_ERR_STATE; }
  if (!out_dev) { set_err("bad sample arguments"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  return sample_common(h, h->logits, h->ldl, 1, mse_dev ? frames_dev : nullptr, h->lastB, h->lastT, deterministic, seed, out_dev, mse_dev, (cudaStream_t)stream);
}

// ============================================================================ optimizer (train.py:225-226; model.py:336)
extern "C" int wn_adam_init(wn_handle* h, float lr, float beta1, float beta2, float eps, float clipnorm) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (lr < 0.f || beta1 < 0.f || beta1 >= 1.f || beta2 < 0.f || beta2 >= 1.f || eps <= 0.f || clipnorm < 0.f) { set_err("bad Adam hyper-parameters"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  h->opt_lr = lr; h->opt_b1 = beta1; h->opt_b2 = beta2; h->opt_eps = eps; h->opt_clipnorm = clipnorm; h->opt_t = 0;
  const size_t bytes = (size_t)h->n_scalars * 4;
  if (!h->opt_m) {
    CK(cudaMalloc(&h->opt_m, bytes)); CK(cudaMalloc(&h->opt_v, bytes));
    std::vector<OptChunk> ch; std::vector<int> first;
    for (size_t v = 0; v < h->params.size(); ++v) {
      first.push_back((int)ch.size());
      for (long long o = 0; o < h->params[v].count; o += OPT_CHUNK)
        ch.push_back(OptChunk{(int)v, (int)std::min<long long>(OPT_CHUNK, h->params[v].count - o), h->params[v].offset + o});
    }
    first.push_back((int)ch.size());
    h->opt_n_chunks = (int)ch.size();
    CK(cudaMalloc(&h->opt_chunks, ch.size() * sizeof(OptChunk)));
    CK(cudaMalloc(&h->opt_var_first, first.size() * sizeof(int)));
    CK(cudaMalloc(&h->opt_partial, ch.size() * 4));
    CK(cudaMalloc(&h->opt_scale, h->params.size() * 4));
    CK(cudaMalloc(&h->opt_norms, h->params.size() * 4));
    CK(cudaMemcpy(h->opt_chunks, ch.data(), ch.size() * sizeof(OptChunk), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->opt_var_first, first.data(), first.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  CK(cudaMemset(h->opt_m, 0, bytes)); CK(cudaMemset(h->opt_v, 0, bytes));
  return WN_OK;
}
// per-variable tf.clip_by_norm of the gradients in place (Keras clips each replica's gradients before the cross-replica sum)
extern "C" int wn_clip_grads(wn_handle* h, void* stream) {
  if (!h || !h->opt_m) { set_err("call wn_adam_init first"); return WN_ERR_STATE; }
  if (h->opt_clipnorm <= 0.f) return WN_OK;
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  opt_sumsq_kernel<<<h->opt_n_chunks, 256, 0, st>>>(h->d_grads, h->opt_chunks, h->opt_partial);
  const int nv = (int)h->params.size();
  opt_clip_scale_kernel<<<cdiv(nv, 128), 128, 0, st>>>(h->opt_partial, h->opt_var_first, nv, h->opt_clipnorm, h->opt_scale, h->opt_norms);
  opt_clip_apply_kernel<<<h->opt_n_chunks, 256, 0, st>>>(h->d_grads, h->opt_chunks, h->opt_scale);
  CK(cudaGetLastError());
  return WN_OK;
}
// one Adam update from wn_grads_dev (already clipped / all-reduced by the caller); lr < 0 keeps the current learning rate.
// Re-packs the kernel-side weight copies.
extern "C" int wn_adam_step(wn_handle* h, float lr, void* stream) {
  if (!h || !h->opt_m) { set_err("call wn_adam_init first"); return WN_ERR_STATE; }
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (lr >= 0.f) h->opt_lr = lr;
  h->opt_t += 1;
  const double b1t = pow((double)h->opt_b1, (double)h->opt_t), b2t = pow((double)h->opt_b2, (double)h->opt_t);
  const float alpha = (float)((double)h->opt_lr * sqrt(1.0 - b2t) / (1.0 - b1t));
  opt_adam_kernel<<<cdiv(h->n_scalars, 256), 256, 0, st>>>(h->d_params, h->d_grads, h->opt_m, h->opt_v, h->n_scalars, alpha, 1.0f - h->opt_b1,
                                                          1.0f - h->opt_b2, h->opt_eps);
  CK(cudaGetLastError());
  return wn_params_changed(h, stream);
}
extern "C" int wn_adam_state(wn_handle* h, float** m_dev, float** v_dev, float** grad_norms_dev, int64_t* step) {
  if (!h || !h->opt_m) { set_err("call wn_adam_init first"); return WN_ERR_STATE; }
  if (m_dev) *m_dev = h->opt_m;
  if (v_dev) *v_dev = h->opt_v;
  if (grad_norms_dev) *grad_norms_dev = h->opt_norms;
  if (step) *step = h->opt_t;
  return WN_OK;
}

// optimizer state of another handle of the same model (a rebuild for a larger workspace keeps training where it was)
extern "C" int wn_adam_restore(wn_handle* h, const float* m_dev, const float* v_dev, int64_t step) {
  if (!h || !h->opt_m) { set_err("call wn_adam_init first"); return WN_ERR_STATE; }
  if (!m_dev || !v_dev || step < 0) { set_err("bad optimizer state"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  const size_t bytes = (size_t)h->n_scalars * 4;
  CK(cudaMemcpy(h->opt_m, m_dev, bytes, cudaMemcpyDeviceToDevice));
  CK(cudaMemcpy(h->opt_v, v_dev, bytes, cudaMemcpyDeviceToDevice));
  h->opt_t = step;
  return WN_OK;
}

extern "C" int wn_set_dropout_masks(wn_handle* h, const uint8_t* keep_host, int B, int T) {
  RET(check_bt(h, B, T));
  if (h->cfg.dropout <= 0.f || !h->drop_mask) { set_err("model was built with dropout == 0"); return WN_ERR_STATE; }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  drop_graphs(h);
  h->fwd_valid = false;
  if (!keep_host) { h->drop_injected = false; return WN_OK; }
  const size_t n = (size_t)B * T * h->R, slab = (size_t)h->maxB * h->maxT * h->R;
  for (int l = 0; l < h->L; ++l) CK(cudaMemcpy(h->drop_mask + l * slab, keep_host + l * n, n, cudaMemcpyHostToDevice));
  h->drop_injected = true;
  h->drop_B = B; h->drop_T = T;
  return WN_OK;
}
// a training pass reads the keep-mask of (b, t) at row b*T + t of its own T: injected masks belong to the shape they were packed for
static int check_injected_mask_shape(wn_handle* h, int B, int T, bool training) {
  if (!training || h->cfg.dropout <= 0.f || !h->drop_injected || (B == h->drop_B && T == h->drop_T)) return WN_OK;
  set_err("dropout masks were injected for (batch, time) = (%d, %d); a training pass at (%d, %d) needs masks of its own shape "
          "(or none: wn_set_dropout_masks(NULL) returns to Philox masks)", h->drop_B, h->drop_T, B, T);
  return WN_ERR_STATE;
}
extern "C" int wn_set_dropout_seed(wn_handle* h, uint64_t seed) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  drop_graphs(h);
  h->drop_seed = seed;
  h->drop_injected = false;
  if (h->d_drop_ctr) CK(cudaMemset(h->d_drop_ctr, 0, 8));
  return WN_OK;
}

extern "C" int wn_quantize(const float* x_dev, int64_t* idx_dev, int64_t n, int bits, void* stream) {
  if (n == 0) return WN_OK;  /* empty input: nothing to do */
  if (!x_dev || !idx_dev || n < 0 || bits < 1 || bits > 16) { set_err("bad quantize arguments"); return WN_ERR_VALUE; }
  RET(use_device_of(idx_dev));
  quantize_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(x_dev, (long long*)idx_dev, n, bits);
  CK(cudaGetLastError());
  return WN_OK;
}

// fresh Philox keep-masks for a training pass (unless the caller injected masks): bumps the device step counter
// only_block >= 0: the mask of that block alone (layer API: the other blocks' masks may still be waiting for their backward)
static void draw_dropout_masks(wn_handle* h, cudaStream_t st, int B, int Tn, int only_block = -1) {
  if (!h->drop_active || h->drop_injected) return;
  const size_t rows_cap = (size_t)h->maxB * h->maxT;
  const long long n8 = ((long long)B * Tn * h->R + 7) / 8;     // (the slabs are 16-byte aligned and padded: a last partial group stays inside)
  { LaunchScope ls(h, st, CLS_MISC); dropout_step_bump<<<1, 1, 0, st>>>(h->d_drop_ctr); }
  LaunchScope ls(h, st, CLS_MISC);
  dropout_mask_philox<<<dim3(cdiv(n8, 256), only_block >= 0 ? 1 : h->L), 256, 0, st>>>(h->drop_mask, n8, (long long)rows_cap * h->R, h->cfg.dropout,
                                                                                    h->drop_seed, h->d_drop_ctr, only_block >= 0 ? only_block : 0);
}

template <class T>
static int forward_entry(wn_handle* h, const float* x, const float* cond, int B, int Tn, int training, float* out, cudaStream_t st) {
  // WaveNet.call(inputs, training): Keras Dropout is active only under training=True (layers.py:195-196)
  h->drop_active = training && h->cfg.dropout > 0.f;
  draw_dropout_masks(h, st, B, Tn);
  RET(model_forward<T>(h, st, x, Tn, cond, B, Tn));
  if (h->cfg.sampling_function == WN_CATEGORICAL) {
    RET(loss_forward<T>(h, st, nullptr, B, Tn, 0.f, false, out, nullptr));
  } else {
    CK(cudaMemcpyAsync(out, h->logits, (size_t)B * Tn * h->Cout * 4, cudaMemcpyDeviceToDevice, st));
  }
  return WN_OK;
}

extern "C" int wn_forward_ex(wn_handle* h, const float* x_dev, const float* cond_dev, int B, int T, int training, float* out_dev, void* stream) {
  RET(check_bt(h, B, T));
  if (!h->cfg.has_head || !h->cfg.has_input_conv) { set_err("wn_forward needs a full model handle"); return WN_ERR_STATE; }
  if (h->cfg.conditioning && !cond_dev) { set_err("Conditioning must be provided."); return WN_ERR_VALUE; }
  if (training && h->cfg.dropout >= 1.f) { set_err("dropout must be < 1 for training"); return WN_ERR_VALUE; }
  RET(check_injected_mask_shape(h, B, T, training != 0));
  CK(cudaSetDevice(h->cfg.device));
  h->launches = 0;
  h->fwd_valid = false;
  cudaStream_t st = (cudaStream_t)stream;
  int r = h->cfg.precision == WN_BF16 ? forward_entry<bf16>(h, x_dev, cond_dev, B, T, training, out_dev, st)
                                      : forward_entry<float>(h, x_dev, cond_dev, B, T, training, out_dev, st);
  h->drop_active = false;
  RET(r);
  CK(cudaGetLastError());
  // (lastB / lastT stay those of the last train/test step: wn_sample_last_step reads them)
  h->fwd = wn_handle::FwdRecord{B, T, training != 0, x_dev, T, cond_dev};
  h->fwd_valid = true;
  return WN_OK;
}

// d loss / d cond_in of the model: without a mapping MLP that is h->dcond; with one, cond_backward leaves the gradient of the first
// mapping layer's pre-activation in the buffer its ping-pong ends on (d0 = dcond, then d1 = cond_dact, d2 = cond_dact2, alternating)
static int cond_input_grad(wn_handle* h, cudaStream_t st, int B, float* dcond) {
  const int n = (int)h->map_w.size();
  if (n == 0) {
    CK(cudaMemcpyAsync(dcond, h->dcond, (size_t)B * h->cfg.cond_in * 4, cudaMemcpyDeviceToDevice, st));
    return WN_OK;
  }
  const float* dpre = n == 1 ? h->dcond : (n - 1) % 2 == 1 ? h->cond_dact : h->cond_dact2;
  const int K = h->cfg.cond_in, N = h->map_width[0];
  LaunchScope ls(h, st, CLS_MISC);
  dense_small_dgrad<<<cdiv(B * K, 4), 128, 0, st>>>(dpre, N, P_(h, h->map_w[0]), dcond, K, B, K, N, 0);
  return WN_OK;
}

template <class T>
static int backward_entry(wn_handle* h, const float* dpred, float* dcond, float* dx, bool param_grads, cudaStream_t st) {
  const int B = h->fwd.B, Tn = h->fwd.T;
  const long long rows = (long long)B * Tn;
  {
    // dlogits = the adjoint of what wn_forward_ex returned: the softmax's VJP, or dpred itself for the raw mixture parameters
    OuterLabel ol(h, "pred_vjp");
    LaunchScope ls(h, st, CLS_LOSS);
    if (h->cfg.sampling_function == WN_CATEGORICAL) {
      if (h->Cout == 256 && h->ldl == 256 && h->ldd % 4 == 0)
        softmax_vjp_reg_kernel<T, 2><<<cdiv(rows, 8), 256, 0, st>>>(h->logits, dpred, rows, (T*)h->dlogits, h->ldd);
      else
        softmax_vjp_kernel<T><<<cdiv(rows, 8), 256, 0, st>>>(h->logits, h->Cout, dpred, rows, (T*)h->dlogits, h->ldd);
    } else {
      convert_pad_kernel<float, T><<<cdiv(rows * h->ldd, 256), 256, 0, st>>>(dpred, h->Cout, (T*)h->dlogits, h->ldd, rows);
    }
  }
  RET(model_backward<T>(h, st, h->fwd.x, h->fwd.ldx, h->fwd.cond, B, Tn, 0.f, dx, param_grads));
  if (dcond) RET(cond_input_grad(h, st, B, dcond));
  return WN_OK;
}

extern "C" int wn_backward_ex(wn_handle* h, const float* dpred_dev, float* dcond_dev, float* dx_dev, int param_grads, void* stream) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (!dpred_dev || ((uintptr_t)dpred_dev & 15) != 0) { set_err("dpred must be a 16-byte aligned device buffer"); return WN_ERR_VALUE; }
  if (dcond_dev && !h->cfg.conditioning) { set_err("the model has no conditioning input"); return WN_ERR_VALUE; }
  if (!param_grads && !dx_dev && !dcond_dev) { set_err("wn_backward_ex without parameter gradients needs dx or dcond: nothing to compute"); return WN_ERR_VALUE; }
  if (!h->fwd_valid) { set_err("wn_backward needs a wn_forward_ex since the handle's activations or weights last changed"); return WN_ERR_STATE; }
  CK(cudaSetDevice(h->cfg.device));
  h->launches = 0;
  cudaStream_t st = (cudaStream_t)stream;
  // the stack-backward plans are keyed on drop_active, and the forward's keep-masks are still in drop_mask
  h->drop_active = h->fwd.training && h->cfg.dropout > 0.f;
  h->ar_now = false;
  h->lastB = h->fwd.B; h->lastT = h->fwd.T;     // wn_debug_tensor reads the pass just differentiated
  int r = h->cfg.precision == WN_BF16 ? backward_entry<bf16>(h, dpred_dev, dcond_dev, dx_dev, param_grads != 0, st)
                                      : backward_entry<float>(h, dpred_dev, dcond_dev, dx_dev, param_grads != 0, st);
  h->drop_active = false;
  RET(r);
  CK(cudaGetLastError());
  return WN_OK;
}
extern "C" int wn_backward(wn_handle* h, const float* dpred_dev, float* dcond_dev, void* stream) {
  return wn_backward_ex(h, dpred_dev, dcond_dev, nullptr, 1, stream);
}
extern "C" int wn_forward(wn_handle* h, const float* x_dev, const float* cond_dev, int B, int T, float* out_dev, void* stream) {
  return wn_forward_ex(h, x_dev, cond_dev, B, T, 0, out_dev, stream);
}

// WaveNet.loss_fn(target, pred) (model.py:505-551) on materialised predictions, per (b, t), no reduction
extern "C" int wn_loss_fn(wn_handle* h, const void* target_dev, int target_is_int64, const float* pred_dev, int B, int T, float* out_dev, void* stream) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (!h->cfg.has_head) { set_err("wn_loss_fn needs a full model handle"); return WN_ERR_STATE; }
  if (B < 1 || T < 1 || !target_dev || !pred_dev || !out_dev) { set_err("bad loss_fn arguments"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  const wn_config& c = h->cfg;
  const long long rows = (long long)B * T;
  if (c.sampling_function == WN_CATEGORICAL) {
    ce_probs_rows_kernel<<<cdiv(rows, 8), 256, 0, st>>>(pred_dev, h->Cout, target_is_int64 ? (const long long*)target_dev : nullptr,
                                                       target_is_int64 ? nullptr : (const float*)target_dev, c.bits, rows, out_dev);
  } else {
    if (target_is_int64) { set_err("mixture losses take the waveform itself as target (model.py:155)"); return WN_ERR_VALUE; }
    mixture_loss_launch<float>(st, nullptr, pred_dev, h->Cout, c.num_mixtures, (const float*)target_dev, T, rows, c.bits,
                               c.sampling_function == WN_GAUSSIAN ? 2 : 1, 1.0f, nullptr, 0, nullptr, T, 0, out_dev);
  }
  CK(cudaGetLastError());
  return WN_OK;
}

// MirroredStrategy's gradient reduction (train.py:203, model.py:336): the loss is already divided by the GLOBAL batch
// (model.py:328), so the replicas' gradients are SUMMED — one ncclAllReduce over the flat fp32 buffer, in place
static int allreduce_grads(wn_handle* h, cudaStream_t st) {
  if (!h->comm) { set_err("no communicator: call wn_comm_init / wn_comm_attach first"); return WN_ERR_STATE; }
  if (h->ar_early_lo >= 0 && h->ar_early_hi > h->ar_early_lo) {
    // model_backward already reduced scalars [lo, hi) on comm_stream, bucket by bucket: join, then the two slices around them
    const long long lo = h->ar_early_lo, hi = h->ar_early_hi;
    h->ar_early_lo = h->ar_early_hi = -1;
    CK(cudaEventRecord(h->ev_comm_done, h->comm_stream));
    CK(cudaStreamWaitEvent(st, h->ev_comm_done, 0));
    g_nccl.GroupStart();
    int r = 0;
    if (lo > 0) { h->launches++; r = g_nccl.AllReduce(h->d_grads, h->d_grads, (size_t)lo, WN_NCCL_FLOAT32, WN_NCCL_SUM, h->comm, st); }
    if (r == 0 && hi < h->n_scalars) {
      h->launches++;
      r = g_nccl.AllReduce(h->d_grads + hi, h->d_grads + hi, (size_t)(h->n_scalars - hi), WN_NCCL_FLOAT32, WN_NCCL_SUM, h->comm, st);
    }
    const int r2 = g_nccl.GroupEnd();
    if (r != 0 || r2 != 0) { set_err("ncclAllReduce failed (%d): %s", r != 0 ? r : r2, nccl_errstr(r != 0 ? r : r2)); return WN_ERR_CUDA; }
    return WN_OK;
  }
  h->launches++;
  const int r = g_nccl.AllReduce(h->d_grads, h->d_grads, (size_t)h->n_scalars, WN_NCCL_FLOAT32, WN_NCCL_SUM, h->comm, st);
  if (r != 0) { set_err("ncclAllReduce failed (%d): %s", r, nccl_errstr(r)); return WN_ERR_CUDA; }
  return WN_OK;
}

extern "C" int wn_nccl_unique_id(uint8_t* id128) {
  if (!id128) { set_err("null argument"); return WN_ERR_VALUE; }
  char err[256];
  if (nccl_load(err, sizeof(err)) != 0) { set_err("%s", err); return WN_ERR_CUDA; }
  wn_ncclUniqueId id;
  const int r = g_nccl.GetUniqueId(&id);
  if (r != 0) { set_err("ncclGetUniqueId failed (%d): %s", r, nccl_errstr(r)); return WN_ERR_CUDA; }
  memcpy(id128, id.internal, 128);
  return WN_OK;
}
extern "C" int wn_comm_init(wn_handle* h, const uint8_t* id128, int nranks, int rank) {
  if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) { set_err("bad communicator arguments"); return WN_ERR_VALUE; }
  char err[256];
  if (nccl_load(err, sizeof(err)) != 0) { set_err("%s", err); return WN_ERR_CUDA; }
  CK(cudaSetDevice(h->cfg.device));
  if (h->comm && h->comm_owned) g_nccl.CommDestroy(h->comm);
  h->comm = nullptr;
  wn_ncclUniqueId id;
  memcpy(id.internal, id128, 128);
  wn_ncclComm_t c = nullptr;
  const int r = g_nccl.CommInitRank(&c, nranks, id, rank);
  if (r != 0) { set_err("ncclCommInitRank failed (%d): %s", r, nccl_errstr(r)); return WN_ERR_CUDA; }
  h->comm = c; h->comm_owned = true; h->comm_nranks = nranks; h->comm_rank = rank;
  cudaDeviceSynchronize();
  drop_graphs(h);
  return WN_OK;
}
extern "C" int wn_comm_attach(wn_handle* h, void* nccl_comm, int nranks, int rank) {
  if (!h || nranks < 1) { set_err("bad communicator arguments"); return WN_ERR_VALUE; }
  char err[256];
  if (nccl_comm && nccl_load(err, sizeof(err)) != 0) { set_err("%s", err); return WN_ERR_CUDA; }
  if (h->comm && h->comm_owned) g_nccl.CommDestroy(h->comm);
  h->comm = (wn_ncclComm_t)nccl_comm; h->comm_owned = false; h->comm_nranks = nccl_comm ? nranks : 1; h->comm_rank = rank;
  cudaDeviceSynchronize();
  drop_graphs(h);
  return WN_OK;
}
extern "C" int wn_comm_fuse_allreduce(wn_handle* h, int on) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if ((on != 0) != (h->ar_in_step != 0)) { h->ar_in_step = on ? 1 : 0; cudaDeviceSynchronize(); drop_graphs(h); }
  return WN_OK;
}
extern "C" int wn_allreduce_grads(wn_handle* h, void* stream) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (h->comm_nranks <= 1) return WN_OK;
  CK(cudaSetDevice(h->cfg.device));
  return allreduce_grads(h, (cudaStream_t)stream);
}
extern "C" const char* wn_nccl_info(void) {
  static char buf[400];
  char err[256];
  if (nccl_load(err, sizeof(err)) != 0) { snprintf(buf, sizeof(buf), "unavailable: %s", err); return buf; }
  int v = 0;
  if (g_nccl.GetVersion) g_nccl.GetVersion(&v);
  snprintf(buf, sizeof(buf), "NCCL %d from %s", v, g_nccl.where);
  return buf;
}

template <class T>
static int step_entry(wn_handle* h, const float* frames, const float* cond, int B, int Tn, int nrep, float* loss, cudaStream_t st, bool train) {
  const float scale = 1.0f / ((float)B * (float)nrep);
  h->drop_active = train && h->cfg.dropout > 0.f;
  draw_dropout_masks(h, st, B, Tn);
  RET(model_forward<T>(h, st, frames, Tn + 1, cond, B, Tn));
  RET(loss_forward<T>(h, st, frames, B, Tn, scale, train, nullptr, loss));
  if (train) {
    const float l2coef = h->cfg.l2_reg_factor > 0.f ? 2.0f * h->cfg.l2_reg_factor / (float)nrep : 0.f;
    h->ar_now = h->ar_in_step && h->comm && h->comm_nranks > 1 && nrep > 1;
    RET(model_backward<T>(h, st, frames, Tn + 1, cond, B, Tn, l2coef));
    if (h->ar_now) RET(allreduce_grads(h, st));
    h->ar_now = false;
  }
  return WN_OK;
}

static int step_common(wn_handle* h, const float* frames_dev, const float* cond_dev, int B, int T, int n_replicas, float* loss_dev, void* stream, bool train) {
  RET(check_bt(h, B, T));
  if (!h->cfg.has_head || !h->cfg.has_input_conv) { set_err("train/test step needs a full model handle"); return WN_ERR_STATE; }
  if (h->cfg.conditioning && !cond_dev) { set_err("Conditioning must be provided."); return WN_ERR_VALUE; }
  if (n_replicas < 1 || !frames_dev || !loss_dev) { set_err("bad step arguments"); return WN_ERR_VALUE; }
  if (train && h->cfg.dropout >= 1.f) { set_err("dropout must be < 1 for training"); return WN_ERR_VALUE; }
  RET(check_injected_mask_shape(h, B, T, train));
  CK(cudaSetDevice(h->cfg.device));
  h->fwd_valid = false;
  cudaStream_t st = (cudaStream_t)stream;
  auto run = [&](cudaStream_t s) -> int {
    h->launches = 0;
    return h->cfg.precision == WN_BF16 ? step_entry<bf16>(h, frames_dev, cond_dev, B, T, n_replicas, loss_dev, s, train)
                                       : step_entry<float>(h, frames_dev, cond_dev, B, T, n_replicas, loss_dev, s, train);
  };
  // The step is ~350 dependent launches: replay it as one CUDA graph from the second identical call on
  // (first call runs eagerly and warms function attributes and the tensor-map cache).
  if (h->use_graphs && h->prof_tag == 0) {
    wn_handle::StepGraph* sg = nullptr;
    for (auto& g : h->graphs)
      if (g.frames == frames_dev && g.cond == cond_dev && g.B == B && g.T == T && g.nrep == n_replicas && g.loss == loss_dev && g.train == train) { sg = &g; break; }
    if (!sg) {
      if (h->graphs.size() >= 8) drop_graphs(h);
      h->graphs.push_back({frames_dev, cond_dev, B, T, n_replicas, loss_dev, train, 0, 0, nullptr});
      sg = &h->graphs.back();
    }
    // the legacy default stream cannot be captured: run the graph on the handle's stream, ordered by events
    const bool legacy = st == nullptr || st == cudaStreamLegacy;
    cudaStream_t gs = legacy ? h->own_stream : st;
    if (sg->seen >= 1 && !sg->exec) {
      cudaGraph_t graph = nullptr;
      if (cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        int r = run(gs);
        cudaError_t e = cudaStreamEndCapture(gs, &graph);
        if (r == WN_OK && e == cudaSuccess && graph && cudaGraphInstantiate(&sg->exec, graph, 0) == cudaSuccess) {
          sg->launches = h->launches;
        } else {
          sg->exec = nullptr;
          h->use_graphs = 0;       // fall back to eager launches for good
          cudaGetLastError();
        }
        if (graph) cudaGraphDestroy(graph);
      } else {
        h->use_graphs = 0;
        cudaGetLastError();
      }
    }
    if (sg->exec) {
      if (legacy) { CK(cudaEventRecord(h->ev_in, st)); CK(cudaStreamWaitEvent(gs, h->ev_in, 0)); }
      CK(cudaGraphLaunch(sg->exec, gs));
      if (legacy) { CK(cudaEventRecord(h->ev_out, gs)); CK(cudaStreamWaitEvent(st, h->ev_out, 0)); }
      h->launches = sg->launches;
      h->lastB = B; h->lastT = T;
      return WN_OK;
    }
    sg->seen++;
  }
  RET(run(st));
  CK(cudaGetLastError());
  h->lastB = B; h->lastT = T;
  return WN_OK;
}

extern "C" int wn_train_step(wn_handle* h, const float* frames_dev, const float* cond_dev, int B, int T, int n_replicas, float* loss_dev, void* stream) {
  return step_common(h, frames_dev, cond_dev, B, T, n_replicas, loss_dev, stream, true);
}
extern "C" int wn_test_step(wn_handle* h, const float* frames_dev, const float* cond_dev, int B, int T, int n_replicas, float* loss_dev, void* stream) {
  return step_common(h, frames_dev, cond_dev, B, T, n_replicas, loss_dev, stream, false);
}

extern "C" int wn_train_step_host(wn_handle* h, const float* frames_host, const float* cond_host, int B, int T, int n_replicas, float* loss_host) {
  RET(check_bt(h, B, T));
  if (!frames_host || !loss_host) { set_err("bad step arguments"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  h->fwd_valid = false;
  cudaStream_t st = h->own_stream;
  const size_t fb = (size_t)B * (T + 1) * 4;
  memcpy(h->pin_frames, frames_host, fb);
  CK(cudaMemcpyAsync(h->d_frames, h->pin_frames, fb, cudaMemcpyHostToDevice, st));
  const float* dc = nullptr;
  if (h->cfg.conditioning) {
    if (!cond_host) { set_err("Conditioning must be provided."); return WN_ERR_VALUE; }
    const size_t cbz = (size_t)B * h->cfg.cond_in * 4;
    memcpy(h->pin_cond, cond_host, cbz);
    CK(cudaMemcpyAsync(h->d_cond_in, h->pin_cond, cbz, cudaMemcpyHostToDevice, st));
    dc = h->d_cond_in;
  }
  RET(step_common(h, h->d_frames, dc, B, T, n_replicas, h->d_loss, st, true));
  CK(cudaMemcpyAsync(h->pin_loss, h->d_loss, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  loss_host[0] = h->pin_loss[0];
  loss_host[1] = h->pin_loss[1];
  return WN_OK;
}

// ---------------------------------------------------------------- layer-level API
template <class T>
static int layer_fwd_entry(wn_handle* h, int l, const float* x, const float* cond, bool seq, int B, int Tn, int training, float* x_out,
                           float* skip, cudaStream_t st) {
  // WaveNetLayer.call(inputs, training): Keras Dropout is active only under training=True (layers.py:195-196)
  h->drop_active = training && h->cfg.dropout > 0.f;
  h->layer_drop[l] = h->drop_active;
  draw_dropout_masks(h, st, B, Tn, l);
  const long long nR = (long long)B * Tn * h->R;
  // keep a private copy of the block input (needed by the backward pass); block l > 0 keeps it where the model does, in xout[l-1]
  void* xin = l == 0 ? h->layer_in : h->xout[l - 1];
  {
    LaunchScope ls(h, st, CLS_MISC);
    convert_kernel<float, T><<<cdiv(nR, 256), 256, 0, st>>>(x, (T*)xin, nR);
  }
  bool has_cb = false;
  h->layer_cseq[l] = nullptr;
  if (seq) {
    // (B,T,Cc) sequence: the bf16 tier contracts a zero-padded bf16 copy, the fp32 tier the caller's buffer itself
    const BlockP& b = h->blocks[l];
    const void* cs = cond;
    if constexpr (sizeof(T) == 2) {
      LaunchScope ls(h, st, CLS_MISC);
      const long long rows = (long long)B * Tn;
      convert_pad_kernel<float, bf16><<<cdiv(rows * h->Ccs, 256), 256, 0, st>>>(cond, h->Cc, (bf16*)h->cseq[l], h->Ccs, rows);
      cs = h->cseq[l];
    }
    {
      LaunchScope ls(h, st, CLS_MISC);
      add2_kernel<float><<<cdiv(2 * h->D, 256), 256, 0, st>>>(P_(h, b.stack.back().b_idx), P_(h, b.cb_idx), h->cseq_bias + (size_t)l * 2 * h->D,
                                                              2 * h->D);
    }
    h->layer_cseq[l] = cs;
    h->cond_seq = cs;
  } else if (h->blocks[l].has_cond) {
    if (!cond) { set_err("Conditioning must be provided."); return WN_ERR_VALUE; }
    h->last_cond = cond;
    cond_bias_block(h, st, l, cond, B);
    has_cb = true;
  }
  RET(block_forward<T>(h, st, l, xin, has_cb, B, Tn));
  {
    LaunchScope ls(h, st, CLS_MISC);
    convert_kernel<T, float><<<cdiv(nR, 256), 256, 0, st>>>((const T*)h->xout[l], x_out, nR);
  }
  if (skip) {
    const BlockP& b = h->blocks[l];
    RET((skip_gemm<T, float>(h, st, l, 1, skip, h->Sp, P_(h, b.has_skip ? b.conv_skip.b_idx : b.conv1.b_idx), B, Tn)));
  }
  return WN_OK;
}

static int layer_forward_call(wn_handle* h, int block, const float* x_dev, const float* cond_dev, bool seq, int B, int T, int training,
                              float* x_out_dev, float* skip_dev, void* stream) {
  CK(cudaSetDevice(h->cfg.device));
  h->launches = 0;
  h->fwd_valid = false;
  cudaStream_t st = (cudaStream_t)stream;
  int r = h->cfg.precision == WN_BF16 ? layer_fwd_entry<bf16>(h, block, x_dev, cond_dev, seq, B, T, training, x_out_dev, skip_dev, st)
                                      : layer_fwd_entry<float>(h, block, x_dev, cond_dev, seq, B, T, training, x_out_dev, skip_dev, st);
  h->drop_active = false;
  h->cond_seq = nullptr;
  RET(r);
  CK(cudaGetLastError());
  h->lastB = B; h->lastT = T;
  h->layer_fwd_valid[block] = true;
  return WN_OK;
}
extern "C" int wn_layer_forward_ex(wn_handle* h, int block, const float* x_dev, const float* cond_dev, int B, int T, int training, float* x_out_dev,
                                   float* skip_dev, void* stream) {
  RET(check_bt(h, B, T));
  if (block < 0 || block >= h->L || !x_dev || !x_out_dev) { set_err("bad layer arguments"); return WN_ERR_VALUE; }
  if (training && h->cfg.dropout >= 1.f) { set_err("dropout must be < 1 for training"); return WN_ERR_VALUE; }
  RET(check_injected_mask_shape(h, B, T, training != 0));
  return layer_forward_call(h, block, x_dev, cond_dev, false, B, T, training, x_out_dev, skip_dev, stream);
}
extern "C" int wn_layer_forward_seq(wn_handle* h, int block, const float* x_dev, const float* cond_dev, int B, int T, int training,
                                    float* x_out_dev, float* skip_dev, void* stream) {
  RET(check_bt(h, B, T));
  if (block < 0 || block >= h->L || !x_dev || !x_out_dev) { set_err("bad layer arguments"); return WN_ERR_VALUE; }
  if (!cond_dev) { set_err("conditioning sequence is NULL"); return WN_ERR_VALUE; }
  if (!h->blocks[block].has_cond) { set_err("block %d was built without conditioning", block); return WN_ERR_VALUE; }
  if (h->Ccs == 0) { set_err("conditioning sequences are built for layer handles (has_head = 0) only"); return WN_ERR_UNSUPPORTED; }
  if (training && h->cfg.dropout >= 1.f) { set_err("dropout must be < 1 for training"); return WN_ERR_VALUE; }
  RET(check_injected_mask_shape(h, B, T, training != 0));
  return layer_forward_call(h, block, x_dev, cond_dev, true, B, T, training, x_out_dev, skip_dev, stream);
}
extern "C" int wn_layer_forward(wn_handle* h, int block, const float* x_dev, const float* cond_dev, int B, int T, float* x_out_dev, float* skip_dev,
                                void* stream) {
  return wn_layer_forward_ex(h, block, x_dev, cond_dev, B, T, 0, x_out_dev, skip_dev, stream);
}

template <class T>
static int layer_bwd_entry(wn_handle* h, int l, const float* dxo, const float* dsk, float* dx, float* dcond, cudaStream_t st) {
  h->drop_active = h->layer_drop[l];   // adjoint of the forward this block last ran (its keep-mask is still in drop_mask)
  h->cond_seq = h->layer_cseq[l];      // ... and its conditioning sequence, if it had one
  const int B = h->lastB, Tn = h->lastT;
  const long long nR = (long long)B * Tn * h->R, nS = (long long)B * Tn * h->Sp;
  const void *dxo_t = nullptr, *dsk_t = nullptr;
  if (dxo) {
    LaunchScope ls(h, st, CLS_MISC);
    convert_kernel<float, T><<<cdiv(nR, 256), 256, 0, st>>>(dxo, (T*)h->dxA, nR);
    dxo_t = h->dxA;
  }
  if (dsk) {
    LaunchScope ls(h, st, CLS_MISC);
    convert_kernel<float, T><<<cdiv(nS, 256), 256, 0, st>>>(dsk, (T*)h->dskip, nS);
    dsk_t = h->dskip;
  }
  const void* xin = l == 0 ? h->layer_in : h->xout[l - 1];
  RET(block_backward<T>(h, st, l, xin, dxo_t, h->R, dsk_t, h->Sp, dx ? h->dxB : nullptr, h->R, B, Tn, 0.f, BlockBwdMode{}));
  if (dx) {
    LaunchScope ls(h, st, CLS_MISC);
    convert_kernel<T, float><<<cdiv(nR, 256), 256, 0, st>>>((const T*)h->dxB, dx, nR);
  }
  if (h->cond_seq) {
    const BlockP& b = h->blocks[l];
    const int n = 2 * h->D, Cc = h->Cc;
    // d Wc = sum_{b,t} c^T dz and d bc = column sums of dz: the sequence against the gate adjoint block_backward left in h->dz
    // (bf16: the contraction runs over the padded width, its first Cc rows are d Wc)
    WgradH w{};
    w.B = B; w.T = Tn; w.N = n; w.G = h->dz; w.ldg = n; w.nseg = 1; w.seg[0] = SegH{h->cond_seq, h->Ccs, 0, h->Ccs};
    w.dst = sizeof(T) == 2 ? h->cseq_dw : G_(h, b.cw_idx); w.w = P_(h, b.cw_idx); w.l2coef = 0.f; w.bias_dst = G_(h, b.cb_idx);
    RET(run_wgrad<T>(h, st, CLS_GEMM, w));
    if (sizeof(T) == 2) CK(cudaMemcpyAsync(G_(h, b.cw_idx), h->cseq_dw, (size_t)Cc * n * 4, cudaMemcpyDeviceToDevice, st));
    if (dcond) {
      // d cond = dz Wc^T (B,T,Cc), fp32 straight into the caller's buffer
      GemmH g;
      g.B = B; g.T = Tn; g.N = Cc; g.nseg = 1;
      g.seg[0] = SegH{h->dz, n, 0, n};
      g.W32 = b.Wct; g.Npad = b.Ccpad;
      g.W16 = b.Wct16; g.ktot16 = n; g.N16 = b.Cc16; g.tile16 = b.tileCc16;
      typename EpiBiasActRes<T, float, sizeof(T) == 2>::Params ep{};
      ep.out = dcond; ep.ldo = Cc; ep.bias = nullptr; ep.cbias = nullptr; ep.act = ACT_LINEAR; ep.res = nullptr; ep.N = Cc; ep.vec = vec_ok<float>(Cc);
      RET((run_conv_gemm<T, EpiBiasActRes<T, float, sizeof(T) == 2>>(h, st, CLS_GEMM, g, ep)));
    }
  } else if (h->blocks[l].has_cond) {
    RET(cond_backward(h, st, nullptr, h->last_cond, B, l, 1, false, h->dcond, 0.f));
    if (dcond) CK(cudaMemcpyAsync(dcond, h->dcond, (size_t)B * h->Cc * 4, cudaMemcpyDeviceToDevice, st));
  }
  return WN_OK;
}

extern "C" int wn_layer_backward(wn_handle* h, int block, const float* dx_out_dev, const float* dskip_dev, float* dx_dev, float* dcond_dev, void* stream) {
  if (!h) { set_err("null handle"); return WN_ERR_VALUE; }
  if (block < 0 || block >= h->L) { set_err("bad block index"); return WN_ERR_VALUE; }
  if (!h->layer_fwd_valid[block]) { set_err("wn_layer_backward before wn_layer_forward"); return WN_ERR_STATE; }
  if (!dx_out_dev && !dskip_dev) { set_err("need at least one upstream gradient"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  h->launches = 0;
  cudaStream_t st = (cudaStream_t)stream;
  int r = h->cfg.precision == WN_BF16 ? layer_bwd_entry<bf16>(h, block, dx_out_dev, dskip_dev, dx_dev, dcond_dev, st)
                                      : layer_bwd_entry<float>(h, block, dx_out_dev, dskip_dev, dx_dev, dcond_dev, st);
  h->drop_active = false;
  h->cond_seq = nullptr;
  RET(r);
  CK(cudaGetLastError());
  return WN_OK;
}

// ---------------------------------------------------------------- kernel-level test hooks (bf16 tier)
// Raw contractions of gemm_tc.cuh without a model around them, so tests can compare each
// tcgen05 mainloop against a plain torch fp32 matmul on the same bf16 inputs.
// Test hook: an intermediate tensor of the LAST step (wn_train_step / wn_forward), converted to fp32 on the host, rows = B*T of
// that step.  name: "h0" | "z" (l) | "g" (l) | "xout" (l) | "skipsum" | "hact" (i) | "logits" | "dlogits" | "dskip" |
// "dz" (l) | "dx" (l: d x_out of block l) — the last two only when the step kept them (grouped weight gradients).
// Returns the row width (columns copied per row), or a negative status.
extern "C" int wn_debug_tensor(wn_handle* h, const char* name, int index, float* out_host, int64_t capacity) {
  if (!h || !name || !out_host) { set_err("bad debug_tensor arguments"); return WN_ERR_VALUE; }
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  const long long rows = (long long)h->lastB * h->lastT;
  const size_t rows_cap = (size_t)h->maxB * h->maxT;
  const bool bf = h->cfg.precision == WN_BF16;
  const size_t es = bf ? 2 : 4;
  const std::string n(name);
  const void* src = nullptr; int width = 0, ld = 0; bool f32 = false;
  const bool lok = index >= 0 && index < h->L;
  if (n == "h0") { src = h->h0; width = ld = h->R; }
  else if (n == "z" && lok) { src = h->zbuf[index]; width = ld = 2 * h->D; }
  else if (n == "g" && lok) { src = (const char*)h->G_all + (size_t)index * rows_cap * h->D * es; width = ld = h->D; }
  else if (n == "xout" && lok) { src = h->xout[index]; width = ld = h->R; }
  else if (n == "skipsum") { src = h->skipsum; width = ld = h->Sp; }
  else if (n == "hact" && index >= 0 && index < (int)h->hact.size()) { src = h->hact[index]; width = ld = h->head[index].cout; }
  else if (n == "act" && index >= 0 && index / 16 < h->L && index % 16 < (int)h->acts[index / 16].size()) {   // output of pre-stack conv j of block l: index = 16 l + j
    src = h->acts[index / 16][index % 16]; width = ld = h->D;
  }
  else if (n == "logits") { src = h->logits; width = h->Cout; ld = h->ldl; f32 = true; }
  else if (n == "dlogits") { src = h->dlogits; width = h->Cout; ld = h->ldd; }
  else if (n == "dskip") { src = h->dskip; width = ld = h->Sp; }
  else if (n == "dz" && lok && h->dz_all) { src = (const char*)h->dz_all + (size_t)index * rows_cap * 2 * h->D * es; width = ld = 2 * h->D; }
  else if (n == "dx" && lok && h->dx_all) { src = (const char*)h->dx_all + (size_t)index * rows_cap * h->R * es; width = ld = h->R; }
  if (!src || rows < 1) { set_err("debug_tensor: no tensor '%s'[%d] in this handle / step", name, index); return WN_ERR_STATE; }
  if ((long long)capacity < rows * width) { set_err("debug_tensor: capacity %lld < %lld", (long long)capacity, rows * width); return WN_ERR_VALUE; }
  const size_t e2 = f32 ? 4 : es;
  std::vector<char> tmp((size_t)rows * ld * e2);
  CK(cudaMemcpy(tmp.data(), src, tmp.size(), cudaMemcpyDeviceToHost));
  for (long long r = 0; r < rows; ++r)
    for (int c = 0; c < width; ++c) {
      const char* p = tmp.data() + ((size_t)r * ld + c) * e2;
      float v;
      if (e2 == 4) memcpy(&v, p, 4);
      else { uint16_t u; memcpy(&u, p, 2); uint32_t w = (uint32_t)u << 16; memcpy(&v, &w, 4); }
      out_host[r * width + c] = v;
    }
  return width;
}

extern "C" int wn_debug_conv_gemm(const void* a_bf16_dev, int lda, int B, int T, int nseg, const int* shifts, int K, const void* w_bf16_dev, int N,
                                  int N16, int tile, float* out_dev, void* stream) {
  if (!a_bf16_dev || !w_bf16_dev || !out_dev || !shifts || nseg < 1 || nseg > TC_MAX_SEG) { set_err("bad debug gemm arguments"); return WN_ERR_VALUE; }
  if (tc_init() != 0) { set_err("cannot resolve cuTensorMapEncodeTiled from the driver"); return WN_ERR_CUDA; }
  static TmapCache cache;
  cache.maps.clear();
  TcGemmDesc d{};
  d.B = B; d.T = T; d.nseg = nseg; d.n_outer = 1; d.outer_stride = 0;
  for (int s = 0; s < nseg; ++s) d.seg[s] = TcSeg{(const bf16*)a_bf16_dev, lda, shifts[s], K};
  d.W = (const bf16*)w_bf16_dev; d.ktot = nseg * K; d.N16 = N16; d.tileN = tile;
  typedef EpiBiasActRes<bf16, float, true> E;
  E::Params ep{};
  ep.out = out_dev; ep.ldo = N; ep.act = ACT_LINEAR; ep.N = N; ep.vec = (N % 4) == 0;
  int r = tc_conv_gemm<E>(cache, (cudaStream_t)stream, d, ep);
  if (r != 0) { set_err("tcgen05 conv_gemm launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  return WN_OK;
}

extern "C" int wn_debug_wgrad(const void* a_bf16_dev, int lda, const void* g_bf16_dev, int ldg, int B, int T, int nseg, const int* shifts, int K, int N,
                              float* out_dev, void* stream) {
  if (!a_bf16_dev || !g_bf16_dev || !out_dev || !shifts || nseg < 1 || nseg > TC_MAX_SEG) { set_err("bad debug wgrad arguments"); return WN_ERR_VALUE; }
  if (tc_init() != 0) { set_err("cannot resolve cuTensorMapEncodeTiled from the driver"); return WN_ERR_CUDA; }
  static TmapCache cache;
  cache.maps.clear();
  cudaStream_t st = (cudaStream_t)stream;
  const long long kn = (long long)nseg * K * N;
  float* partial = nullptr;
  CK(cudaMalloc(&partial, (size_t)kn * WN_MAX_WGRAD_SPLITS * 4));
  TcWgradDesc d{};
  d.B = B; d.T = T; d.N = N; d.G = (const bf16*)g_bf16_dev; d.ldg = ldg; d.nseg = nseg; d.ktot = nseg * K; d.partial = partial;
  for (int s = 0; s < nseg; ++s) d.seg[s] = TcSeg{(const bf16*)a_bf16_dev, lda, shifts[s], K};
  d.cs_partial = nullptr;
  TcWgradPlan plan{};
  int r = tc_wgrad(cache, st, d, &plan);
  if (r != 0) { cudaFree(partial); set_err("tcgen05 wgrad launch failed (%d): %s", r, tc_last_error()); return WN_ERR_CUDA; }
  reduce_parts<<<cdiv(kn, 256), 256, 0, st>>>(partial, plan.nsplit, kn, out_dev, kn, nullptr, 0.f);
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(partial);
  CK(e);
  return WN_OK;
}

// micro-benchmark hook: `reps` back-to-back launches of one mainloop on caller buffers, CUDA-event timed.
// which: 0 = conv GEMM (bf16 out, no bias), 1 = wgrad (+finish), 2 = wgrad kernel alone
extern "C" int wn_debug_bench(int which, int reps, const void* a_bf16_dev, int lda, const void* g_or_w_bf16_dev, int ldg, int B, int T, int nseg,
                              const int* shifts, int K, int N, void* out_dev, int ldo, float* ms_out) {
  if (tc_init() != 0) { set_err("cannot resolve cuTensorMapEncodeTiled from the driver"); return WN_ERR_CUDA; }
  static TmapCache cache;
  cache.maps.clear();
  cudaStream_t st = nullptr;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  float* partial = nullptr;
  const long long kn = (long long)nseg * K * N;
  if (which >= 1) CK(cudaMalloc(&partial, (size_t)kn * WN_MAX_WGRAD_SPLITS * 4));
  int rc = 0;
  for (int it = -2; it < reps && rc == 0; ++it) {
    if (it == 0) cudaEventRecord(e0, st);
    if (which == 0) {
      TcGemmDesc d{};
      d.B = B; d.T = T; d.nseg = nseg; d.n_outer = 1;
      for (int s = 0; s < nseg; ++s) d.seg[s] = TcSeg{(const bf16*)a_bf16_dev, lda, shifts[s], K};
      d.W = (const bf16*)g_or_w_bf16_dev; d.ktot = nseg * K; d.N16 = N; d.tileN = 0;
      TcEpiBiasActRes<true>::Params q{nullptr, nullptr, 0, ACT_LINEAR, N};
      TcEpiIo in[2] = {{}, {}};
      TcEpiIo out[3] = {{(const bf16*)out_dev, ldo, N, 0}, {}, {}};
      rc = tc_conv_gemm_staged<TcEpiBiasActRes<true>>(cache, st, d, q, in, 0u, out);
    } else {
      TcWgradDesc d{};
      d.B = B; d.T = T; d.N = N; d.G = (const bf16*)g_or_w_bf16_dev; d.ldg = ldg; d.nseg = nseg; d.ktot = nseg * K; d.partial = partial;
      for (int s = 0; s < nseg; ++s) d.seg[s] = TcSeg{(const bf16*)a_bf16_dev, lda, shifts[s], K};
      TcWgradPlan plan{};
      rc = tc_wgrad(cache, st, d, &plan);
      if (rc == 0 && which == 1) reduce_parts<<<cdiv(kn, 256), 256, 0, st>>>(partial, plan.nsplit, kn, (float*)out_dev, kn, nullptr, 0.f);
    }
  }
  cudaEventRecord(e1, st);
  cudaError_t e = cudaStreamSynchronize(st);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  if (ms_out) *ms_out = ms / (reps > 0 ? reps : 1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (partial) cudaFree(partial);
  if (rc != 0) { set_err("debug bench launch failed (%d): %s", rc, tc_last_error()); return WN_ERR_CUDA; }
  CK(e);
  return WN_OK;
}

// ---------------------------------------------------------------- introspection
extern "C" int64_t wn_last_launch_count(const wn_handle* h) { return h ? h->launches : 0; }
// number of blocks whose gated conv + conv1 ran as ONE fused launch in the last enqueued forward (0 = separate kernels)
extern "C" int wn_fused_forward_blocks(const wn_handle* h) { return h ? h->fused_fwd_launches : 0; }
extern "C" int wn_stack_forward_layers(const wn_handle* h) { return h ? h->stack_fwd_layers : 0; }
extern "C" int wn_stack_backward_layers(const wn_handle* h) { return h ? h->stack_bwd_layers : 0; }
extern "C" int wn_allreduce_buckets(const wn_handle* h) { return h ? h->last_ar_buckets : 0; }
extern "C" int wn_grouped_wgrad_tiles(const wn_handle* h, int* side_launches) {
  if (side_launches) *side_launches = h ? h->wg_last_side : 0;
  return h ? h->wg_last_tiles : 0;
}
// grouped weight gradients of the last backward pass: output tiles, fp32 partial tiles the finish launch reads (tiles x row
// splits), side launches
extern "C" int wn_grouped_wgrad_info(const wn_handle* h, int* tiles, int* partial_tiles, int* side_launches) {
  if (!h) return WN_ERR_VALUE;
  if (tiles) *tiles = h->wg_last_tiles;
  if (side_launches) *side_launches = h->wg_last_side;
  if (partial_tiles) *partial_tiles = h->wg_last_partials;
  return WN_OK;
}
// per-launch record of the last wn_profile_end: returns the number of timed launches; i in [0,n): duration + label
extern "C" int wn_profile_get(wn_handle* h, int i, double* ms, char* label, int label_len) {
  if (!h) return WN_ERR_VALUE;
  if (i >= 0 && i < (int)h->prof_ms.size()) {
    if (ms) *ms = h->prof_ms[i];
    if (label && label_len > 0) snprintf(label, label_len, "%s", h->prof_last_labels[i] ? h->prof_last_labels[i] : "");
  }
  return (int)h->prof_ms.size();
}
extern "C" int wn_profile_begin(wn_handle* h, int tag) {
  if (!h) return WN_ERR_VALUE;
  h->prof_tag = tag; h->prof_used = 0; h->prof_launches = 0;
  return WN_OK;
}
extern "C" int wn_profile_end(wn_handle* h, double* ms, int64_t* launches) {
  if (!h) return WN_ERR_VALUE;
  CK(cudaDeviceSynchronize());
  double tot = 0;
  h->prof_ms.assign(h->prof_used, 0.f);
  h->prof_last_labels.assign(h->prof_labels.begin(), h->prof_labels.begin() + h->prof_used);
  for (size_t i = 0; i < h->prof_used; ++i) {
    float t = 0;
    cudaEventElapsedTime(&t, h->prof_events[i].first, h->prof_events[i].second);
    h->prof_ms[i] = t;
    tot += t;
  }
  if (ms) *ms = tot;
  if (launches) *launches = h->prof_launches;
  h->prof_tag = 0; h->prof_used = 0;
  return WN_OK;
}
