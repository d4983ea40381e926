// gemm_tc.cuh — bf16 tcgen05/TMEM/TMA mainloops (the throughput tier).
//
// Same two contractions as gemm_simt.cuh, re-designed for sm_100a:
//
//   tc_conv_gemm : out[(b,t), n] = sum_seg A_seg[(b, t+shift_seg), :] . W[n, kofs_seg + :]
//     The dilated causal conv is a dense contraction over the [x_{t-d}, x_t] channel concat
//     that is never materialised: each tap is its own TMA box of the SAME activation tensor,
//     fetched through a (C, T, B, slab) tensor map at time coordinate t0+shift.  Rows outside
//     [0,T) are out of bounds for the map and arrive as zeros: causal padding and batch
//     isolation cost nothing and are exact.  Persistent, warp-specialised CTA:
//       warp 0      TMA producer  (A box 128 rows x 64 ch, W box BN rows x 64 k; 128B swizzle)
//       warp 1      tcgen05.mma issuer (one elected lane; M=128, N=BN, K=16 per instruction)
//       warp 2      TMEM allocator (2 accumulator stages x BN fp32 columns)
//       warps 4..   epilogue: tcgen05.ld -> fused epilogue functor (epilogues.cuh) -> HBM
//     smem ring full/empty mbarriers (TMA <-> MMA), TMEM full/empty mbarriers (MMA <-> epilogue),
//     so the epilogue of tile i overlaps the mainloop of tile i+1.
//
//   tc_wgrad : dW[kofs_seg + c, n] = sum_{b,t} A_seg[(b, t+shift_seg), c] * G[(b,t), n]
//     Time is the contraction dimension, so both operands are MN-major straight from their
//     (B,T,C) layout (no transposes): A box = 64 time rows x 64 channels.  Split over row ranges;
//     fp32 partials reduced by a second deterministic kernel (no atomics).
#pragma once
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"
#include "tc_epilogues.cuh"

#define WN_MAX_WGRAD_SPLITS 64
#define TC_MAX_TAPS 4
// + 1: the gated conv of a layer called with a conditioning sequence contracts it as one more segment (shift 0)
#define TC_MAX_SEG (TC_MAX_TAPS + 1)

struct TcSeg { const bf16* A; int lda; int shift; int K; };
// L2 policy per tensor of a launch: 0 = normal, 1 = evict_first (streaming), 2 = evict_last (the next kernel reads it)
enum { TC_L2_NORMAL = 0, TC_L2_FIRST = 1, TC_L2_LAST = 2 };
static inline unsigned long long tc_policy(int code) {
  return code == TC_L2_FIRST ? TC_POL_FIRST : (code == TC_L2_LAST ? TC_POL_LAST : TC_POL_NORMAL);
}
struct TcGemmDesc {
  int B, T, nseg; TcSeg seg[TC_MAX_SEG]; int n_outer; long long outer_stride;
  const bf16* W; int ktot; int N16; int tileN;
  int l2_a = 0, l2_in[2] = {0, 0}, l2_out[3] = {0, 0, 0};   // TC_L2_* codes: activation operand, epilogue inputs, outputs
  int l2_seg[TC_MAX_SEG] = {-1, -1, -1, -1, -1};            // per-segment override of l2_a (-1: none)
};
struct TcWgradDesc {
  int l2_a = 0, l2_g = 0;
  int B, T, N; const bf16* G; int ldg; int nseg; TcSeg seg[TC_MAX_SEG]; int ktot; float* partial;
  float* cs_partial;   // optional: per-(split, batch slot) column sums of G, [nsplit][slots][N] (bias / conditioning gradients)
};
struct TcWgradPlan { int nsplit, chunks_per_split, chunks_t, slots, mtiles; };

// Channel widths: multiples of 32 (the reference's default width, defaults.yaml:10).  A 64-channel k-block of a narrower
// tensor is padded in SHARED memory, not in HBM: the TMA box reaches past the tensor's channel extent and the out-of-bounds
// half arrives as zeros (same mechanism as the causal padding in time); the weight box of the same k-block then also covers
// the next tap's rows, which meet those zeros.  Output panels are 32 columns wide.
static inline int tc_check_config(int R, int D, int S, int K) {
  if (R % 32 || D % 32 || S % 32) return -1;
  if (K > TC_MAX_TAPS) return -2;
  return 0;
}
// column tiling of an N-wide output: N16 = padded width, tile = CTA tile width (64/128/256).
// gate == true: n = 2D and a tile must hold matching filter and gate halves (tile/2 | D).
static inline void tc_pick_tile(int n, bool gate, int* n16, int* tile) {
  int t;
  if (gate) t = ((n / 2) % 128 == 0) ? 256 : 128;
  else t = n > 128 ? 256 : (n > 64 ? 128 : 64);
  *tile = t;
  *n16 = (n + t - 1) / t * t;
}

// ---------------------------------------------------------------- gate weight pack (transposed + interleaved)
// dst[n'][k] = W[k][src(n')] : tile-interleaved columns [filter ch0.. | gate ch0..) per tile of width `tile`
__global__ void tc_pack_gate_T_kernel(const float* __restrict__ src, int ktot, int cout, bf16* __restrict__ dst, int ld, int tile, int D, int n16) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n16 * ktot) return;
  const int np = (int)(i / ktot), k = (int)(i % ktot);
  const int half = tile >> 1;
  const int ti = np / tile, j = np % tile;
  const int ch = ti * half + (j % half);
  float v = 0.f;
  if (ch < D) v = src[(long long)k * cout + (j < half ? ch : D + ch)];
  dst[(long long)np * ld + k] = __float2bfloat16_rn(v);
}
static inline void tc_pack_gate_T(cudaStream_t st, const float* src, int ktot, int cout, bf16* dst, int ld, int tile, int D, int n16) {
  const long long total = (long long)n16 * ktot;
  tc_pack_gate_T_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, ktot, cout, dst, ld, tile, D, n16);
}

// cluster shape + programmatic dependent launch of the GEMM-class kernels
static inline int tc_launch_attrs(cudaLaunchAttribute* attr, int cluster) {
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  return 2;
}

// ---------------------------------------------------------------- conv GEMM kernel
struct TcGemmParams {
  int B, T;
  int tiles_t;      // ceil(T / 128)
  int n_tiles;      // N16 / BN
  int num_tiles;    // B * tiles_t * n_tiles
  int nseg;
  int segK[TC_MAX_SEG];
  int segShift[TC_MAX_SEG];
  int n_outer;
};

template <int BN> struct TcGemmCfg {
  static constexpr int BM = 128, BK = 64;
  static constexpr int A_BYTES = BM * BK * 2;           // 16 KB
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN == 256) ? 4 : 6;
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <class Epi, int BN, int NEPI>
__global__ void __launch_bounds__(128 + 32 * NEPI, 1)
tc_conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                    const __grid_constant__ CUtensorMap tmA3, const __grid_constant__ CUtensorMap tmA4, const __grid_constant__ CUtensorMap tmW, const TcGemmParams p,
                    const typename Epi::Params ep) {
  using Cfg = TcGemmCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_ptr = (uint32_t*)(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    if (p.nseg > 1) tma_prefetch_desc(&tmA1);
    if (p.nseg > 2) tma_prefetch_desc(&tmA2);
    if (p.nseg > 3) tma_prefetch_desc(&tmA3);
    if (p.nseg > 4) tma_prefetch_desc(&tmA4);
    tma_prefetch_desc(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], NEPI); }
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
        const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * Cfg::BM, n0 = nt * BN;
        int wk = 0;
        for (int o = 0; o < p.n_outer; ++o) {
          for (int s = 0; s < p.nseg; ++s) {
            const CUtensorMap* tm = s == 0 ? &tmA0 : (s == 1 ? &tmA1 : (s == 2 ? &tmA2 : (s == 3 ? &tmA3 : &tmA4)));
            const int kseg = p.segK[s], tcoord = t0 + p.segShift[s];
            for (int k0 = 0; k0 < kseg; k0 += Cfg::BK) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
              tma_load_4d(sa, tm, &full_bar[stage], k0, tcoord, b, o);
              tma_load_2d(sa + Cfg::A_BYTES, &tmW, &full_bar[stage], wk + k0, n0);
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            wk += kseg;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = umma_idesc_bf16(128, BN, 0, 0);
    int stage = 0; uint32_t phase = 0;
    int as = 0; uint32_t aphase = 0;
    int ksteps = 0;
    for (int s = 0; s < p.nseg; ++s) ksteps += (p.segK[s] + Cfg::BK - 1) / Cfg::BK;
    ksteps *= p.n_outer;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[as], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
      for (int ks = 0; ks < ksteps; ++ks) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t adesc = umma_smem_desc(sa, 16, 1024);
          const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES, 16, 1024);
#pragma unroll
          for (int k = 0; k < Cfg::BK / 16; ++k)   // +32 bytes (>>4 = 2) per K=16 step inside the 128B swizzle row
            umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (ks | k) != 0);
          umma_commit(&empty_bar[stage]);
          if (ks == ksteps - 1) umma_commit(&tfull_bar[as]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int e = warp - 4;
    const int quarter = warp & 3;            // TMEM lane quarter this warp may access
    const int q = e >> 2;                    // column-chunk phase when NEPI == 8
    constexpr int nq = NEPI / 4;
    int as = 0; uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
      const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * Cfg::BM, n0 = nt * BN;
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const int t = t0 + quarter * 32 + lane;
      TmemAccRow acc{tmem_base + (uint32_t)(as * BN) + ((uint32_t)(quarter * 32) << 16), t < p.T};
      Epi::row(ep, acc, b, (long long)b * p.T + (t < p.T ? t : 0), n0, BN, q, nq);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

static int g_tc_num_sms = 0;
static inline int tc_num_sms() {
  if (g_tc_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_tc_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_tc_num_sms <= 0) g_tc_num_sms = 148;
  }
  return g_tc_num_sms;
}

// activation operand map: (C = K channels, T, B, slabs) with box (64, rows, 1, 1)
static inline const CUtensorMap* tc_act_map(TmapCache& tc, const bf16* A, int lda, int K, int T, int B, int n_outer, long long outer_stride,
                                            int box_rows) {
  uint64_t dims[4] = {(uint64_t)K, (uint64_t)T, (uint64_t)B, (uint64_t)(n_outer > 0 ? n_outer : 1)};
  uint64_t str[3] = {(uint64_t)lda * 2, (uint64_t)T * lda * 2, (uint64_t)(n_outer > 1 ? outer_stride * 2 : (long long)B * T * lda * 2)};
  uint32_t box[4] = {64, (uint32_t)box_rows, 1, 1};
  return tc.get(A, 4, dims, str, box);
}

// the same tensor seen as 64-channel atoms: (64 ch, T, C/64 atoms, B) with box (64, rows, atoms, 1).  One TMA op then
// fills `atoms` consecutive [rows][128 B] slabs (8 KB apart for 64 rows) = the MN-major operand layout of the wgrad,
// instead of one op per atom: a TMA issue costs the producer thread ~150-200 cycles (timeline, profiles/README.md)
static inline const CUtensorMap* tc_atom_map(TmapCache& tc, const bf16* A, int lda, int K, int T, int B, int box_rows, int atoms) {
  uint64_t dims[4] = {64, (uint64_t)T, (uint64_t)(K / 64), (uint64_t)B};
  uint64_t str[3] = {(uint64_t)lda * 2, 128, (uint64_t)T * lda * 2};
  uint32_t box[4] = {64, (uint32_t)box_rows, (uint32_t)atoms, 1};
  return tc.get(A, 4, dims, str, box);
}

// Persistent kernels walk their tiles round-robin: with 256 tiles on 74 CTA pairs the last of 4 rounds keeps 34 pairs busy.
// The same 4 rounds fit on 64 pairs; the SMs left over can run other work (the side-stream weight gradients) meanwhile.
// g_tc_balance: 0 = always the whole GPU, 1 = the fewest CTAs (pairs) that keep the number of rounds.
// The switch belongs to the pass a host thread is enqueuing (set by a TcBalanceScope around the backward chain), so it is per
// thread: handles driven from different threads do not see each other's setting.
static thread_local int g_tc_balance = 0;
static inline int tc_balanced_slots(int tiles, int slots) {
  if (!g_tc_balance || tiles <= slots) return slots;
  const int rounds = (tiles + slots - 1) / slots;
  return (tiles + rounds - 1) / rounds;
}
// sets the switch for one phase of a pass; every exit of the phase, an error return too, restores the whole GPU
struct TcBalanceScope {
  explicit TcBalanceScope(bool on) { g_tc_balance = on ? 1 : 0; }
  ~TcBalanceScope() { g_tc_balance = 0; }
};

template <class Epi, int BN, int NEPI>
static int tc_conv_gemm_launch(TmapCache& tc, cudaStream_t st, const TcGemmDesc& d, const typename Epi::Params& ep) {
  using Cfg = TcGemmCfg<BN>;
  const CUtensorMap* ma[TC_MAX_SEG] = {};
  for (int s = 0; s < d.nseg; ++s) {
    ma[s] = tc_act_map(tc, d.seg[s].A, d.seg[s].lda, d.seg[s].K, d.T, d.B, s == 0 ? d.n_outer : 1, d.outer_stride, 128);
    if (!ma[s]) return -10;
  }
  for (int s = d.nseg; s < TC_MAX_SEG; ++s) ma[s] = ma[0];
  uint64_t wd[2] = {(uint64_t)d.ktot, (uint64_t)d.N16};
  uint64_t ws[1] = {(uint64_t)d.ktot * 2};
  uint32_t wb[2] = {64, (uint32_t)BN};
  const CUtensorMap* mw = tc.get(d.W, 2, wd, ws, wb);
  if (!mw) return -11;
  TcGemmParams p{};
  p.B = d.B; p.T = d.T; p.tiles_t = (d.T + 127) / 128; p.n_tiles = d.N16 / BN; p.num_tiles = d.B * p.tiles_t * p.n_tiles;
  p.nseg = d.nseg; p.n_outer = d.n_outer > 0 ? d.n_outer : 1;
  for (int s = 0; s < d.nseg; ++s) { p.segK[s] = d.seg[s].K; p.segShift[s] = d.seg[s].shift; }
  auto kern = tc_conv_gemm_kernel<Epi, BN, NEPI>;
  static unsigned long long attr_devs = 0ull;   // per template instantiation
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  const int grid = p.num_tiles < tc_num_sms() ? p.num_tiles : tc_num_sms();
  kern<<<grid, 128 + 32 * NEPI, Cfg::SMEM_BYTES, st>>>(*ma[0], *ma[1], *ma[2], *ma[3], *ma[4], *mw, p, ep);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "conv_gemm launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

template <class Epi> static int tc_conv_gemm(TmapCache& tc, cudaStream_t st, const TcGemmDesc& d, const typename Epi::Params& ep) {
  int tile = d.tileN;
  if (tile == 0) tile = d.N16 % 256 == 0 ? 256 : (d.N16 % 128 == 0 ? 128 : 64);
  if (d.N16 % tile != 0 || d.nseg < 1 || d.nseg > TC_MAX_SEG) { snprintf(g_tc_err, sizeof(g_tc_err), "bad tiling N16=%d tile=%d nseg=%d", d.N16, tile, d.nseg); return -1; }
  constexpr int NEPI = Epi::kHeavy ? 8 : 4;
  switch (tile) {
    case 256: return tc_conv_gemm_launch<Epi, 256, NEPI>(tc, st, d, ep);
    case 128: return tc_conv_gemm_launch<Epi, 128, NEPI>(tc, st, d, ep);
    case 64: return tc_conv_gemm_launch<Epi, 64, NEPI>(tc, st, d, ep);
  }
  return -2;
}

// ---------------------------------------------------------------- conv GEMM kernel, TMA-staged epilogue
// Same mainloop; the epilogue moves every HBM tensor through shared memory (tc_epilogues.cuh):
//   warp 3      epilogue-input producer: TMA loads of 128x32 half-panels (residual / cached z / ...)
//   warps 4..11 epilogue: tcgen05.ld -> functor -> bf16 -> swizzled st.shared; one thread issues the
//               TMA stores (bulk async groups, double-buffered output slots, one named barrier per step)
struct TcEpiIo { const bf16* base; int ld; int C; int col_off; };
struct TcStagedParams {
  uint32_t in_mask;
  int in_col[2];
  int out_col[3];
  unsigned long long pol_a, pol_w, pol_in[2], pol_out[3];   // L2 cache policies (TC_POL_*)
  unsigned long long pol_seg[TC_MAX_SEG];                    // per-segment policy of the activation operand
};

// IN_PANELS: capacity of the epilogue-input ring in half-panels (slots = IN_PANELS / active inputs, decided at
// run time); OUT_SLOTS: output slots of NOUT half-panels each.
// CTA pairs (cta_group::2): a pair works on 256 rows x BN columns; each CTA stages its own 128 rows of A and HALF
// of the W tile, so one k-step moves 32 KB per SM instead of 48 KB for the same FLOPs (the conv GEMMs at
// cta_group::1 top out on L2 -> SM bandwidth, profiles/README.md).
template <int BN, int NIN, int NOUT, int IN_PANELS, int OUT_SLOTS_> struct TcStagedCfg {
  static constexpr int BM = 128, BK = 64;
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = (BN / 2) * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int PANEL = 128 * 64;                 // 128 rows x 32 bf16
  static constexpr int IN_MAX = IN_PANELS > 0 ? IN_PANELS : 1, OUT_SLOTS = OUT_SLOTS_;
  static constexpr int STAGING = (IN_PANELS + OUT_SLOTS * NOUT) * PANEL;
  static constexpr int MAX_SMEM = 232448;
  static constexpr int ST0 = (MAX_SMEM - 4096 - STAGING) / STAGE_BYTES;
  static constexpr int STAGES = ST0 > 6 ? 6 : ST0;
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING + 1024 + 512 + 2048 /*bias tables (double-buffered)*/;
  static_assert(STAGES >= 2, "not enough shared memory for the mainloop ring");
};

template <class Epi, int BN>
__global__ void __launch_bounds__(384, 1)
tc_conv_gemm_staged_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                           const __grid_constant__ CUtensorMap tmA3, const __grid_constant__ CUtensorMap tmA4, const __grid_constant__ CUtensorMap tmW,
                           const __grid_constant__ CUtensorMap tmI0, const __grid_constant__ CUtensorMap tmI1,
                           const __grid_constant__ CUtensorMap tmO0, const __grid_constant__ CUtensorMap tmO1, const __grid_constant__ CUtensorMap tmO2,
                           const TcGemmParams p, const TcStagedParams sp, const typename Epi::Params ep) {
  constexpr int NIN = Epi::NIN, NOUT = Epi::NOUT;
  using Cfg = TcStagedCfg<BN, NIN, NOUT, Epi::kInPanels, Epi::kOutSlots>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int NEPI = 8;
  constexpr int STEPS = Epi::kGate ? BN / 64 : BN / 32;   // 32 output columns per step
  // CTA pair: rank 0 leads (issues the MMAs, owns the barriers the pair synchronises on)
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int tile_first = (int)blockIdx.x / 2, tile_stride = (int)gridDim.x / 2;
  const int pair_row0 = (int)crank * Cfg::BM;     // first row of this CTA inside the pair's 256-row tile
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* in_ring = smem + STAGES * Cfg::STAGE_BYTES;
  uint8_t* out_ring = in_ring + Epi::kInPanels * Cfg::PANEL;
  uint64_t* full_bar = (uint64_t*)(out_ring + Cfg::OUT_SLOTS * NOUT * Cfg::PANEL);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* in_full = tempty_bar + 2;
  uint64_t* in_empty = in_full + Cfg::IN_MAX;
  uint64_t* out_empty = in_empty + Cfg::IN_MAX;          // output slot has been read by its TMA stores
  uint32_t* tmem_ptr = (uint32_t*)(out_empty + Cfg::OUT_SLOTS);
  float* bias_s = (float*)(((uintptr_t)(tmem_ptr + 4) + 15) & ~(uintptr_t)15);   // per-tile bias table (<= 256 floats)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool use_in = NIN > 0 && sp.in_mask != 0;
  // active inputs are packed densely: slot = nact consecutive half-panels, so fewer inputs => a deeper ring
  const int nact = NIN > 0 ? __popc(sp.in_mask) : 0;
  const int in_slots = nact > 0 ? Epi::kInPanels / nact : 1;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA0);
    if (p.nseg > 1) tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmO0);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], NEPI * 2); }
    for (int i = 0; i < Cfg::IN_MAX; ++i) { mbar_init(&in_full[i], 1); mbar_init(&in_empty[i], NEPI); }
    for (int i = 0; i < Cfg::OUT_SLOTS; ++i) mbar_init(&out_empty[i], 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc_pair<Cfg::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // the peer's barriers are initialised before anything is signalled across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // everything above touched only shared memory / TMEM; global data of the previous kernel is read below
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer (mainloop operands) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = tile_first; tile < p.num_tiles; tile += tile_stride) {
        const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
        const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (Cfg::BM * 2) + pair_row0, n0 = nt * BN;
        int wk = 0;
        for (int o = 0; o < p.n_outer; ++o) {
          for (int s = 0; s < p.nseg; ++s) {
            const CUtensorMap* tm = s == 0 ? &tmA0 : (s == 1 ? &tmA1 : (s == 2 ? &tmA2 : (s == 3 ? &tmA3 : &tmA4)));
            const int kseg = p.segK[s], tcoord = t0 + p.segShift[s];
            const unsigned long long pol_as = sp.pol_seg[s];
            for (int k0 = 0; k0 < kseg; k0 += Cfg::BK) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              // the leader's barrier counts the bytes of both CTAs' operand halves
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
              tma_load_4d_pair_h(sa, tm, &full_bar[stage], k0, tcoord, b, o, pol_as);
              tma_load_2d_pair_h(sa + Cfg::A_BYTES, &tmW, &full_bar[stage], wk + k0, n0 + (int)crank * (BN / 2), sp.pol_w);
              if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            wk += kseg;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA of a pair only) =====================
    constexpr uint32_t idesc = umma_idesc_bf16(256, BN, 0, 0);
    if (leader) {
    int stage = 0; uint32_t phase = 0;
    int as = 0; uint32_t aphase = 0;
    int ksteps = 0;
    for (int s = 0; s < p.nseg; ++s) ksteps += (p.segK[s] + Cfg::BK - 1) / Cfg::BK;
    ksteps *= p.n_outer;
#ifdef TC_TIMELINE
    long long tl_m[8][3]; int tl_mi = 0;
#endif
    for (int tile = tile_first; tile < p.num_tiles; tile += tile_stride) {
#ifdef TC_TIMELINE
      const long long tl_a = clock64();
#endif
      mbar_wait(&tempty_bar[as], aphase ^ 1);
      tc_fence_after();
#ifdef TC_TIMELINE
      const long long tl_b = clock64();
#endif
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
      for (int ks = 0; ks < ksteps; ++ks) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t adesc = umma_smem_desc(sa, 16, 1024);
          const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES, 16, 1024);
#pragma unroll
          for (int k = 0; k < Cfg::BK / 16; ++k)
            umma_bf16_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (ks | k) != 0);
          umma_commit_pair(&empty_bar[stage]);
          if (ks == ksteps - 1) umma_commit_pair(&tfull_bar[as]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
#ifdef TC_TIMELINE
      if (tl_mi < 8) { tl_m[tl_mi][0] = tl_a; tl_m[tl_mi][1] = tl_b; tl_m[tl_mi][2] = clock64(); ++tl_mi; }
#endif
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
#ifdef TC_TIMELINE
    if (blockIdx.x == 0 && lane == 0)
      for (int i = 0; i < tl_mi; ++i) printf("MMA tile %d: wait_tempty %lld issue %lld (t0 %lld)\n", i, tl_m[i][1] - tl_m[i][0], tl_m[i][2] - tl_m[i][1], tl_m[i][0] - tl_m[0][0]);
#endif
    }
  } else if (warp == 2) {
    // ===================== output store warp =====================
    // waits for the 8 epilogue warps to fill an output slot (named barrier per slot), issues its TMA stores, and
    // frees the slot of the previous step once those stores have read shared memory
    int oslot = 0, prev = -1;
    for (int tile = tile_first; tile < p.num_tiles; tile += tile_stride) {
      const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
      const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (Cfg::BM * 2) + pair_row0;
      const int tile_col0 = Epi::kGate ? nt * (BN / 2) : nt * BN;
#pragma unroll 1
      for (int step = 0; step < STEPS; ++step) {
        const int col0 = tile_col0 + step * 32;
        named_bar_sync(3 + oslot, NEPI * 32 + 32);
        if (lane == 0) {
          const uint8_t* ob = out_ring + oslot * NOUT * Cfg::PANEL;
          tma_store_3d_h(ob, &tmO0, sp.out_col[0] + col0, t0, b, sp.pol_out[0]);
          if (NOUT > 1) tma_store_3d_h(ob + Cfg::PANEL, &tmO1, sp.out_col[1] + col0, t0, b, sp.pol_out[1]);
          if (NOUT > 2) tma_store_3d_h(ob + 2 * Cfg::PANEL, &tmO2, sp.out_col[2] + col0, t0, b, sp.pol_out[2]);
          bulk_commit_group();
          if (prev >= 0) { bulk_wait_group_read<1>(); mbar_arrive(&out_empty[prev]); }
          prev = oslot;
        }
        __syncwarp();
        if (++oslot == Cfg::OUT_SLOTS) oslot = 0;
      }
    }
    if (lane == 0) bulk_wait_group<0>();
  } else if (warp == 3) {
    // ===================== epilogue-input producer =====================
    if (NIN > 0 && use_in && lane == 0) {
      int islot = 0; uint32_t iphase = 0;
      for (int tile = tile_first; tile < p.num_tiles; tile += tile_stride) {
        const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
        const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (Cfg::BM * 2) + pair_row0;
        const int tile_col0 = Epi::kGate ? nt * (BN / 2) : nt * BN;
        for (int step = 0; step < STEPS; ++step) {
          mbar_wait(&in_empty[islot], iphase ^ 1);
          mbar_expect_tx(&in_full[islot], (uint32_t)(nact * Cfg::PANEL));
          uint8_t* dst = in_ring + islot * nact * Cfg::PANEL;
          if (sp.in_mask & 1u) { tma_load_3d_h(dst, &tmI0, &in_full[islot], sp.in_col[0] + tile_col0 + step * 32, t0, b, sp.pol_in[0]); dst += Cfg::PANEL; }
          if (NIN > 1 && (sp.in_mask & 2u)) tma_load_3d_h(dst, &tmI1, &in_full[islot], sp.in_col[1] + tile_col0 + step * 32, t0, b, sp.pol_in[1]);
          if (++islot == in_slots) { islot = 0; iphase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int e = warp - 4;
    const int quarter = warp & 3;
    const int q = e >> 2;                         // which 16-column chunk of the 32-column step
    const int row = quarter * 32 + lane;          // TMEM lane == tile row
    const uint32_t row_off = (uint32_t)row * 64u;
    const uint32_t sw = (uint32_t)((row >> 1) & 3);
    const uint32_t u0 = (uint32_t)(2 * q), u1 = u0 + 1;   // 16-byte units of this chunk inside the 64-byte row
    const uint32_t off0 = row_off + ((u0 ^ sw) << 4), off1 = row_off + ((u1 ^ sw) << 4);
    int as = 0; uint32_t aphase = 0;
    int islot = 0; uint32_t iphase = 0;
    int oslot = 0; uint32_t ophase = 0;
#ifdef TC_TIMELINE
    long long tl_e[8][3]; int tl_ei = 0;
#endif
    for (int tile = tile_first; tile < p.num_tiles; tile += tile_stride) {
#ifdef TC_TIMELINE
      const long long tl_a = clock64();
#endif
      const int nt = tile % p.n_tiles, mt = tile / p.n_tiles;
      const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (Cfg::BM * 2) + pair_row0;
      const int tile_col0 = Epi::kGate ? nt * (BN / 2) : nt * BN;
      const int bsafe = b < p.B ? b : p.B - 1;
      constexpr int NBIAS = Epi::kBiasFloats(BN);
      float bias_reg = 0.f;
      if (NBIAS > 0 && (int)threadIdx.x - 128 < NBIAS) bias_reg = Epi::bias_load(ep, bsafe, tile_col0, BN, (int)threadIdx.x - 128);
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
#ifdef TC_TIMELINE
      const long long tl_b = clock64();
#endif
      // table double-buffered by tile parity: since the TMA-store warp took over, the epilogue warps only meet at this
      // barrier (once per tile), so a warp running ahead must not overwrite entries the others still read
      float* const bs = bias_s + as * 256;
      if (NBIAS > 0) {
        if ((int)threadIdx.x - 128 < NBIAS) bs[threadIdx.x - 128] = bias_reg;
        named_bar_sync(2, NEPI * 32);
      }
      TmemAccRow acc{tmem_base + (uint32_t)(as * BN) + ((uint32_t)(quarter * 32) << 16), true};
#ifdef TC_TIMELINE
      long long ph[6] = {0, 0, 0, 0, 0, 0};
#define TL_MARK(i) { const long long tl_now = clock64(); ph[i] += tl_now - tl_prev; tl_prev = tl_now; }
      long long tl_prev = clock64();
#else
#define TL_MARK(i)
#endif
#pragma unroll 1
      for (int step = 0; step < STEPS; ++step) {
        const int col0 = tile_col0 + step * 32;
        float in[NIN > 0 ? NIN : 1][16];
        float out[NOUT][16];
        if (NIN > 0 && use_in) {
          mbar_wait(&in_full[islot], iphase);
          const uint8_t* ib = in_ring + islot * nact * Cfg::PANEL;
#pragma unroll
          for (int k = 0; k < NIN; ++k) {
            if ((sp.in_mask >> k) & 1u) {
              const uint4 a = *reinterpret_cast<const uint4*>(ib + off0);
              const uint4 c = *reinterpret_cast<const uint4*>(ib + off1);
              ib += Cfg::PANEL;
              const uint32_t w[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                in[k][2 * j] = __uint_as_float(w[j] << 16);
                in[k][2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&in_empty[islot]);
          if (++islot == in_slots) { islot = 0; iphase ^= 1; }
        }
        TL_MARK(0)
        Epi::chunk(ep, acc, bsafe, step * 32 + q * 16, BN / 2, col0 + q * 16, sp.in_mask, in, out, bs);
        TL_MARK(1)
        uint8_t* ob = out_ring + oslot * NOUT * Cfg::PANEL;
        mbar_wait(&out_empty[oslot], ophase ^ 1);     // the TMA stores of this slot's previous use have read it
#pragma unroll
        for (int k = 0; k < NOUT; ++k) {
          uint4 a, c;
          a.x = pack_bf16x2(out[k][0], out[k][1]); a.y = pack_bf16x2(out[k][2], out[k][3]);
          a.z = pack_bf16x2(out[k][4], out[k][5]); a.w = pack_bf16x2(out[k][6], out[k][7]);
          c.x = pack_bf16x2(out[k][8], out[k][9]); c.y = pack_bf16x2(out[k][10], out[k][11]);
          c.z = pack_bf16x2(out[k][12], out[k][13]); c.w = pack_bf16x2(out[k][14], out[k][15]);
          *reinterpret_cast<uint4*>(ob + k * Cfg::PANEL + off0) = a;
          *reinterpret_cast<uint4*>(ob + k * Cfg::PANEL + off1) = c;
        }
        fence_proxy_async();
        TL_MARK(2)
        // hand the slot to the store warp (warp 2) and move on: no epilogue thread waits for TMA issue or read-back
        named_bar_arrive(3 + oslot, NEPI * 32 + 32);
        TL_MARK(3)
        TL_MARK(4)
        TL_MARK(5)
        if (++oslot == Cfg::OUT_SLOTS) { oslot = 0; ophase ^= 1; }
      }
#ifdef TC_TIMELINE
      if (blockIdx.x == 0 && (threadIdx.x == 128 || threadIdx.x == 320) && tl_ei >= 2 && tl_ei < 4)
        printf("  EPI phases thr %d tile %d: in %lld chunk %lld pack+sts+fence %lld wait_read %lld bar %lld tma %lld\n", threadIdx.x, tl_ei, ph[0], ph[1], ph[2],
               ph[3], ph[4], ph[5]);
      if (tl_ei < 8) { tl_e[tl_ei][0] = tl_a; tl_e[tl_ei][1] = tl_b; tl_e[tl_ei][2] = clock64(); ++tl_ei; }
#endif
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_relaxed(&tempty_bar[as], 0u);      // the leader's MMA warp waits for both CTAs' epilogues
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
#ifdef TC_TIMELINE
    if (blockIdx.x == 0 && threadIdx.x == 128)
      for (int i = 0; i < tl_ei; ++i) printf("EPI tile %d: wait_tfull %lld work %lld (t0 %lld)\n", i, tl_e[i][1] - tl_e[i][0], tl_e[i][2] - tl_e[i][1], tl_e[i][0] - tl_e[0][0]);
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();       // nobody leaves (or frees TMEM) while the pair may still signal / read
  if (warp == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
}

// half-panel map over a (B,T,ld) bf16 tensor restricted to C columns: box (32 cols, 128 rows, 1), 64B swizzle
static inline const CUtensorMap* tc_panel_map(TmapCache& tc, const TcEpiIo& io, int T, int B) {
  uint64_t dims[3] = {(uint64_t)io.C, (uint64_t)T, (uint64_t)B};
  uint64_t str[2] = {(uint64_t)io.ld * 2, (uint64_t)T * io.ld * 2};
  uint32_t box[3] = {32, 128, 1};
  return tc.get(io.base, 3, dims, str, box, 64);
}

template <class Epi, int BN>
static int tc_conv_gemm_staged_launch(TmapCache& tc, cudaStream_t st, const TcGemmDesc& d, const typename Epi::Params& ep, const TcEpiIo* ins,
                                      uint32_t in_mask, const TcEpiIo* outs) {
  using Cfg = TcStagedCfg<BN, Epi::NIN, Epi::NOUT, Epi::kInPanels, Epi::kOutSlots>;
  const CUtensorMap* ma[TC_MAX_SEG] = {};
  for (int s = 0; s < d.nseg; ++s) {
    ma[s] = tc_act_map(tc, d.seg[s].A, d.seg[s].lda, d.seg[s].K, d.T, d.B, s == 0 ? d.n_outer : 1, d.outer_stride, 128);
    if (!ma[s]) return -10;
  }
  for (int s = d.nseg; s < TC_MAX_SEG; ++s) ma[s] = ma[0];
  uint64_t wd[2] = {(uint64_t)d.ktot, (uint64_t)d.N16};
  uint64_t ws[1] = {(uint64_t)d.ktot * 2};
  uint32_t wb[2] = {64, (uint32_t)(BN / 2)};
  const CUtensorMap* mw = tc.get(d.W, 2, wd, ws, wb);
  if (!mw) return -11;
  TcStagedParams sp{};
  sp.in_mask = in_mask;
  sp.pol_a = tc_policy(d.l2_a); sp.pol_w = tc_policy(TC_L2_LAST);
  for (int s = 0; s < TC_MAX_SEG; ++s) sp.pol_seg[s] = tc_policy(d.l2_seg[s] >= 0 ? d.l2_seg[s] : d.l2_a);      // weights: every CTA re-reads them all kernel long
  for (int k = 0; k < 2; ++k) sp.pol_in[k] = tc_policy(d.l2_in[k]);
  for (int k = 0; k < 3; ++k) sp.pol_out[k] = tc_policy(d.l2_out[k]);
  const CUtensorMap* mo[3] = {nullptr, nullptr, nullptr};
  const CUtensorMap* mi[2] = {nullptr, nullptr};
  for (int k = 0; k < Epi::NOUT; ++k) {
    mo[k] = tc_panel_map(tc, outs[k], d.T, d.B);
    if (!mo[k]) return -14;
    sp.out_col[k] = outs[k].col_off;
  }
  for (int k = Epi::NOUT; k < 3; ++k) mo[k] = mo[0];
  for (int k = 0; k < Epi::NIN; ++k) {
    if ((in_mask >> k) & 1u) {
      mi[k] = tc_panel_map(tc, ins[k], d.T, d.B);
      if (!mi[k]) return -15;
      sp.in_col[k] = ins[k].col_off;
    }
  }
  for (int k = 0; k < 2; ++k) if (!mi[k]) mi[k] = mo[0];
  TcGemmParams p{};
  p.B = d.B; p.T = d.T; p.tiles_t = (d.T + 255) / 256; p.n_tiles = d.N16 / BN; p.num_tiles = d.B * p.tiles_t * p.n_tiles;
  p.nseg = d.nseg; p.n_outer = d.n_outer > 0 ? d.n_outer : 1;
  for (int s = 0; s < d.nseg; ++s) { p.segK[s] = d.seg[s].K; p.segShift[s] = d.seg[s].shift; }
  auto kern = tc_conv_gemm_staged_kernel<Epi, BN>;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  const int slots = tc_balanced_slots(p.num_tiles, tc_num_sms() / 2);      // one CTA pair per pair of SMs (a TPC)
  const int grid = (p.num_tiles < slots ? p.num_tiles : slots) * 2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(384); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 2);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, *ma[0], *ma[1], *ma[2], *ma[3], *ma[4], *mw, *mi[0], *mi[1], *mo[0], *mo[1], *mo[2], p, sp, ep);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "staged conv_gemm launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

template <class Epi>
static int tc_conv_gemm_staged(TmapCache& tc, cudaStream_t st, const TcGemmDesc& d, const typename Epi::Params& ep, const TcEpiIo* ins, uint32_t in_mask,
                               const TcEpiIo* outs) {
  int tile = d.tileN;
  if (tile == 0) tile = d.N16 % 256 == 0 ? 256 : (d.N16 % 128 == 0 ? 128 : 64);
  if (d.N16 % tile != 0 || d.nseg < 1 || d.nseg > TC_MAX_SEG) { snprintf(g_tc_err, sizeof(g_tc_err), "bad tiling N16=%d tile=%d nseg=%d", d.N16, tile, d.nseg); return -1; }
  switch (tile) {
    case 256: return tc_conv_gemm_staged_launch<Epi, 256>(tc, st, d, ep, ins, in_mask, outs);
    case 128: return tc_conv_gemm_staged_launch<Epi, 128>(tc, st, d, ep, ins, in_mask, outs);
    case 64: return tc_conv_gemm_staged_launch<Epi, 64>(tc, st, d, ep, ins, in_mask, outs);
  }
  return -2;
}

// ---------------------------------------------------------------- wgrad kernel
struct TcWgradParams {
  int B, T, N;
  int chunks_t;          // ceil(T / 64)
  int total_chunks;      // B * chunks_t
  int chunks_per_split;
  int ktot;
  int nseg;
  int segK[TC_MAX_SEG];
  int segShift[TC_MAX_SEG];
  float* partial;        // [nsplit][ktot][N]
  float* cs_partial;     // [nsplit][slots][N] or null
  int slots;
  unsigned long long pol_a, pol_g;   // L2 cache policies of the two operands
};

template <int BN> struct TcWgradCfg {
  static constexpr int BKT = 64;                         // time rows per stage
  static constexpr int A_BYTES = 2 * 64 * BKT * 2;       // two 64-channel atoms: 16 KB
  static constexpr int G_BYTES = (BN / 64) * 64 * BKT * 2;
  static constexpr int STAGE_BYTES = A_BYTES + G_BYTES;
  static constexpr int STAGES = (BN == 256) ? 4 : 6;
  static constexpr int TMEM_COLS = BN < 32 ? 32 : BN;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
};

// grid: x = 128-row tiles of the (seg, channel) axis, y = BN-wide tiles of N, z = row-range split
template <int BN>
__global__ void __launch_bounds__(256, 1)
tc_wgrad_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                const __grid_constant__ CUtensorMap tmA3, const __grid_constant__ CUtensorMap tmA4, const __grid_constant__ CUtensorMap tmG, const TcWgradParams p) {
  using Cfg = TcWgradCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint32_t* tmem_ptr = (uint32_t*)(tfull_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // locate segment / channel offset of this m tile
  int mt = blockIdx.x, s = 0, koff = 0;
  while (true) {
    const int nt = (p.segK[s] + 127) >> 7;
    if (mt < nt) break;
    mt -= nt; koff += p.segK[s]; ++s;
  }
  const int k0 = mt << 7;
  const int n0 = blockIdx.y * BN;
  const int c_begin = blockIdx.z * p.chunks_per_split;
  const int c_end = min(p.total_chunks, c_begin + p.chunks_per_split);
  const int nchunks = c_end - c_begin;

  // The otherwise idle epilogue warps also reduce the columns of G (bias / conditioning gradients)
  // straight from the TMA-staged G tiles in shared memory; the gridDim.x CTAs that share a G tile
  // split its 64 time rows between them so no CTA becomes the long pole.
  const bool do_cs = p.cs_partial != nullptr;
  const int cs_r0 = (Cfg::BKT * (int)blockIdx.x) / (int)gridDim.x, cs_r1 = (Cfg::BKT * ((int)blockIdx.x + 1)) / (int)gridDim.x;
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], do_cs ? 5 : 1); }
    mbar_init(tfull_bar, 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc<Cfg::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      const CUtensorMap* tm = s == 0 ? &tmA0 : (s == 1 ? &tmA1 : (s == 2 ? &tmA2 : (s == 3 ? &tmA3 : &tmA4)));
      tma_prefetch_desc(tm);
      tma_prefetch_desc(&tmG);
      const int shift = p.segShift[s];
      int stage = 0; uint32_t phase = 0;
      for (int ch = c_begin; ch < c_end; ++ch) {
        const int b = ch / p.chunks_t, t0 = (ch % p.chunks_t) * Cfg::BKT;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
        mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
        tma_load_4d_h(sa, tm, &full_bar[stage], k0, t0 + shift, b, 0, p.pol_a);
        tma_load_4d_h(sa + 8192, tm, &full_bar[stage], k0 + 64, t0 + shift, b, 0, p.pol_a);
#pragma unroll
        for (int j = 0; j < BN / 64; ++j) tma_load_4d_h(sa + Cfg::A_BYTES + j * 8192, &tmG, &full_bar[stage], n0 + 64 * j, t0, b, 0, p.pol_g);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(128, BN, 1, 1);   // both operands MN-major
    int stage = 0; uint32_t phase = 0;
    for (int it = 0; it < nchunks; ++it) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
        // MN-major, 128B swizzle: 64-wide channel atoms 8192 B apart (LBO), 8 time rows = 1024 B (SBO)
        const uint64_t adesc = umma_smem_desc(sa, 8192, 1024);
        const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES, 8192, 1024);
#pragma unroll
        for (int k = 0; k < Cfg::BKT / 16; ++k)   // 16 time rows = 2048 bytes (>>4 = 128) per step
          umma_bf16(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, (it | k) != 0);
        umma_commit(&empty_bar[stage]);
        if (it == nchunks - 1) umma_commit(tfull_bar);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp >= 4) {
    if (do_cs) {
      // thread -> two adjacent columns (one bf16x2 word); rows past T are TMA zero fill
      const int tid = threadIdx.x - 128;
      const int c = 2 * tid;                         // column inside the BN tile
      const bool act = c < BN;
      const int atom = c >> 6, cc = c & 63;
      const uint32_t col_off = (uint32_t)(atom * 8192 + (cc & 7) * 2);
      const uint32_t chunk = (uint32_t)(cc >> 3);
      float s0 = 0.f, s1 = 0.f;
      int stage = 0; uint32_t phase = 0;
      int cur_b = c_begin / p.chunks_t;
      const int b_first = cur_b;
      for (int ch = c_begin; ch < c_end; ++ch) {
        const int b = ch / p.chunks_t;
        if (b != cur_b) {
          if (act && n0 + c < p.N) {
            float* o = p.cs_partial + (((long long)blockIdx.z * gridDim.x + blockIdx.x) * p.slots + (cur_b - b_first)) * p.N + n0 + c;
            o[0] = s0;
            if (n0 + c + 1 < p.N) o[1] = s1;
          }
          s0 = s1 = 0.f; cur_b = b;
        }
        mbar_wait(&full_bar[stage], phase);
        if (act) {
          const uint8_t* g = smem + stage * Cfg::STAGE_BYTES + Cfg::A_BYTES + col_off;
#pragma unroll 8
          for (int r = cs_r0; r < cs_r1; ++r) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(g + r * 128 + ((chunk ^ (uint32_t)(r & 7)) << 4));
            s0 += __uint_as_float(w << 16);
            s1 += __uint_as_float(w & 0xffff0000u);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (nchunks > 0 && act && n0 + c < p.N) {
        float* o = p.cs_partial + (((long long)blockIdx.z * gridDim.x + blockIdx.x) * p.slots + (cur_b - b_first)) * p.N + n0 + c;
        o[0] = s0;
        if (n0 + c + 1 < p.N) o[1] = s1;
      }
    }
    const int quarter = warp & 3;
    const int k = k0 + quarter * 32 + lane;        // channel index inside the segment
    float* out = p.partial + ((long long)blockIdx.z * p.ktot + koff + k) * p.N;
    const bool valid = k < p.segK[s];
    if (nchunks > 0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    for (int c = 0; c < BN; c += 16) {
      const int n = n0 + c;
      if (n >= p.N) break;
      float v[16];
      if (nchunks > 0) tmem_ld16(taddr + (uint32_t)c, v);
      else {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = 0.f;
      }
      if (valid) {
        const int nv = min(16, p.N - n);
        if (nv == 16 && ((p.N & 3) == 0)) {
#pragma unroll
          for (int i = 0; i < 4; ++i) reinterpret_cast<float4*>(out + n)[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) if (i < nv) out[n + i] = v[i];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------- wgrad kernel, CTA pairs (cta_group::2)
// Same contraction, M = 256 channels per pair: CTA rank r stages ITS 128 channels of A and ITS half of the BN columns
// of G, so one 64-row step moves 32 KB per SM instead of 48 KB (the cta_group::1 kernel is bound by L2 -> SM
// bandwidth: 387 MB per dilated wgrad launch).  The leader's barrier counts both CTAs' TMA bytes; the column sums
// read the local G half after the MMAs of the stage have completed (mma_done), then release the stage.
// Requires every segment width to be a multiple of 256 (pair tiles never straddle a segment).
// NH: BN-wide column blocks per pair: 1 here, 2 in the two-accumulator units of the grouped kernel (gemm_tc_wgroup.cuh).
template <int BN, int NH = 1> struct TcWgradPairCfg {
  static constexpr int BKT = 64;
  static constexpr int A_BYTES = 2 * 64 * BKT * 2;               // two 64-channel atoms: 16 KB
  static constexpr int G_ATOMS = BN / 2 / 64;                    // 64-column atoms of this CTA's half of ONE column block
  static constexpr int GH_BYTES = G_ATOMS * 64 * BKT * 2;
  static constexpr int G_BYTES = NH * GH_BYTES;
  static constexpr int STAGE_BYTES = A_BYTES + G_BYTES;
  static constexpr int STAGES = NH == 2 ? 4 : 6;
  static constexpr int TMEM_COLS = BN * NH < 32 ? 32 : BN * NH;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 1024 + 2048;   // align slack, barriers, column-sum scratch
};

template <int BN>
__global__ void __launch_bounds__(256, 1)
tc_wgrad_pair_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                     const __grid_constant__ CUtensorMap tmA3, const __grid_constant__ CUtensorMap tmA4, const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmP,
                     const TcWgradParams p) {
  using Cfg = TcWgradPairCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int HALF = BN / 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* mma_done = empty_bar + STAGES;
  uint64_t* tfull_bar = mma_done + STAGES;
  uint32_t* tmem_ptr = (uint32_t*)(tfull_bar + 1);
  float* cs_s = (float*)(smem + STAGES * Cfg::STAGE_BYTES + 1024);      // [RH][HALF] column-sum hand-over between row halves

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
#ifdef TC_TIMELINE
  long long te0 = 0, te1 = 0;
#endif
  // segment / channel offset of this pair's m tile
  int mp = (int)blockIdx.x >> 1, s = 0, koff = 0;
  while (true) {
    const int nt = p.segK[s] >> 8;
    if (mp < nt) break;
    mp -= nt; koff += p.segK[s]; ++s;
  }
  const int k0 = (mp << 8) + (int)crank * 128;
  const int n0 = blockIdx.y * BN;
  const int gcol0 = n0 + (int)crank * HALF;           // first column of this CTA's half of the column block
  const int c_begin = blockIdx.z * p.chunks_per_split;
  const int c_end = min(p.total_chunks, c_begin + p.chunks_per_split);
  const int nchunks = c_end - c_begin;
  const bool do_cs = p.cs_partial != nullptr;
  // the pairs of this (n tile, split) share the G tile: each takes a slice of its 64 time rows for the column sums
  const int npairs = (int)gridDim.x >> 1, pidx = (int)blockIdx.x >> 1;
  const int cs_r0 = (Cfg::BKT * pidx) / npairs, cs_r1 = (Cfg::BKT * (pidx + 1)) / npairs;

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], do_cs ? 4 : 1); mbar_init(&mma_done[i], 1); }
    mbar_init(tfull_bar, 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc_pair<Cfg::TMEM_COLS>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_launch_dependents();
  pdl_wait();

  if (warp == 0) {
    if (lane == 0) {
      const CUtensorMap* tm = s == 0 ? &tmA0 : (s == 1 ? &tmA1 : (s == 2 ? &tmA2 : (s == 3 ? &tmA3 : &tmA4)));
      tma_prefetch_desc(tm);
      tma_prefetch_desc(&tmG);
      const int shift = p.segShift[s];
      int stage = 0; uint32_t phase = 0;
#ifdef TC_TIMELINE
      long long tw = 0, tt0 = clock64();
#endif
      for (int ch = c_begin; ch < c_end; ++ch) {
        const int b = ch / p.chunks_t, t0 = (ch % p.chunks_t) * Cfg::BKT;
#ifdef TC_TIMELINE
        const long long ta = clock64();
#endif
        mbar_wait(&empty_bar[stage], phase ^ 1);
#ifdef TC_TIMELINE
        tw += clock64() - ta;
#endif
        uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
        if (leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
        // one op per operand: boxes of 2 (A) and G_ATOMS (G) 64-channel atoms (tc_atom_map)
        tma_load_4d_pair_h(sa, tm, &full_bar[stage], 0, t0 + shift, k0 >> 6, b, p.pol_a);
        tma_load_4d_pair_h(sa + Cfg::A_BYTES, &tmG, &full_bar[stage], 0, t0, gcol0 >> 6, b, p.pol_g);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
#ifdef TC_TIMELINE
      if (blockIdx.x < 2 && blockIdx.y == 0 && blockIdx.z == 0) printf("WG producer blk %d: chunks %d total %lld wait_empty %lld\n", blockIdx.x, nchunks, clock64() - tt0, tw);
#endif
    }
  } else if (warp == 1) {
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BN, 1, 1);   // both operands MN-major
      int stage = 0; uint32_t phase = 0;
#ifdef TC_TIMELINE
      long long tw = 0, tt0 = clock64(), tfirst = 0;
#endif
      for (int it = 0; it < nchunks; ++it) {
#ifdef TC_TIMELINE
        const long long ta = clock64();
#endif
        mbar_wait(&full_bar[stage], phase);
#ifdef TC_TIMELINE
        if (it == 0) tfirst = clock64() - ta; else tw += clock64() - ta;
#endif
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t adesc = umma_smem_desc(sa, 8192, 1024);
          const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES, 8192, 1024);
#pragma unroll
          for (int k = 0; k < Cfg::BKT / 16; ++k)
            umma_bf16_pair(tmem_base, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, (it | k) != 0);
          // with column sums the stage is released by the summing warps, which first wait for these MMAs
          umma_commit_pair(do_cs ? &mma_done[stage] : &empty_bar[stage]);
          if (it == nchunks - 1) umma_commit_pair(tfull_bar);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
#ifdef TC_TIMELINE
      if (blockIdx.x < 2 && blockIdx.y == 0 && blockIdx.z == 0 && lane == 0) printf("WG mma blk %d: chunks %d total %lld first_wait %lld wait_full(rest) %lld\n", blockIdx.x, nchunks, clock64() - tt0, tfirst, tw);
#endif
    }
  } else if (warp >= 4) {
    if (do_cs) {
      // 128 threads: column pair (tid & 63 .. of HALF/2 pairs) x row half (tid >> 6) of this pair's row slice
      const int tid = threadIdx.x - 128;
      constexpr int NPAIR = HALF / 2;
      const int pr = tid % NPAIR, rh = tid / NPAIR;          // rh in [0, 128 / NPAIR)
      constexpr int RH = 128 / NPAIR;
      const int c = 2 * pr;
      const int atom = c >> 6, cc = c & 63;
      const uint32_t col_off = (uint32_t)(atom * 8192 + (cc & 7) * 2);
      const uint32_t chunk = (uint32_t)(cc >> 3);
      const int len = cs_r1 - cs_r0;
      const int r_lo = cs_r0 + (len * rh) / RH, r_hi = cs_r0 + (len * (rh + 1)) / RH;
      float s0 = 0.f, s1 = 0.f;
      int stage = 0; uint32_t phase = 0;
      int cur_b = c_begin / p.chunks_t;
      const int b_first = cur_b;
      auto flush = [&](int slot) {
        // combine the row halves in a fixed order, write this CTA's columns and zero the peer's half
        cs_s[rh * HALF + c] = s0; cs_s[rh * HALF + c + 1] = s1;
        named_bar_sync(7, 128);
        if (rh == 0) {
          float* o = p.cs_partial + (((long long)blockIdx.z * gridDim.x + blockIdx.x) * p.slots + slot) * p.N;
          float t0 = 0.f, t1 = 0.f;
#pragma unroll
          for (int h2 = 0; h2 < RH; ++h2) { t0 += cs_s[h2 * HALF + c]; t1 += cs_s[h2 * HALF + c + 1]; }
          const int mine = gcol0 + c, other = n0 + (1 - (int)crank) * HALF + c;
          if (mine < p.N) o[mine] = t0;
          if (mine + 1 < p.N) o[mine + 1] = t1;
          if (other < p.N) o[other] = 0.f;
          if (other + 1 < p.N) o[other + 1] = 0.f;
        }
        named_bar_sync(7, 128);
      };
      for (int ch = c_begin; ch < c_end; ++ch) {
        const int b = ch / p.chunks_t;
        if (b != cur_b) {
          flush(cur_b - b_first);
          s0 = s1 = 0.f;
          cur_b = b;
        }
        mbar_wait(&mma_done[stage], phase);
        const uint8_t* g = smem + stage * Cfg::STAGE_BYTES + Cfg::A_BYTES + col_off;
#pragma unroll 8
        for (int r = r_lo; r < r_hi; ++r) {
          const uint32_t w = *reinterpret_cast<const uint32_t*>(g + r * 128 + ((chunk ^ (uint32_t)(r & 7)) << 4));
          s0 += __uint_as_float(w << 16);
          s1 += __uint_as_float(w & 0xffff0000u);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (nchunks > 0) flush(cur_b - b_first);
    }
    const int quarter = warp & 3;
    const int k = k0 + quarter * 32 + lane;        // channel index inside the segment
    float* out = p.partial + ((long long)blockIdx.z * p.ktot + koff + k) * p.N;
    const bool valid = k < p.segK[s];
#ifdef TC_TIMELINE
    te0 = clock64();
#endif
    if (nchunks > 0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
#ifdef TC_TIMELINE
    te1 = clock64();
#endif
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    // partial tile (128 channels x BN fp32) -> the operand ring (free now: every MMA has completed and read it) as BN/32
    // boxes of 128 rows x 32 floats, 128B swizzle -> TMA stores.  Row-per-thread global stores took 9.5 k cycles here.
    {
      const int r = quarter * 32 + lane;
      const uint32_t rsw = (uint32_t)(r & 7);
      uint8_t* const rowp = smem + (uint32_t)r * 128u;
      for (int c = 0; c < BN; c += 16) {
        float v[16];
        if (nchunks > 0) tmem_ld16(taddr + (uint32_t)c, v);
        else {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = 0.f;
        }
        uint8_t* const boxp = rowp + (c >> 5) * 16384;
        const uint32_t j0 = (uint32_t)((c & 31) >> 2);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          *reinterpret_cast<float4*>(boxp + (((j0 + i) ^ rsw) << 4)) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      fence_proxy_async();
      named_bar_sync(6, 128);
      if (threadIdx.x == 128) {
        const int row0 = koff + k0;
#pragma unroll
        for (int bx = 0; bx < BN / 32; ++bx)
          if (n0 + bx * 32 < p.N) tma_store_3d_h(smem + bx * 16384, &tmP, n0 + bx * 32, row0, (int)blockIdx.z, TC_POL_LAST);
        bulk_commit_group();
      }
      if (threadIdx.x == 128) bulk_wait_group<0>();
    }
  }
#ifdef TC_TIMELINE
  if (warp == 4 && lane == 0 && blockIdx.x < 2 && blockIdx.y == 0 && blockIdx.z == 0) printf("WG epi blk %d: wait_tfull(after cs) %lld store %lld\n", blockIdx.x, te1 - te0, clock64() - te1);
#endif
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
}

template <int BN>
static int tc_wgrad_pair_launch(TmapCache& tc, cudaStream_t st, const TcWgradDesc& d, TcWgradPlan* plan) {
  using Cfg = TcWgradPairCfg<BN>;
  const CUtensorMap* ma[TC_MAX_SEG] = {};
  int mpairs = 0;
  for (int s = 0; s < d.nseg; ++s) {
    ma[s] = tc_atom_map(tc, d.seg[s].A, d.seg[s].lda, d.seg[s].K, d.T, d.B, 64, 2);
    if (!ma[s]) return -10;
    mpairs += d.seg[s].K / 256;
  }
  for (int s = d.nseg; s < TC_MAX_SEG; ++s) ma[s] = ma[0];
  const CUtensorMap* mg = tc_atom_map(tc, d.G, d.ldg, d.N, d.T, d.B, 64, Cfg::G_ATOMS);
  if (!mg) return -11;
  TcWgradParams p{};
  p.B = d.B; p.T = d.T; p.N = d.N; p.chunks_t = (d.T + 63) / 64; p.total_chunks = d.B * p.chunks_t; p.ktot = d.ktot; p.nseg = d.nseg;
  for (int s = 0; s < d.nseg; ++s) { p.segK[s] = d.seg[s].K; p.segShift[s] = d.seg[s].shift; }
  p.partial = d.partial;
  p.pol_a = tc_policy(d.l2_a); p.pol_g = tc_policy(d.l2_g);
  const int ntiles = (d.N + BN - 1) / BN;
  int nsplit = (tc_num_sms() / 2) / (mpairs * ntiles);     // one wave of CTA pairs
  if (nsplit < 1) nsplit = 1;
  if (nsplit > WN_MAX_WGRAD_SPLITS) nsplit = WN_MAX_WGRAD_SPLITS;
  if (nsplit > p.total_chunks) nsplit = p.total_chunks;
  p.chunks_per_split = (p.total_chunks + nsplit - 1) / nsplit;
  nsplit = (p.total_chunks + p.chunks_per_split - 1) / p.chunks_per_split;
  p.slots = (p.chunks_per_split + p.chunks_t - 2) / p.chunks_t + 1;
  p.cs_partial = d.cs_partial;
  plan->nsplit = nsplit; plan->chunks_per_split = p.chunks_per_split; plan->chunks_t = p.chunks_t; plan->slots = p.slots; plan->mtiles = 2 * mpairs;
  // partials [nsplit][ktot][N] fp32 as a TMA-store target: boxes of 32 floats x 128 rows
  uint64_t pd[3] = {(uint64_t)d.N, (uint64_t)d.ktot, (uint64_t)nsplit};
  uint64_t ps[2] = {(uint64_t)d.N * 4, (uint64_t)d.ktot * d.N * 4};
  uint32_t pb[3] = {32, 128, 1};
  const CUtensorMap* mp = tc.get(d.partial, 3, pd, ps, pb, 128, true);
  if (!mp) return -14;
  auto kern = tc_wgrad_pair_kernel<BN>;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * mpairs, ntiles, nsplit); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 2);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, *ma[0], *ma[1], *ma[2], *ma[3], *ma[4], *mg, *mp, p);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "wgrad launch (cta pairs): %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

template <int BN>
static int tc_wgrad_launch(TmapCache& tc, cudaStream_t st, const TcWgradDesc& d, TcWgradPlan* plan) {
  using Cfg = TcWgradCfg<BN>;
  const CUtensorMap* ma[TC_MAX_SEG] = {};
  int mtiles = 0;
  for (int s = 0; s < d.nseg; ++s) {
    ma[s] = tc_act_map(tc, d.seg[s].A, d.seg[s].lda, d.seg[s].K, d.T, d.B, 1, 0, 64);
    if (!ma[s]) return -10;
    mtiles += (d.seg[s].K + 127) / 128;
  }
  for (int s = d.nseg; s < TC_MAX_SEG; ++s) ma[s] = ma[0];
  // No clusters along the m-tiles that share a G tile.  Measured on B200 (C2 dilated wgrad, profiles/README.md): multicasting
  // the G tile to clusters of 4 is SLOWER (43 vs 37 us in isolation, +1.9 ms per step in situ: lock-step coupling, 2 KB boxes,
  // remote barrier arrivals, and only 132 SMs host 4-clusters) — L2 already coalesces same-line requests of neighbouring SMs.
  const CUtensorMap* mg = tc_act_map(tc, d.G, d.ldg, d.N, d.T, d.B, 1, 0, 64);
  if (!mg) return -11;
  TcWgradParams p{};
  p.B = d.B; p.T = d.T; p.N = d.N; p.chunks_t = (d.T + 63) / 64; p.total_chunks = d.B * p.chunks_t; p.ktot = d.ktot; p.nseg = d.nseg;
  for (int s = 0; s < d.nseg; ++s) { p.segK[s] = d.seg[s].K; p.segShift[s] = d.seg[s].shift; }
  p.partial = d.partial;
  p.pol_a = tc_policy(d.l2_a); p.pol_g = tc_policy(d.l2_g);
  const int ntiles = (d.N + BN - 1) / BN;
  int nsplit = tc_num_sms() / (mtiles * ntiles);   // one wave: never more CTAs than can be resident
  if (nsplit < 1) nsplit = 1;
  if (nsplit > WN_MAX_WGRAD_SPLITS) nsplit = WN_MAX_WGRAD_SPLITS;
  if (nsplit > p.total_chunks) nsplit = p.total_chunks;
  p.chunks_per_split = (p.total_chunks + nsplit - 1) / nsplit;
  nsplit = (p.total_chunks + p.chunks_per_split - 1) / p.chunks_per_split;
  p.slots = (p.chunks_per_split + p.chunks_t - 2) / p.chunks_t + 1;
  p.cs_partial = d.cs_partial;
  plan->nsplit = nsplit; plan->chunks_per_split = p.chunks_per_split; plan->chunks_t = p.chunks_t; plan->slots = p.slots; plan->mtiles = mtiles;
  auto kern = tc_wgrad_kernel<BN>;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(mtiles, ntiles, nsplit); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 1);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, *ma[0], *ma[1], *ma[2], *ma[3], *ma[4], *mg, p);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "wgrad launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

static inline int tc_wgrad(TmapCache& tc, cudaStream_t st, const TcWgradDesc& d, TcWgradPlan* plan) {
  if (d.nseg < 1 || d.nseg > TC_MAX_SEG) return -1;
  // CTA pairs when the pair's 256-channel tiles fit the segments exactly
  bool pair_ok = d.N > 64 && d.N % 64 == 0;
  for (int s = 0; s < d.nseg; ++s) pair_ok = pair_ok && d.seg[s].K % 256 == 0;
  if (pair_ok) {
    // one column block per pair.  Two 256-column blocks (N = 512, all of TMEM) move a third less L2 -> SM traffic per FLOP,
    // but need twice the splits (37 instead of 18) and therefore twice the partial bytes to write and to reduce: measured
    // SLOWER on C2 (7.41 vs 7.31 ms/step)
    return d.N > 128 ? tc_wgrad_pair_launch<256>(tc, st, d, plan) : tc_wgrad_pair_launch<128>(tc, st, d, plan);
  }
  if (d.N > 128) return tc_wgrad_launch<256>(tc, st, d, plan);
  if (d.N > 64) return tc_wgrad_launch<128>(tc, st, d, plan);
  return tc_wgrad_launch<64>(tc, st, d, plan);
}
// upper bound of cs_partial rows for a (B, T) problem: nsplit * slots <= this
static inline long long tc_wgrad_cs_rows(int B, int T, int max_mtiles) {
  return ((long long)WN_MAX_WGRAD_SPLITS * 2 + B + 2) * (max_mtiles > 0 ? max_mtiles : 1);
}

// Second stage of the wgrad: deterministic sum of the split partials (no atomics), written in
// Keras layout.  The N output columns may belong to two variables (conv1 | conv_skip share one
// launch): columns [0,N0) -> dst0 [ktot][N0], columns [N0,N) -> dst1 [ktot][N-N0].  Optional
// L2 term dst += l2coef * w.  Blocks past the weight part finish the column sums of G:
// bias gradients (total over all rows) and the conditioning per-batch sums.
struct TcWgradFinish {
  const float* partial; int nsplit; int ktot; int N; int N0;
  float* dst0; float* dst1; const float* w0; const float* w1; float l2coef;
  const float* cs; int slots; int cps; int chunks_t; int B; int mtiles;
  float* bias0; float* bias1; float* per_batch; int ldpb;
  int wblocks;   // blocks of the weight part
};
__device__ __forceinline__ void tc_wgrad_finish_body(const TcWgradFinish& f, const int bid, float (*red)[33]) {
  if (bid < f.wblocks) {
    const long long j = (long long)bid * 256 + threadIdx.x;
    const long long n_all = (long long)f.ktot * f.N;
    if (j >= n_all) return;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    const float* p = f.partial + j;
    int i = 0;
    for (; i + 3 < f.nsplit; i += 4) {
      s0 += p[(long long)i * n_all]; s1 += p[(long long)(i + 1) * n_all];
      s2 += p[(long long)(i + 2) * n_all]; s3 += p[(long long)(i + 3) * n_all];
    }
    for (; i < f.nsplit; ++i) s0 += p[(long long)i * n_all];
    float s = (s0 + s1) + (s2 + s3);
    const int k = (int)(j / f.N), n = (int)(j % f.N);
    if (n < f.N0) {
      const long long o = (long long)k * f.N0 + n;
      if (f.w0) s = fmaf(f.l2coef, f.w0[o], s);
      f.dst0[o] = s;
    } else {
      const long long o = (long long)k * (f.N - f.N0) + (n - f.N0);
      if (f.w1) s = fmaf(f.l2coef, f.w1[o], s);
      f.dst1[o] = s;
    }
    return;
  }
  // ---- column sums: 32 columns x 8 batch lanes per block
  const int nl = threadIdx.x & 31, bl = threadIdx.x >> 5;
  const int n = (bid - f.wblocks) * 32 + nl;
  float tot = 0.f;
  if (n < f.N) {
    for (int b = bl; b < f.B; b += 8) {
      const int z0 = (b * f.chunks_t) / f.cps, z1 = min(f.nsplit - 1, ((b + 1) * f.chunks_t - 1) / f.cps);
      float sb = 0.f;
      for (int z = z0; z <= z1; ++z) {
        const int b_first = (z * f.cps) / f.chunks_t;
        for (int m = 0; m < f.mtiles; ++m) sb += f.cs[(((long long)z * f.mtiles + m) * f.slots + (b - b_first)) * f.N + n];
      }
      if (f.per_batch) f.per_batch[(long long)b * f.ldpb + n] = sb;
      tot += sb;
    }
  }
  red[bl][nl] = tot;
  __syncthreads();
  if (bl == 0 && n < f.N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][nl];
    if (n < f.N0) { if (f.bias0) f.bias0[n] = t; }
    else if (f.bias1) f.bias1[n - f.N0] = t;
  }
}

__global__ void __launch_bounds__(256) tc_wgrad_finish(const TcWgradFinish f) {
  __shared__ float red[8][33];
  pdl_launch_dependents();
  pdl_wait();
  tc_wgrad_finish_body(f, (int)blockIdx.x, red);
}
