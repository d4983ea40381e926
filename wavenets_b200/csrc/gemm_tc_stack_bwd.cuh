// gemm_tc_stack_bwd.cuh — the backward chain of the whole residual stack (the autodiff of the block loop of WaveNet.call,
// model.py:229-234,335, i.e. of WaveNetLayer.call, layers.py:199-224, for every block) as ONE persistent launch: the mirror
// image of gemm_tc_stack.cuh.
//
// Per block l (from the last to the first) and 256-row tile m (CTA pair, 128 rows per CTA):
//
//   dg   = [d x_out_l | d skip] . [Wr^T ; Ws^T]                      DG tile   (M = 256, N = D, K = R + S)
//   d z  = gate'(z_l) * dg                                           DG epilogue: z_f / z_s panels arrive by TMA, d z goes
//                                                                    K-major, 128B-swizzled into the operand ring in shared
//                                                                    memory (and from there, by TMA, to HBM once: the
//                                                                    grouped weight gradients read it later)
//   d x_out_{l-1} = d x_out_l                                        OUT tile: the residual gradient is added in the OUT epilogue
//                                                                    (d x_out panels arrive by TMA in the ring the P, Q panels use)
//                 + d z[t]       . W_{K-1}^T                         ... the un-shifted tap straight from the operand ring
//                 + d z[t + s_k] . W_k^T,  k < K-1                   ... the anti-causal taps by TMA from HBM / L2 (rows of
//                                                                    LATER tiles of the same block, and the peer's half)
//
// Before: per block one gate-adjoint launch (reads d x_out, d skip and z, writes d z) and one dgrad launch (reads d z twice and
// d x_out again), 60 launches with their fill and drain, d z making an extra L2 -> SM trip.  Here a CTA pair walks the
// (block, tile) list of all blocks, blocks descending, tiles of a sequence in DESCENDING time order, so that every
// dependency points to a smaller tile id:
//   DG(l, m)        needs d x_out_l rows of tile m            <- OUT(l+1, m)           flags_dx[l+1][m]
//   shifted taps    need d z_l rows t0+s .. t0+s+255          <- DG epilogue (l, m') with m' >= m (its own tile included)
// Tiles are published like in the forward kernel (TMA stores complete -> proxy fence -> red.release.gpu) and acquired by the
// producer warp before the first dependent load.  All CTAs are resident (grid <= SMs, 1 CTA per SM), ids ascend per pair.
//
// TMEM: columns [0, D) = DG accumulator, [256, 256 + R) = OUT accumulator (one stage each: the OUT accumulator is held from
// the first un-shifted tap product until its epilogue has read it; the next tile's DG products run under that epilogue).
// Warps: 0 TMA producer (operand ring) | 1 MMA issuer (leader CTA) | 2 TMEM allocator, then TMA-store warp + tile publisher |
//        3 z-panel producer | 4-11 epilogue (DG: gate adjoint; OUT: pack) | 12 pair hand-off of the d z slabs
#pragma once
#include "gemm_tc_stack.cuh"

// in-kernel phase accounting (clock64 sums over all tiles of one CTA, printed by CTAs 0 and 41): -DTC_TIMELINE builds only
#ifdef TC_TIMELINE
#define SBT_DECL(n) long long sbt[n] = {}; long long sbt_prev = clock64();
#define SBT(i) { const long long sbt_now = clock64(); sbt[i] += sbt_now - sbt_prev; sbt_prev = sbt_now; }
#else
#define SBT_DECL(n)
#define SBT(i)
#endif

struct alignas(128) TcStackBwdLayer {
  CUtensorMap tmDX, tmDS, tmWdg, tmZf, tmZs, tmDZ, tmWb, tmDXp, tmO;   // tmZf / tmZs: the cached gate derivative coefficients P / Q; tmDXp: d x_out as 32-column panels
  int shift[TC_MAX_TAPS];      // row shift of tap k (k < nseg - 1: positive; tap nseg - 1: 0)
  int has_dx, has_ds, has_res;
  int wait_dx;                // d x_out_l is written by this launch (every block but the last): acquire its tile flag first
  const uint8_t* mask;        // dropout keep-mask of this block's conv branch [b*T+t][R], or null
  // multi-dilation blocks (layers.py:64-88): a "layer" of the launch is one CONV.  kind 0 = the block's gated conv (DG tile +
  // gate adjoint + OUT tile), kind 1 = a plain conv in front of it: one OUT-type tile whose taps ALL come from L2 (tmDZ = the
  // gradient wrt this conv's output, written by layer + 1 of this launch; kb_tap 64-wide k blocks per tap).
  // OUT epilogue: out_mode 1 adds the residual gradient (tmDXp = d x_out of the block, guarded by flags_dx[in_flag_layer] when
  // >= 0), out_mode 2 multiplies by act'(y) of the conv in front (tmDXp = its cached bf16 output), 0 neither.
  int kind, out_mode, act, kb_tap, in_flag_layer;
  int alias;                  // skip_channels=None: the skip IS conv1's output, d(conv1 output) = d x_out + d skip — both DG segments
                              // meet the same Wr^T columns (no materialised sum)
};

struct TcStackBwdParams {
  int B, T, tiles_t, num_mtiles, L;
  int nseg;                   // taps of the gated conv
  int kb_dx, kb_ds;           // 64-wide k blocks of the DG contraction over d x_out (R) and d skip (S)
  unsigned long long pol_dx, pol_ds, pol_w, pol_z, pol_dz_ld, pol_dz_st, pol_o;
  float drop_scale;           // 1 / (1 - rate)
  int band, nbands;           // tile order: bands of `band` m tiles (the last one may be shorter); within a band all layers, last to first
};

// No separate d z operand buffer: an un-shifted-tap k-step only loads weights, so the A half of its ring stage is idle — the DG
// epilogue writes the d z slab straight into it (and the TMA store to HBM reads it from there).  Against a 64 KB operand buffer
// beside a 3-stage ring, the same shared memory as 5 ring stages holds up to five slabs in flight between epilogue and MMA instead
// of two slab pairs, and deepens the ring for the DG / shifted-tap k-steps.  Measured (in-kernel phase accounting, C2): DG k-steps
// 9.3 k -> 7.0 k cycles per tile, step -0.3 .. -0.9 % same-box; the pair hand-off chain (epilogue -> hand-off warp ->
// cluster-scope arrive -> MMA) still paces the un-shifted tap at ~10 k cycles per tile.  The peer's hand-off arrive keeps its
// cluster-scope release: without it the hand-off waits drop by 25 % but the step stays within noise, and the hand-off would lean
// on shared-memory writes being physically complete before the local barrier that the hand-off warp acquires, not on the PTX
// memory model.
template <int D_, int R_> struct TcStackBwdCfg {
  static constexpr int BM = 128, BK = 64;
  static constexpr int A_BYTES = BM * BK * 2;                  // 16 KB
  static constexpr int B_BYTES = 128 * BK * 2;                 // this CTA's half of a 256-row weight tile: 16 KB
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = 5;
  static constexpr int NSLAB = 2 * D_ / 64;                    // 64-column slabs of d z (filter slabs first, then gate slabs)
  static constexpr int NPAIR = D_ / 64;                        // slab pairs (f_p, s_p) = two 32-channel epilogue steps each
  static constexpr int PANEL = 128 * 64;                       // 128 rows x 32 bf16
  static constexpr int IN_SLOTS = 3, OUT_SLOTS = 2;            // z ring: (z_f, z_s) panels per slot; out ring: one d x panel per slot
  static constexpr int TMEM_COLS = 512;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + IN_SLOTS * 2 * PANEL + OUT_SLOTS * PANEL + 512;
  static_assert(D_ % 128 == 0 && D_ <= 256 && R_ % 64 == 0 && R_ <= 256, "stack backward kernel: D in {128,256}, R <= 256");
  static_assert(SMEM_BYTES <= 232448, "stack backward kernel does not fit shared memory");
};

template <int D_, int R_>
__global__ void __launch_bounds__(416, 1)
tc_stack_bwd_kernel(const TcStackBwdLayer* __restrict__ layers, int* __restrict__ flags_dx, int* __restrict__ flags_dz, const TcStackBwdParams p) {
  using Cfg = TcStackBwdCfg<D_, R_>;
  constexpr int STAGES = Cfg::STAGES, NEPI = 8, NPAIR = Cfg::NPAIR;
  constexpr int KB_Z = Cfg::NSLAB;
  extern __shared__ __align__(1024) uint8_t smem_sb[];
  uint8_t* smem = smem_sb;
  if ((smem_u32(smem) & 1023u) != 0u) { if (threadIdx.x == 0) printf("libwavenet_b200: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
  uint8_t* in_ring = smem + STAGES * Cfg::STAGE_BYTES;
  uint8_t* out_ring = in_ring + Cfg::IN_SLOTS * 2 * Cfg::PANEL;
  uint64_t* full_bar = (uint64_t*)(out_ring + Cfg::OUT_SLOTS * Cfg::PANEL);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* dg_full = empty_bar + STAGES;            // DG accumulator complete (both CTAs)
  uint64_t* dg_empty = dg_full + 1;                  // leader's: both CTAs' epilogues have read the DG accumulator
  uint64_t* out_full = dg_empty + 1;
  uint64_t* out_empty = out_full + 1;
  uint64_t* in_full = out_empty + 1;                 // [IN_SLOTS]
  uint64_t* in_empty = in_full + Cfg::IN_SLOTS;
  uint64_t* oslot_empty = in_empty + Cfg::IN_SLOTS;  // [OUT_SLOTS] output panel has been read by its TMA store
  // per ring stage — a_done (local, 8 epilogue warps: this CTA's d z slab is in the stage's A half), a_ready (leader's, both CTAs),
  // sfree (local: the TMA store of the slab has read the stage)
  uint64_t* a_done = oslot_empty + Cfg::OUT_SLOTS;
  uint64_t* a_ready = a_done + STAGES;
  uint64_t* sfree = a_ready + STAGES;
  uint32_t* tmem_ptr = (uint32_t*)(sfree + STAGES);
  // k-steps of a tile in ring order (all roles walk the same sequence): DG, un-shifted tap (one per d z slab), shifted taps / plain taps
  auto tile_ksteps = [&](const TcStackBwdLayer& Ly, int& n_dg, int& n_un, int& n_sh) {
    if (Ly.kind) { n_dg = 0; n_un = 0; n_sh = p.nseg * Ly.kb_tap; }
    else { n_dg = (Ly.has_dx ? p.kb_dx : 0) + (Ly.has_ds ? p.kb_ds : 0); n_un = KB_Z; n_sh = (p.nseg - 1) * KB_Z; }
  };
  auto ring_adv = [&](int& rs, uint32_t& rp, int n) { rs += n; while (rs >= STAGES) { rs -= STAGES; rp ^= 1u; } };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int tile_first = (int)blockIdx.x >> 1, tile_stride = (int)gridDim.x >> 1;
  const int pair_row0 = (int)crank * Cfg::BM;
  const int total_tiles = p.L * p.num_mtiles;
  const int n_tiles = tile_first < total_tiles ? (total_tiles - tile_first + tile_stride - 1) / tile_stride : 0;

  // tile id -> (layer, m tile).  Within a layer the tiles of a sequence run in descending time order (the anti-causal taps read
  // d z of LATER rows).  The m tiles are cut into bands: a band walks all layers, last to first, before the next band starts, so
  // that what a tile re-reads — d skip of its rows (the same for every layer) and d x_out written one layer earlier — was touched
  // `band` tiles ago instead of `num_mtiles` tiles ago and is still in L2 (layer-major order: 50 % L2 hit rate, 4.9 GB read from
  // DRAM per C2 pass against 2 GB of cached P, Q; bands of 128: 3.5 GB).  Dependencies still point to smaller ids: (l + 1, m)
  // earlier in the same band, (l, m') with m' < m in the same band or in an earlier one.
  auto locate = [&](int j, int& ly, int& mt, int& b, int& tb) {
    const int gt = tile_first + j * tile_stride;
    const int full = (p.nbands - 1) * p.band * p.L;      // tiles of the bands in front of the last one
    int lr, mr;
    if (gt < full) {
      const int k = gt / (p.band * p.L), r = gt - k * (p.band * p.L);
      lr = r / p.band; mr = k * p.band + (r - lr * p.band);
    } else {
      const int wl = p.num_mtiles - (p.nbands - 1) * p.band, r = gt - full;
      lr = r / wl; mr = (p.nbands - 1) * p.band + (r - lr * wl);
    }
    ly = p.L - 1 - lr;
    b = mr / p.tiles_t;
    tb = p.tiles_t - 1 - (mr - b * p.tiles_t);
    mt = b * p.tiles_t + tb;
  };

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(dg_full, 1); mbar_init(dg_empty, NEPI * 2); mbar_init(out_full, 1); mbar_init(out_empty, NEPI * 2);
    for (int i = 0; i < Cfg::IN_SLOTS; ++i) { mbar_init(&in_full[i], 1); mbar_init(&in_empty[i], NEPI); }
    for (int i = 0; i < Cfg::OUT_SLOTS; ++i) mbar_init(&oslot_empty[i], 1);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&a_done[i], NEPI); mbar_init(&a_ready[i], 2); mbar_init(&sfree[i], 1); }
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

  auto wait_flag = [&](const int* f, int ly, int mt) {
    const long long spin0 = clock64();
    while (ld_acquire_gpu(f) < 2) {
      __nanosleep(32);
      if (clock64() - spin0 > 6000000000ll) { printf("libwavenet_b200: stack backward waited > 3 s for tile (%d, %d)\n", ly, mt); __trap(); }
    }
  };

  if (warp == 0) {
    // ===================== TMA producer (operand ring) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      auto next = [&]() { if (++stage == STAGES) { stage = 0; phase ^= 1; } };
      // a stage whose last use carried a d z slab is free again once the slab's TMA store has read it (bit per stage:
      // un_pend = that wait is outstanding, un_wpar = parity to wait for, un_npar = parity of the stage's next slab use)
      uint32_t un_pend = 0u, un_wpar = 0u, un_npar = 0u;
      auto stage_wait = [&]() {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if ((un_pend >> stage) & 1u) { mbar_wait(&sfree[stage], (un_wpar >> stage) & 1u); un_pend &= ~(1u << stage); }
      };
      SBT_DECL(4)
      constexpr int WDG_BYTES = (D_ / 2) * 64 * 2, WB_BYTES = (R_ / 2) * 64 * 2;
      for (int j = 0; j < n_tiles; ++j) {
        int ly, mt, b, tb;
        locate(j, ly, mt, b, tb);
        const TcStackBwdLayer& Ly = layers[ly];
        const int t0 = tb * (2 * Cfg::BM) + pair_row0;
        if (Ly.kind) {
          // ---- plain conv: every tap reads the gradient wrt this conv's output, tiles of layer + 1 of this launch
          for (int s = 0; s < p.nseg; ++s) {
            const int lo = tb * (2 * Cfg::BM) + Ly.shift[s];
            const int t_lo = lo / (2 * Cfg::BM);
            int t_hi = (lo + 2 * Cfg::BM - 1) / (2 * Cfg::BM);
            if (t_hi > p.tiles_t - 1) t_hi = p.tiles_t - 1;
            SBT(0)
            for (int tt = t_lo; tt <= t_hi; ++tt) wait_flag(flags_dx + (size_t)(ly + 1) * p.num_mtiles + b * p.tiles_t + tt, ly + 1, b * p.tiles_t + tt);
            SBT(1)
          }
          fence_proxy_async_global();
          for (int s = 0; s < p.nseg; ++s)
            for (int kb = 0; kb < Ly.kb_tap; ++kb) {
              stage_wait();
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + WB_BYTES));
              tma_load_3d_pair_h(sa, &Ly.tmDZ, &full_bar[stage], kb * 64, t0 + Ly.shift[s], b, p.pol_dz_ld);
              tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmWb, &full_bar[stage], (s * Ly.kb_tap + kb) * 64, (int)crank * (R_ / 2), p.pol_w);
              next();
            }
          continue;
        }
        // ---- DG: [d x_out | d skip] . Wdg
        if (Ly.has_dx) {
          if (Ly.wait_dx) {
            // d x_out_l tile m was written by the OUT tile (l+1, m) of this launch
            SBT(0)
            wait_flag(flags_dx + (size_t)(ly + 1) * p.num_mtiles + mt, ly + 1, mt);
            fence_proxy_async_global();
            SBT(1)
          }
          for (int kb = 0; kb < p.kb_dx; ++kb) {
            stage_wait();
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (leader) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + WDG_BYTES));
            tma_load_4d_pair_h(sa, &Ly.tmDX, &full_bar[stage], kb * 64, t0, b, 0, p.pol_dx);
            tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmWdg, &full_bar[stage], kb * 64, (int)crank * (D_ / 2), p.pol_w);
            next();
          }
        }
        if (Ly.has_ds) {
          const int k0 = (Ly.has_dx && !Ly.alias) ? p.kb_dx * 64 : 0;
          for (int kb = 0; kb < p.kb_ds; ++kb) {
            stage_wait();
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (leader) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + WDG_BYTES));
            tma_load_4d_pair_h(sa, &Ly.tmDS, &full_bar[stage], kb * 64, t0, b, 0, p.pol_ds);
            tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmWdg, &full_bar[stage], k0 + kb * 64, (int)crank * (D_ / 2), p.pol_w);
            next();
          }
        }
        // ---- OUT, un-shifted tap: only the weights (the A half receives a d z slab from the epilogue), slab pairs in production order
        const int kloc = (p.nseg - 1) * 2 * D_;
        for (int pr = 0; pr < NPAIR; ++pr) {
          for (int hh = 0; hh < 2; ++hh) {
            const int slab = hh == 0 ? pr : NPAIR + pr;
            stage_wait();
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (leader) mbar_expect_tx(&full_bar[stage], 2 * WB_BYTES);
            tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmWb, &full_bar[stage], kloc + slab * 64, (int)crank * (R_ / 2), p.pol_w);
            un_wpar = (un_wpar & ~(1u << stage)) | (((un_npar >> stage) & 1u) << stage);
            un_npar ^= 1u << stage; un_pend |= 1u << stage;
            next();
          }
        }
        // ---- OUT, shifted taps: d z rows of this and of later tiles of the same sequence, written by this launch
        for (int s = 0; s < p.nseg - 1; ++s) {
          const int lo = tb * (2 * Cfg::BM) + Ly.shift[s];
          const int t_lo = lo / (2 * Cfg::BM);
          int t_hi = (lo + 2 * Cfg::BM - 1) / (2 * Cfg::BM);
          if (t_hi > p.tiles_t - 1) t_hi = p.tiles_t - 1;
          SBT(0)
          for (int tt = t_lo; tt <= t_hi; ++tt) wait_flag(flags_dz + (size_t)ly * p.num_mtiles + b * p.tiles_t + tt, ly, b * p.tiles_t + tt);
          fence_proxy_async_global();
          SBT(2)
          for (int kb = 0; kb < KB_Z; ++kb) {
            stage_wait();
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (leader) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + WB_BYTES));
            tma_load_3d_pair_h(sa, &Ly.tmDZ, &full_bar[stage], kb * 64, t0 + Ly.shift[s], b, p.pol_dz_ld);
            tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmWb, &full_bar[stage], s * 2 * D_ + kb * 64, (int)crank * (R_ / 2), p.pol_w);
            next();
          }
        }
      }
      SBT(0)
#ifdef TC_TIMELINE
      if (blockIdx.x == 0 || blockIdx.x == 41)
        printf("SBWD cta %d producer: tiles %d  ring+issue %lld  wait_flag_dx %lld  wait_flag_dz %lld\n", blockIdx.x, n_tiles, sbt[0], sbt[1], sbt[2]);
#endif
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (leader) {
      constexpr uint32_t idesc_g = umma_idesc_bf16(256, D_, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16(256, R_, 0, 0);
      const uint32_t t_dg = tmem_base, t_out = tmem_base + 256u;
      int stage = 0; uint32_t phase = 0;
      uint32_t ng = 0u;                  // gated tiles so far
      uint32_t ar_par = 0u;              // per stage, parity of its next a_ready phase
      SBT_DECL(10)
      auto kstep = [&](uint32_t d_tmem, uint32_t idesc, bool first, uint64_t* extra) {
#ifdef TC_TIMELINE
        const long long w0 = clock64();
#endif
        mbar_wait(&full_bar[stage], phase);
#ifdef TC_TIMELINE
        sbt[9] += clock64() - w0;
#endif
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint64_t adesc = umma_smem_desc(sa, 16, 1024);
          const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES, 16, 1024);
#pragma unroll
          for (int k = 0; k < Cfg::BK / 16; ++k)
            umma_bf16_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (first && k == 0) ? 0u : 1u);
          umma_commit_pair(&empty_bar[stage]);
          if (extra) umma_commit_pair(extra);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      };
      for (int j = 0; j < n_tiles; ++j) {
        int ly, mt, b, tb;
        locate(j, ly, mt, b, tb);
        const TcStackBwdLayer& Ly = layers[ly];
        const uint32_t par = (uint32_t)(j & 1);
        if (Ly.kind) {
          // ---- plain conv: one OUT-type tile, all k-steps from the ring
          SBT(2)
          mbar_wait(out_empty, par ^ 1);
          SBT(3)
          tc_fence_after();
          const int ks_p = p.nseg * Ly.kb_tap;
          for (int ks = 0; ks < ks_p; ++ks) kstep(t_out, idesc_o, ks == 0, ks == ks_p - 1 ? out_full : nullptr);
          SBT(7)
          continue;
        }
        const uint32_t gpar = ng & 1u; ++ng;      // the DG accumulator hand-shakes count gated tiles only
        // ---- DG
        SBT(0)
        mbar_wait(dg_empty, gpar ^ 1);
        SBT(1)
        tc_fence_after();
        const int ks_dg = (Ly.has_dx ? p.kb_dx : 0) + (Ly.has_ds ? p.kb_ds : 0);
        for (int ks = 0; ks < ks_dg; ++ks) kstep(t_dg, idesc_g, ks == 0, ks == ks_dg - 1 ? dg_full : nullptr);
        // ---- OUT
        SBT(2)
        mbar_wait(out_empty, par ^ 1);
        SBT(3)
        tc_fence_after();
        const int ks_sh = (p.nseg - 1) * KB_Z;
        for (int q = 0; q < KB_Z; ++q) {
          // one hand-off per slab PAIR, on the barrier of the filter slab's stage: both CTAs' two slabs are in their stages' A halves
          if ((q & 1) == 0) { mbar_wait(&a_ready[stage], (ar_par >> stage) & 1u); ar_par ^= 1u << stage; }
          SBT(5)
          tc_fence_after();
          const bool last = ks_sh == 0 && q == KB_Z - 1;
          kstep(t_out, idesc_o, q == 0, last ? out_full : nullptr);
          SBT(6)
        }
        for (int ks = 0; ks < ks_sh; ++ks) kstep(t_out, idesc_o, false, ks == ks_sh - 1 ? out_full : nullptr);
        SBT(7)
      }
#ifdef TC_TIMELINE
      if (lane == 0 && (blockIdx.x == 0 || blockIdx.x == 40))
        printf("SBWD cta %d mma: tiles %d  wait_dg_empty %lld  DG ksteps %lld  wait_out_empty %lld  wait_a_ready %lld  unshifted %lld  shifted %lld  (of the ksteps: wait_full_bar %lld)\n",
               blockIdx.x, n_tiles, sbt[1], sbt[2], sbt[3], sbt[5], sbt[6], sbt[7], sbt[9]);
#endif
    }
  } else if (warp == 2) {
    // ===================== TMA-store warp + tile publisher =====================
    int oslot = 0;
    uint64_t* pend = nullptr;       // barrier(s) to release once the previously committed store group has read shared memory
    uint64_t* pend2 = nullptr;
    auto committed = [&](uint64_t* rel, uint64_t* rel2 = nullptr) {
      bulk_commit_group();
      if (pend) { bulk_wait_group_read<1>(); mbar_arrive(pend); if (pend2) mbar_arrive(pend2); }
      pend = rel; pend2 = rel2;
    };
    int s_rs = 0; uint32_t s_rp = 0u;      // ring position at the start of the current tile
    auto publish = [&](int* flag) {
      // every store of this thread so far has landed -> visible to the async proxy of other SMs -> count this CTA in
      bulk_wait_group<0>();
      if (pend) { mbar_arrive(pend); if (pend2) mbar_arrive(pend2); pend = nullptr; pend2 = nullptr; }
      fence_proxy_async_global();
      __threadfence();
      red_release_gpu_add(flag, 1);
    };
    for (int j = 0; j < n_tiles; ++j) {
      int ly, mt, b, tb;
      locate(j, ly, mt, b, tb);
      const TcStackBwdLayer& Ly = layers[ly];
      const int t0 = tb * (2 * Cfg::BM) + pair_row0;
      int n_dg, n_un, n_sh;
      tile_ksteps(Ly, n_dg, n_un, n_sh);
      if (!Ly.kind) {
      int u_rs = s_rs; uint32_t u_rp = s_rp;
      ring_adv(u_rs, u_rp, n_dg);      // stage of the first un-shifted-tap k-step
      for (int pr = 0; pr < NPAIR; ++pr) {
        named_bar_sync(8 + pr, NEPI * 32 + 32);
        const int sf = u_rs; ring_adv(u_rs, u_rp, 1);
        const int ss = u_rs; ring_adv(u_rs, u_rp, 1);
        if (lane == 0) {
          tma_store_3d_h(smem + sf * Cfg::STAGE_BYTES, &Ly.tmDZ, pr * 64, t0, b, p.pol_dz_st);
          tma_store_3d_h(smem + ss * Cfg::STAGE_BYTES, &Ly.tmDZ, D_ + pr * 64, t0, b, p.pol_dz_st);
          committed(&sfree[sf], &sfree[ss]);
        }
        __syncwarp();
      }
      if (lane == 0) publish(flags_dz + (size_t)ly * p.num_mtiles + mt);
      __syncwarp();
      }
      for (int step = 0; step < R_ / 32; ++step) {
        named_bar_sync(3 + oslot, NEPI * 32 + 32);
        if (lane == 0) {
          tma_store_3d_h(out_ring + oslot * Cfg::PANEL, &Ly.tmO, step * 32, t0, b, p.pol_o);
          committed(&oslot_empty[oslot]);
        }
        __syncwarp();
        if (++oslot == Cfg::OUT_SLOTS) oslot = 0;
      }
      if (lane == 0) publish(flags_dx + (size_t)ly * p.num_mtiles + mt);
      __syncwarp();
      ring_adv(s_rs, s_rp, n_dg + n_un + n_sh);
    }
    if (lane == 0) bulk_wait_group<0>();
  } else if (warp == 3) {
    // ===================== z-panel producer (gate adjoint inputs) =====================
    if (lane == 0) {
      int islot = 0; uint32_t iphase = 0;
      for (int j = 0; j < n_tiles; ++j) {
        int ly, mt, b, tb;
        locate(j, ly, mt, b, tb);
        const TcStackBwdLayer& Ly = layers[ly];
        const int t0 = tb * (2 * Cfg::BM) + pair_row0;
        if (!Ly.kind)
        for (int step = 0; step < D_ / 32; ++step) {
          mbar_wait(&in_empty[islot], iphase ^ 1);
          mbar_expect_tx(&in_full[islot], 2u * Cfg::PANEL);
          uint8_t* dst = in_ring + islot * 2 * Cfg::PANEL;
          tma_load_3d_h(dst, &Ly.tmZf, &in_full[islot], step * 32, t0, b, p.pol_z);
          tma_load_3d_h(dst + Cfg::PANEL, &Ly.tmZs, &in_full[islot], step * 32, t0, b, p.pol_z);
          if (++islot == Cfg::IN_SLOTS) { islot = 0; iphase ^= 1; }
        }
        if (Ly.out_mode) {
          // OUT epilogue input, one panel per slot: the residual gradient d x_out of the block, or the cached output of the conv in
          // front (activation adjoint)
          if (Ly.in_flag_layer >= 0) {
            wait_flag(flags_dx + (size_t)Ly.in_flag_layer * p.num_mtiles + mt, Ly.in_flag_layer, mt);      // (long set, by transitivity of the operand waits)
            fence_proxy_async_global();
          }
          for (int step = 0; step < R_ / 32; ++step) {
            mbar_wait(&in_empty[islot], iphase ^ 1);
            mbar_expect_tx(&in_full[islot], (uint32_t)Cfg::PANEL);
            tma_load_3d_h(in_ring + islot * 2 * Cfg::PANEL, &Ly.tmDXp, &in_full[islot], step * 32, t0, b, p.pol_dx);
            if (++islot == Cfg::IN_SLOTS) { islot = 0; iphase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 12) {
    // ===================== pair hand-off of the d z slabs =====================
    if (lane == 0) {
      int h_rs = 0; uint32_t h_rp = 0u, ad_par = 0u;      // ring position, per-stage parity of the next a_done phase
      for (int j = 0; j < n_tiles; ++j) {
        int n_dg, n_un, n_sh;
        { int ly, mt, b, tb; locate(j, ly, mt, b, tb); tile_ksteps(layers[ly], n_dg, n_un, n_sh); }
        int u_rs = h_rs; uint32_t u_rp = h_rp;
        ring_adv(u_rs, u_rp, n_dg);
        for (int q = 0; q < n_un; q += 2) {
          mbar_wait(&a_done[u_rs], (ad_par >> u_rs) & 1u); ad_par ^= 1u << u_rs;
          if (leader) mbar_arrive(&a_ready[u_rs]);
          else mbar_arrive_remote(&a_ready[u_rs], 0u);
          ring_adv(u_rs, u_rp, 2);
        }
        ring_adv(h_rs, h_rp, n_dg + n_un + n_sh);
      }
    }
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue =====================
    const int e = warp - 4;
    const int quarter = warp & 3;
    const int q = e >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t row_off = (uint32_t)row * 64u;
    const uint32_t sw = (uint32_t)((row >> 1) & 3);
    const uint32_t u0 = (uint32_t)(2 * q), u1 = u0 + 1;
    const uint32_t off0 = row_off + ((u0 ^ sw) << 4), off1 = row_off + ((u1 ^ sw) << 4);
    const uint32_t grow = (uint32_t)row * 128u, gsw = (uint32_t)(row & 7);
    int islot = 0; uint32_t iphase = 0;
    int oslot = 0; uint32_t ophase = 0;
    uint32_t nge = 0u;                 // gated tiles so far
    int e_rs = 0; uint32_t e_rp = 0u;                              // ring position at the start of the current tile
    uint32_t eu_pend = 0u, eu_wpar = 0u, eu_npar = 0u;             // per-stage slab-store bookkeeping (see the producer)
    uint8_t* slab_dst[2] = {nullptr, nullptr};                     // A halves of the stages the current slab pair goes to
    int slab_st[2] = {0, 0};
    const TcEpiGateBwd<true>::Params pg{D_};
    const uint32_t lane_base = (uint32_t)(quarter * 32) << 16;
    SBT_DECL(10)
    for (int j = 0; j < n_tiles; ++j) {
      const uint32_t par = (uint32_t)(j & 1);
      int out_mode, out_act, kind;
      int n_dg, n_un, n_sh;
      const uint8_t* mrow = nullptr;       // this row's keep-mask bytes (dropout on the conv branch this tile differentiates)
      {
        int ly, mt, b, tb;
        locate(j, ly, mt, b, tb);
        out_mode = layers[ly].out_mode; out_act = layers[ly].act; kind = layers[ly].kind;
        tile_ksteps(layers[ly], n_dg, n_un, n_sh);
        const int tt = tb * (2 * Cfg::BM) + pair_row0 + row;
        if (layers[ly].mask && tt < p.T && b < p.B) mrow = layers[ly].mask + ((size_t)b * p.T + tt) * R_;
      }
      if (!kind) {
      const uint32_t gpar = nge & 1u; ++nge;      // the DG accumulator hand-shakes count gated tiles only
      // ---- DG epilogue: d z = d g * [P | Q] -> operand ring
      SBT(0)
      mbar_wait(dg_full, gpar);
      SBT(1)
      tc_fence_after();
      int u_rs = e_rs; uint32_t u_rp = e_rp;
      ring_adv(u_rs, u_rp, n_dg);          // stage of the first un-shifted-tap k-step of this tile
      {
        TmemAccRow acc{tmem_base + lane_base, true};
#pragma unroll 1
        for (int step = 0; step < D_ / 32; ++step) {
          const int pr = step >> 1;
          float in[2][16];
          float out[2][16];
          SBT(2)
          mbar_wait(&in_full[islot], iphase);
          SBT(3)
          {
            const uint8_t* ib = in_ring + islot * 2 * Cfg::PANEL;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const uint4 a = *reinterpret_cast<const uint4*>(ib + k * Cfg::PANEL + off0);
              const uint4 c = *reinterpret_cast<const uint4*>(ib + k * Cfg::PANEL + off1);
              const uint32_t w[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                in[k][2 * i] = __uint_as_float(w[i] << 16);
                in[k][2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&in_empty[islot]);
          if (++islot == Cfg::IN_SLOTS) { islot = 0; iphase ^= 1; }
          TcEpiGateBwd<true>::chunk(pg, acc, 0, step * 32 + q * 16, 0, 0, 3u, in, out, nullptr);
          SBT(2)
          if ((step & 1) == 0) {
            // the two ring stages of this slab pair (filter slab, gate slab): free once the MMAs of their previous use have completed
            // and, if that use carried a slab, its TMA store has read it
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              mbar_wait(&empty_bar[u_rs], u_rp ^ 1u);
              if ((eu_pend >> u_rs) & 1u) { mbar_wait(&sfree[u_rs], (eu_wpar >> u_rs) & 1u); eu_pend &= ~(1u << u_rs); }
              eu_wpar = (eu_wpar & ~(1u << u_rs)) | (((eu_npar >> u_rs) & 1u) << u_rs);
              eu_npar ^= 1u << u_rs; eu_pend |= 1u << u_rs;
              slab_st[k] = u_rs; slab_dst[k] = smem + u_rs * Cfg::STAGE_BYTES;
              ring_adv(u_rs, u_rp, 1);
            }
          }
          SBT(4)
          {
            // channels [ch, ch+16) of this row: 16-byte units (ch % 64) / 8 and +1 of the 128B-swizzled 64-column slab
            const int ch = (step & 1) * 32 + q * 16;
            const uint32_t j0 = (uint32_t)(ch >> 3);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              uint8_t* gs = slab_dst[k] + grow;
              uint4 a, c;
              a.x = pack_bf16x2(out[k][0], out[k][1]); a.y = pack_bf16x2(out[k][2], out[k][3]);
              a.z = pack_bf16x2(out[k][4], out[k][5]); a.w = pack_bf16x2(out[k][6], out[k][7]);
              c.x = pack_bf16x2(out[k][8], out[k][9]); c.y = pack_bf16x2(out[k][10], out[k][11]);
              c.z = pack_bf16x2(out[k][12], out[k][13]); c.w = pack_bf16x2(out[k][14], out[k][15]);
              *reinterpret_cast<uint4*>(gs + ((j0 ^ gsw) << 4)) = a;
              *reinterpret_cast<uint4*>(gs + (((j0 + 1) ^ gsw) << 4)) = c;
            }
          }
          if (step & 1) {
            // slab pair complete in this CTA: store warp (HBM copy) and, through the hand-off warp, the MMA side
            fence_proxy_async();
            named_bar_arrive(8 + pr, NEPI * 32 + 32);
            __syncwarp();
            if (lane == 0) mbar_arrive(&a_done[slab_st[0]]);      // (the pair's hand-off rides on the filter slab's stage)
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_relaxed(dg_empty, 0u);
      }
      // ---- OUT epilogue: d x_out_{l-1} (or the gradient wrt the output of the conv in front)
      SBT(2)
      mbar_wait(out_full, par);
      SBT(5)
      tc_fence_after();
      {
        TmemAccRow acc{tmem_base + 256u + lane_base, true};
#pragma unroll 1
        for (int step = 0; step < R_ / 32; ++step) {
          float v[16];
          acc.load16(step * 32 + q * 16, v);
          if (mrow) {
            // adjoint of the inverted dropout (layers.py:195-196): the conv branch saw keep * x / (1 - rate)
            const uint4 mk = __ldg(reinterpret_cast<const uint4*>(mrow + step * 32 + q * 16));
            const uint32_t mw[4] = {mk.x, mk.y, mk.z, mk.w};
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = ((mw[i >> 2] >> (8 * (i & 3))) & 0xffu) ? v[i] * p.drop_scale : 0.f;
          }
          if (out_mode) {
            mbar_wait(&in_full[islot], iphase);
            const uint8_t* ib = in_ring + islot * 2 * Cfg::PANEL;
            const uint4 a = *reinterpret_cast<const uint4*>(ib + off0);
            const uint4 c = *reinterpret_cast<const uint4*>(ib + off1);
            const uint32_t w[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
            float y[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              y[2 * i] = __uint_as_float(w[i] << 16);
              y[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
            }
            if (out_mode == 1) {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] += y[i];          // residual gradient
            } else {
              wn_act_grad16(out_act, y, v);                       // activation adjoint from the cached output of the conv in front
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&in_empty[islot]);
            if (++islot == Cfg::IN_SLOTS) { islot = 0; iphase ^= 1; }
          }
          uint8_t* ob = out_ring + oslot * Cfg::PANEL;
          SBT(6)
          mbar_wait(&oslot_empty[oslot], ophase ^ 1);
          SBT(7)
          uint4 a, c;
          a.x = pack_bf16x2(v[0], v[1]); a.y = pack_bf16x2(v[2], v[3]); a.z = pack_bf16x2(v[4], v[5]); a.w = pack_bf16x2(v[6], v[7]);
          c.x = pack_bf16x2(v[8], v[9]); c.y = pack_bf16x2(v[10], v[11]); c.z = pack_bf16x2(v[12], v[13]); c.w = pack_bf16x2(v[14], v[15]);
          *reinterpret_cast<uint4*>(ob + off0) = a;
          *reinterpret_cast<uint4*>(ob + off1) = c;
          fence_proxy_async();
          named_bar_arrive(3 + oslot, NEPI * 32 + 32);
          if (++oslot == Cfg::OUT_SLOTS) { oslot = 0; ophase ^= 1; }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote_relaxed(out_empty, 0u);
      ring_adv(e_rs, e_rp, n_dg + n_un + n_sh);
      SBT(6)
    }
#ifdef TC_TIMELINE
    if (lane == 0 && warp == 4 && (blockIdx.x == 0 || blockIdx.x == 41))
      printf("SBWD cta %d epilogue warp 4: wait_dg_full %lld  DG epi work %lld (+ wait z panels %lld, wait slab slot %lld)  wait_out_full %lld  OUT epi work %lld (+ wait out slot %lld)\n",
             blockIdx.x, sbt[1], sbt[2], sbt[3], sbt[4], sbt[5], sbt[6], sbt[7]);
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------- host side
struct TcStackBwdDesc {       // one block
  int B, T, nseg, shift[TC_MAX_TAPS], D, R, S;
  const bf16* dxo;            // d x_out_l (B,T,R) or null (last block under use_skip)
  const bf16* dskip; int lds; // d skip (B,T,S) or null
  const bf16* z;              // cached gate pre-activations (B,T,2D)
  bf16* dz;                   // (B,T,2D), kept for the grouped weight gradients
  bf16* dx;                   // d x_out_{l-1} (B,T,R)
  const bf16* Wdg; int k_dg;  // [D][k_dg] = [Wr^T | Ws^T] rows (first k = R, or S when dxo == null and the pointer is offset)
  const bf16* Wb; int k_b;    // [R][k_b]: dgrad operand of the gated conv, contraction (tap, 2D)
  int has_res;                // use_residual: d x_out_{l-1} += d x_out_l
  const uint8_t* mask; float drop_scale;    // dropout on this block's conv branch (null / 0 = off)
  // multi-dilation blocks: one desc per CONV, in forward order.  plain != 0: a conv in front of the gated conv —
  //   gin (B,T,D) = gradient wrt this conv's output (written by the desc behind this one), Wb its dgrad operand [Cin][nseg*D],
  //   dx (B,T,Cin) the gradient wrt its input.
  // OUT epilogue input `ein` (B,T,R), both kinds: out_mode 1 = residual gradient d x_out of the block (ein_layer = index of the desc
  // whose tile writes it, or -1: written before the launch), out_mode 2 = cached output of the conv in front (activation adjoint), 0 none
  int plain; const bf16* gin;
  int out_mode, act, ein_layer; const bf16* ein;
  int alias;                  // d skip is a second DG segment against the SAME weight columns as d x_out (Wdg = Wr^T only)
};

struct TcStackBwdPlan {
  int B = 0, T = 0, L = 0, num_mtiles = 0; bool drop = false;
  TcStackBwdLayer* d_layers = nullptr; int* d_flags = nullptr;
  void release() { cudaFree(d_layers); cudaFree(d_flags); d_layers = nullptr; d_flags = nullptr; }
};

template <int D_, int R_>
static int tc_stack_bwd_build_t(TmapCache& tc, const std::vector<TcStackBwdDesc>& descs, TcStackBwdPlan* plan) {
  std::vector<TcStackBwdLayer> tab(descs.size());
  for (size_t l = 0; l < descs.size(); ++l) {
    const TcStackBwdDesc& d = descs[l];
    TcStackBwdLayer& t = tab[l];
    memset(&t, 0, sizeof(t));
    const TcEpiIo xo{d.dx, d.R, d.R, 0};
    const CUtensorMap* mO = tc_panel_map(tc, xo, d.T, d.B);
    uint64_t bd[2] = {(uint64_t)d.k_b, (uint64_t)d.R}, bs[1] = {(uint64_t)d.k_b * 2};
    uint32_t bb[2] = {64, (uint32_t)(R_ / 2)};
    const CUtensorMap* mWb = tc.get(d.Wb, 2, bd, bs, bb);
    if (!mO || !mWb) return -10;
    t.tmO = *mO; t.tmWb = *mWb; t.tmDXp = *mO;
    for (int s = 0; s < TC_MAX_TAPS; ++s) t.shift[s] = s < d.nseg ? d.shift[s] : 0;
    t.mask = d.mask;
    t.kind = d.plain ? 1 : 0; t.out_mode = d.out_mode; t.act = d.act; t.in_flag_layer = d.out_mode == 1 ? d.ein_layer : -1;
    if (d.out_mode) {
      const TcEpiIo ei{d.ein, d.R, d.R, 0};
      const CUtensorMap* mp = tc_panel_map(tc, ei, d.T, d.B);
      if (!mp) return -10;
      t.tmDXp = *mp;
    }
    if (d.plain) {
      const CUtensorMap* mG = tc_slab_map(tc, d.gin, d.D, d.D, d.T, d.B);
      if (!mG) return -10;
      t.tmDZ = *mG; t.kb_tap = d.D / 64;
      t.tmDX = *mG; t.tmDS = *mG; t.tmWdg = *mWb; t.tmZf = *mO; t.tmZs = *mO;       // placeholders (a plain layer never touches them)
      continue;
    }
    const CUtensorMap* mDZ = tc_slab_map(tc, d.dz, 2 * d.D, 2 * d.D, d.T, d.B);
    const TcEpiIo zf{d.z, 2 * d.D, d.D, 0}, zs{d.z + d.D, 2 * d.D, d.D, 0};
    const CUtensorMap* mZf = tc_panel_map(tc, zf, d.T, d.B);
    const CUtensorMap* mZs = tc_panel_map(tc, zs, d.T, d.B);
    uint64_t wd[2] = {(uint64_t)d.k_dg, (uint64_t)d.D}, ws[1] = {(uint64_t)d.k_dg * 2};
    uint32_t wb[2] = {64, (uint32_t)(D_ / 2)};
    const CUtensorMap* mWdg = tc.get(d.Wdg, 2, wd, ws, wb);
    if (!mDZ || !mZf || !mZs || !mWdg) return -10;
    t.tmDZ = *mDZ; t.tmZf = *mZf; t.tmZs = *mZs; t.tmWdg = *mWdg;
    t.tmDX = *mDZ; t.tmDS = *mDZ;       // placeholders for absent operands (never dereferenced)
    if (d.dxo) {
      const CUtensorMap* m = tc_act_map(tc, d.dxo, d.R, d.R, d.T, d.B, 1, 0, 128);
      if (!m) return -10;
      t.tmDX = *m;
    }
    if (d.dskip) {
      const CUtensorMap* m = tc_act_map(tc, d.dskip, d.lds, d.S, d.T, d.B, 1, 0, 128);
      if (!m) return -10;
      t.tmDS = *m;
    }
    t.has_dx = d.dxo != nullptr; t.has_ds = d.dskip != nullptr; t.has_res = d.out_mode == 1 ? 1 : 0; t.alias = d.alias;
    t.wait_dx = (d.dxo != nullptr && l + 1 < descs.size()) ? 1 : 0;
  }
  const TcStackBwdDesc& d0 = descs[0];
  plan->release();
  plan->B = d0.B; plan->T = d0.T; plan->L = (int)descs.size(); plan->num_mtiles = d0.B * ((d0.T + 255) / 256); plan->drop = false;
  for (const TcStackBwdDesc& d : descs) if (d.mask) plan->drop = true;
  if (cudaMalloc((void**)&plan->d_layers, tab.size() * sizeof(TcStackBwdLayer)) != cudaSuccess ||
      cudaMemcpy(plan->d_layers, tab.data(), tab.size() * sizeof(TcStackBwdLayer), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMalloc((void**)&plan->d_flags, (size_t)2 * plan->L * plan->num_mtiles * sizeof(int)) != cudaSuccess) {
    snprintf(g_tc_err, sizeof(g_tc_err), "stack backward: plan allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    plan->release();
    return -23;
  }
  return 0;
}

template <int D_, int R_>
static int tc_stack_bwd_launch_t(cudaStream_t st, const TcStackBwdPlan& plan, const TcStackBwdDesc& d0) {
  using Cfg = TcStackBwdCfg<D_, R_>;
  TcStackBwdParams p{};
  p.B = d0.B; p.T = d0.T; p.tiles_t = (d0.T + 255) / 256; p.num_mtiles = d0.B * p.tiles_t; p.L = plan.L;
  p.nseg = d0.nseg; p.kb_dx = d0.R / 64; p.kb_ds = d0.S / 64; p.drop_scale = d0.drop_scale;
  p.pol_dx = tc_policy(TC_L2_NORMAL); p.pol_ds = tc_policy(TC_L2_LAST); p.pol_w = tc_policy(TC_L2_LAST); p.pol_z = tc_policy(TC_L2_FIRST);
  p.pol_dz_ld = tc_policy(TC_L2_NORMAL); p.pol_dz_st = tc_policy(TC_L2_LAST); p.pol_o = tc_policy(TC_L2_LAST);
  auto kern = tc_stack_bwd_kernel<D_, R_>;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  const int pairs = tc_num_sms() / 2;
  if (p.num_mtiles <= pairs) return -100;
  {
    // bands of ~128 m tiles, every band longer than the launch has pairs (a tile then never waits for a tile of the round its own
    // pair is in).
    // (Tried and dropped: issuing DG of a pair's next tile between the un-shifted and the shifted taps of the current one, to
    // fill the d z round trip through L2 — the OUT epilogue then no longer runs under those DG products: 1.79 -> 2.03 ms.)
    constexpr int band_target = 128;
    int nb = p.num_mtiles / band_target;
    if (nb < 1) nb = 1;
    for (; nb > 1; --nb) {
      const int bw = (p.num_mtiles + nb - 1) / nb;
      if (bw > pairs && p.num_mtiles - (nb - 1) * bw > pairs) break;
    }
    p.nbands = nb; p.band = (p.num_mtiles + nb - 1) / nb;
  }
  {
    // every CTA pair of the launch must be resident at the same time (tiles wait for tiles of other pairs)
    static int max_clusters_dev[64];
    static unsigned long long mc_devs = 0ull;
    int& max_clusters = max_clusters_dev[tc_current_device()];
    if (tc_first_use_on_device(&mc_devs)) {
      cudaLaunchConfig_t oc{};
      oc.gridDim = dim3(tc_num_sms()); oc.blockDim = dim3(416); oc.dynamicSmemBytes = Cfg::SMEM_BYTES;
      cudaLaunchAttribute oa[1];
      oa[0].id = cudaLaunchAttributeClusterDimension;
      oa[0].val.clusterDim.x = 2; oa[0].val.clusterDim.y = 1; oa[0].val.clusterDim.z = 1;
      oc.attrs = oa; oc.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, kern, &oc) != cudaSuccess) { n = 0; cudaGetLastError(); }
      max_clusters = n;
    }
    if (pairs > max_clusters) return -100;
  }
  const size_t nflags = (size_t)plan.L * plan.num_mtiles;
  if (cudaMemsetAsync(plan.d_flags, 0, 2 * nflags * sizeof(int), st) != cudaSuccess) return -14;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(416); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 2);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, (const TcStackBwdLayer*)plan.d_layers, plan.d_flags, plan.d_flags + nflags, p);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "stack backward launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

static inline int tc_stack_bwd_build(TmapCache& tc, const std::vector<TcStackBwdDesc>& descs, TcStackBwdPlan* plan) {
  const TcStackBwdDesc& d = descs[0];
  if (d.D == 256 && d.R == 256) return tc_stack_bwd_build_t<256, 256>(tc, descs, plan);
  return -100;
}
static inline int tc_stack_bwd_launch(cudaStream_t st, const TcStackBwdPlan& plan, const TcStackBwdDesc& d) {
  if (d.D == 256 && d.R == 256) return tc_stack_bwd_launch_t<256, 256>(st, plan, d);
  return -100;
}
