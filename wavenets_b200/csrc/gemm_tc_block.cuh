// gemm_tc_block.cuh — fused forward of one WaveNet block's tail (layers.py:199-224) on CTA pairs:
//
//   z = [x_{t-(K-1)d}, .., x_t] . Wg + b (+ conditioning bias)      gated dilated conv   (GATE tiles)
//   g = tanh(z_f) * sigmoid(z_s)                                     gate, in the GATE epilogue
//   x_out = [g | x] . [Wr ; I] + br                                  conv1 + residual     (OUT tile)
//
// in ONE persistent kernel: g never makes the HBM round trip between the two GEMMs (it is still written once, for the
// skip sum and the backward pass), conv1 stops being a separate launch with its own fill / drain, and the residual
// comes through the contraction (identity block), so no epilogue input ring is needed at all.
//
// A CTA pair owns 256 rows (128 per CTA).  Per m tile it runs NT1 = 2D/256 GATE tiles and one OUT tile through the same
// two TMEM accumulator stages (stage = running tile counter & 1):
//   warp 0   TMA producer: GATE k-steps load A (tap box 128x64) + this CTA's half of the Wg tile; OUT k-steps over g
//            load only the [Wr ; I] half-tile, OUT k-steps over x load x + [Wr ; I]
//   warp 1   MMA issuer (leader CTA): GATE as in gemm_tc.cuh; OUT takes its A operand for the first D/64 k-steps from
//            the g buffer in shared memory (K-major, 128B swizzle, written by the GATE epilogue), after `g_full`
//   warp 2   TMEM allocator, then TMA-store warp: z_f / z_s panels, x_out panels, and g straight out of the g buffer
//   warp 3   pair hand-off: waits until this CTA's epilogue has completed g, then arrives on the leader's g_full
//   warps 4-11  epilogue: GATE: tcgen05.ld -> +bias -> z_f, z_s (staged, TMA store) and g -> g buffer;
//               OUT: tcgen05.ld -> +bias -> x_out (staged, TMA store)
#pragma once
#include "gemm_tc.cuh"

// Tile order of one CTA pair over its m tiles m_0 .. m_{n-1} (software pipelined so that the tensor pipe never waits
// for the gate epilogue that completes g):  G_0(m_0) .. G_{NT1-1}(m_0), then for every further m tile
// G_0(m_{j+1}), OUT(m_j), G_1(m_{j+1}) [, ..], and OUT(m_{n-1}) last.  OUT(m_j) is issued behind G_0(m_{j+1}); the
// epilogue of G_h(m_{j+1}) may overwrite its half of the g buffer once OUT(m_j) has consumed it (g_cons[h]).
// kind < NT1: gate tile `kind`; kind == NT1: OUT tile.  j: index of the m tile in this CTA's list.
template <int NT1> __device__ __forceinline__ void blk_tile(int pos, int n, int& kind, int& j) {
  if (pos < NT1) { kind = pos; j = 0; return; }
  const int q = (pos - NT1) / (NT1 + 1), r = (pos - NT1) % (NT1 + 1);
  if (q >= n - 1) { kind = NT1; j = n - 1; return; }
  if (r == 0) { kind = 0; j = q + 1; }
  else if (r == 1) { kind = NT1; j = q; }
  else { kind = r - 1; j = q + 1; }
}

struct TcBlockParams {
  int B, T, tiles_t, num_mtiles;
  int nseg, shift[TC_MAX_TAPS];   // taps of the gated conv (all on the same input tensor)
  int Cin, D, R, has_res;
  const float* bias_g; const float* cbias; const float* bias_r;   // [2D], [B][2D] or null, [R]
  unsigned long long pol_a, pol_w, pol_z, pol_g, pol_o;
  float drop_scale;              // 1 / (1 - rate) of the inverted dropout (stack forward with dropout only)
};

template <int D_, int R_> struct TcBlockCfg {
  static constexpr int BM = 128, BK = 64, BN = 256;
  static constexpr int A_BYTES = BM * BK * 2;                  // 16 KB
  static constexpr int B_BYTES = (BN / 2) * BK * 2;            // this CTA's half of a 256-wide weight tile: 16 KB
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = 4;
  static constexpr int G_BYTES = BM * D_ * 2;                  // 64 KB for D = 256
  static constexpr int PANEL = 128 * 64;                       // 128 rows x 32 bf16
  static constexpr int OUT_SLOTS = 2, SLOT_PANELS = 2;
  static constexpr int NT1 = 2 * D_ / BN;                      // GATE tiles per m tile
  static constexpr int TMEM_COLS = 512;
  // the dynamic shared memory is declared __align__(1024) (128B-swizzled TMA tiles need it), so no alignment slack:
  // 4 x 32 KB ring + 64 KB g + 32 KB staging + 2.5 KB = 231,936 B of the 232,448 B a CTA may have
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + G_BYTES + OUT_SLOTS * SLOT_PANELS * PANEL + 512 /*barriers*/ + 2048 /*bias tables*/;
  static_assert(D_ % 128 == 0 && D_ <= 256 && R_ % 64 == 0 && R_ <= 256, "fused block kernel: D in {128,256}, R <= 256");
  static_assert(SMEM_BYTES <= 232448, "fused block kernel does not fit shared memory");
};

template <int D_, int R_>
__global__ void __launch_bounds__(384, 1)
tc_block_fwd_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW1,
                    const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmZf, const __grid_constant__ CUtensorMap tmZs,
                    const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmO, const TcBlockParams p) {
  using Cfg = TcBlockCfg<D_, R_>;
  constexpr int STAGES = Cfg::STAGES, NEPI = 8, NT1 = Cfg::NT1;
  constexpr int KB_G = D_ / 64, KB_X = R_ / 64;
  extern __shared__ __align__(1024) uint8_t smem_blk[];
  uint8_t* smem = smem_blk;
  if ((smem_u32(smem) & 1023u) != 0u) { if (threadIdx.x == 0) printf("libwavenet_b200: dynamic shared memory is not 1024-byte aligned\n"); __trap(); }
  uint8_t* gbuf = smem + STAGES * Cfg::STAGE_BYTES;                       // [D/64][128 rows][128 B], 128B swizzle
  uint8_t* out_ring = gbuf + Cfg::G_BYTES;
  uint64_t* full_bar = (uint64_t*)(out_ring + Cfg::OUT_SLOTS * Cfg::SLOT_PANELS * Cfg::PANEL);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* out_empty = tempty_bar + 2;
  uint64_t* g_done = out_empty + Cfg::OUT_SLOTS;     // local: this CTA's epilogue has written (and fenced) all of g
  uint64_t* g_full = g_done + 1;                     // leader's: both CTAs' g buffers are complete
  uint64_t* g_free = g_full + 1;                     // local: the TMA stores of g have read the buffer
  uint64_t* g_cons = g_free + 1;                     // [2] local: OUT has consumed the slabs written by gate tile h
  uint32_t* tmem_ptr = (uint32_t*)(g_cons + 2);
  float* bias_s = (float*)(((uintptr_t)(tmem_ptr + 4) + 15) & ~(uintptr_t)15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int tile_first = (int)blockIdx.x >> 1, tile_stride = (int)gridDim.x >> 1;
  const int pair_row0 = (int)crank * Cfg::BM;
  const int kb_a = p.Cin / 64;                        // k-blocks per tap of the gated conv
  const int n_mt = tile_first < p.num_mtiles ? (p.num_mtiles - tile_first + tile_stride - 1) / tile_stride : 0;
  const int n_pos = n_mt * (NT1 + 1);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmW1); tma_prefetch_desc(&tmW2); tma_prefetch_desc(&tmX);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], NEPI * 2); }
    for (int i = 0; i < Cfg::OUT_SLOTS; ++i) mbar_init(&out_empty[i], 1);
    mbar_init(g_done, NEPI); mbar_init(g_full, 2); mbar_init(g_free, 1); mbar_init(&g_cons[0], 1); mbar_init(&g_cons[1], 1);
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
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      auto next = [&]() { if (++stage == STAGES) { stage = 0; phase ^= 1; } };
      constexpr int W2_BYTES = (R_ / 2) * 64 * 2;
      for (int pos = 0; pos < n_pos; ++pos) {
        int kind, j;
        blk_tile<NT1>(pos, n_mt, kind, j);
        const int mt = tile_first + j * tile_stride;
        const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (2 * Cfg::BM) + pair_row0;
        if (kind < NT1) {
          int wk = 0;
          for (int s = 0; s < p.nseg; ++s) {
            for (int kb = 0; kb < kb_a; ++kb) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
              tma_load_4d_pair_h(sa, &tmA, &full_bar[stage], kb * 64, t0 + p.shift[s], b, 0, p.pol_a);
              tma_load_2d_pair_h(sa + Cfg::A_BYTES, &tmW1, &full_bar[stage], wk + kb * 64, kind * Cfg::BN + (int)crank * (Cfg::BN / 2), p.pol_w);
              next();
            }
            wk += p.Cin;
          }
        } else {
          // OUT tile: [g | x] . [Wr ; I]; this CTA's half of the R output columns
          for (int kb = 0; kb < KB_G; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
            if (leader) mbar_expect_tx(&full_bar[stage], 2 * W2_BYTES);
            tma_load_2d_pair_h(sa + Cfg::A_BYTES, &tmW2, &full_bar[stage], kb * 64, (int)crank * (R_ / 2), p.pol_w);
            next();
          }
          if (p.has_res) {
            for (int kb = 0; kb < KB_X; ++kb) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + W2_BYTES));
              tma_load_4d_pair_h(sa, &tmX, &full_bar[stage], kb * 64, t0, b, 0, p.pol_a);
              tma_load_2d_pair_h(sa + Cfg::A_BYTES, &tmW2, &full_bar[stage], D_ + kb * 64, (int)crank * (R_ / 2), p.pol_w);
              next();
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (leader) {
      constexpr uint32_t idesc_g = umma_idesc_bf16(256, Cfg::BN, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16(256, R_, 0, 0);
      int stage = 0; uint32_t phase = 0;
      int as = 0; uint32_t aphase = 0;
      uint32_t gphase = 0;
      const int ksteps_g = p.nseg * kb_a;
      const int ksteps_o = KB_G + (p.has_res ? KB_X : 0);
#ifdef TC_TIMELINE
      long long tl_rec[12][4]; int tl_n = 0; const long long tl_start = clock64();
#endif
      for (int pos = 0; pos < n_pos; ++pos) {
        {
          int kind, j;
          blk_tile<NT1>(pos, n_mt, kind, j);
          const bool is_out = kind == NT1;
          const int ksteps = is_out ? ksteps_o : ksteps_g;
#ifdef TC_TIMELINE
          const long long tl0 = clock64();
#endif
          mbar_wait(&tempty_bar[as], aphase ^ 1);
#ifdef TC_TIMELINE
          const long long tl1 = clock64();
#endif
          if (is_out) { mbar_wait(g_full, gphase); gphase ^= 1; }     // both CTAs' g tiles are in shared memory
#ifdef TC_TIMELINE
          const long long tl2 = clock64();
#endif
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(as * Cfg::BN);
          for (int ks = 0; ks < ksteps; ++ks) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
              const uint32_t a_addr = (is_out && ks < KB_G) ? smem_u32(gbuf) + (uint32_t)ks * (uint32_t)Cfg::A_BYTES : sa;
              const uint64_t adesc = umma_smem_desc(a_addr, 16, 1024);
              const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES, 16, 1024);
#pragma unroll
              for (int k = 0; k < Cfg::BK / 16; ++k)
                umma_bf16_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), is_out ? idesc_o : idesc_g, (ks | k) != 0);
              umma_commit_pair(&empty_bar[stage]);
              if (ks == ksteps - 1) umma_commit_pair(&tfull_bar[as]);
              // the slabs of g written by gate tile h have been read once k-step (h+1)*KB_G/NT1 - 1 of OUT is done
              if (is_out && ks < KB_G && (ks + 1) % (KB_G / NT1) == 0) umma_commit_pair(&g_cons[(ks + 1) / (KB_G / NT1) - 1]);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
#ifdef TC_TIMELINE
          if (tl_n < 12) { tl_rec[tl_n][0] = tl1 - tl0; tl_rec[tl_n][1] = tl2 - tl1; tl_rec[tl_n][2] = clock64() - tl2; tl_rec[tl_n][3] = tl0 - tl_start; ++tl_n; }
#endif
          if (++as == 2) { as = 0; aphase ^= 1; }
        }
      }
#ifdef TC_TIMELINE
      if (blockIdx.x == 0 && lane == 0)
        for (int i = 0; i < tl_n; ++i) printf("BLK mma tile %d: t0 %lld wait_tempty %lld wait_g %lld issue %lld\n", i, tl_rec[i][3], tl_rec[i][0], tl_rec[i][1], tl_rec[i][2]);
#endif
    }
  } else if (warp == 2) {
    // ===================== TMA-store warp =====================
    int oslot = 0, prev = -1;
    auto step_store = [&](const CUtensorMap* m0, const CUtensorMap* m1, int c0, int t0, int b, unsigned long long pol) {
      named_bar_sync(3 + oslot, NEPI * 32 + 32);
      if (lane == 0) {
        const uint8_t* ob = out_ring + oslot * Cfg::SLOT_PANELS * Cfg::PANEL;
        tma_store_3d_h(ob, m0, c0, t0, b, pol);
        if (m1) tma_store_3d_h(ob + Cfg::PANEL, m1, c0, t0, b, pol);
        bulk_commit_group();
        if (prev >= 0) { bulk_wait_group_read<1>(); mbar_arrive(&out_empty[prev]); }
        prev = oslot;
      }
      __syncwarp();
      if (++oslot == Cfg::OUT_SLOTS) oslot = 0;
    };
    for (int pos = 0; pos < n_pos; ++pos) {
      int kind, j;
      blk_tile<NT1>(pos, n_mt, kind, j);
      const int mt = tile_first + j * tile_stride;
      const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (2 * Cfg::BM) + pair_row0;
      if (kind < NT1) {
        for (int step = 0; step < Cfg::BN / 64; ++step) step_store(&tmZf, &tmZs, kind * (Cfg::BN / 2) + step * 32, t0, b, p.pol_z);
        if (kind == NT1 - 1) {
          // g: the whole 128 x D tile straight out of the operand buffer (same 128B-swizzled K-major slabs as a TMA box)
          named_bar_sync(8, NEPI * 32 + 32);
          if (lane == 0) {
#pragma unroll
            for (int kb = 0; kb < KB_G; ++kb) tma_store_3d_h(gbuf + kb * Cfg::A_BYTES, &tmG, kb * 64, t0, b, p.pol_g);
            bulk_commit_group();
            // the very next epilogue tile overwrites g: wait until every store group issued so far has read shared memory
            bulk_wait_group_read<0>();
            if (prev >= 0) { mbar_arrive(&out_empty[prev]); prev = -1; }
            mbar_arrive(g_free);
          }
          __syncwarp();
        }
      } else {
        for (int step = 0; step < R_ / 32; ++step) step_store(&tmO, nullptr, step * 32, t0, b, p.pol_o);
      }
    }
    if (lane == 0) bulk_wait_group<0>();
  } else if (warp == 3) {
    // ===================== pair hand-off of g =====================
    if (lane == 0) {
      uint32_t dphase = 0;
      for (int j = 0; j < n_mt; ++j) {
        mbar_wait(g_done, dphase); dphase ^= 1;
        if (leader) mbar_arrive(g_full);
        else mbar_arrive_remote(g_full, 0u);
      }
    }
  } else {
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
    int as = 0; uint32_t aphase = 0;
    int oslot = 0; uint32_t ophase = 0;

#ifdef TC_TIMELINE
    long long tl_rec[12][3]; int tl_n = 0; const long long tl_start = clock64();
#endif
    const TcEpiGate<true>::Params pg{p.bias_g, p.cbias, D_};
    const TcEpiBiasActRes<true>::Params po{p.bias_r, nullptr, 0, ACT_LINEAR, R_};
    for (int pos = 0; pos < n_pos; ++pos) {
      int nt, j;
      blk_tile<NT1>(pos, n_mt, nt, j);
      const int mt = tile_first + j * tile_stride;
      const int b = mt / p.tiles_t;
      const int bsafe = b < p.B ? b : p.B - 1;
      {
        const bool is_out = nt == NT1;
        const int tid = (int)threadIdx.x - 128;
        float bias_reg = 0.f;
        if (is_out) { if (tid < R_) bias_reg = TcEpiBiasActRes<true>::bias_load(po, bsafe, 0, R_, tid); }
        else bias_reg = TcEpiGate<true>::bias_load(pg, bsafe, nt * (Cfg::BN / 2), Cfg::BN, tid);
#ifdef TC_TIMELINE
        const long long te0 = clock64();
#endif
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
#ifdef TC_TIMELINE
        const long long te1 = clock64();
#endif
        // table double-buffered by tile parity: a warp that runs ahead into the next tile must not overwrite entries
        // other warps still read (the epilogue warps only meet at this barrier, once per tile)
        float* const bs = bias_s + as * 256;
        bs[tid] = bias_reg;
        named_bar_sync(2, NEPI * 32);
        TmemAccRow acc{tmem_base + (uint32_t)(as * Cfg::BN) + ((uint32_t)(quarter * 32) << 16), true};
        if (!is_out) {
          if (j > 0) {
            // this tile's half of the g buffer still holds the previous m tile's g: wait until OUT has consumed it and
            // (first gate tile) until the TMA stores of that g have read the buffer
            mbar_wait(&g_cons[nt], (uint32_t)((j - 1) & 1));
            if (nt == 0) mbar_wait(g_free, (uint32_t)((j - 1) & 1));
          }
#pragma unroll 1
          for (int step = 0; step < Cfg::BN / 64; ++step) {
            float in[1][16];
            float out[3][16];
            TcEpiGate<true>::chunk(pg, acc, bsafe, step * 32 + q * 16, Cfg::BN / 2, 0, 0u, in, out, bs);
            uint8_t* ob = out_ring + oslot * Cfg::SLOT_PANELS * Cfg::PANEL;
            mbar_wait(&out_empty[oslot], ophase ^ 1);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              uint4 a, c;
              a.x = pack_bf16x2(out[k][0], out[k][1]); a.y = pack_bf16x2(out[k][2], out[k][3]);
              a.z = pack_bf16x2(out[k][4], out[k][5]); a.w = pack_bf16x2(out[k][6], out[k][7]);
              c.x = pack_bf16x2(out[k][8], out[k][9]); c.y = pack_bf16x2(out[k][10], out[k][11]);
              c.z = pack_bf16x2(out[k][12], out[k][13]); c.w = pack_bf16x2(out[k][14], out[k][15]);
              *reinterpret_cast<uint4*>(ob + k * Cfg::PANEL + off0) = a;
              *reinterpret_cast<uint4*>(ob + k * Cfg::PANEL + off1) = c;
            }
            {
              // g channels [ch, ch+16) of this row -> operand buffer: slab ch/64, 16-byte units (ch%64)/8 and +1, 128B swizzle
              const int ch = nt * (Cfg::BN / 2) + step * 32 + q * 16;
              uint8_t* gs = gbuf + (ch >> 6) * Cfg::A_BYTES + grow;
              const uint32_t j0 = (uint32_t)((ch & 63) >> 3);
              uint4 a, c;
              a.x = pack_bf16x2(out[2][0], out[2][1]); a.y = pack_bf16x2(out[2][2], out[2][3]);
              a.z = pack_bf16x2(out[2][4], out[2][5]); a.w = pack_bf16x2(out[2][6], out[2][7]);
              c.x = pack_bf16x2(out[2][8], out[2][9]); c.y = pack_bf16x2(out[2][10], out[2][11]);
              c.z = pack_bf16x2(out[2][12], out[2][13]); c.w = pack_bf16x2(out[2][14], out[2][15]);
              *reinterpret_cast<uint4*>(gs + ((j0 ^ gsw) << 4)) = a;
              *reinterpret_cast<uint4*>(gs + (((j0 + 1) ^ gsw) << 4)) = c;
            }
            fence_proxy_async();
            named_bar_arrive(3 + oslot, NEPI * 32 + 32);
            if (++oslot == Cfg::OUT_SLOTS) { oslot = 0; ophase ^= 1; }
          }
          if (nt == NT1 - 1) {
            // g is complete in this CTA (every writer fenced above): let the store warp and the MMA side know
            named_bar_arrive(8, NEPI * 32 + 32);
            __syncwarp();
            if (lane == 0) mbar_arrive(g_done);
          }
        } else {
#pragma unroll 1
          for (int step = 0; step < R_ / 32; ++step) {
            float in[1][16];
            float out[1][16];
            TcEpiBiasActRes<true>::chunk(po, acc, bsafe, step * 32 + q * 16, 0, 0, 0u, in, out, bs);
            uint8_t* ob = out_ring + oslot * Cfg::SLOT_PANELS * Cfg::PANEL;
            mbar_wait(&out_empty[oslot], ophase ^ 1);
            uint4 a, c;
            a.x = pack_bf16x2(out[0][0], out[0][1]); a.y = pack_bf16x2(out[0][2], out[0][3]);
            a.z = pack_bf16x2(out[0][4], out[0][5]); a.w = pack_bf16x2(out[0][6], out[0][7]);
            c.x = pack_bf16x2(out[0][8], out[0][9]); c.y = pack_bf16x2(out[0][10], out[0][11]);
            c.z = pack_bf16x2(out[0][12], out[0][13]); c.w = pack_bf16x2(out[0][14], out[0][15]);
            *reinterpret_cast<uint4*>(ob + off0) = a;
            *reinterpret_cast<uint4*>(ob + off1) = c;
            fence_proxy_async();
            named_bar_arrive(3 + oslot, NEPI * 32 + 32);
            if (++oslot == Cfg::OUT_SLOTS) { oslot = 0; ophase ^= 1; }
          }
        }
#ifdef TC_TIMELINE
        if (tl_n < 12) { tl_rec[tl_n][0] = te1 - te0; tl_rec[tl_n][1] = clock64() - te1; tl_rec[tl_n][2] = te0 - tl_start; ++tl_n; }
#endif
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote_relaxed(&tempty_bar[as], 0u);
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
#ifdef TC_TIMELINE
    if (blockIdx.x == 0 && threadIdx.x == 128)
      for (int i = 0; i < tl_n; ++i) printf("BLK epi tile %d: t0 %lld wait_tfull %lld work %lld\n", i, tl_rec[i][2], tl_rec[i][0], tl_rec[i][1]);
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
}

struct TcBlockDesc {
  int B, T, nseg, shift[TC_MAX_TAPS], Cin, D, R, has_res;
  const bf16* A; int lda;            // input of the gated conv (B,T,Cin)
  const bf16* X; int ldx;            // residual / block input (B,T,R)
  const bf16* W1; int k1;            // gate weights, tile-interleaved [2D][nseg*Cin]
  const bf16* W2;                    // [R][D + R] = [Wr^T | I]
  bf16* z; bf16* g; bf16* xout;      // (B,T,2D), (B,T,D), (B,T,R)
  const float* bias_g; const float* cbias; const float* bias_r;
  // training-mode dropout of the NEXT block's conv branch (layers.py:195-196), applied where x_out is produced (stack forward
  // only): keep-mask bytes [b*T+t][R] of the next block, its masked-and-scaled input (B,T,R), 1 / (1 - rate); null / 0 = off
  const uint8_t* mask_next; bf16* xdrop_next; float drop_scale;
  // stack forward only: plain != 0 describes a conv IN FRONT of the gated conv of a multi-dilation block (layers.py:64-74):
  // xout = act(A taps . W1^T + bias_g), W1 [D][nseg*Cin]; X, W2, z, g, cbias, bias_r unused
  int plain, act;
};

// SW128 tile map over a (B,T,ld) tensor for 64-channel x 128-row boxes (TMA store of the g operand slabs)
static inline const CUtensorMap* tc_slab_map(TmapCache& tc, const bf16* base, int ld, int C, int T, int B) {
  uint64_t dims[3] = {(uint64_t)C, (uint64_t)T, (uint64_t)B};
  uint64_t str[2] = {(uint64_t)ld * 2, (uint64_t)T * ld * 2};
  uint32_t box[3] = {64, 128, 1};
  return tc.get(base, 3, dims, str, box, 128);
}

template <int D_, int R_>
static int tc_block_fwd_launch(TmapCache& tc, cudaStream_t st, const TcBlockDesc& d) {
  using Cfg = TcBlockCfg<D_, R_>;
  const CUtensorMap* mA = tc_act_map(tc, d.A, d.lda, d.Cin, d.T, d.B, 1, 0, 128);
  const CUtensorMap* mX = tc_act_map(tc, d.X, d.ldx, d.R, d.T, d.B, 1, 0, 128);
  uint64_t w1d[2] = {(uint64_t)d.k1, (uint64_t)(2 * d.D)}, w1s[1] = {(uint64_t)d.k1 * 2};
  uint32_t w1b[2] = {64, 128};
  const CUtensorMap* mW1 = tc.get(d.W1, 2, w1d, w1s, w1b);
  uint64_t w2d[2] = {(uint64_t)(d.D + d.R), (uint64_t)d.R}, w2s[1] = {(uint64_t)(d.D + d.R) * 2};
  uint32_t w2b[2] = {64, (uint32_t)(R_ / 2)};
  const CUtensorMap* mW2 = tc.get(d.W2, 2, w2d, w2s, w2b);
  const TcEpiIo zf{d.z, 2 * d.D, d.D, 0}, zs{d.z + d.D, 2 * d.D, d.D, 0}, xo{d.xout, d.R, d.R, 0};
  const CUtensorMap* mZf = tc_panel_map(tc, zf, d.T, d.B);
  const CUtensorMap* mZs = tc_panel_map(tc, zs, d.T, d.B);
  const CUtensorMap* mO = tc_panel_map(tc, xo, d.T, d.B);
  const CUtensorMap* mG = tc_slab_map(tc, d.g, d.D, d.D, d.T, d.B);
  if (!mA || !mX || !mW1 || !mW2 || !mZf || !mZs || !mO || !mG) return -10;
  TcBlockParams p{};
  p.B = d.B; p.T = d.T; p.tiles_t = (d.T + 255) / 256; p.num_mtiles = d.B * p.tiles_t;
  p.nseg = d.nseg;
  for (int s = 0; s < d.nseg; ++s) p.shift[s] = d.shift[s];
  p.Cin = d.Cin; p.D = d.D; p.R = d.R; p.has_res = d.has_res;
  p.bias_g = d.bias_g; p.cbias = d.cbias; p.bias_r = d.bias_r;
  p.pol_a = tc_policy(TC_L2_NORMAL); p.pol_w = tc_policy(TC_L2_LAST);
  p.pol_z = tc_policy(TC_L2_FIRST); p.pol_g = tc_policy(TC_L2_FIRST); p.pol_o = tc_policy(TC_L2_LAST);
  auto kern = tc_block_fwd_kernel<D_, R_>;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  const int slots = tc_balanced_slots(p.num_mtiles, tc_num_sms() / 2);
  const int grid = (p.num_mtiles < slots ? p.num_mtiles : slots) * 2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(384); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 2);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, *mA, *mX, *mW1, *mW2, *mZf, *mZs, *mG, *mO, p);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "fused block forward launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

// supported shapes: D in {128, 256}, R in {128, 256}, Cin % 64 == 0; returns -100 when the caller should use the
// separate gate / conv1 kernels instead
static inline int tc_block_fwd(TmapCache& tc, cudaStream_t st, const TcBlockDesc& d) {
  if (d.Cin % 64 != 0 || d.nseg < 1 || d.nseg > TC_MAX_TAPS) return -100;
  if (d.D == 256 && d.R == 256) return tc_block_fwd_launch<256, 256>(tc, st, d);
  if (d.D == 128 && d.R == 128) return tc_block_fwd_launch<128, 128>(tc, st, d);
  return -100;
}
