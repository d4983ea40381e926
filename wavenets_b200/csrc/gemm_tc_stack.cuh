// gemm_tc_stack.cuh — the fused block forward of gemm_tc_block.cuh (layers.py:199-224) over the WHOLE residual stack
// (the block loop of WaveNet.call, model.py:229-234) as ONE persistent launch.
//
// Per-block launches walk 256 row tiles on 74 CTA pairs in 4 rounds (the last a third full) and pay a launch, a fill and a
// drain per block.  Here a CTA pair walks the (layer, m tile) list of all L layers in layer-major order with the same
// software-pipelined tile order; per-layer tensor maps, tap shifts and bias pointers come from a table in global memory.
// Tile (l, m) reads x_out tiles of layer l-1 (its own rows and the rows its causal taps reach back to, same sequence);
// those were written by OTHER pairs of this launch, so every CTA publishes a tile (TMA stores complete -> proxy fence ->
// release add on flags[l][m]) and a producer acquires the 2-4 flags its boxes touch before the first load of an m tile.
// Dependencies point to smaller ids and every pair walks its ids in ascending order with all CTAs resident (grid <= SMs,
// 1 CTA per SM), so the wait graph has no cycle as long as a layer has more m tiles than the launch has pairs (the
// pipelined order issues G_0 of a pair's NEXT tile before OUT of its current one: that next tile must not depend on it).
//
// Multiple dilations per block (layers.py:64-88,199-200; the reference's shipped topology is 5 blocks x 5): a "layer" of the
// launch is one CONV of the model.  The convs in front of a block's gated conv (Conv1D + bias + activation) are PLAIN layers:
// one 256 x 256 tile per m tile (same operand loads as a gate tile of the kind-0 half, K = taps * Cin), whose epilogue
// applies bias and activation and stores the bf16 output for the next conv (and for the backward pass).  The block's last
// conv is the GATED layer as before; its residual operand X is the BLOCK input (the previous block's x_out), its A operand
// the previous conv's output.  flags[layer][m] therefore count conv outputs, of either kind.
#pragma once
#include "gemm_tc_block.cuh"

// in-kernel phase accounting (clock64 sums over all tiles of one CTA, printed by a few CTAs): -DTC_TIMELINE builds only
#ifdef TC_TIMELINE
#define SFT_DECL(n) long long sft[n] = {}; long long sft_prev = clock64();
#define SFT(i) { const long long sft_now = clock64(); sft[i] += sft_now - sft_prev; sft_prev = sft_now; }
#else
#define SFT_DECL(n)
#define SFT(i)
#endif

#define TC_STACK_MAX_LAYERS 256
struct alignas(128) TcStackLayer {
  CUtensorMap tmA, tmX, tmW1, tmW2, tmZf, tmZs, tmG, tmO, tmOd;
  int shift[TC_MAX_TAPS];
  const float* bias_g; const float* cbias; const float* bias_r;
  const uint8_t* mask_next;      // dropout keep-mask of the next block's conv branch, or null (tmOd: its masked input)
  int kind;                      // 0: gated conv + gate + conv1 (+ residual) = block tail; 1: plain conv + bias + activation
  int act;                       // activation of a plain layer (ACT_*)
};

// Sub-tile sequence of one CTA pair over its (layer, m tile) list t_0 .. t_{n-1}: first(t_0), rest(t_0), then for every j:
// first(t_{j+1}), OUT(t_j), rest(t_{j+1}).  first = gate sub-tile 0 or the PLAIN tile; rest = gate sub-tiles 1..NT1-1; OUT only
// for gated tiles.  (All gated: the order of gemm_tc_block.cuh's blk_tile.)  kind < NT1: gate sub-tile; NT1: OUT; NT1 + 1: PLAIN.
// kmask: one bit per layer (1 = plain), in shared memory (the sequence is walked by four roles on their critical paths: no
// global loads here)
template <int NT1> struct TcStackSeq {
  const uint32_t* kmask; int n, tile_first, tile_stride, num_mtiles;
  int j, ph, r;
  __device__ __forceinline__ TcStackSeq(const uint32_t* km, int n_, int tf, int ts, int nm) : kmask(km), n(n_), tile_first(tf), tile_stride(ts), num_mtiles(nm), j(0), ph(0), r(1) {}
  __device__ __forceinline__ bool plain(int jj) const {
    const int ly = (tile_first + jj * tile_stride) / num_mtiles;
    return ((kmask[ly >> 5] >> (ly & 31)) & 1u) != 0u;
  }
  __device__ __forceinline__ bool next(int& kind, int& jj) {
    for (;;) {
      switch (ph) {
        case 0:
          if (n <= 0) return false;
          ph = 1; r = 1; kind = plain(0) ? NT1 + 1 : 0; jj = 0; return true;
        case 1:
          if (!plain(0) && r < NT1) { kind = r++; jj = 0; return true; }
          ph = 2; j = 0; break;
        case 2:
          ph = 3;
          if (j + 1 < n) { kind = plain(j + 1) ? NT1 + 1 : 0; jj = j + 1; return true; }
          break;
        case 3:
          ph = 4; r = 1;
          if (!plain(j)) { kind = NT1; jj = j; return true; }
          break;
        default:
          if (j + 1 < n && !plain(j + 1) && r < NT1) { kind = r++; jj = j + 1; return true; }
          if (++j >= n) return false;
          ph = 2; break;
      }
    }
  }
};

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add(int* p, int v) {
  asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// orders async-proxy (TMA) accesses to global memory against generic-proxy ones of this thread
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

template <int D_, int R_>
__global__ void __launch_bounds__(384, 1)
tc_stack_fwd_kernel(const TcStackLayer* __restrict__ layers, const int L, int* __restrict__ flags, const TcBlockParams p) {

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
  uint32_t* kmask = (uint32_t*)(bias_s + 512);       // [TC_STACK_MAX_LAYERS / 32] layer kinds, behind the two bias tables

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int tile_first = (int)blockIdx.x >> 1, tile_stride = (int)gridDim.x >> 1;
  const int pair_row0 = (int)crank * Cfg::BM;
  const int kb_a = p.Cin / 64;                        // k-blocks per tap of the gated conv
  const int total_tiles = L * p.num_mtiles;            // (layer, m tile) in layer-major order: dependencies always point to smaller ids
  const int n_mt = tile_first < total_tiles ? (total_tiles - tile_first + tile_stride - 1) / tile_stride : 0;
  constexpr int K_OUT = NT1, K_PLAIN = NT1 + 1;

  if (warp == 0 && lane == 0 && n_mt > 0) {
    const TcStackLayer& L0 = layers[tile_first / p.num_mtiles];
    tma_prefetch_desc(&L0.tmA); tma_prefetch_desc(&L0.tmW1); tma_prefetch_desc(&L0.tmW2); tma_prefetch_desc(&L0.tmX);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], NEPI * 2); }
    for (int i = 0; i < Cfg::OUT_SLOTS; ++i) mbar_init(&out_empty[i], 1);
    mbar_init(g_done, NEPI); mbar_init(g_full, 2); mbar_init(g_free, 1); mbar_init(&g_cons[0], 1); mbar_init(&g_cons[1], 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc_pair<Cfg::TMEM_COLS>(tmem_ptr);
  if (threadIdx.x >= 128 && threadIdx.x < 128 + TC_STACK_MAX_LAYERS / 32) {
    // layer kinds (the table was written by the host when the plan was built, long before this launch)
    const int w = (int)threadIdx.x - 128;
    uint32_t m = 0u;
    for (int l = w * 32; l < L && l < w * 32 + 32; ++l) if (layers[l].kind != 0) m |= 1u << (l & 31);
    kmask[w] = m;
  }
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
      TcStackSeq<NT1> seq(kmask, n_mt, tile_first, tile_stride, p.num_mtiles);
      int kind, j;
      SFT_DECL(4)
      while (seq.next(kind, j)) {
        const int gt = tile_first + j * tile_stride, ly = gt / p.num_mtiles, mt = gt - ly * p.num_mtiles;
        const TcStackLayer& Ly = layers[ly];
        const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (2 * Cfg::BM) + pair_row0;
        SFT(0)
        if (kind != K_OUT) {
          const int wrow = kind == K_PLAIN ? 0 : kind * Cfg::BN;      // first weight row (output column) of this sub-tile
          if ((kind == 0 || kind == K_PLAIN) && ly > 0) {
            // the rows the taps (and the residual) read are x_out tiles of the previous layer, written by other CTA pairs
            // of this launch: wait for both CTAs of each of those tiles (ids are smaller than this tile's: no cycles)
            const int tb = mt % p.tiles_t, row0 = tb * (2 * Cfg::BM);
            const int* fl = flags + (size_t)(ly - 1) * p.num_mtiles + (mt - tb);
            for (int s = 0; s < p.nseg; ++s) {
              const int lo = row0 + Ly.shift[s], hi = lo + 2 * Cfg::BM - 1;
              if (hi < 0) continue;
              const int t_lo = lo < 0 ? 0 : lo / (2 * Cfg::BM);
              int t_hi = hi / (2 * Cfg::BM);
              if (t_hi > p.tiles_t - 1) t_hi = p.tiles_t - 1;
              for (int tt = t_lo; tt <= t_hi; ++tt) {
                const long long spin0 = clock64();
                while (ld_acquire_gpu(fl + tt) < 2) {
                  __nanosleep(32);
                  // every CTA of the launch is resident by construction; if that ever fails, fail loudly instead of hanging
                  if (clock64() - spin0 > 6000000000ll) { printf("libwavenet_b200: stack forward waited > 3 s for tile (%d, %d)\n", ly - 1, mt - tb + tt); __trap(); }
                }
              }
            }
            fence_proxy_async_global();
            SFT(1)
          }
          int wk = 0;
          for (int s = 0; s < p.nseg; ++s) {
            for (int kb = 0; kb < kb_a; ++kb) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
              tma_load_4d_pair_h(sa, &Ly.tmA, &full_bar[stage], kb * 64, t0 + Ly.shift[s], b, 0, p.pol_a);
              tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmW1, &full_bar[stage], wk + kb * 64, wrow + (int)crank * (Cfg::BN / 2), p.pol_w);
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
            tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmW2, &full_bar[stage], kb * 64, (int)crank * (R_ / 2), p.pol_w);
            next();
          }
          if (p.has_res) {
            for (int kb = 0; kb < KB_X; ++kb) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * (Cfg::A_BYTES + W2_BYTES));
              tma_load_4d_pair_h(sa, &Ly.tmX, &full_bar[stage], kb * 64, t0, b, 0, p.pol_a);
              tma_load_2d_pair_h(sa + Cfg::A_BYTES, &Ly.tmW2, &full_bar[stage], D_ + kb * 64, (int)crank * (R_ / 2), p.pol_w);
              next();
            }
          }
        }
      }
      SFT(0)
#ifdef TC_TIMELINE
      if (blockIdx.x == 0 || blockIdx.x == 41) printf("SFWD cta %d producer: tiles %d  ring+issue %lld  wait_flags %lld\n", blockIdx.x, n_mt, sft[0], sft[1]);
#endif
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
      TcStackSeq<NT1> seq(kmask, n_mt, tile_first, tile_stride, p.num_mtiles);
      int kind, j;
      SFT_DECL(8)
      while (seq.next(kind, j)) {
        {
          const bool is_out = kind == K_OUT;
          const int ksteps = is_out ? ksteps_o : ksteps_g;
          SFT(0)
          mbar_wait(&tempty_bar[as], aphase ^ 1);
          SFT(1)
          if (is_out) { mbar_wait(g_full, gphase); gphase ^= 1; }     // both CTAs' g tiles are in shared memory
          SFT(2)
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(as * Cfg::BN);
          for (int ks = 0; ks < ksteps; ++ks) {
            mbar_wait(&full_bar[stage], phase);
            SFT(3)
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
          if (++as == 2) { as = 0; aphase ^= 1; }
        }
      }
#ifdef TC_TIMELINE
      if (lane == 0 && (blockIdx.x == 0 || blockIdx.x == 40))
        printf("SFWD cta %d mma: tiles %d  wait_tempty %lld  wait_g_full %lld  wait_full_bar %lld  issue+other %lld\n", blockIdx.x, n_mt, sft[1], sft[2], sft[3], sft[0]);
#endif
    }
  } else if (warp == 2) {
    // ===================== TMA-store warp =====================
    int oslot = 0, prev = -1, pend_flag = -1, pend_new = -1;
    const bool delay_publish = p.num_mtiles > 2 * tile_stride;
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
    TcStackSeq<NT1> seq(kmask, n_mt, tile_first, tile_stride, p.num_mtiles);
    int kind, j;
    while (seq.next(kind, j)) {
      const int gt = tile_first + j * tile_stride, ly = gt / p.num_mtiles, mt = gt - ly * p.num_mtiles;
      const TcStackLayer& Ly = layers[ly];
      const int b = mt / p.tiles_t, t0 = (mt % p.tiles_t) * (2 * Cfg::BM) + pair_row0;
      if (kind == K_PLAIN) {
        // plain conv: 256 output channels, one panel per step; the tile is the next conv's operand
        for (int step = 0; step < Cfg::BN / 32; ++step) step_store(&Ly.tmO, nullptr, step * 32, t0, b, p.pol_o);
        if (ly + 1 < L) pend_new = ly * p.num_mtiles + mt;
      } else if (kind < NT1) {
        for (int step = 0; step < Cfg::BN / 64; ++step) step_store(&Ly.tmZf, &Ly.tmZs, kind * (Cfg::BN / 2) + step * 32, t0, b, p.pol_z);
        if (kind == NT1 - 1) {
          // g: the whole 128 x D tile straight out of the operand buffer (same 128B-swizzled K-major slabs as a TMA box)
          named_bar_sync(8, NEPI * 32 + 32);
          if (lane == 0) {
#pragma unroll
            for (int kb = 0; kb < KB_G; ++kb) tma_store_3d_h(gbuf + kb * Cfg::A_BYTES, &Ly.tmG, kb * 64, t0, b, p.pol_g);
            bulk_commit_group();
            // the very next epilogue tile overwrites g: wait until every store group issued so far has read shared memory
            bulk_wait_group_read<0>();
            if (prev >= 0) { mbar_arrive(&out_empty[prev]); prev = -1; }
            mbar_arrive(g_free);
          }
          __syncwarp();
        }
      } else {
        // (with dropout: second panel = the next block's conv-branch input keep * x_out / (1 - rate), layers.py:195-196)
        for (int step = 0; step < R_ / 32; ++step) step_store(&Ly.tmO, Ly.mask_next ? &Ly.tmOd : nullptr, step * 32, t0, b, p.pol_o);
        // this CTA's 128 rows of x_out are the next layer's operand: published behind the NEXT tile's stores (below), so
        // that the store warp never waits for a write to land while the epilogue warps are filling the output slots
        if (ly + 1 < L) pend_new = ly * p.num_mtiles + mt;
      }
      if (pend_flag >= 0) {
        // every sub-tile commits at least BN/64 = 4 store groups: once at most 4 are pending, the groups of the sub-tile
        // before this one (the OUT / PLAIN tile whose flag is pending) have completed
        if (lane == 0) {
          bulk_wait_group<4>();
          fence_proxy_async_global();
          __threadfence();
          red_release_gpu_add(flags + pend_flag, 1);
        }
        __syncwarp();
      }
      pend_flag = pend_new; pend_new = -1;
      if (pend_flag >= 0 && !delay_publish) {
        // The sub-tile behind this one may belong to this pair's tile id + 2 * stride (a plain tile has no second sub-tile),
        // which reads layer - 1 tiles down to id + 2 * stride - num_mtiles: with num_mtiles <= 2 * stride that can be THIS
        // tile, so its flag cannot wait for that sub-tile's stores
        if (lane == 0) {
          bulk_wait_group<0>();
          fence_proxy_async_global();
          __threadfence();
          red_release_gpu_add(flags + pend_flag, 1);
        }
        __syncwarp();
        pend_flag = -1;
      }
    }
    if (lane == 0) {
      bulk_wait_group<0>();
      if (pend_flag >= 0) {
        fence_proxy_async_global();
        __threadfence();
        red_release_gpu_add(flags + pend_flag, 1);
      }
    }
    if (lane == 0) bulk_wait_group<0>();
  } else if (warp == 3) {
    // ===================== pair hand-off of g =====================
    if (lane == 0) {
      uint32_t dphase = 0;
      for (int j = 0; j < n_mt; ++j) {
        { const int ly = (tile_first + j * tile_stride) / p.num_mtiles; if ((kmask[ly >> 5] >> (ly & 31)) & 1u) continue; }     // plain convs produce no g
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
    int ng = 0, ng_j = -1;      // gated tiles of this CTA before tile ng_j (the g buffer hand-shakes count gated tiles only)
    SFT_DECL(8)

    TcStackSeq<NT1> seq(kmask, n_mt, tile_first, tile_stride, p.num_mtiles);
    int nt, j;
    while (seq.next(nt, j)) {
      const int gt = tile_first + j * tile_stride, ly = gt / p.num_mtiles, mt = gt - ly * p.num_mtiles;
      const TcStackLayer& Ly = layers[ly];
      const int b = mt / p.tiles_t;
      const int bsafe = b < p.B ? b : p.B - 1;
      const bool is_plain = nt == K_PLAIN;
      if (nt == 0) {
        // first sub-tile of a gated tile: ng = number of gated tiles this CTA has started before it
        if (ng_j >= 0) ++ng;
        ng_j = j;
      }
      const TcEpiGate<true>::Params pg{Ly.bias_g, Ly.cbias, D_};
      // OUT: conv1 bias, linear; PLAIN: the conv's own bias and activation (both 256 = BN columns wide)
      const TcEpiBiasActRes<true>::Params po{is_plain ? Ly.bias_g : Ly.bias_r, nullptr, 0, is_plain ? Ly.act : ACT_LINEAR, is_plain ? Cfg::BN : R_};
      {
        const bool is_out = nt == K_OUT || is_plain;      // one-panel-per-step epilogue
        const int tid = (int)threadIdx.x - 128;
        float bias_reg = 0.f;
        if (is_out) { if (tid < po.N) bias_reg = TcEpiBiasActRes<true>::bias_load(po, bsafe, 0, po.N, tid); }
        else bias_reg = TcEpiGate<true>::bias_load(pg, bsafe, nt * (Cfg::BN / 2), Cfg::BN, tid);
#ifdef TC_TIMELINE
        const int wb = is_plain ? 7 : (nt == K_OUT ? 6 : 5);
#endif
        SFT(4)            // sequence + layer-table reads + bias loads of this sub-tile
        mbar_wait(&tfull_bar[as], aphase);
        SFT(1)
        tc_fence_after();
        // table double-buffered by tile parity: a warp that runs ahead into the next tile must not overwrite entries
        // other warps still read (the epilogue warps only meet at this barrier, once per tile)
        float* const bs = bias_s + as * 256;
        bs[tid] = bias_reg;
        named_bar_sync(2, NEPI * 32);
        TmemAccRow acc{tmem_base + (uint32_t)(as * Cfg::BN) + ((uint32_t)(quarter * 32) << 16), true};
        if (!is_out) {
          if (ng > 0) {
            // this tile's half of the g buffer still holds the previous gated tile's g: wait until OUT has consumed it and
            // (first gate tile) until the TMA stores of that g have read the buffer
            SFT(wb)
            mbar_wait(&g_cons[nt], (uint32_t)((ng - 1) & 1));
            if (nt == 0) mbar_wait(g_free, (uint32_t)((ng - 1) & 1));
            SFT(2)
          }
#pragma unroll 1
          for (int step = 0; step < Cfg::BN / 64; ++step) {
            float in[1][16];
            float out[3][16];
            TcEpiGate<true>::chunk(pg, acc, bsafe, step * 32 + q * 16, Cfg::BN / 2, 0, 0u, in, out, bs);
            uint8_t* ob = out_ring + oslot * Cfg::SLOT_PANELS * Cfg::PANEL;
            SFT(wb)
            mbar_wait(&out_empty[oslot], ophase ^ 1);
            SFT(3)
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
          const uint8_t* const mask_next = is_plain ? nullptr : Ly.mask_next;
#pragma unroll 1
          for (int step = 0; step < po.N / 32; ++step) {
            float in[1][16];
            float out[1][16];
            TcEpiBiasActRes<true>::chunk(po, acc, bsafe, step * 32 + q * 16, 0, 0, 0u, in, out, bs);
            uint4 mk = make_uint4(0u, 0u, 0u, 0u);
            if (mask_next) {
              const int tt = (mt % p.tiles_t) * (2 * Cfg::BM) + pair_row0 + row;
              if (tt < p.T && b < p.B)
                mk = __ldg(reinterpret_cast<const uint4*>(mask_next + ((size_t)b * p.T + tt) * R_ + step * 32 + q * 16));
            }
            uint8_t* ob = out_ring + oslot * Cfg::SLOT_PANELS * Cfg::PANEL;
            SFT(wb)
            mbar_wait(&out_empty[oslot], ophase ^ 1);
            SFT(3)
            uint4 a, c;
            a.x = pack_bf16x2(out[0][0], out[0][1]); a.y = pack_bf16x2(out[0][2], out[0][3]);
            a.z = pack_bf16x2(out[0][4], out[0][5]); a.w = pack_bf16x2(out[0][6], out[0][7]);
            c.x = pack_bf16x2(out[0][8], out[0][9]); c.y = pack_bf16x2(out[0][10], out[0][11]);
            c.z = pack_bf16x2(out[0][12], out[0][13]); c.w = pack_bf16x2(out[0][14], out[0][15]);
            *reinterpret_cast<uint4*>(ob + off0) = a;
            *reinterpret_cast<uint4*>(ob + off1) = c;
            if (mask_next) {
              // keep * (the bf16 value just stored) / (1 - rate), rounded once more: what dropout_apply makes of x_out
              const uint32_t xw[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
              const uint32_t mw[4] = {mk.x, mk.y, mk.z, mk.w};
              uint32_t dw[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const uint32_t k0 = (mw[i >> 1] >> (16 * (i & 1))) & 0xffu, k1 = (mw[i >> 1] >> (16 * (i & 1) + 8)) & 0xffu;
                const float v0 = k0 ? __uint_as_float(xw[i] << 16) * p.drop_scale : 0.f;
                const float v1 = k1 ? __uint_as_float(xw[i] & 0xffff0000u) * p.drop_scale : 0.f;
                dw[i] = pack_bf16x2(v0, v1);
              }
              *reinterpret_cast<uint4*>(ob + Cfg::PANEL + off0) = make_uint4(dw[0], dw[1], dw[2], dw[3]);
              *reinterpret_cast<uint4*>(ob + Cfg::PANEL + off1) = make_uint4(dw[4], dw[5], dw[6], dw[7]);
            }
            fence_proxy_async();
            named_bar_arrive(3 + oslot, NEPI * 32 + 32);
            if (++oslot == Cfg::OUT_SLOTS) { oslot = 0; ophase ^= 1; }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote_relaxed(&tempty_bar[as], 0u);
        if (++as == 2) { as = 0; aphase ^= 1; }
#ifdef TC_TIMELINE
        SFT(wb)
#endif
      }
    }
#ifdef TC_TIMELINE
    if (lane == 0 && warp == 4 && (blockIdx.x == 0 || blockIdx.x == 41))
      printf("SFWD cta %d epilogue warp 4: setup(seq, table, bias) %lld  wait_tfull %lld  wait_g_cons/free %lld  wait_out_slot %lld  work: gate sub-tiles %lld  OUT %lld  plain %lld\n",
             blockIdx.x, sft[4], sft[1], sft[2], sft[3], sft[5], sft[6], sft[7]);
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
}


struct TcStackPlan {
  int B = 0, T = 0, L = 0, num_mtiles = 0; bool cb = false, drop = false;
  TcStackLayer* d_layers = nullptr; int* d_flags = nullptr;
  void release() { cudaFree(d_layers); cudaFree(d_flags); d_layers = nullptr; d_flags = nullptr; }
};

// layers[l]: the TcBlockDesc of conv layer l (a block's gated conv + tail, or one of the plain convs in front of it); same
// Cin = D = R, taps and B, T for every layer
template <int D_, int R_>
static int tc_stack_build_t(TmapCache& tc, const std::vector<TcBlockDesc>& descs, TcStackPlan* plan) {
  std::vector<TcStackLayer> tab(descs.size());
  for (size_t l = 0; l < descs.size(); ++l) {
    const TcBlockDesc& d = descs[l];
    TcStackLayer& t = tab[l];
    memset(&t, 0, sizeof(t));
    const CUtensorMap* mA = tc_act_map(tc, d.A, d.lda, d.Cin, d.T, d.B, 1, 0, 128);
    uint64_t w1d[2] = {(uint64_t)d.k1, (uint64_t)(d.plain ? d.D : 2 * d.D)}, w1s[1] = {(uint64_t)d.k1 * 2};
    uint32_t w1b[2] = {64, 128};
    const CUtensorMap* mW1 = tc.get(d.W1, 2, w1d, w1s, w1b);
    const TcEpiIo xo{d.xout, d.plain ? d.D : d.R, d.plain ? d.D : d.R, 0};
    const CUtensorMap* mO = tc_panel_map(tc, xo, d.T, d.B);
    if (!mA || !mW1 || !mO) return -10;
    t.tmA = *mA; t.tmW1 = *mW1; t.tmO = *mO; t.tmOd = *mO;
    t.tmX = *mA; t.tmW2 = *mW1; t.tmZf = *mO; t.tmZs = *mO; t.tmG = *mO;      // placeholders (a plain layer never touches them)
    t.kind = d.plain ? 1 : 0; t.act = d.act;
    if (!d.plain) {
      const CUtensorMap* mX = tc_act_map(tc, d.X, d.ldx, d.R, d.T, d.B, 1, 0, 128);
      uint64_t w2d[2] = {(uint64_t)(d.D + d.R), (uint64_t)d.R}, w2s[1] = {(uint64_t)(d.D + d.R) * 2};
      uint32_t w2b[2] = {64, (uint32_t)(R_ / 2)};
      const CUtensorMap* mW2 = tc.get(d.W2, 2, w2d, w2s, w2b);
      const TcEpiIo zf{d.z, 2 * d.D, d.D, 0}, zs{d.z + d.D, 2 * d.D, d.D, 0};
      const CUtensorMap* mZf = tc_panel_map(tc, zf, d.T, d.B);
      const CUtensorMap* mZs = tc_panel_map(tc, zs, d.T, d.B);
      const CUtensorMap* mG = tc_slab_map(tc, d.g, d.D, d.D, d.T, d.B);
      if (!mX || !mW2 || !mZf || !mZs || !mG) return -10;
      t.tmX = *mX; t.tmW2 = *mW2; t.tmZf = *mZf; t.tmZs = *mZs; t.tmG = *mG;
      if (d.mask_next && d.xdrop_next) {
        const TcEpiIo xd{d.xdrop_next, d.R, d.R, 0};
        const CUtensorMap* mOd = tc_panel_map(tc, xd, d.T, d.B);
        if (!mOd) return -10;
        t.tmOd = *mOd; t.mask_next = d.mask_next;
      }
    }
    for (int s = 0; s < TC_MAX_TAPS; ++s) t.shift[s] = s < d.nseg ? d.shift[s] : 0;
    t.bias_g = d.bias_g; t.cbias = d.cbias; t.bias_r = d.bias_r;
  }
  const TcBlockDesc& d0 = descs[0];
  if (descs.size() > TC_STACK_MAX_LAYERS) return -100;
  plan->release();
  plan->B = d0.B; plan->T = d0.T; plan->L = (int)descs.size(); plan->num_mtiles = d0.B * ((d0.T + 255) / 256); plan->cb = false; plan->drop = false;
  for (const TcBlockDesc& d : descs) { if (d.cbias) plan->cb = true; if (d.mask_next) plan->drop = true; }
  if (cudaMalloc((void**)&plan->d_layers, tab.size() * sizeof(TcStackLayer)) != cudaSuccess ||
      cudaMemcpy(plan->d_layers, tab.data(), tab.size() * sizeof(TcStackLayer), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMalloc((void**)&plan->d_flags, (size_t)plan->L * plan->num_mtiles * sizeof(int)) != cudaSuccess) {
    snprintf(g_tc_err, sizeof(g_tc_err), "stack forward: plan allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    plan->release();
    return -23;
  }
  return 0;
}

// pairs a stack launch would use; the launch is only valid when a layer has MORE m tiles than that
static inline int tc_stack_pairs(int num_mtiles) { return tc_balanced_slots(num_mtiles, tc_num_sms() / 2); }

template <int D_, int R_>
static int tc_stack_launch_t(cudaStream_t st, const TcStackPlan& plan, const TcBlockDesc& d0) {
  using Cfg = TcBlockCfg<D_, R_>;
  TcBlockParams p{};
  p.B = d0.B; p.T = d0.T; p.tiles_t = (d0.T + 255) / 256; p.num_mtiles = d0.B * p.tiles_t;
  p.nseg = d0.nseg;
  p.Cin = d0.Cin; p.D = d0.D; p.R = d0.R; p.has_res = d0.has_res; p.drop_scale = d0.drop_scale;
  p.pol_a = tc_policy(TC_L2_NORMAL); p.pol_w = tc_policy(TC_L2_LAST);
  p.pol_z = tc_policy(TC_L2_FIRST); p.pol_g = tc_policy(TC_L2_FIRST); p.pol_o = tc_policy(TC_L2_LAST);
  auto kern = tc_stack_fwd_kernel<D_, R_>;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  const int pairs = tc_stack_pairs(p.num_mtiles);
  if (p.num_mtiles <= pairs) return -100;
  {
    // every CTA pair of the launch must be resident at the same time (tiles wait for tiles of other pairs)
    static int max_clusters_dev[64];
    static unsigned long long mc_devs = 0ull;
    int& max_clusters = max_clusters_dev[tc_current_device()];
    if (tc_first_use_on_device(&mc_devs)) {
      cudaLaunchConfig_t oc{};
      oc.gridDim = dim3(tc_num_sms()); oc.blockDim = dim3(384); oc.dynamicSmemBytes = Cfg::SMEM_BYTES;
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
  if (cudaMemsetAsync(plan.d_flags, 0, (size_t)plan.L * plan.num_mtiles * sizeof(int), st) != cudaSuccess) return -14;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * pairs); cfg.blockDim = dim3(384); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 2);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, (const TcStackLayer*)plan.d_layers, plan.L, plan.d_flags, p);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "stack forward launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

static inline int tc_stack_build(TmapCache& tc, const std::vector<TcBlockDesc>& descs, TcStackPlan* plan) {
  const TcBlockDesc& d = descs[0];
  if (d.D == 256 && d.R == 256) return tc_stack_build_t<256, 256>(tc, descs, plan);
  if (d.D == 128 && d.R == 128) return tc_stack_build_t<128, 128>(tc, descs, plan);
  return -100;
}
static inline int tc_stack_launch(cudaStream_t st, const TcStackPlan& plan, const TcBlockDesc& d) {
  if (d.D == 256 && d.R == 256) return tc_stack_launch_t<256, 256>(st, plan, d);
  if (d.D == 128 && d.R == 128) return tc_stack_launch_t<128, 128>(st, plan, d);
  return -100;
}
