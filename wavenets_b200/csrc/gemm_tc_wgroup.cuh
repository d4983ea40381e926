// Grouped weight-gradient launch (bf16 tcgen05 tier, CTA pairs).
//
// Reference: the filter gradients `tape.gradient(loss, trainable_variables)` of every WaveNetLayer (model.py:335) —
// conv backprop-filter of the gated dilated conv (layers.py:199-200), conv1 (layers.py:213) and conv_skip (layers.py:216).
//
// The per-block wgrad launches of gemm_tc.cuh split the (b, t) contraction 18-37 ways to fill the GPU with ONE problem:
// every launch then pays fill/drain, the fp32 partial round trip and a finish launch (profiles/README.md: ~59 us of the
// 95 us a block's weight gradients take are such overhead).  Nothing consumes a weight gradient before the end of the
// backward pass, so here ALL of them run in ONE launch after the dgrad chain: every 256 x 256 output tile of every block
// is a job, split over the rows only as far as the tail of the last wave asks for (1-4 ways), each (job, split) = a
// "unit" = one CTA pair running the same mainloop as tc_wgrad_pair_kernel over 250-1000 64-row chunks instead of 27-56.
// The operands (d z_l, d x_out_l for every block) are kept by the backward chain instead of living in ping-pong buffers.
// Units and tensor maps come from tables in global memory (built once per (B, T) on the host).  Deterministic: the
// finish kernel sums the splits of a tile in a fixed order, no atomics.
#pragma once
#include <algorithm>
#include <map>
#include <tuple>
#include <unordered_map>
#include <vector>

struct TcWgUnit {            // 64 B: one CTA pair's work = one 256-channel A tile against ONE or TWO 256-column G tiles
  int a_map, a_atom;         // tensor-map index (tc_atom_map boxes: 64 rows x 2 atoms) / first 64-channel atom of the 256 A channels
  int shift;                 // time shift of the A rows (causal tap)
  int nh;                    // G tiles (1 or 2): two tiles share every A load -> a quarter less L2 -> SM traffic per product
  int g_map[2], g_atom[2];   // per G tile: tensor map, first 64-column atom
  int out_tile[2];           // [256][256] fp32 partial tile of each product
  int cs_row0[2];            // first row of this unit's column-sum rows of each G tile (< 0: no column sums for it):
                             // cs[(cs_row0 + batch - first batch) * 256 + col]
  int c_begin, c_end;        // 64-row chunks [c_begin, c_end) of the flattened (b, t) axis
  int cs_r0, cs_r1;          // rows of every 64-row chunk this unit adds up for the column sums
  int share_g, shift2;       // share_g != 0 (nh == 2): the two products are two TAPS of one conv against the SAME G tile — the second
                             // A tile (same channels, time shift shift2) takes the second G slot of the stage; one G load for two
                             // products (the plain convs of a multi-dilation block have one 256-column G tile and K taps)
};

struct TcWgGroupParams {
  const CUtensorMap* maps;
  const TcWgUnit* units;
  float* cs;
  int chunks_t;              // ceil(T / 64)
  int unit_base;             // this launch works on units [unit_base, unit_base + gridDim.x / 2)
};

__global__ void __launch_bounds__(256, 1)
tc_wgrad_group_kernel(const __grid_constant__ CUtensorMap tmP, const TcWgGroupParams p) {
  using Cfg = TcWgradPairCfg<256, 2>;     // 4 stages of 16 KB (A) + 2 x 16 KB (G) per CTA, all 512 TMEM columns
  constexpr int STAGES = Cfg::STAGES;
  constexpr int BN = 256, HALF = 128, NH = 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* mma_done = empty_bar + STAGES;
  uint64_t* tfull_bar = mma_done + STAGES;
  uint32_t* tmem_ptr = (uint32_t*)(tfull_bar + 1);
  float* cs_s = (float*)(smem + STAGES * Cfg::STAGE_BYTES + 1024);      // [RH][NH * HALF] column-sum hand-over between row halves

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const TcWgUnit u = p.units[p.unit_base + (blockIdx.x >> 1)];
  const int nchunks = u.c_end - u.c_begin;
  const bool cs_on[2] = {u.cs_r1 > u.cs_r0 && u.cs_row0[0] >= 0, u.nh > 1 && u.cs_r1 > u.cs_r0 && u.cs_row0[1] >= 0};
  const bool do_cs = cs_on[0] || cs_on[1];

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
      const CUtensorMap* tmA = p.maps + u.a_map;
      const CUtensorMap* tmG0 = p.maps + u.g_map[0];
      const CUtensorMap* tmG1 = p.maps + u.g_map[1];
      tma_prefetch_desc(tmA);
      tma_prefetch_desc(tmG0);
      if (u.nh > 1) tma_prefetch_desc(tmG1);
      const int a_atom = u.a_atom + 2 * (int)crank, g_atom0 = u.g_atom[0] + 2 * (int)crank, g_atom1 = u.g_atom[1] + 2 * (int)crank;
      const uint32_t tx = 2u * (uint32_t)(Cfg::A_BYTES + u.nh * Cfg::GH_BYTES);
      int stage = 0; uint32_t phase = 0;
      int b = u.c_begin / p.chunks_t, ct = u.c_begin % p.chunks_t;
      for (int ch = u.c_begin; ch < u.c_end; ++ch) {
        const int t0 = ct * Cfg::BKT;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
        if (leader) mbar_expect_tx(&full_bar[stage], tx);
        // sibling units (other taps / column tiles of the same block) read the same boxes at about the same time: normal policy
        tma_load_4d_pair_h(sa, tmA, &full_bar[stage], 0, t0 + u.shift, a_atom, b, TC_POL_NORMAL);
        tma_load_4d_pair_h(sa + Cfg::A_BYTES, tmG0, &full_bar[stage], 0, t0, g_atom0, b, TC_POL_NORMAL);
        if (u.nh > 1) {
          if (u.share_g) tma_load_4d_pair_h(sa + Cfg::A_BYTES + Cfg::GH_BYTES, tmA, &full_bar[stage], 0, t0 + u.shift2, a_atom, b, TC_POL_NORMAL);
          else tma_load_4d_pair_h(sa + Cfg::A_BYTES + Cfg::GH_BYTES, tmG1, &full_bar[stage], 0, t0, g_atom1, b, TC_POL_NORMAL);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
        if (++ct == p.chunks_t) { ct = 0; ++b; }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BN, 1, 1);   // both operands MN-major
      int stage = 0; uint32_t phase = 0;
      for (int it = 0; it < nchunks; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          for (int hh = 0; hh < u.nh; ++hh) {
            const uint64_t adesc = umma_smem_desc((u.share_g && hh) ? sa + Cfg::A_BYTES + Cfg::GH_BYTES : sa, 8192, 1024);
            const uint64_t bdesc = umma_smem_desc(sa + Cfg::A_BYTES + (u.share_g ? 0 : hh) * Cfg::GH_BYTES, 8192, 1024);
#pragma unroll
            for (int k = 0; k < Cfg::BKT / 16; ++k)
              umma_bf16_pair(tmem_base + (uint32_t)(hh * BN), adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, (it | k) != 0);
          }
          // with column sums the stage is released by the summing warps, which first wait for these MMAs
          umma_commit_pair(do_cs ? &mma_done[stage] : &empty_bar[stage]);
          if (it == nchunks - 1) umma_commit_pair(tfull_bar);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    if (do_cs) {
      // 128 threads: 64 column pairs of this CTA's 128 columns of each G tile x 2 row halves of the unit's row slice
      const int tid = threadIdx.x - 128;
      constexpr int NPAIR = HALF / 2;
      constexpr int RH = 128 / NPAIR;
      const int pr = tid % NPAIR, rh = tid / NPAIR;
      const int c = 2 * pr;
      const int atom = c >> 6, cc = c & 63;
      const uint32_t col_off = (uint32_t)(atom * 8192 + (cc & 7) * 2);
      const uint32_t chunk = (uint32_t)(cc >> 3);
      const int len = u.cs_r1 - u.cs_r0;
      const int r_lo = u.cs_r0 + (len * rh) / RH, r_hi = u.cs_r0 + (len * (rh + 1)) / RH;
      float s0[NH] = {0.f, 0.f}, s1[NH] = {0.f, 0.f};
      int stage = 0; uint32_t phase = 0;
      int cur_b = u.c_begin / p.chunks_t;
      const int b_first = cur_b;
      auto flush = [&](int slot) {
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) { cs_s[(rh * NH + hh) * HALF + c] = s0[hh]; cs_s[(rh * NH + hh) * HALF + c + 1] = s1[hh]; }
        named_bar_sync(7, 128);
        if (rh == 0) {
#pragma unroll
          for (int hh = 0; hh < NH; ++hh) {
            if (!cs_on[hh]) continue;
            float t0 = 0.f, t1 = 0.f;
#pragma unroll
            for (int h2 = 0; h2 < RH; ++h2) { t0 += cs_s[(h2 * NH + hh) * HALF + c]; t1 += cs_s[(h2 * NH + hh) * HALF + c + 1]; }
            float* o = p.cs + (long long)(u.cs_row0[hh] + slot) * BN + (int)crank * HALF + c;
            o[0] = t0; o[1] = t1;
          }
        }
        named_bar_sync(7, 128);
      };
      int ct = u.c_begin % p.chunks_t, b = cur_b;
      for (int ch = u.c_begin; ch < u.c_end; ++ch) {
        if (b != cur_b) {
          flush(cur_b - b_first);
#pragma unroll
          for (int hh = 0; hh < NH; ++hh) s0[hh] = s1[hh] = 0.f;
          cur_b = b;
        }
        mbar_wait(&mma_done[stage], phase);
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) {
          if (!cs_on[hh]) continue;
          const uint8_t* g = smem + stage * Cfg::STAGE_BYTES + Cfg::A_BYTES + hh * Cfg::GH_BYTES + col_off;
#pragma unroll 8
          for (int r = r_lo; r < r_hi; ++r) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(g + r * 128 + ((chunk ^ (uint32_t)(r & 7)) << 4));
            s0[hh] += __uint_as_float(w << 16);
            s1[hh] += __uint_as_float(w & 0xffff0000u);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
        if (++ct == p.chunks_t) { ct = 0; ++b; }
      }
      if (nchunks > 0) flush(cur_b - b_first);
    }
    const int quarter = warp & 3;
    if (nchunks > 0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    // partial tiles (this CTA's 128 channels x 256 fp32 each) -> the operand ring (free: every MMA has completed) as 8 boxes of
    // 128 rows x 32 floats, 128B swizzle -> TMA stores
    {
      const int r = quarter * 32 + lane;
      const uint32_t rsw = (uint32_t)(r & 7);
      uint8_t* const rowp = smem + (uint32_t)r * 128u;
#pragma unroll 1
      for (int hh = 0; hh < u.nh; ++hh) {
        if (hh > 0) {
          // the staging area is reused: its TMA stores must have read it
          if (threadIdx.x == 128) bulk_wait_group_read<0>();
          named_bar_sync(6, 128);
        }
        for (int c = 0; c < BN; c += 16) {
          float v[16];
          if (nchunks > 0) tmem_ld16(taddr + (uint32_t)(hh * BN + c), v);
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
#pragma unroll
          for (int bx = 0; bx < BN / 32; ++bx) tma_store_3d_h(smem + bx * 16384, &tmP, bx * 32, (int)crank * 128, u.out_tile[hh], TC_POL_NORMAL);
          bulk_commit_group();
        }
      }
      if (threadIdx.x == 128) bulk_wait_group<0>();
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------- finish: split sums -> Keras layouts, column sums -> biases
struct TcWgFinTile {        // one 256 x 256 output tile
  float* dst;               // &grad[row0 * ld + col0] (Keras layout [ktot][N])
  const float* w;           // matching weights for the L2 term, or null
  int ld;
  int tile0, nsplit;        // partial tiles tile0 .. tile0 + nsplit - 1
  int pad;
};
#define TC_WG_MAX_CS_SRC 32
struct TcWgFinCs {          // column sums of one 256-column tile of a G tensor
  float* bias;              // [256] or null
  float* per_batch;         // &per_batch[col0], row stride ldpb, or null
  int ldpb, nsrc;
  int row0[TC_WG_MAX_CS_SRC], b_first[TC_WG_MAX_CS_SRC], nb[TC_WG_MAX_CS_SRC];   // source units: cs rows, first batch, batches covered
};
struct TcWgFinParams {
  const float* partial; const float* cs;
  const TcWgFinTile* tiles; int ntiles;
  const TcWgFinCs* css; int ncs;
  float l2coef; int B;
};
// grid: ntiles * 64 blocks (4 rows x 256 columns each, float4 per thread) + ncs blocks
__global__ void __launch_bounds__(256) tc_wgrad_group_finish(const TcWgFinParams f) {
  pdl_launch_dependents();
  pdl_wait();
  const int bid = (int)blockIdx.x;
  if (bid < f.ntiles * 64) {
    const TcWgFinTile t = f.tiles[bid >> 6];
    const int r = ((bid & 63) << 2) + (threadIdx.x >> 6), c = (threadIdx.x & 63) << 2;
    const float4* src = reinterpret_cast<const float4*>(f.partial + ((long long)t.tile0 << 16) + r * 256 + c);
    float4 s = src[0];
    for (int i = 1; i < t.nsplit; ++i) {
      const float4 v = src[(long long)i << 14];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    const long long o = (long long)r * t.ld + c;
    if (t.w) {
      const float4 w = *reinterpret_cast<const float4*>(t.w + o);
      s.x = fmaf(f.l2coef, w.x, s.x); s.y = fmaf(f.l2coef, w.y, s.y); s.z = fmaf(f.l2coef, w.z, s.z); s.w = fmaf(f.l2coef, w.w, s.w);
    }
    *reinterpret_cast<float4*>(t.dst + o) = s;
    return;
  }
  const TcWgFinCs& e = f.css[bid - f.ntiles * 64];
  const int n = threadIdx.x;
  float tot = 0.f;
  for (int b = 0; b < f.B; ++b) {
    float sb = 0.f;
    for (int s = 0; s < e.nsrc; ++s) {
      const int k = b - e.b_first[s];
      if (k >= 0 && k < e.nb[s]) sb += f.cs[(long long)(e.row0[s] + k) * 256 + n];
    }
    if (e.per_batch) e.per_batch[(long long)b * e.ldpb + n] = sb;
    tot += sb;
  }
  if (e.bias) e.bias[n] = tot;
}

// ---------------------------------------------------------------- host side: plan
struct TcWgJobDesc {         // one weight-gradient problem dW[k * Cin + c, n] = sum_{b,t} A[(b, t + shift_k), c] * G[(b, t), n]
  const bf16* A; int lda; int cin; int ntaps; int shift[TC_MAX_TAPS];
  const bf16* G; int ldg; int N;
  float* dst; const float* w;            // [ntaps * cin][N] fp32 gradient (Keras layout), weights for L2 (or null)
  float* bias;                           // [N] column sums of G, or null
  float* per_batch; int ldpb;            // [B][ldpb] per-batch column sums of G, or null
  // acc_prev: this problem's product is ADDED to the previous problem's gradient (same dst; both one 256 x 256 tile): its partial
  // tiles follow the previous problem's and the finish sums them all — conv1 under skip_channels=None sees d x_out + d skip
  // (layers.py:217-218), two G tensors against the same A.  bias_add_G: the column sums of that other G tensor are added to `bias`.
  bool acc_prev = false; const bf16* bias_add_G = nullptr;
  int bucket = 0;                        // final-launch jobs only: the final launch runs as one launch + finish per bucket, in bucket
                                         // order, so that the gradients of bucket k can be all-reduced while bucket k + 1 is computed
  int group = -1;                        // -1: the launch at the end of the backward pass; g >= 0: side launch g (one per block
                                         // that hands its weight gradients to the SMs the dgrad chain leaves idle)
  // several problems may share one G (conv_skip of every block reads d skip): the column sums are computed once, by the
  // first problem that names the tensor, and the finish writes them to every bias that asks for them
};

struct TcWgGroupPlan {
  int B = 0, T = 0;
  int nunits = 0, ntiles = 0, nfin = 0, ncs = 0, nsplit = 1, npartial = 0;   // ntiles: 256 x 256 products; nfin: gradient tiles the finish writes
  int final_units = 0;                                   // units [0, final_units): the launch at the end
  struct Bucket { int unit0, nunits, tile0, ntiles, cs0, ncs; };
  std::vector<Bucket> buckets;                           // the final launch, bucket by bucket (tiles / column-sum entries of a bucket are contiguous)
  std::vector<std::pair<int, int>> side;                 // per side group: (first unit, units)
  CUtensorMap* d_maps = nullptr; TcWgUnit* d_units = nullptr; TcWgFinTile* d_tiles = nullptr; TcWgFinCs* d_css = nullptr;
  float* d_partial = nullptr; float* d_cs = nullptr;
  CUtensorMap tmP;
  void release() {
    cudaFree(d_maps); cudaFree(d_units); cudaFree(d_tiles); cudaFree(d_css); cudaFree(d_partial); cudaFree(d_cs);
    d_maps = nullptr; d_units = nullptr; d_tiles = nullptr; d_css = nullptr; d_partial = nullptr; d_cs = nullptr;
  }
};

// every problem must have cin % 256 == 0 and N % 256 == 0
static inline bool tc_wgrad_group_ok(int cin, int N) { return cin % 256 == 0 && N % 256 == 0; }

static int tc_wgrad_group_build(TmapCache& tc, const std::vector<TcWgJobDesc>& jobs_in, int B, int T, int force_split, bool pair_tiles, int side_pairs, TcWgGroupPlan* plan) {
  plan->release();
  plan->B = B; plan->T = T;
  // final-launch jobs in bucket order (stable), side-launch jobs behind them
  std::vector<TcWgJobDesc> jobs(jobs_in);
  std::stable_sort(jobs.begin(), jobs.end(), [](const TcWgJobDesc& a, const TcWgJobDesc& b) {
    const int ka = a.group >= 0 ? (1 << 20) + a.group : a.bucket, kb = b.group >= 0 ? (1 << 20) + b.group : b.bucket;
    return ka < kb;
  });
  int nbuckets = 1;
  for (const auto& j : jobs) if (j.group < 0 && j.bucket + 1 > nbuckets) nbuckets = j.bucket + 1;
  std::vector<CUtensorMap> maps;
  std::map<std::tuple<const void*, int, int>, int> map_of;
  auto map_idx = [&](const bf16* p, int ld, int width) -> int {
    const auto key = std::make_tuple((const void*)p, ld, width);
    auto it = map_of.find(key);
    if (it != map_of.end()) return it->second;
    const CUtensorMap* m = tc_atom_map(tc, p, ld, width, T, B, 64, 2);
    if (!m) return -1;
    maps.push_back(*m);
    map_of[key] = (int)maps.size() - 1;
    return (int)maps.size() - 1;
  };
  const int chunks_t = (T + 63) / 64, total_chunks = B * chunks_t;
  // ---- 256 x 256 output tiles, column-sum entries
  struct Tile { int a_map, a_atom, shift, g_map, g_atom; int cs_entry; int cs_r0, cs_r1; bool used; int group; int bucket; };
  std::vector<int> cs_bucket;                            // bucket of every TcWgFinCs entry (side-launch jobs: the last bucket)
  std::vector<Tile> tl;
  std::vector<TcWgFinTile> tiles;
  std::vector<TcWgFinCs> css;
  std::unordered_map<const void*, int> cs_of;            // G tensor -> index of its first TcWgFinCs entry (one per 256 columns)
  std::vector<int> fin_of;                               // tile -> index of the finish tile that sums its partials
  std::vector<std::pair<int, const void*>> cs_extra;     // (column-sum entry, other G tensor whose sums are added to it)
  for (const auto& j : jobs) {
    if (j.acc_prev && (j.cin != 256 || j.N != 256 || j.ntaps != 1 || tiles.empty() || tiles.back().dst != j.dst)) {
      snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad: an accumulating problem must be one 256 x 256 tile behind the problem it adds to");
      return -25;
    }
    if (!tc_wgrad_group_ok(j.cin, j.N)) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad: widths %d x %d not multiples of 256", j.cin, j.N); return -20; }
    const int am = map_idx(j.A, j.lda, j.cin), gm = map_idx(j.G, j.ldg, j.N);
    if (am < 0 || gm < 0) return -21;
    const bool want_cs = j.bias || j.per_batch;
    bool own_cs = false;
    int cs0 = -1;
    if (want_cs) {
      auto it = cs_of.find(j.G);
      own_cs = it == cs_of.end();
      if (own_cs) { cs0 = (int)css.size(); cs_of[j.G] = cs0; } else cs0 = it->second;
      // (a later problem on the same G gets copies of the owner's entries with its own destinations, see below)
      if (own_cs)
        for (int nt = 0; nt < j.N / 256; ++nt) {
          TcWgFinCs e{};
          e.bias = j.bias ? j.bias + nt * 256 : nullptr;
          e.per_batch = j.per_batch ? j.per_batch + nt * 256 : nullptr;
          e.ldpb = j.ldpb; e.nsrc = 0;
          if (j.bias_add_G && nt == 0) cs_extra.push_back(std::make_pair((int)css.size(), (const void*)j.bias_add_G));
          css.push_back(e);
          cs_bucket.push_back(j.group < 0 ? j.bucket : nbuckets - 1);
        }
    }
    // the tiles that share a G tile split the 64 rows of a chunk between them for the column sums
    const int sharers = j.ntaps * (j.cin / 256);
    int sh = 0;
    for (int k = 0; k < j.ntaps; ++k)
      for (int mt = 0; mt < j.cin / 256; ++mt, ++sh)
        for (int nt = 0; nt < j.N / 256; ++nt) {
          if (j.acc_prev) {
            fin_of.push_back((int)tiles.size() - 1);      // no finish tile of its own: its partials extend the previous one's
          } else {
            TcWgFinTile ft{};
            ft.dst = j.dst + ((long long)(k * j.cin + mt * 256)) * j.N + nt * 256;
            ft.w = j.w ? j.w + ((long long)(k * j.cin + mt * 256)) * j.N + nt * 256 : nullptr;
            ft.ld = j.N; ft.tile0 = 0; ft.nsplit = 0;
            tiles.push_back(ft);
            fin_of.push_back((int)tiles.size() - 1);
          }
          Tile t{};
          t.a_map = am; t.a_atom = mt * 4; t.shift = j.shift[k]; t.g_map = gm; t.g_atom = nt * 4;
          t.cs_entry = own_cs ? cs0 + nt : -1;
          t.cs_r0 = (64 * sh) / sharers; t.cs_r1 = (64 * (sh + 1)) / sharers;
          t.used = false; t.group = j.group; t.bucket = j.group < 0 ? j.bucket : nbuckets - 1;
          tl.push_back(t);
        }
    if (want_cs && !own_cs) {
      // same column sums, another destination: the sources are copied from the owner once they are known (second pass)
      for (int nt = 0; nt < j.N / 256; ++nt) {
        TcWgFinCs e{};
        e.bias = j.bias ? j.bias + nt * 256 : nullptr;
        e.per_batch = j.per_batch ? j.per_batch + nt * 256 : nullptr;
        e.ldpb = j.ldpb; e.nsrc = -1 - (cs0 + nt);      // marks "copy of entry cs0 + nt"
        css.push_back(e);
        cs_bucket.push_back(j.group < 0 ? j.bucket : nbuckets - 1);
      }
    }
  }
  const int ntiles = (int)tl.size();
  // ---- pair up tiles that read the same A tile (same rows, channels and shift): one unit, one A load for two products.
  // Column-sum duty needs equal row slices in both halves (the unit has one [cs_r0, cs_r1)); otherwise the second loses it...
  // so only tiles with the same slice (or no duty on one side) are paired.
  static_assert(TcWgradPairCfg<256, 2>::A_BYTES == TcWgradPairCfg<256, 2>::GH_BYTES, "share_g units put an A tile into a G slot");
  struct UnitT { int t[2]; int nh; int share_g; };
  std::vector<UnitT> ut;
  for (int i = 0; i < ntiles; ++i) {
    if (tl[i].used) continue;
    tl[i].used = true;
    UnitT uu{{i, -1}, 1, 0};
    if (pair_tiles)
      for (int k = i + 1; k < ntiles && k < i + 64; ++k) {
        if (tl[k].used) continue;
        const Tile &x = tl[i], &y = tl[k];
        if (x.a_map != y.a_map || x.a_atom != y.a_atom || x.shift != y.shift || x.group != y.group || x.bucket != y.bucket) continue;
        const bool cx = x.cs_entry >= 0, cy = y.cs_entry >= 0;
        if (cx && cy && (x.cs_r0 != y.cs_r0 || x.cs_r1 != y.cs_r1)) continue;
        uu.t[1] = k; uu.nh = 2; tl[k].used = true;
        break;
      }
    if (pair_tiles && uu.nh == 1)
      // no partner on the same A tile: two taps of the same conv against the same G tile (same A channels, another time shift)
      for (int k = i + 1; k < ntiles && k < i + 64; ++k) {
        if (tl[k].used) continue;
        const Tile &x = tl[i], &y = tl[k];
        if (x.g_map != y.g_map || x.g_atom != y.g_atom || x.a_map != y.a_map || x.a_atom != y.a_atom || x.shift == y.shift || x.group != y.group || x.bucket != y.bucket) continue;
        // column-sum duty: both name the same G tile; their row slices must be adjacent (the unit sums one range)
        if (x.cs_entry != y.cs_entry || (x.cs_entry >= 0 && x.cs_r1 != y.cs_r0)) continue;
        uu.t[1] = k; uu.nh = 2; uu.share_g = 1; tl[k].used = true;
        break;
      }
    ut.push_back(uu);
  }
  // ---- launch order: the units of the final launch first, then every side group's units side by side
  int ngroups = 0;
  for (const auto& t : tl) if (t.group + 1 > ngroups) ngroups = t.group + 1;
  std::vector<std::vector<int>> by_group(ngroups + 1);     // [0]: final, [1 + g]: side group g
  for (int i = 0; i < (int)ut.size(); ++i) by_group[tl[ut[i].t[0]].group + 1].push_back(i);
  // ---- splits of the final launch, per bucket: simulate the block scheduler (units in launch order onto the earliest free CTA pair)
  const int npairs = tc_num_sms() / 2;
  auto norm_split = [&](int s) { const int cps = (total_chunks + s - 1) / s; return (total_chunks + cps - 1) / cps; };
  auto pick_split = [&](const std::vector<int>& us) -> int {
    int ns = 1;
    if (force_split > 0) ns = force_split;
    else if (!us.empty()) {
      double best = 1e30;
      for (int s = 1; s <= 8; ++s) {
        if (s > total_chunks) break;
        std::vector<double> free_at(npairs, 0.0);
        for (int z0 : us)
          for (int z = 0; z < s; ++z) {
            auto it = std::min_element(free_at.begin(), free_at.end());
            // mainloop chunks x products (+ a per-unit fixed cost: fill, partial store and its later reduction, in chunk units)
            *it += (double)total_chunks / s * (ut[z0].nh == 2 ? 1.55 : 1.0) + 12.0 * ut[z0].nh;
          }
        const double mk = *std::max_element(free_at.begin(), free_at.end());
        if (mk < best * 0.995) { best = mk; ns = s; }
      }
    }
    if (ns > total_chunks) ns = total_chunks;
    if (ns > 8) ns = 8;
    return norm_split(ns);
  };
  std::vector<std::vector<int>> by_bucket(nbuckets);
  for (int ui : by_group[0]) by_bucket[tl[ut[ui].t[0]].bucket].push_back(ui);
  std::vector<int> split_bk(nbuckets, 1);
  for (int b = 0; b < nbuckets; ++b) split_bk[b] = pick_split(by_bucket[b]);
  const int nsplit = split_bk[0];
  std::vector<int> split_of(ngroups + 1, nsplit);
  for (int g = 0; g < ngroups; ++g) {
    // a side launch never asks for more CTA pairs than the dgrad chain leaves free
    const int n = (int)by_group[1 + g].size();
    int s = n > 0 ? side_pairs / n : 1;
    if (s < 1) s = 1;
    if (s > 8) s = 8;
    if (s > total_chunks) s = total_chunks;
    split_of[1 + g] = norm_split(s);
  }
  // partial tiles: one per (work tile, row split), in work-tile order; a finish tile sums the partials of its work tile(s) —
  // an accumulating problem's tile directly follows the tile it adds to, so the range stays contiguous
  std::vector<int> part0(ntiles, 0);
  int npart_total = 0;
  {
    int t0 = 0;
    for (int i = 0; i < ntiles; ++i) {
      const int s = tl[i].group < 0 ? split_bk[tl[i].bucket] : split_of[tl[i].group + 1];
      part0[i] = t0;
      TcWgFinTile& ft = tiles[fin_of[i]];
      if (ft.nsplit == 0) { ft.tile0 = t0; ft.nsplit = s; } else ft.nsplit += s;
      t0 += s;
    }
    npart_total = t0;
  }
  std::vector<TcWgUnit> units;
  int cs_rows = 0;
  plan->side.assign(ngroups, std::make_pair(0, 0));
  plan->buckets.assign(nbuckets, TcWgGroupPlan::Bucket{0, 0, 0, 0, 0, 0});
  // (launch order of the final group: bucket by bucket)
  {
    std::vector<int> ordered;
    for (int b = 0; b < nbuckets; ++b) for (int ui : by_bucket[b]) ordered.push_back(ui);
    by_group[0] = ordered;
  }
  for (int gi = 0; gi <= ngroups; ++gi) {
    const int first = (int)units.size();
    for (int ui : by_group[gi]) {
      const UnitT& uu = ut[ui];
      const int gs = gi == 0 ? split_bk[tl[uu.t[0]].bucket] : split_of[gi];
      const int cps = (total_chunks + gs - 1) / gs;
      if (gi == 0) {
        TcWgGroupPlan::Bucket& bk = plan->buckets[tl[uu.t[0]].bucket];
        if (bk.nunits == 0) bk.unit0 = (int)units.size();
        bk.nunits += gs;
      }
      for (int z = 0; z < gs; ++z) {
        TcWgUnit u{};
        const Tile& t0 = tl[uu.t[0]];
        u.a_map = t0.a_map; u.a_atom = t0.a_atom; u.shift = t0.shift; u.nh = uu.nh;
        u.c_begin = z * cps; u.c_end = std::min(total_chunks, (z + 1) * cps);
        const int b0 = u.c_begin / chunks_t, b1 = (u.c_end - 1) / chunks_t;
        u.cs_r0 = u.cs_r1 = 0;
        u.share_g = uu.share_g; u.shift2 = uu.share_g ? tl[uu.t[1]].shift : 0;
        for (int hh = 0; hh < 2; ++hh) {
          const Tile& t = tl[uu.t[hh] >= 0 ? uu.t[hh] : uu.t[0]];
          u.g_map[hh] = t.g_map; u.g_atom[hh] = t.g_atom; u.out_tile[hh] = uu.t[hh] >= 0 ? part0[uu.t[hh]] + z : 0;
          u.cs_row0[hh] = -1;
          if (uu.share_g && hh == 1) continue;      // one G tile: its column sums belong to slot 0 (rows of both taps' slices)
          if (uu.t[hh] >= 0 && t.cs_entry >= 0 && t.cs_r1 > t.cs_r0) {
            u.cs_r0 = t.cs_r0; u.cs_r1 = (uu.share_g && tl[uu.t[1]].cs_entry >= 0) ? tl[uu.t[1]].cs_r1 : t.cs_r1;
            TcWgFinCs& e = css[t.cs_entry];
            if (e.nsrc >= TC_WG_MAX_CS_SRC) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad: too many column-sum sources"); return -22; }
            u.cs_row0[hh] = cs_rows;
            e.row0[e.nsrc] = cs_rows; e.b_first[e.nsrc] = b0; e.nb[e.nsrc] = b1 - b0 + 1; e.nsrc++;
            cs_rows += b1 - b0 + 1;
          }
        }
        units.push_back(u);
      }
    }
    if (gi == 0) plan->final_units = (int)units.size();
    else plan->side[gi - 1] = std::make_pair(first, (int)units.size() - first);
  }
  for (auto& e : css)
    if (e.nsrc < 0) {
      const TcWgFinCs& o = css[-1 - e.nsrc];
      e.nsrc = o.nsrc;
      for (int i = 0; i < o.nsrc; ++i) { e.row0[i] = o.row0[i]; e.b_first[i] = o.b_first[i]; e.nb[i] = o.nb[i]; }
    }
  // tiles and column-sum entries were created in job order = bucket order (side-launch jobs last: finished with the last bucket)
  for (int b = 0; b < nbuckets; ++b) {
    TcWgGroupPlan::Bucket& bk = plan->buckets[b];
    bk.tile0 = 0; bk.ntiles = 0; bk.cs0 = (int)css.size(); bk.ncs = 0;
    // (finish tiles of the bucket: those of its work tiles, a contiguous range)
    int f_lo = (int)tiles.size(), f_hi = -1;
    for (int i = 0; i < ntiles; ++i) if (tl[i].bucket == b) { f_lo = std::min(f_lo, fin_of[i]); f_hi = std::max(f_hi, fin_of[i]); }
    if (f_hi >= f_lo) { bk.tile0 = f_lo; bk.ntiles = f_hi - f_lo + 1; }
    for (int i = 0; i < (int)css.size(); ++i) if (cs_bucket[i] == b) { if (bk.ncs == 0) bk.cs0 = i; bk.ncs++; }
    if (bk.ntiles == 0) bk.tile0 = 0;
    if (bk.ncs == 0) bk.cs0 = 0;
  }
  // column sums of another G tensor added to a bias (conv1 under skip_channels=None: d x_out + d skip): its owner's sources join
  for (const auto& ce : cs_extra) {
    auto it = cs_of.find(ce.second);
    if (it == cs_of.end()) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad: no problem computes the column sums a bias adds"); return -26; }
    TcWgFinCs& e = css[ce.first];
    const TcWgFinCs& o = css[it->second];
    if (o.nsrc < 0 || e.nsrc < 0 || e.nsrc + o.nsrc > TC_WG_MAX_CS_SRC) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad: too many column-sum sources"); return -22; }
    for (int i = 0; i < o.nsrc; ++i) { e.row0[e.nsrc] = o.row0[i]; e.b_first[e.nsrc] = o.b_first[i]; e.nb[e.nsrc] = o.nb[i]; e.nsrc++; }
  }
  plan->nunits = (int)units.size(); plan->ntiles = ntiles; plan->nfin = (int)tiles.size(); plan->ncs = (int)css.size(); plan->nsplit = nsplit;
  auto up = [&](void** d, const void* src, size_t bytes) -> bool {
    if (bytes == 0) { *d = nullptr; return true; }
    if (cudaMalloc(d, bytes) != cudaSuccess) return false;
    return cudaMemcpy(*d, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  bool ok = up((void**)&plan->d_maps, maps.data(), maps.size() * sizeof(CUtensorMap)) && up((void**)&plan->d_units, units.data(), units.size() * sizeof(TcWgUnit)) &&
            up((void**)&plan->d_tiles, tiles.data(), tiles.size() * sizeof(TcWgFinTile)) && up((void**)&plan->d_css, css.data(), css.size() * sizeof(TcWgFinCs));
  const size_t npart = (size_t)npart_total;
  plan->npartial = (int)npart;
  ok = ok && cudaMalloc((void**)&plan->d_partial, npart * 65536 * 4) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&plan->d_cs, (size_t)(cs_rows > 0 ? cs_rows : 1) * 256 * 4) == cudaSuccess;
  if (!ok) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad: plan allocation failed: %s", cudaGetErrorString(cudaGetLastError())); plan->release(); return -23; }
  uint64_t pd[3] = {256, 256, (uint64_t)npart};
  uint64_t ps[2] = {256 * 4, 65536 * 4};
  uint32_t pb[3] = {32, 128, 1};
  const CUtensorMap* mp = tc.get(plan->d_partial, 3, pd, ps, pb, 128, true);
  if (!mp) { plan->release(); return -24; }
  plan->tmP = *mp;
  return 0;
}

static int tc_wgrad_group_launch(cudaStream_t st, const TcWgGroupPlan& plan, int unit_base, int nunits) {
  if (nunits <= 0) return 0;
  using Cfg = TcWgradPairCfg<256, 2>;
  auto kern = tc_wgrad_group_kernel;
  static unsigned long long attr_devs = 0ull;
  if (tc_first_use_on_device(&attr_devs)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "cudaFuncSetAttribute(smem=%d): %s", Cfg::SMEM_BYTES, cudaGetErrorString(e)); return -12; }
  }
  TcWgGroupParams p{};
  p.maps = plan.d_maps; p.units = plan.d_units; p.cs = plan.d_cs; p.chunks_t = (plan.T + 63) / 64; p.unit_base = unit_base;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * nunits); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = Cfg::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 2);
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, plan.tmP, p);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}

// bucket < 0: every tile and column-sum entry of the plan; else those of one bucket of the final launch
static int tc_wgrad_group_finish_launch(cudaStream_t st, const TcWgGroupPlan& plan, float l2coef, int bucket = -1) {
  TcWgFinParams f{};
  f.partial = plan.d_partial; f.cs = plan.d_cs; f.tiles = plan.d_tiles; f.ntiles = plan.nfin; f.css = plan.d_css; f.ncs = plan.ncs;
  if (bucket >= 0) {
    const TcWgGroupPlan::Bucket& bk = plan.buckets[bucket];
    f.tiles = plan.d_tiles + bk.tile0; f.ntiles = bk.ntiles; f.css = plan.d_css + bk.cs0; f.ncs = bk.ncs;
  }
  f.l2coef = l2coef; f.B = plan.B;
  if (f.ntiles * 64 + f.ncs <= 0) return 0;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(f.ntiles * 64 + f.ncs); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  cfg.attrs = attr; cfg.numAttrs = tc_launch_attrs(attr, 1);
  cudaError_t e = cudaLaunchKernelEx(&cfg, tc_wgrad_group_finish, f);
  if (e != cudaSuccess) { snprintf(g_tc_err, sizeof(g_tc_err), "grouped wgrad finish launch: %s", cudaGetErrorString(e)); return -13; }
  return 0;
}
