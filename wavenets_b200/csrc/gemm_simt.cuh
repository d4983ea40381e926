// gemm_simt.cuh — fp32 FFMA mainloops (the <=1e-4 parity tier; also serves channel widths the
// tcgen05 path does not tile, e.g. the reference default R=32).
//
// Two contractions cover the whole training pass:
//   conv_gemm : out[(b,t), n]   = sum_seg  A_seg[(b, t+shift_seg), :] . W_seg[:, n]   (+ epilogue)
//               forward dilated causal convs (shift = -(K-1-k)*d, reference layers.py:199-200 /
//               Keras Conv1D padding='causal'), their dgrads (shift = +(K-1-k)*d), all 1x1 convs.
//               Rows with t+shift outside [0,T) read as zero PER BATCH ROW (causal padding and
//               batch isolation).
//   wgrad     : dW[seg.koff + c, n] = sum_{b,t} A_seg[(b, t+shift_seg), c] * G[(b,t), n]
//               (contraction over time), split over row ranges with a deterministic 2-stage
//               reduction (no atomics).
#pragma once
#include "common.cuh"

#define WN_MAX_TAPS 4
// + 1: the gated conv of a layer called with a conditioning sequence contracts it as one more segment (shift 0)
#define WN_MAX_SEG (WN_MAX_TAPS + 1)

struct SegF {
  const float* A;   // [(b*T + t) * lda + c]
  int lda;
  int shift;        // row (time) shift
  int K;            // contraction width (channels)
};

struct ConvGemmArgsF {
  int B, T;
  int Npad;                 // packed weight row length (multiple of 64)
  int nseg;
  SegF seg[WN_MAX_SEG];
  int n_outer;              // >1: seg[0] is repeated over n_outer slabs (skip-sum over blocks)
  long long a_outer_stride; // elements between slabs of seg[0].A
  const float* W;           // [ktot][Npad], rows ordered (outer, seg, c)
};

struct SmemAccRow {
  const float* rowp;
  __device__ __forceinline__ void load16(int c, float* v) const {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = rowp[c + i];
  }
  __device__ __forceinline__ int clip(int nv) const { return nv; }
};

// tile 64 rows x 64 cols, 256 threads, 4x4 micro-tile, K chunks of 16
template <class Epi>
__global__ void __launch_bounds__(256) conv_gemm_simt(ConvGemmArgsF a, typename Epi::Params ep) {
  __shared__ __align__(16) float As[16][68];
  __shared__ __align__(16) float Bs[16][64];
  __shared__ float Cs[64][65];
  const int tid = threadIdx.x;
  const int tiles_per_b = (a.T + 63) >> 6;
  const int b = blockIdx.x / tiles_per_b;
  const int t0 = (blockIdx.x % tiles_per_b) << 6;
  const int n0 = blockIdx.y << 6;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int lr = tid >> 2, lk = (tid & 3) << 2;   // A loader: row lr, k offset lk..lk+3
  const int wk = tid >> 4, wn = (tid & 15) << 2;  // W loader: k row wk, cols wn..wn+3
  // Software pipeline over the K chunks of all (outer, segment) pairs: the global loads of chunk i+1 are issued before the FMAs of
  // chunk i.  At the reference's default width a CTA runs 8 chunks of 16 k: un-pipelined, every chunk paid a full global-load
  // round trip between two barriers, which is most of an 11 us launch (the fp32 tier's C1 step is ~140 such launches).
  // (Tried and dropped: programmatic dependent launch for these kernels — 1.02 -> 1.43 ms per C1 step inside the step graph.)
  struct Chunk { int o, s, k0, wrow; };
  auto first = [&]() { return Chunk{0, 0, 0, 0}; };
  auto valid = [&](const Chunk& c) { return c.o < a.n_outer; };
  auto advance = [&](Chunk c) {
    c.k0 += 16;
    if (c.k0 >= a.seg[c.s].K) {
      c.wrow += a.seg[c.s].K; c.k0 = 0; ++c.s;
      if (c.s >= a.nseg) { c.s = 0; ++c.o; }
    }
    return c;
  };
  auto fetch = [&](const Chunk& c, float (&ra)[4], float4& rw) {
    const SegF sg = a.seg[c.s];
    const float* Ab = sg.A + (c.s == 0 ? (long long)c.o * a.a_outer_stride : 0);
    const int ta = t0 + lr + sg.shift;
    const bool rok = (ta >= 0) && (ta < a.T);
    const float* arow = Ab + ((long long)b * a.T + ta) * sg.lda;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = c.k0 + lk + i;
      ra[i] = (rok && k < sg.K) ? arow[k] : 0.f;
    }
    const int k = c.k0 + wk;
    rw = make_float4(0.f, 0.f, 0.f, 0.f);
    if (k < sg.K) rw = *reinterpret_cast<const float4*>(a.W + (long long)(c.wrow + k) * a.Npad + n0 + wn);
  };
  Chunk cur = first();
  float ra[4]; float4 rw;
  if (valid(cur)) fetch(cur, ra, rw);
  while (valid(cur)) {
#pragma unroll
    for (int i = 0; i < 4; ++i) As[lk + i][lr] = ra[i];
    *reinterpret_cast<float4*>(&Bs[wk][wn]) = rw;
    __syncthreads();
    const Chunk nxt = advance(cur);
    if (valid(nxt)) fetch(nxt, ra, rw);      // in flight while this chunk is multiplied
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty << 2]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx << 2]);
      const float aa[4] = {av.x, av.y, av.z, av.w};
      const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
    __syncthreads();
    cur = nxt;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) Cs[(ty << 2) + i][(tx << 2) + j] = acc[i][j];
  __syncthreads();
  const int r = tid & 63, q = tid >> 6;
  const int t = t0 + r;
  if (t < a.T) {
    SmemAccRow ar{&Cs[r][0]};
    Epi::row(ep, ar, b, (long long)b * a.T + t, n0, 64, q, 4);
  }
}

struct WgradArgsF {
  int B, T;
  int N;            // G columns
  const float* G;   // [(b*T+t)*ldg + n]
  int ldg;
  int nseg;
  SegF seg[WN_MAX_SEG];  // A operands; output rows are (seg, c)
  int ktot;
  float* partial;   // [nsplit][ktot (+ 1)][N]
  int chunks_per_split;  // 16-row chunks handled by one blockIdx.z
  int cs_row;       // != 0: row ktot of every partial holds the column sums of G over the split's rows (bias gradient rides along:
                    // the G tile is in shared memory anyway — two extra launches per conv otherwise, and the fp32 tier at the
                    // reference's default width is launch bound: 209 launches per C1 step)
};

// output tile 64 (k) x 64 (n); rows consumed in chunks of 16
__global__ void __launch_bounds__(256) wgrad_simt(WgradArgsF a) {
  __shared__ __align__(16) float As[16][64];
  __shared__ __align__(16) float Gs[16][64];
  const int tid = threadIdx.x;
  // locate the segment / k offset of this k tile
  int kt = blockIdx.x, s = 0, koff = 0;
  while (true) {
    const int nt = (a.seg[s].K + 63) >> 6;
    if (kt < nt) break;
    kt -= nt; koff += a.seg[s].K; ++s;
  }
  const SegF sg = a.seg[s];
  const int k0 = kt << 6;
  const int n0 = blockIdx.y << 6;
  const int ty = tid >> 4, tx = tid & 15;
  const int lr = tid >> 4, lc = (tid & 15) << 2;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int chunks_per_b = (a.T + 15) >> 4;
  const int total = a.B * chunks_per_b;
  const bool do_cs = a.cs_row != 0 && blockIdx.x == 0 && tid < 64;      // one k tile per (n tile, split) sums the columns
  float csum = 0.f;
  const int c_begin = blockIdx.z * a.chunks_per_split;
  const int c_end = min(total, c_begin + a.chunks_per_split);
  // same software pipeline over the 16-row chunks: the loads of chunk ch+1 fly while chunk ch is multiplied
  float ra[4], rg[4];
  auto fetch = [&](int ch) {
    const int b = ch / chunks_per_b;
    const int t = ((ch % chunks_per_b) << 4) + lr;
    const int ta = t + sg.shift;
    const bool aok = (t < a.T) && (ta >= 0) && (ta < a.T);
    const float* arow = sg.A + ((long long)b * a.T + ta) * sg.lda + k0 + lc;
    const float* grow = a.G + ((long long)b * a.T + t) * a.ldg + n0 + lc;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ra[i] = (aok && (k0 + lc + i) < sg.K) ? arow[i] : 0.f;
      rg[i] = ((t < a.T) && (n0 + lc + i) < a.N) ? grow[i] : 0.f;
    }
  };
  if (c_begin < c_end) fetch(c_begin);
  for (int ch = c_begin; ch < c_end; ++ch) {
#pragma unroll
    for (int i = 0; i < 4; ++i) { As[lr][lc + i] = ra[i]; Gs[lr][lc + i] = rg[i]; }
    __syncthreads();
    if (ch + 1 < c_end) fetch(ch + 1);
    if (do_cs) {
#pragma unroll
      for (int r = 0; r < 16; ++r) csum += Gs[r][tid];
    }
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      const float4 av = *reinterpret_cast<const float4*>(&As[r][ty << 2]);
      const float4 gv = *reinterpret_cast<const float4*>(&Gs[r][tx << 2]);
      const float aa[4] = {av.x, av.y, av.z, av.w};
      const float gg[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], gg[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* out = a.partial + (long long)blockIdx.z * (a.ktot + (a.cs_row ? 1 : 0)) * a.N;
  if (do_cs && n0 + tid < a.N) out[(long long)a.ktot * a.N + n0 + tid] = csum;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = k0 + (ty << 2) + i;
    if (k >= sg.K) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + (tx << 2) + j;
      if (n < a.N) out[(long long)(koff + k) * a.N + n] = acc[i][j];
    }
  }
}
