// kernels_misc.cuh — HBM-bound kernels around the GEMMs: input causal conv, bias/conditioning
// reductions, output head losses (softmax-256 CE, mixture of logistics / normals), quantiser,
// weight packing, tiny dense layers of the conditioning MLP.  All coalesced along channels,
// vectorised where layout allows, reductions via warp shuffles + deterministic 2-stage sums.
#pragma once
#include "common.cuh"

// (b, t) of a flattened row; 32-bit division whenever the row count allows (a 64-bit division is ~100 instructions)
__device__ __forceinline__ void wn_row_bt(long long row, long long rows, int Tn, long long& b, long long& t) {
  if (rows <= 0x7fffffffLL) {
    const unsigned r = (unsigned)row, q = r / (unsigned)Tn;
    b = q; t = r - q * (unsigned)Tn;
  } else {
    b = row / Tn; t = row % Tn;
  }
}

// ------------------------------------------------------------------ input causal conv (model.py:84-88,228)
// h[b,t,c] = sum_k W[k,0,c] * x[b, t-(K-1-k)] + bias[c] ; x (B,T) fp32 with row stride ldx
template <class T>
__global__ void input_conv_fwd(const float* __restrict__ x, int ldx, const float* __restrict__ W, const float* __restrict__ bias,
                               T* __restrict__ h, int B, int Tn, int R, int K) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)B * Tn * R;
  if (i >= total) return;
  const int c = (int)(i % R);
  const long long row = i / R;
  const int t = (int)(row % Tn), b = (int)(row / Tn);
  float v = bias[c];
  for (int k = 0; k < K; ++k) {
    const int ts = t - (K - 1 - k);
    if (ts >= 0) v = fmaf(W[k * R + c], x[(long long)b * ldx + ts], v);
  }
  h[i] = from_f<T>(v);
}

// 8 channels per thread held across ROWS_PER_BLOCK rows: the K taps and the bias of those channels are loaded once
// into registers (the per-row variant below re-loads 8*(K+1) floats for every 16-byte store)
#define ICF_ROWS 64
template <class T>
__global__ void __launch_bounds__(256) input_conv_fwd_rows(const float* __restrict__ x, int ldx, const float* __restrict__ W, const float* __restrict__ bias,
                                                           T* __restrict__ h, int B, int Tn, int R, int K) {
  const int r8 = R >> 3;                       // channel groups per row
  const int groups = 256 / r8 > 0 ? 256 / r8 : 1;   // rows processed side by side (r8 <= 256)
  const int cg = threadIdx.x % r8, rg = threadIdx.x / r8;
  if (rg >= groups) return;
  const int c = cg << 3;
  float w[4][8], bv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) bv[j] = bias[c + j];
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) w[k][j] = k < K ? W[k * R + c + j] : 0.f;
  const long long rows = (long long)B * Tn;
  const long long r_end = min(rows, ((long long)blockIdx.x + 1) * ICF_ROWS);
#pragma unroll 4
  for (long long row = (long long)blockIdx.x * ICF_ROWS + rg; row < r_end; row += groups) {
    long long bq, tq;
    wn_row_bt(row, rows, Tn, bq, tq);          // (two 64-bit divisions per row were most of this kernel's instructions)
    const int t = (int)tq, b = (int)bq;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = bv[j];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int ts = t - (K - 1 - k);
      if (k < K && ts >= 0) {
        const float xv = x[(long long)b * ldx + ts];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(w[k][j], xv, v[j]);
      }
    }
    T* o = h + row * R + c;
    if constexpr (sizeof(T) == 2) {
      uint4 q;
      q.x = pack_bf16x2(v[0], v[1]); q.y = pack_bf16x2(v[2], v[3]); q.z = pack_bf16x2(v[4], v[5]); q.w = pack_bf16x2(v[6], v[7]);
      *reinterpret_cast<uint4*>(o) = q;
    } else {
      reinterpret_cast<float4*>(o)[0] = make_float4(v[0], v[1], v[2], v[3]);
      reinterpret_cast<float4*>(o)[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

// same, 8 channels per thread (R % 8 == 0): 16/32-byte stores, no per-element div/mod
template <class T>
__global__ void __launch_bounds__(256) input_conv_fwd_vec8(const float* __restrict__ x, int ldx, const float* __restrict__ W, const float* __restrict__ bias,
                                                           T* __restrict__ h, int B, int Tn, int R, int K) {
  const int r8 = R >> 3;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * Tn * r8) return;
  const int c = (int)(i % r8) << 3;
  const long long row = i / r8;
  const int t = (int)(row % Tn), b = (int)(row / Tn);
  float v[16];
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = bias[c + j];
#pragma unroll
  for (int j = 8; j < 16; ++j) v[j] = 0.f;
  for (int k = 0; k < K; ++k) {
    const int ts = t - (K - 1 - k);
    if (ts >= 0) {
      const float xv = x[(long long)b * ldx + ts];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(W[k * R + c + j], xv, v[j]);
    }
  }
  T* o = h + row * R + c;
  if constexpr (sizeof(T) == 2) {
    uint4 q;
    q.x = pack_bf16x2(v[0], v[1]); q.y = pack_bf16x2(v[2], v[3]); q.z = pack_bf16x2(v[4], v[5]); q.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(o) = q;
  } else {
    reinterpret_cast<float4*>(o)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(o)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
}

// stage 1 of input conv wgrad: partial[(chunk)][k][c] = sum_{t in chunk} dh[b,t,c] * x[b,t-(K-1-k)], k==K => bias
template <class T>
__global__ void input_conv_bwd_stage1(const float* __restrict__ x, int ldx, const T* __restrict__ dh, int lddh, float* __restrict__ partial,
                                      int B, int Tn, int R, int K, int rows_per_chunk) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= R) return;
  const int b = blockIdx.z;
  const int t0 = blockIdx.y * rows_per_chunk, t1 = min(Tn, t0 + rows_per_chunk);
  float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  for (int t = t0; t < t1; ++t) {
    const float d = to_f(dh[((long long)b * Tn + t) * lddh + c]);
    for (int k = 0; k < K; ++k) {
      const int ts = t - (K - 1 - k);
      if (ts >= 0) acc[k] = fmaf(d, x[(long long)b * ldx + ts], acc[k]);
    }
    acc[K] += d;
  }
  const long long chunk = (long long)b * gridDim.y + blockIdx.y;
  for (int k = 0; k <= K; ++k) partial[(chunk * (K + 1) + k) * R + c] = acc[k];
}

// wide variant (R even, R/2 <= 256): one block = ICB_ROWS flattened (b,t) rows x all channels; a thread owns a channel
// pair (one 32-bit load per row for bf16) for every `groups`-th row, then the row groups are summed through shared
// memory in a fixed order.  partial[block][k][c], k == K => bias.
#define ICB_ROWS 128
template <class T>
__global__ void __launch_bounds__(256) input_conv_bwd_stage1_wide(const float* __restrict__ x, int ldx, const T* __restrict__ dh, int lddh,
                                                                  float* __restrict__ partial, int B, int Tn, int R, int K) {
  __shared__ float red[256][11];
  const int cp_n = R >> 1;
  const int groups = 256 / cp_n;
  const int cp = threadIdx.x % cp_n, rg = threadIdx.x / cp_n;
  float acc[5][2];
#pragma unroll
  for (int k = 0; k < 5; ++k) acc[k][0] = acc[k][1] = 0.f;
  const long long rows = (long long)B * Tn;
  const long long r_end = min(rows, ((long long)blockIdx.x + 1) * ICB_ROWS);
  if (rg < groups) {
    // (b, t) of the first row once, then stepped: two 64-bit divisions per row were most of this kernel's time
    long long row = (long long)blockIdx.x * ICB_ROWS + rg;
    int t = (int)(row % Tn), b = (int)(row / Tn);
#pragma unroll 4
    for (; row < r_end; row += groups, t += groups) {
      while (t >= Tn) { t -= Tn; ++b; }
      float d0, d1;
      if constexpr (sizeof(T) == 2) {
        const uint32_t wv = *reinterpret_cast<const uint32_t*>(dh + row * lddh + 2 * cp);
        d0 = __uint_as_float(wv << 16); d1 = __uint_as_float(wv & 0xffff0000u);
      } else {
        const float2 wv = *reinterpret_cast<const float2*>(dh + row * lddh + 2 * cp);
        d0 = wv.x; d1 = wv.y;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int ts = t - (K - 1 - k);
        if (k < K && ts >= 0) {
          const float xv = x[(long long)b * ldx + ts];
          acc[k][0] = fmaf(d0, xv, acc[k][0]); acc[k][1] = fmaf(d1, xv, acc[k][1]);
        }
      }
      acc[4][0] += d0; acc[4][1] += d1;
    }
  }
#pragma unroll
  for (int k = 0; k < 5; ++k) { red[threadIdx.x][2 * k] = acc[k][0]; red[threadIdx.x][2 * k + 1] = acc[k][1]; }
  __syncthreads();
  if (rg == 0) {
    float* out = partial + (long long)blockIdx.x * (K + 1) * R;
    for (int k = 0; k <= K; ++k) {
      const int kk = k < K ? k : 4;
      float s0 = 0.f, s1 = 0.f;
      for (int g = 0; g < groups; ++g) { s0 += red[g * cp_n + cp][2 * kk]; s1 += red[g * cp_n + cp][2 * kk + 1]; }
      out[k * R + 2 * cp] = s0; out[k * R + 2 * cp + 1] = s1;
    }
  }
}

// input conv dgrad, the adjoint of input_conv_fwd onto the 1-channel signal:
//   dx[b,s] = sum_k [s+(K-1-k) < T] * q_k(b, s+(K-1-k)),   q_k(b,t) = sum_c dh[b,t,c] * W[k,0,c]
// One CTA = ICD_ROWS positions of one sequence.  Every dh row the CTA needs (its own rows plus the K-1 halo rows after them,
// cut at the sequence end so the next batch row is never read) is read once, by one warp: each lane holds V channels per
// 16-byte load (V = 1: the scalar path for widths and strides that are not multiples of 16 bytes) and K partial dot products,
// then a butterfly shuffle sums the lanes.  Fixed summation order everywhere: bit-reproducible.  dx (B,T) fp32, row stride T.
#define ICD_ROWS 64
#define ICD_MAXK 4
#define ICD_RPW ((ICD_ROWS + ICD_MAXK - 1 + 7) / 8)     // q rows per warp (8 warps)
template <class T, int V>
__global__ void __launch_bounds__(256) input_conv_dgrad(const T* __restrict__ dh, int lddh, const float* __restrict__ W, float* __restrict__ dx,
                                                        int Tn, int R, int K) {
  __shared__ float q[ICD_MAXK][ICD_ROWS + ICD_MAXK - 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y, t0 = blockIdx.x * ICD_ROWS;
  const int nq = min(ICD_ROWS + K - 1, Tn - t0);
  const T* base = dh + ((long long)b * Tn + t0) * lddh;
  float acc[ICD_RPW][ICD_MAXK];
#pragma unroll
  for (int i = 0; i < ICD_RPW; ++i)
#pragma unroll
    for (int k = 0; k < ICD_MAXK; ++k) acc[i][k] = 0.f;
  for (int c = lane * V; c < R; c += 32 * V) {
    float w[ICD_MAXK][V];
#pragma unroll
    for (int k = 0; k < ICD_MAXK; ++k)
#pragma unroll
      for (int j = 0; j < V; ++j) w[k][j] = k < K ? W[k * R + c + j] : 0.f;
    // every row's load first (rows past nq read as zero): one memory latency per chunk, not one per row
    using Vec = std::conditional_t<V == 8, uint4, std::conditional_t<V == 4, float4, T>>;
    Vec raw[ICD_RPW];
#pragma unroll
    for (int i = 0; i < ICD_RPW; ++i) {
      const int r = warp + 8 * i;
      if (r < nq) raw[i] = *reinterpret_cast<const Vec*>(base + (long long)r * lddh + c);
      else raw[i] = Vec{};
    }
#pragma unroll
    for (int i = 0; i < ICD_RPW; ++i) {
      float d[V];
      if constexpr (V == 8) {
        const uint32_t a[4] = {raw[i].x, raw[i].y, raw[i].z, raw[i].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { d[2 * j] = __uint_as_float(a[j] << 16); d[2 * j + 1] = __uint_as_float(a[j] & 0xffff0000u); }
      } else if constexpr (V == 4) {
        d[0] = raw[i].x; d[1] = raw[i].y; d[2] = raw[i].z; d[3] = raw[i].w;
      } else {
        d[0] = to_f(raw[i]);
      }
#pragma unroll
      for (int k = 0; k < ICD_MAXK; ++k)
#pragma unroll
        for (int j = 0; j < V; ++j) acc[i][k] = fmaf(d[j], w[k][j], acc[i][k]);
    }
  }
#pragma unroll
  for (int i = 0; i < ICD_RPW; ++i)
#pragma unroll
    for (int k = 0; k < ICD_MAXK; ++k) {
      const int r = warp + 8 * i;
      if (k >= K || r >= nq) continue;      // (warp-uniform)
      float v = acc[i][k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) q[k][r] = v;
    }
  __syncthreads();
  const int sl = threadIdx.x;
  if (sl < ICD_ROWS && t0 + sl < Tn) {
    float s = 0.f;
    for (int k = 0; k < K; ++k) {
      const int r = sl + K - 1 - k;     // (r < nq <=> t0 + r < T: a tap past the sequence end contributes zero)
      if (r < nq) s += q[k][r];
    }
    dx[(long long)b * Tn + t0 + sl] = s;
  }
}

// per-batch column sums of several (B,T,N) slabs in one launch: out[l*out_slab + b*ldpb + n] = sum_t G[l*slab + (b*T+t)*ldg + n].
// One CTA = 64 columns (a column pair per lane) of one (slab, batch row): 8 row lanes walk T in 4 independent chains and meet in
// shared memory in a fixed order (bit-reproducible).  N and ldg even.
template <class T>
__global__ void __launch_bounds__(256) colsum_per_batch_slabs(const T* __restrict__ G, long long slab, int ldg, int Tn, int N, float* __restrict__ out,
                                                              long long out_slab, int ldpb) {
  __shared__ float sh[8][64];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n = blockIdx.x * 64 + 2 * tx;
  const int b = blockIdx.y, l = blockIdx.z;
  float s[4][2] = {};
  if (n < N) {
    const T* p = G + l * slab + ((long long)b * Tn + ty) * ldg + n;
    int t = ty;
    for (; t + 24 < Tn; t += 32, p += 32LL * ldg) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float2 v;
        if constexpr (sizeof(T) == 2) {
          const uint32_t w = *reinterpret_cast<const uint32_t*>(p + 8LL * u * ldg);
          v = make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
        } else {
          v = *reinterpret_cast<const float2*>(p + 8LL * u * ldg);
        }
        s[u][0] += v.x; s[u][1] += v.y;
      }
    }
    for (; t < Tn; t += 8, p += 8LL * ldg) { s[0][0] += to_f(p[0]); s[0][1] += to_f(p[1]); }
  }
  sh[ty][2 * tx] = (s[0][0] + s[1][0]) + (s[2][0] + s[3][0]);
  sh[ty][2 * tx + 1] = (s[0][1] + s[1][1]) + (s[2][1] + s[3][1]);
  __syncthreads();
  if (ty < 2) {
    const int c = 2 * tx + ty;
    float r = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) r += sh[k][c];
    if (blockIdx.x * 64 + c < N) out[l * out_slab + (long long)b * ldpb + blockIdx.x * 64 + c] = r;
  }
}

// ------------------------------------------------------------------ generic deterministic reductions
// out[j] = scale * sum_{i<n_parts} partial[i*stride + j]  (+ addend[j]*add_coef), j < n
__global__ void reduce_parts(const float* __restrict__ partial, int n_parts, long long stride, float* __restrict__ out, long long n,
                             const float* __restrict__ addend, float add_coef) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  float s = 0.f;
  for (int i = 0; i < n_parts; ++i) s += partial[i * stride + j];
  if (addend) s = fmaf(add_coef, addend[j], s);
  out[j] = s;
}

// two destinations: out0[j] for j < n0 (+ addend0[j]*add_coef), out1[j - n0] for n0 <= j < n0 + n1 (a filter gradient with its bias row)
__global__ void reduce_parts2(const float* __restrict__ partial, int n_parts, long long stride, float* __restrict__ out0, long long n0,
                              float* __restrict__ out1, long long n1, const float* __restrict__ addend0, float add_coef) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n0 + n1) return;
  float s0 = 0.f, s1 = 0.f;
  int i = 0;
  for (; i + 1 < n_parts; i += 2) { s0 += partial[i * stride + j]; s1 += partial[(i + 1) * stride + j]; }
  if (i < n_parts) s0 += partial[i * stride + j];
  float s = s0 + s1;
  if (j < n0) {
    if (addend0) s = fmaf(add_coef, addend0[j], s);
    out0[j] = s;
  } else {
    out1[j - n0] = s;
  }
}

// same contract for MANY partials (hundreds): 32 outputs x 8 partial-lanes per block, fixed summation order
__global__ void __launch_bounds__(256) reduce_parts_tall(const float* __restrict__ partial, int n_parts, long long stride, float* __restrict__ out,
                                                         long long n, const float* __restrict__ addend, float add_coef) {
  __shared__ float red[8][33];
  const int jl = threadIdx.x & 31, pl = threadIdx.x >> 5;
  const long long j = (long long)blockIdx.x * 32 + jl;
  float s0 = 0.f, s1 = 0.f;
  if (j < n) {
    int i = pl;
    for (; i + 8 < n_parts; i += 16) { s0 += partial[i * stride + j]; s1 += partial[(i + 8) * stride + j]; }
    if (i < n_parts) s0 += partial[i * stride + j];
  }
  red[pl][jl] = s0 + s1;
  __syncthreads();
  if (pl == 0 && j < n) {
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += red[q][jl];
    if (addend) s = fmaf(add_coef, addend[j], s);
    out[j] = s;
  }
}

// column sums of G (B,T,N): stage 1 -> partial[b][chunk][n]
// block = 32 columns x 8 row lanes: a warp reads 32 consecutive columns of one row (coalesced), every thread adds up
// rows_per_chunk / 8 rows in 4 independent chains, the 8 lanes meet in shared memory.  (One thread per column walking 256 rows
// took 25.7 us per call at N = 32 — the reference's default width —, 30 % of the fp32 tier's C1 step: launch list r2m.)
template <class T>
__global__ void __launch_bounds__(256) colsum_stage1(const T* __restrict__ G, int ldg, float* __restrict__ partial, int Tn, int N, int rows_per_chunk) {
  __shared__ float sh[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + tx;
  const int b = blockIdx.z;
  const int t0 = blockIdx.y * rows_per_chunk, t1 = min(Tn, t0 + rows_per_chunk);
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  if (n < N) {
    const T* p = G + ((long long)b * Tn + t0 + ty) * ldg + n;
    int t = t0 + ty;
    for (; t + 24 < t1; t += 32, p += 32LL * ldg) {
      s0 += to_f(p[0]); s1 += to_f(p[8LL * ldg]); s2 += to_f(p[16LL * ldg]); s3 += to_f(p[24LL * ldg]);
    }
    for (; t < t1; t += 8, p += 8LL * ldg) s0 += to_f(p[0]);
  }
  sh[ty][tx] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (ty == 0 && n < N) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += sh[k][tx];
    partial[((long long)b * gridDim.y + blockIdx.y) * N + n] = s;
  }
}
// stage 2: per_batch[b][n] (optional) and total[n] (optional) from partial[b][chunk][n]; same 32 x 8 layout, the 8 lanes
// split the chunks of a batch row
__global__ void __launch_bounds__(256) colsum_stage2(const float* __restrict__ partial, int B, int chunks, int N, float* __restrict__ per_batch, int ldpb,
                                                    float* __restrict__ total) {
  __shared__ float sh[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + tx;
  float tot = 0.f;
  for (int b = 0; b < B; ++b) {
    float s = 0.f;
    if (n < N)
      for (int c = ty; c < chunks; c += 8) s += partial[((long long)b * chunks + c) * N + n];
    sh[ty][tx] = s;
    __syncthreads();
    if (ty == 0 && n < N) {
      float r = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) r += sh[k][tx];
      if (per_batch) per_batch[(long long)b * ldpb + n] = r;
      tot += r;
    }
    __syncthreads();
  }
  if (ty == 0 && n < N && total) total[n] = tot;
}

// ------------------------------------------------------------------ elementwise helpers
template <class TI, class TO>
__global__ void convert_kernel(const TI* __restrict__ in, TO* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = from_f<TO>(to_f(in[i]));
}
// out[r][c] = in[r][c] for c < cin, 0 for cin <= c < cout: rows of width cin widened to cout (zero padding)
template <class TI, class TO>
__global__ void convert_pad_kernel(const TI* __restrict__ in, int cin, TO* __restrict__ out, int cout, long long rows) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cout) return;
  const long long r = i / cout;
  const int c = (int)(i % cout);
  out[i] = from_f<TO>(c < cin ? to_f(in[r * cin + c]) : 0.f);
}
template <class T>
__global__ void add2_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = from_f<T>(to_f(a[i]) + (b ? to_f(b[i]) : 0.f));
}

// ------------------------------------------------------------------ dropout (layers.py:109-112,195-196)
// Inverted dropout on the conv branch of a block (the residual is taken before it, layers.py:192-193).
// Keep-masks are one byte per element, [block][b*T+t][r]; either injected by the caller (parity tests: TF's RNG
// stream cannot be reproduced) or drawn here with Philox-4x32-10 keyed by (seed, step counter): counter-based,
// so the backward pass re-reads the same bytes and a replayed CUDA graph still gets fresh masks every step.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
  }
  return c;
}
__global__ void dropout_step_bump(unsigned long long* ctr) { ctr[0] += 1ull; }
// n8 = groups of 8 elements per block slab; slab stride in bytes between blocks.  One Philox call serves 8 elements, 16 random
// bits each: keep <=> u16 >= round(rate * 65536) (the drop probability is exact to 2^-17; 32 bits per element made this kernel
// compute bound: 0.72 ms per C2 step for 492 MB of masks, ~70 integer operations per call)
// layer0 = block index of slab blockIdx.y == 0 (the layer API draws one block's mask at a time)
__global__ void dropout_mask_philox(uint8_t* __restrict__ mask, long long n8, long long slab_stride, float rate, unsigned long long seed,
                                    const unsigned long long* __restrict__ step_ctr, int layer0) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const unsigned long long step = step_ctr[0];
  const uint4 r = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), blockIdx.y + layer0, (uint32_t)step),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(step >> 32)));
  const uint32_t thr = (uint32_t)fminf(fmaxf(rate * 65536.0f + 0.5f, 0.0f), 65536.0f);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  uint32_t lo = 0u, hi = 0u;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t a = (w[k] & 0xffffu) >= thr ? 1u : 0u, b = (w[k] >> 16) >= thr ? 1u : 0u;
    const uint32_t two = a | (b << 8);
    if (k < 2) lo |= two << (16 * k); else hi |= two << (16 * (k - 2));
  }
  reinterpret_cast<uint2*>(mask + (long long)(blockIdx.y + layer0) * slab_stride)[i] = make_uint2(lo, hi);
}
// xd = keep ? x / (1 - rate) : 0
template <class T>
__global__ void dropout_apply(const T* __restrict__ x, const uint8_t* __restrict__ keep, T* __restrict__ xd, long long n, float inv) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) xd[i] = from_f<T>(keep[i] ? to_f(x[i]) * inv : 0.f);
}
// dx[row][c] = (keep ? draw / (1 - rate) : 0) + add[row][c]   (add: residual gradient, may be null)
template <class T>
__global__ void dropout_bwd(const T* __restrict__ draw, const uint8_t* __restrict__ keep, const T* __restrict__ add, int ld_add,
                            T* __restrict__ out, int ld_out, long long rows, int R, float inv) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * R) return;
  const long long row = i / R;
  const int c = (int)(i % R);
  float v = keep[i] ? to_f(draw[i]) * inv : 0.f;
  if (add) v += to_f(add[row * ld_add + c]);
  out[row * ld_out + c] = from_f<T>(v);
}

// dst[i][i] = 1 for i < n (row stride ld): identity block of the residual-in-the-GEMM operand
__global__ void set_identity_bf16(bf16* __restrict__ dst, int ld, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[(long long)i * ld + i] = __float2bfloat16_rn(1.0f);
}

// ------------------------------------------------------------------ weight packing
// dst[r][c] (ld = dst_ld, pre-zeroed) from Keras-layout src (rows x cols, row-major):
//   mode 0: dst[r][c]  = src[r][c]
//   mode 1: dst[c][r]  = src[r][c]                       (transpose, for dgrad)
//   mode 2: gate interleave with tile width `tile`: dst col n' = tile_i*tile + j ;
//           ch = tile_i*(tile/2) + (j % (tile/2)) ; src col = j < tile/2 ? ch : D + ch
template <class TO>
__global__ void pack_weight(const float* __restrict__ src, int rows, int cols, TO* __restrict__ dst, int dst_ld, int mode, int tile, int D,
                            int dst_cols) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (mode == 2) {
    const long long total = (long long)rows * dst_cols;
    if (i >= total) return;
    const int r = (int)(i / dst_cols), np = (int)(i % dst_cols);
    const int half = tile >> 1;
    const int ti = np / tile, j = np % tile;
    const int ch = ti * half + (j % half);
    float v = 0.f;
    if (ch < D) v = src[(long long)r * cols + (j < half ? ch : D + ch)];
    dst[(long long)r * dst_ld + np] = from_f<TO>(v);
  } else {
    const long long total = (long long)rows * cols;
    if (i >= total) return;
    const int r = (int)(i / cols), c = (int)(i % cols);
    const float v = src[i];
    if (mode == 0) dst[(long long)r * dst_ld + c] = from_f<TO>(v);
    else dst[(long long)c * dst_ld + r] = from_f<TO>(v);
  }
}

// all weight re-packs of a handle in ONE launch (after every optimizer step): a table of jobs, each job = one former
// pack_weight / tc_pack_gate_T / set_identity launch; a block finds its job by binary search over first-block indices
struct PackJob {
  const float* src; void* dst;
  int rows, cols, dst_ld, mode, tile, D, dst_cols;   // modes 0,1,2 as pack_weight; 3 = gate transposed+interleaved; 4 = identity
  long long first, total;                              // first block index, number of elements
};
template <class TO>
__global__ void __launch_bounds__(256) pack_all_kernel(const PackJob* __restrict__ jobs, int n) {
  const long long gb = blockIdx.x;
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].first <= gb) lo = mid; else hi = mid - 1;
  }
  const PackJob j = jobs[lo];
  const long long i = (gb - j.first) * 256 + threadIdx.x;
  if (i >= j.total) return;
  TO* dst = (TO*)j.dst;
  if (j.mode == 2) {
    const int r = (int)(i / j.dst_cols), np = (int)(i % j.dst_cols);
    const int half = j.tile >> 1;
    const int ti = np / j.tile, jj = np % j.tile;
    const int ch = ti * half + (jj % half);
    float v = 0.f;
    if (ch < j.D) v = j.src[(long long)r * j.cols + (jj < half ? ch : j.D + ch)];
    dst[(long long)r * j.dst_ld + np] = from_f<TO>(v);
  } else if (j.mode == 3) {
    // rows = ktot, cols = cout, dst_cols = n16: dst[np][k] = src[k][col(np)]
    const int np = (int)(i / j.rows), k = (int)(i % j.rows);
    const int half = j.tile >> 1;
    const int ti = np / j.tile, jj = np % j.tile;
    const int ch = ti * half + (jj % half);
    float v = 0.f;
    if (ch < j.D) v = j.src[(long long)k * j.cols + (jj < half ? ch : j.D + ch)];
    dst[(long long)np * j.dst_ld + k] = from_f<TO>(v);
  } else if (j.mode == 4) {
    dst[i * j.dst_ld + i] = from_f<TO>(1.0f);
  } else {
    const int r = (int)(i / j.cols), c = (int)(i % j.cols);
    const float v = j.src[i];
    if (j.mode == 0) dst[(long long)r * j.dst_ld + c] = from_f<TO>(v);
    else dst[(long long)c * j.dst_ld + r] = from_f<TO>(v);
  }
}

// ------------------------------------------------------------------ tiny dense layers (conditioning MLP, model.py:141-148)
// y[b][n] = act(sum_k x[b][k] W[k][n] + bias[n])
__global__ void dense_small_fwd(const float* __restrict__ x, int ldx, const float* __restrict__ W, const float* __restrict__ bias,
                                float* __restrict__ y, int ldy, int B, int K, int N, int act) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * N) return;
  const int b = i / N, n = i % N;
  float s = bias ? bias[n] : 0.f;
  for (int k = 0; k < K; ++k) s = fmaf(x[(long long)b * ldx + k], W[(long long)k * N + n], s);
  y[(long long)b * ldy + n] = wn_act<false>(act, s);
}
// dpre[b][n] = dy[b][n] * act'(y[b][n])   (in place on dy)
__global__ void dense_small_actgrad(float* __restrict__ dy, const float* __restrict__ y, int n_total, int act) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_total) dy[i] *= wn_act_grad_from_out(act, y[i]);
}
// dW[k][n] = sum_b x[b][k] dpre[b][n] ; db[n] = sum_b dpre[b][n]  (thread per (k,n), k==K => bias)
__global__ void dense_small_wgrad(const float* __restrict__ x, int ldx, const float* __restrict__ dpre, int ldd, float* __restrict__ dW,
                                  float* __restrict__ db, int B, int K, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (K + 1) * N) return;
  const int k = i / N, n = i % N;
  float s = 0.f;
  for (int b = 0; b < B; ++b) s = fmaf(k < K ? x[(long long)b * ldx + k] : 1.0f, dpre[(long long)b * ldd + n], s);
  if (k < K) dW[(long long)k * N + n] = s;
  else if (db) db[n] = s;
}
// The whole conditioning MLP (model.py:141-148: Dense + activation per mapping layer) in ONE single-block launch each way, for the
// sizes it really has (batch x [109 -> 8 -> 16 -> 32]: ~12 k multiply-adds): per layer the separate kernels above cost three
// dependent launches of a few us at the very start (forward) and the very end (backward: 8 launches behind the last
// weight-gradient kernel) of every step.  Same arithmetic order as dense_small_fwd / _actgrad / _wgrad (bit-identical there);
// the dgrad sums run serially over n instead of as a warp tree.
struct MapArgs {
  int n_layers, B, cond_in, act;
  float l2coef;
  const float* x0;                 // (B, cond_in)
  int width[WN_MAX_LIST];
  const float* W[WN_MAX_LIST];     // (K_i, width_i), K_0 = cond_in, K_i = width_{i-1}
  const float* bias[WN_MAX_LIST];
  float* gW[WN_MAX_LIST];
  float* gb[WN_MAX_LIST];
  float* actv[WN_MAX_LIST];        // (B, width_i): activated outputs (written by the forward, read by the backward)
  float* d0;                       // backward: gradient wrt actv[n_layers - 1] on entry (overwritten)
  float* d1;
  float* d2;
};
// hint: pull n floats towards L2 (one 128-byte line per thread and step) — the layers below run as dependent phases, each of which
// would otherwise meet its operands cold in DRAM (the step's GBs of activations evict the parameters from L2 every step)
__device__ __forceinline__ void wn_prefetch_l2(const float* p, long long n) {
  for (long long i = (long long)threadIdx.x * 32; i < n; i += 256 * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + i));
}
__global__ void __launch_bounds__(256) mapping_fwd_fused(MapArgs a) {
  {
    int k = a.cond_in;
    wn_prefetch_l2(a.x0, (long long)a.B * k);
    for (int i = 0; i < a.n_layers; ++i) { wn_prefetch_l2(a.W[i], (long long)k * a.width[i]); wn_prefetch_l2(a.bias[i], a.width[i]); k = a.width[i]; }
  }
  const float* cur = a.x0;
  int K = a.cond_in;
  for (int i = 0; i < a.n_layers; ++i) {
    const int N = a.width[i];
    const float* W = a.W[i];
    for (int j = threadIdx.x; j < a.B * N; j += 256) {
      const int b = j / N, n = j % N;
      float s = a.bias[i][n];
      // (unrolled: the loads of 8 steps are in flight together, the FMA order stays that of dense_small_fwd)
#pragma unroll 8
      for (int k = 0; k < K; ++k) s = fmaf(cur[(long long)b * K + k], W[(long long)k * N + n], s);
      a.actv[i][j] = wn_act<false>(a.act, s);
    }
    __syncthreads();
    cur = a.actv[i];
    K = N;
  }
}
__global__ void __launch_bounds__(256) mapping_bwd_fused(MapArgs a) {
  {
    int k = a.cond_in;
    wn_prefetch_l2(a.x0, (long long)a.B * k);
    for (int i = 0; i < a.n_layers; ++i) {
      wn_prefetch_l2(a.W[i], (long long)k * a.width[i]);
      wn_prefetch_l2(a.actv[i], (long long)a.B * a.width[i]);
      k = a.width[i];
    }
  }
  float* dcur = a.d0;
  for (int i = a.n_layers - 1; i >= 0; --i) {
    const int N = a.width[i];
    const int K = i > 0 ? a.width[i - 1] : a.cond_in;
    const float* inp = i > 0 ? a.actv[i - 1] : a.x0;
    const float* W = a.W[i];
    for (int j = threadIdx.x; j < a.B * N; j += 256) dcur[j] *= wn_act_grad_from_out(a.act, a.actv[i][j]);
    __syncthreads();
    for (int j = threadIdx.x; j < (K + 1) * N; j += 256) {
      const int k = j / N, n = j % N;
      float s = 0.f;
#pragma unroll 8
      for (int b = 0; b < a.B; ++b) s = fmaf(k < K ? inp[(long long)b * K + k] : 1.0f, dcur[(long long)b * N + n], s);
      if (k < K) a.gW[i][j] = a.l2coef != 0.f ? fmaf(a.l2coef, W[j], s) : s;
      else a.gb[i][n] = s;
    }
    if (i > 0) {
      float* dn = (dcur == a.d1) ? a.d2 : a.d1;
      for (int j = threadIdx.x; j < a.B * K; j += 256) {
        const int b = j / K, k = j % K;
        float s = 0.f;
#pragma unroll 8
        for (int n = 0; n < N; ++n) s = fmaf(dcur[(long long)b * N + n], W[(long long)k * N + n], s);
        dn[j] = s;
      }
      __syncthreads();
      dcur = dn;
    }
  }
}
// dx[b][k] (+)= sum_n dpre[b][n] W[k][n] ; one warp per output, lanes stride over n (coalesced rows of W)
__global__ void __launch_bounds__(128) dense_small_dgrad(const float* __restrict__ dpre, int ldd, const float* __restrict__ W, float* __restrict__ dx,
                                                         int ldx, int B, int K, int N, int accumulate) {
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= B * K) return;
  const int b = i / K, k = i % K;
  float s = 0.f;
  for (int n = lane; n < N; n += 32) s = fmaf(dpre[(long long)b * ldd + n], W[(long long)k * N + n], s);
  s = warp_sum(s);
  if (lane == 0) {
    if (accumulate) dx[(long long)b * ldx + k] += s;
    else dx[(long long)b * ldx + k] = s;
  }
}

// ------------------------------------------------------------------ conditioning, all blocks in one launch
// The per-block conv_cond (layers.py:117-120,203-204) on a time-constant conditioning vector is a
// (B,Cc)x(Cc,2D) product per block; offs[2*l] / offs[2*l+1] = offsets of Wc_l / bc_l in the flat
// parameter (and gradient) buffers.  blockIdx.y = block index l.
// cb[l][b][n] = sum_k cond[b][k] Wc_l[k][n] + bc_l[n]
__global__ void cond_bias_all(const float* __restrict__ cond, int Cc, const float* __restrict__ params, const int* __restrict__ offs,
                              float* __restrict__ cb, long long cb_stride, int B, int N) {
  const int l = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * N) return;
  const int b = i / N, n = i % N;
  const float* W = params + offs[2 * l];
  float s = params[offs[2 * l + 1] + n];
  for (int k = 0; k < Cc; ++k) s = fmaf(cond[(long long)b * Cc + k], W[(long long)k * N + n], s);
  cb[(long long)l * cb_stride + (long long)b * N + n] = s;
}
// dWc_l[k][n] = sum_b cond[b][k] dcb_l[b][n] (+ l2coef * Wc_l[k][n]) ; dbc_l[n] = sum_b dcb_l[b][n]   (k == Cc => bias)
__global__ void cond_wgrad_all(const float* __restrict__ cond, int Cc, const float* __restrict__ dcb, long long dcb_stride,
                               const float* __restrict__ params, float* __restrict__ grads, const int* __restrict__ offs, int B, int N,
                               float l2coef, int l0) {
  const int l = l0 + blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (Cc + 1) * N) return;
  const int k = i / N, n = i % N;
  const float* d = dcb + (long long)l * dcb_stride;
  float s = 0.f;
  for (int b = 0; b < B; ++b) s = fmaf(k < Cc ? cond[(long long)b * Cc + k] : 1.0f, d[(long long)b * N + n], s);
  if (k < Cc) {
    const long long o = offs[2 * l] + (long long)k * N + n;
    grads[o] = l2coef != 0.f ? fmaf(l2coef, params[o], s) : s;
  } else {
    grads[offs[2 * l + 1] + n] = s;
  }
}
// dcond[b][k] = sum_l sum_n dcb_l[b][n] Wc_l[k][n] ; one block per output: 8 warps stride over the blocks l,
// lanes over n; fixed summation order (deterministic)
__global__ void __launch_bounds__(256) cond_dgrad_all(const float* __restrict__ dcb, long long dcb_stride, const float* __restrict__ params,
                                                      const int* __restrict__ offs, float* __restrict__ dcond, int L, int B, int Cc, int N) {
  __shared__ float red[8];
  const int i = blockIdx.x;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = i / Cc, k = i % Cc;
  float s = 0.f;
  for (int l = w; l < L; l += 8) {
    const float* d = dcb + (long long)l * dcb_stride + (long long)b * N;
    const float* W = params + offs[2 * l] + (long long)k * N;
    for (int n = lane; n < N; n += 32) s = fmaf(d[n], W[n], s);
  }
  s = warp_sum(s);
  if (lane == 0) red[w] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) tot += red[j];
    dcond[(long long)b * Cc + k] = tot;
  }
}

// Keras 3's sparse_categorical_crossentropy on the softmax OUTPUT (model.py:114-118,516) [TF-internal, restated — the golden
// case `cat_saturated` executes it from the reference source over the shim]: c = clip(p, 1e-7, 1 - 1e-7), then sparse softmax
// cross entropy with log(c) as logits:  l = log(sum_j c_j) - log(c_y);  the clip passes gradient only where it is inactive:
//   dl/dlogit_k = p_k (in_k / S - [k == y] in_y / c_y - (Pm / S - in_y)),   S = sum_j c_j = 1 + delta,   Pm = sum_j in_j p_j.
// While no p_j of a row leaves [1e-7, 1 - 1e-7] this is lse - logit_y and softmax - onehot, evaluated as before (rows take the
// clipped form warp-uniformly, only when one of their probabilities is clipped).
#define WN_CE_EPS 1e-7f
struct WnCeClip { float S_inv, dot, y_coef; };
// returns the row loss; `loss_unclipped` = lse - logit_y, p_y = the target's probability as the row loop computes it
__device__ __forceinline__ float wn_ce_clip(WnCeClip& cc, float delta, float pm, float p_y, float loss_unclipped) {
  const bool in_y = p_y >= WN_CE_EPS && p_y <= 1.0f - WN_CE_EPS;
  const float c_y = fminf(fmaxf(p_y, WN_CE_EPS), 1.0f - WN_CE_EPS);
  cc.S_inv = 1.0f / (1.0f + delta);
  cc.dot = pm * cc.S_inv - (in_y ? 1.0f : 0.0f);
  cc.y_coef = in_y ? 1.0f / c_y : 0.0f;
  return log1pf(delta) + (in_y ? loss_unclipped : -logf(c_y));
}
__device__ __forceinline__ float wn_ce_clip_grad(const WnCeClip& cc, float p, bool is_target) {
  const bool in = p >= WN_CE_EPS && p <= 1.0f - WN_CE_EPS;
  return p * ((in ? cc.S_inv : 0.0f) - (is_target ? cc.y_coef : 0.0f) - cc.dot);
}

// Row access of the generic softmax kernels below.  C = 2^bits is a multiple of 4 except at C = 2 (1-bit audio), where a float4
// would take the next row's two values (and be 8-byte aligned on odd rows).  There the row is read element by element into a float4
// whose missing lanes hold `pad`: -inf for logits (p = 0, nothing added to the max, the sum or dot) and 0 for dp; the loops skip
// those lanes for the clip sums and the stores.  For C >= 4 this is the plain float4 load.
__device__ __forceinline__ float4 wn_row_ld4(const float* __restrict__ p, int c, int C, float pad) {
  if (C >= 4) return *reinterpret_cast<const float4*>(p + c);
  return make_float4(p[c], c + 1 < C ? p[c + 1] : pad, c + 2 < C ? p[c + 2] : pad, pad);
}

// ------------------------------------------------------------------ softmax-256 cross entropy (model.py:114-118,516)
// One warp per row.  logits fp32 [rows][C]; the target index is quantised on the fly from
// frames[b][t+1] (model.py:319-320).  Writes per-block loss partials, dlogits (= scale *
// (softmax - onehot)) and optionally the probabilities (WaveNet.call output).
template <class TD>
__global__ void __launch_bounds__(256) softmax_ce_kernel(const float* __restrict__ logits, int C, const float* __restrict__ frames, int Tn,
                                                         long long rows, int bits, float scale, TD* __restrict__ dlogits, int ldd,
                                                         float* __restrict__ probs, float* __restrict__ loss_partial) {
  __shared__ float wsum[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  float loss = 0.f;
  if (row < rows) {
    const float* lp = logits + row * C;
    float m = -INFINITY;
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
      m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
    }
    m = warp_max(m);
    float s = 0.f;
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
      s += expf(v.x - m) + expf(v.y - m) + expf(v.z - m) + expf(v.w - m);
    }
    s = warp_sum(s);
    const float lse = m + logf(s);
    const float inv = 1.0f / s;
    // Keras 3 clip (see wn_ce_clip above): delta = sum_j (clip(p_j) - p_j), pm = sum of the un-clipped p_j
    float delta = 0.f, pm = 0.f;
    bool any_out = false;
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
      const float p[4] = {expf(v.x - m) * inv, expf(v.y - m) * inv, expf(v.z - m) * inv, expf(v.w - m) * inv};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (c + i >= C) break;
        const bool in = p[i] >= WN_CE_EPS && p[i] <= 1.0f - WN_CE_EPS;
        any_out |= !in;
        delta += fminf(fmaxf(p[i], WN_CE_EPS), 1.0f - WN_CE_EPS) - p[i];
        pm += in ? p[i] : 0.f;
      }
    }
    const bool clipped = __any_sync(0xffffffffu, any_out);
    WnCeClip cc;
    cc.S_inv = 1.f; cc.dot = 0.f; cc.y_coef = 1.f;
    if (clipped) { delta = warp_sum(delta); pm = warp_sum(pm); }
    int idx = -1;
    if (frames) {
      long long b, t;
      wn_row_bt(row, rows, Tn, b, t);
      idx = wn_quantize_idx(frames[b * (Tn + 1) + t + 1], bits);
      loss = lse - lp[idx];
      if (clipped) loss = wn_ce_clip(cc, delta, pm, expf(lp[idx] - m) * inv, loss);
    } else if (clipped) {
      wn_ce_clip(cc, delta, pm, 0.5f, 0.f);
    }
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
      float p[4] = {expf(v.x - m) * inv, expf(v.y - m) * inv, expf(v.z - m) * inv, expf(v.w - m) * inv};
      if (probs) {
        if (C >= 4) *reinterpret_cast<float4*>(probs + row * C + c) = make_float4(p[0], p[1], p[2], p[3]);
        else for (int i = 0; i < 4 && c + i < C; ++i) probs[row * C + c + i] = p[i];
      }
      if (dlogits) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (c + i < C) dlogits[row * ldd + c + i] = from_f<TD>((clipped ? wn_ce_clip_grad(cc, p[i], c + i == idx) : p[i] - (c + i == idx ? 1.0f : 0.0f)) * scale);
      }
    }
  }
  if (loss_partial) {
    if (lane == 0) wsum[warp] = loss;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += wsum[i];
      loss_partial[blockIdx.x] = t;
    }
  }
}

// register-resident variant for C = 128 * NV4 classes (C = 256 for 8-bit audio): the row is read from memory ONCE,
// exp is evaluated once per element; same arithmetic order as softmax_ce_kernel (bit-identical results)
template <class TD, int NV4>
__global__ void __launch_bounds__(256) softmax_ce_reg_kernel(const float* __restrict__ logits, const float* __restrict__ frames, int Tn, long long rows,
                                                             int bits, float scale, TD* __restrict__ dlogits, int ldd, float* __restrict__ probs,
                                                             float* __restrict__ loss_partial) {
  constexpr int C = 128 * NV4;
  __shared__ float wsum[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  float loss = 0.f;
  if (row < rows) {
    const float* lp = logits + row * C;
    float4 v[NV4];
#pragma unroll
    for (int i = 0; i < NV4; ++i) v[i] = *reinterpret_cast<const float4*>(lp + lane * 4 + i * 128);
    float m = -INFINITY;
#pragma unroll
    for (int i = 0; i < NV4; ++i) m = fmaxf(m, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
    m = warp_max(m);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      v[i].x = expf(v[i].x - m); v[i].y = expf(v[i].y - m); v[i].z = expf(v[i].z - m); v[i].w = expf(v[i].w - m);
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    s = warp_sum(s);
    const float inv = 1.0f / s;
    // Keras 3 clip (see wn_ce_clip above).  Detection costs one min per element: the largest probability of the row is exactly
    // `inv` (its exponent is exp(0) = 1), the smallest is min_j e_j * inv (x -> x * inv is monotonic).
    float emin = INFINITY;
#pragma unroll
    for (int i = 0; i < NV4; ++i) emin = fminf(emin, fminf(fminf(v[i].x, v[i].y), fminf(v[i].z, v[i].w)));
    const bool clipped = __any_sync(0xffffffffu, emin * inv < WN_CE_EPS || inv > 1.0f - WN_CE_EPS);   // warp-uniform
    WnCeClip cc;
    cc.S_inv = 1.f; cc.dot = 0.f; cc.y_coef = 1.f;
    float delta = 0.f, pm = 0.f;     // delta = sum_j (clip(p_j) - p_j), pm = sum of the un-clipped p_j
    if (clipped) {
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const float p[4] = {v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool in = p[j] >= WN_CE_EPS && p[j] <= 1.0f - WN_CE_EPS;
          delta += fminf(fmaxf(p[j], WN_CE_EPS), 1.0f - WN_CE_EPS) - p[j];
          pm += in ? p[j] : 0.f;
        }
      }
      delta = warp_sum(delta); pm = warp_sum(pm);
    }
    int idx = -1;
    if (frames) {
      long long b, t;
      wn_row_bt(row, rows, Tn, b, t);
      idx = wn_quantize_idx(frames[b * (Tn + 1) + t + 1], bits);
      loss = (m + logf(s)) - lp[idx];
      if (clipped) loss = wn_ce_clip(cc, delta, pm, expf(lp[idx] - m) * inv, loss);
    } else if (clipped) {
      wn_ce_clip(cc, delta, pm, 0.5f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const int c = lane * 4 + i * 128;
      const float p[4] = {v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv};
      if (probs) *reinterpret_cast<float4*>(probs + row * C + c) = make_float4(p[0], p[1], p[2], p[3]);
      if (dlogits) {
        float d[4];
        if (clipped) {
#pragma unroll
          for (int j = 0; j < 4; ++j) d[j] = wn_ce_clip_grad(cc, p[j], c + j == idx) * scale;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) d[j] = (p[j] - (c + j == idx ? 1.0f : 0.0f)) * scale;
        }
        if constexpr (sizeof(TD) == 2) {
          uint2 q;
          q.x = pack_bf16x2(d[0], d[1]); q.y = pack_bf16x2(d[2], d[3]);
          *reinterpret_cast<uint2*>(dlogits + row * ldd + c) = q;
        } else {
          *reinterpret_cast<float4*>(dlogits + row * ldd + c) = make_float4(d[0], d[1], d[2], d[3]);
        }
      }
    }
  }
  if (loss_partial) {
    if (lane == 0) wsum[warp] = loss;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += wsum[i];
      loss_partial[blockIdx.x] = t;
    }
  }
}

// ------------------------------------------------------------------ adjoint of the probabilities WaveNet.call returns (model.py:238)
// dlogits[r][c] = p_c (dp_c - sum_j p_j dp_j) for a caller's dp = d loss / d p.  One warp per row; p is recomputed from the logits
// with softmax_ce_kernel's arithmetic, so it is bit-for-bit the p that wn_forward returned.  Columns [C, ldd) are zeroed: the head's
// dgrad contracts over ldd columns on the bf16 tier.
template <class TD>
__global__ void __launch_bounds__(256) softmax_vjp_kernel(const float* __restrict__ logits, int C, const float* __restrict__ dp, long long rows,
                                                          TD* __restrict__ dlogits, int ldd) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const float* lp = logits + row * C;
  const float* gp = dp + row * C;
  float m = -INFINITY;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
    m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
  }
  m = warp_max(m);
  float s = 0.f;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
    s += expf(v.x - m) + expf(v.y - m) + expf(v.z - m) + expf(v.w - m);
  }
  s = warp_sum(s);
  const float inv = 1.0f / s;
  float dot = 0.f;
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
    const float4 g = wn_row_ld4(gp, c, C, 0.f);
    dot += expf(v.x - m) * inv * g.x + expf(v.y - m) * inv * g.y + expf(v.z - m) * inv * g.z + expf(v.w - m) * inv * g.w;
  }
  dot = warp_sum(dot);
  for (int c = lane * 4; c < C; c += 128) {
    const float4 v = wn_row_ld4(lp, c, C, -INFINITY);
    const float4 g = wn_row_ld4(gp, c, C, 0.f);
    const float p[4] = {expf(v.x - m) * inv, expf(v.y - m) * inv, expf(v.z - m) * inv, expf(v.w - m) * inv};
    const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) if (c + i < C) dlogits[row * ldd + c + i] = from_f<TD>(p[i] * (gv[i] - dot));
  }
  for (int c = C + lane; c < ldd; c += 32) dlogits[row * ldd + c] = from_f<TD>(0.f);
}

// register-resident variant for C = 128 * NV4 classes (C = 256 for 8-bit audio): logits and dp are read once; p has the arithmetic
// order of softmax_ce_reg_kernel (bit-identical to softmax_vjp_kernel)
template <class TD, int NV4>
__global__ void __launch_bounds__(256) softmax_vjp_reg_kernel(const float* __restrict__ logits, const float* __restrict__ dp, long long rows,
                                                              TD* __restrict__ dlogits, int ldd) {
  constexpr int C = 128 * NV4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  float4 v[NV4], g[NV4];
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    v[i] = *reinterpret_cast<const float4*>(logits + row * C + lane * 4 + i * 128);
    g[i] = *reinterpret_cast<const float4*>(dp + row * C + lane * 4 + i * 128);
  }
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV4; ++i) m = fmaxf(m, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
  m = warp_max(m);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    v[i].x = expf(v[i].x - m); v[i].y = expf(v[i].y - m); v[i].z = expf(v[i].z - m); v[i].w = expf(v[i].w - m);
    s += v[i].x + v[i].y + v[i].z + v[i].w;
  }
  s = warp_sum(s);
  const float inv = 1.0f / s;
  float dot = 0.f;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    v[i].x *= inv; v[i].y *= inv; v[i].z *= inv; v[i].w *= inv;
    dot += v[i].x * g[i].x + v[i].y * g[i].y + v[i].z * g[i].z + v[i].w * g[i].w;
  }
  dot = warp_sum(dot);
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    const int c = lane * 4 + i * 128;
    const float d[4] = {v[i].x * (g[i].x - dot), v[i].y * (g[i].y - dot), v[i].z * (g[i].z - dot), v[i].w * (g[i].w - dot)};
    if constexpr (sizeof(TD) == 2) {
      uint2 q;
      q.x = pack_bf16x2(d[0], d[1]); q.y = pack_bf16x2(d[2], d[3]);
      *reinterpret_cast<uint2*>(dlogits + row * ldd + c) = q;
    } else {
      *reinterpret_cast<float4*>(dlogits + row * ldd + c) = make_float4(d[0], d[1], d[2], d[3]);
    }
  }
  for (int c = C + lane; c < ldd; c += 32) dlogits[row * ldd + c] = from_f<TD>(0.f);
}

// ------------------------------------------------------------------ WaveNet.loss_fn on materialised probabilities (model.py:516)
// tf.keras.losses.sparse_categorical_crossentropy(target, probs), Keras 3 semantics [TF-internal, restated]: the probabilities
// are clipped to [1e-7, 1 - 1e-7], their logarithm is taken as logits of sparse_softmax_cross_entropy_with_logits:
//   l = log(sum_i clip(p_i)) - log(clip(p_y)).   One warp per row; the target is an int64 class index or, when idx == null,
// a waveform sample quantised like prepare_target (model.py:151-155).
__global__ void __launch_bounds__(256) ce_probs_rows_kernel(const float* __restrict__ probs, int C, const long long* __restrict__ idx,
                                                            const float* __restrict__ wave, int bits, long long rows, float* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const float* p = probs + row * C;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += fminf(fmaxf(p[c], 1e-7f), 1.0f - 1e-7f);
  s = warp_sum(s);
  if (lane == 0) {
    long long y = idx ? idx[row] : (long long)wn_quantize_idx(wave[row], bits);
    y = y < 0 ? 0 : (y >= C ? C - 1 : y);
    out[row] = logf(s) - logf(fminf(fmaxf(p[y], 1e-7f), 1.0f - 1e-7f));
  }
}

// ------------------------------------------------------------------ mixture losses (model.py:517-547)
// pred fp32 [rows][ldp] = [weights M | means M | log-scales M].  kind: 1 logistic, 2 gaussian.  SQRT2PI is the fp32 value of
// sqrt(2*3.14159265359) (model.py:9).
// G lanes per row (G = 4 / 8 / 16 / 32 >= M), lane m owns mixture component m: the three parameter loads and the three
// gradient stores of a row are coalesced, softmax over the weights and the likelihood sum are G-wide shuffle reductions, and
// the chain of exp / log / sigmoid per row is one component long.  (Round 1-2: one thread per row walking all M components
// through local-memory arrays — 53 us per C4 step at 20 % of the warps active, 8 MB read; ncu_full_r3a_c4_mixture_loss.txt.)
#define WN_MAX_MIX 32
template <int G>
__device__ __forceinline__ float wn_group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int G>
__device__ __forceinline__ float wn_group_max(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <class TD, int G>
__global__ void __launch_bounds__(256) mixture_loss_kernel(const float* __restrict__ pred, int ldp, int M, const float* __restrict__ frames,
                                                           int Tn, long long rows, int bits, int kind, float scale, TD* __restrict__ dpred,
                                                           int ldd, float* __restrict__ loss_partial, int frame_stride, int frame_off,
                                                           float* __restrict__ row_out) {
  __shared__ float wsum[8];
  constexpr int RPB = 256 / G;                       // rows per block
  const int gl = threadIdx.x & (G - 1);              // component of this lane
  const long long row = (long long)blockIdx.x * RPB + threadIdx.x / G;
  const bool rok = row < rows;                       // uniform over the G lanes of a row (every lane takes part in the shuffles)
  const bool act = rok && gl < M;
  float loss = 0.f;
  float y = 0.f, w = -INFINITY, mu = 0.f, lsr = 0.f;
  if (rok) {
    long long b, t;
    wn_row_bt(row, rows, Tn, b, t);
    // training / test step: the target of position t is frames[b][t+1] (model.py:319); loss_fn: a dense (B,T) target
    y = frames[b * frame_stride + t + frame_off];
  }
  if (act) {
    const float* p = pred + row * ldp;
    w = p[gl]; mu = p[M + gl]; lsr = p[2 * M + gl];
  }
  const float wmax = wn_group_max<G>(w);
  float pi = act ? expf(w - wmax) : 0.f;
  const float wsumv = wn_group_sum<G>(pi);
  pi = rok ? pi / wsumv : 0.f;
  const float SQRT2PI = 2.50662827463100050242f;
  const float h = 0.5f / (float)(1 << bits);
  const float ls = fmaxf(lsr, -7.0f);
  float comp = 0.f, sc = 1.f, e = 1.f;
  if (act) {
    if (kind == 2) {
      sc = expf(ls);
      const float xx = fminf((y - mu) / sc, 1e8f);
      comp = expf(-0.5f * xx * xx) / (sc * SQRT2PI);
    } else {
      // sigma(a) - sigma(b) == sigma(a) * sigma(-b) * (1 - exp(-(a-b))), a-b = 2h*e: the same
      // quantity as model.py:543-544 without the fp32 cancellation of two nearly equal sigmoids
      e = expf(-ls);
      comp = wn_sigmoid<false>((y - mu + h) * e) * wn_sigmoid<false>(-(y - mu - h) * e) * (-expm1f(-2.0f * h * e));
    }
  }
  const float lik = wn_group_sum<G>(pi * comp);
  if (rok) {
    loss = -logf(lik);
    if (row_out && gl == 0) row_out[row] = loss;
    if (dpred) {
      TD* d = dpred + row * ldd;
      if (act) {
        const float linv = 1.0f / lik;
        const float pass = lsr >= -7.0f ? 1.0f : 0.0f;
        const float r = pi * comp * linv;
        float dmu, dls;
        if (kind == 2) {
          const float xr = (y - mu) / sc;
          const float nc = xr <= 1e8f ? 1.0f : 0.0f;
          const float xx = fminf(xr, 1e8f);
          dmu = -r * xx / sc * nc;
          dls = -r * (xx * xx * nc - 1.0f) * pass;
        } else {
          const float a = (y - mu + h) * e, bq = (y - mu - h) * e, dab = 2.0f * h * e;
          const float sa = wn_sigmoid<false>(a), snb = wn_sigmoid<false>(-bq);
          // sigma'(a) - sigma'(b) = (sigma(a)-sigma(b)) * (1 - sigma(a) - sigma(b)) ; comp holds sigma(a)-sigma(b)
          const float dd = comp * (snb - sa);
          const float dsb = snb * (1.0f - snb);
          const float c = pi * linv;
          dmu = c * e * dd;
          dls = c * (a * dd + dab * dsb) * pass;
        }
        d[gl] = from_f<TD>((pi - r) * scale);
        d[M + gl] = from_f<TD>(dmu * scale);
        d[2 * M + gl] = from_f<TD>(dls * scale);
      }
      for (int m = 3 * M + gl; m < ldd; m += G) d[m] = from_f<TD>(0.f);      // padding columns of the gradient operand
    }
  }
  if (loss_partial) {
    // one value per row (lane 0 of its group), fixed order: warp shuffle tree, then the 8 warps in sequence
    float v = (rok && gl == 0) ? loss : 0.f;
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tot = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) tot += wsum[i];
      loss_partial[blockIdx.x] = tot;
    }
  }
}
// lanes per row for M components
static inline int mixture_lanes(int M) { return M <= 4 ? 4 : (M <= 8 ? 8 : (M <= 16 ? 16 : 32)); }
template <class TD>
static void mixture_loss_launch(cudaStream_t st, int* nparts_out, const float* pred, int ldp, int M, const float* frames, int Tn, long long rows, int bits,
                                int kind, float scale, TD* dpred, int ldd, float* loss_partial, int frame_stride, int frame_off, float* row_out) {
  const int G = mixture_lanes(M);
  const int nparts = (int)((rows + 256 / G - 1) / (256 / G));
  if (nparts_out) *nparts_out = nparts;
#define WN_MIX_GO(GG) mixture_loss_kernel<TD, GG><<<nparts, 256, 0, st>>>(pred, ldp, M, frames, Tn, rows, bits, kind, scale, dpred, ldd, loss_partial, \
                                                                          frame_stride, frame_off, row_out)
  if (G == 4) WN_MIX_GO(4); else if (G == 8) WN_MIX_GO(8); else if (G == 16) WN_MIX_GO(16); else WN_MIX_GO(32);
#undef WN_MIX_GO
}

// final loss: out[0] = scale * sum(partial) (metric 'loss'), out[1] = extra_coef * extra (metric 'reg_loss', model.py:340-344)
// (single block, deterministic)
__global__ void loss_finalize(const float* __restrict__ partial, int n, float scale, const float* __restrict__ extra, float extra_coef,
                              float* __restrict__ out) {
  __shared__ float sh[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += partial[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) { out[0] = v * scale; out[1] = extra ? extra_coef * extra[0] : 0.f; }
  }
}

// sum of squares of a weight tensor (L2 regulariser, model.py:331-334), single block, accumulates
__global__ void sumsq_accum(const float* __restrict__ w, long long n, float* __restrict__ out) {
  __shared__ float sh[32];
  float s = 0.f;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s = fmaf(w[i], w[i], s);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) out[0] += v;
  }
}

// ------------------------------------------------------------------ quantiser (model.py:151-155)
__global__ void quantize_kernel(const float* __restrict__ x, long long* __restrict__ idx, long long n, int bits) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) idx[i] = wn_quantize_idx(x[i], bits);
}

// ------------------------------------------------------------------ optimizer (train.py:225-226, model.py:336)
// tf.keras.optimizers.Adam(learning_rate, clipnorm=1.0) on the flat fp32 buffers.  The flat buffer is cut into chunks
// of OPT_CHUNK elements that never straddle a variable: chunk c = (variable id, first element, count).
#define OPT_CHUNK 4096
struct OptChunk { int var; int count; long long start; };
// per-chunk sum of squares of the gradient (deterministic: fixed tree per chunk)
__global__ void __launch_bounds__(256) opt_sumsq_kernel(const float* __restrict__ g, const OptChunk* __restrict__ chunks, float* __restrict__ partial) {
  const OptChunk c = chunks[blockIdx.x];
  const float* p = g + c.start;
  float s = 0.f;
  for (int i = threadIdx.x; i < c.count; i += 256) s = fmaf(p[i], p[i], s);
  __shared__ float sh[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < 8 ? sh[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) partial[blockIdx.x] = v;
  }
}
// per variable: norm = sqrt(sum of its chunk partials, in chunk order); tf.clip_by_norm scale = clipnorm / max(norm, clipnorm)
__global__ void opt_clip_scale_kernel(const float* __restrict__ partial, const int* __restrict__ var_first_chunk, int n_vars, float clipnorm,
                                      float* __restrict__ scale, float* __restrict__ norms) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_vars) return;
  float s = 0.f;
  for (int c = var_first_chunk[v]; c < var_first_chunk[v + 1]; ++c) s += partial[c];
  const float n = sqrtf(s);
  norms[v] = n;
  scale[v] = clipnorm > 0.f ? clipnorm / fmaxf(n, clipnorm) : 1.0f;
}
__global__ void __launch_bounds__(256) opt_clip_apply_kernel(float* __restrict__ g, const OptChunk* __restrict__ chunks, const float* __restrict__ scale) {
  const OptChunk c = chunks[blockIdx.x];
  const float sc = scale[c.var];
  if (sc == 1.0f) return;
  float* p = g + c.start;
  for (int i = threadIdx.x; i < c.count; i += 256) p[i] *= sc;
}
// Keras 3 Adam.update_step: m += (g - m)(1 - b1); v += (g^2 - v)(1 - b2); w -= alpha * m / (sqrt(v) + eps),
// alpha = lr * sqrt(1 - b2^t) / (1 - b1^t)
__global__ void __launch_bounds__(256) opt_adam_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                       long long n, float alpha, float one_minus_b1, float one_minus_b2, float eps) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i];
  const float mi = fmaf(gi - m[i], one_minus_b1, m[i]);
  const float vi = fmaf(fmaf(gi, gi, -v[i]), one_minus_b2, v[i]);
  m[i] = mi; v[i] = vi;
  w[i] -= alpha * mi / (sqrtf(vi) + eps);
}

// ------------------------------------------------------------------ sample_waveform (model.py:393-503) + MSE metric (model.py:338-346)
// One warp per (b,t) row.  kind 0: categorical over C classes; `is_logits` says whether `pred` holds pre-softmax logits
// (the fused train step keeps those) or probabilities (WaveNet.call output).  deterministic: argmax (first maximum);
// otherwise inverse-CDF draw with a Philox uniform per row (TF's stateless_categorical / seed (4,2) stream cannot be
// reproduced: statistical parity only).  Output idx / 2^(bits-1) - 1.
// kinds 1/2: logistic / gaussian mixtures, pred = [weights M | means M | log-scales M]: component = argmax or a
// categorical draw over softmax(weights); sample = mu (deterministic) or mu + scale*(log u - log(1-u)) / mu + scale*z;
// clipped to [-1,1].  Optional: squared error against y (frames[b][t+1]) accumulated per block -> mse_partial.
__global__ void __launch_bounds__(256) sample_kernel(const float* __restrict__ pred, int ld, int C, int M, int kind, int is_logits, int bits,
                                                     int deterministic, unsigned long long seed, const float* __restrict__ frames, int Tn,
                                                     long long rows, float* __restrict__ out, float* __restrict__ mse_partial,
                                                     const int* __restrict__ ctr_dev = nullptr) {
  __shared__ float wsum[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  float err2 = 0.f;
  if (row < rows) {
    const float* p = pred + row * ld;
    // ctr_dev: device-side step counter (autoregressive generation replays one graph for every step)
    const uint4 rnd = philox4x32_10(make_uint4((uint32_t)row, (uint32_t)(row >> 32), 0x5A17u, ctr_dev ? (uint32_t)*ctr_dev : 0u),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const float u0 = ((float)(rnd.x >> 8) + 0.5f) * (1.0f / 16777216.0f);   // (0,1)
    const float u1 = ((float)(rnd.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(rnd.z >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const int n = kind == 0 ? C : M;
    // softmax statistics of the n selection weights (identity for probabilities)
    float mx = -INFINITY;
    for (int c = lane; c < n; c += 32) mx = fmaxf(mx, p[c]);
    mx = warp_max(mx);
    const bool soft = kind != 0 || is_logits;
    float sum = 0.f;
    for (int c = lane; c < n; c += 32) sum += soft ? expf(p[c] - mx) : p[c];
    sum = warp_sum(sum);
    int sel;
    if (deterministic) {
      // first index attaining the maximum (tf.argmax)
      int best = 0x7fffffff;
      for (int c = lane; c < n; c += 32) if (p[c] == mx) { best = c; break; }
      for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
      sel = best;
    } else {
      // smallest k with cdf(k) > u*sum : lane-strided partial sums in class order chunks of 32
      const float target = u0 * sum;
      float run = 0.f;
      sel = n - 1;
      bool found = false;
      for (int c0 = 0; c0 < n && !found; c0 += 32) {
        const int c = c0 + lane;
        float w = c < n ? (soft ? expf(p[c] - mx) : p[c]) : 0.f;
        float incl = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const float t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        const unsigned hit = __ballot_sync(0xffffffffu, c < n && run + incl > target);
        if (hit) { sel = c0 + __ffs(hit) - 1; found = true; }
        run += __shfl_sync(0xffffffffu, incl, 31);
      }
    }
    float val;
    if (kind == 0) {
      val = (float)sel / exp2f((float)(bits - 1)) - 1.0f;
    } else {
      const float mu = p[M + sel];
      if (deterministic) val = mu;
      else {
        const float sc = expf(p[2 * M + sel]);
        if (kind == 1) val = mu + sc * (logf(u1) - logf(1.0f - u1));
        else val = mu + sc * sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
      }
      val = fminf(fmaxf(val, -1.0f), 1.0f);
    }
    if (lane == 0) {
      out[row] = val;
      if (frames) {
        const long long b = row / Tn, t = row % Tn;
        const float d = frames[b * (Tn + 1) + t + 1] - val;
        err2 = d * d;
      }
    }
  }
  if (mse_partial) {
    if (lane == 0) wsum[warp] = err2;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += wsum[i];
      mse_partial[blockIdx.x] = t;
    }
  }
}

// ------------------------------------------------------------------ device input pipeline (utils.py:31-70, callbacks.py:126-131)
// mu-law companding utils.py:35: sign(x) * log(1 + 255|x|) / log(256).  Evaluated in fp64 and rounded once, i.e. the
// correctly rounded fp32 value of the formula (TF evaluates it with its own fp32 log: <= 1 ulp from this).
__device__ __forceinline__ float wn_mu_law(float x) {
  const double a = fabs((double)x);
  const double y = log(1.0 + 255.0 * a) / 5.545177444479562;   // log(256)
  const float r = (float)y;
  return x > 0.f ? r : (x < 0.f ? -r : 0.f * x);
}
// frames[f][i] = g(speech[f*T + i]), i in [0, T], f in [0, n_frames): tf.signal.frame(frame_length=T+1, frame_step=T)
// (utils.py:36-38), g = optional /2^15 for int16 input (utils.py:52-55) then optional mu-law.  valid[f] = every sample
// finite and within [-1,1] (utils.py:58-70; the length test is always true for un-padded frames).
template <class TIN>
__global__ void preprocess_frames_kernel(const TIN* __restrict__ speech, float in_scale, int T, int n_frames, int apply_mulaw,
                                         float* __restrict__ frames, int* __restrict__ valid) {
  const int f = blockIdx.y;
  int bad = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= T; i += gridDim.x * blockDim.x) {
    float x = (float)speech[(long long)f * T + i] * in_scale;
    if (apply_mulaw) x = wn_mu_law(x);
    frames[(long long)f * (T + 1) + i] = x;
    if (!(isfinite(x) && x >= -1.0f && x <= 1.0f)) bad = 1;
  }
  if (bad) atomicAnd(valid + f, 0);     // idempotent flag clear: order-independent
}
__global__ void fill_int_kernel(int* p, int n, int v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// callbacks.py:126-131: sign(y) * (256^|y| - 1) / 255
__global__ void inverse_mu_law_kernel(const float* __restrict__ y, float* __restrict__ x, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = y[i];
  const float r = (float)((exp(fabs((double)v) * 5.545177444479562) - 1.0) / 255.0);
  x[i] = v > 0.f ? r : (v < 0.f ? -r : 0.f * v);
}
// tf.one_hot(ids, depth): rows of zeros with a one at ids[i] (all zeros when the id is out of range)
__global__ void one_hot_kernel(const int* __restrict__ ids, int n, int depth, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)n * depth) return;
  out[i] = ids[i / depth] == (int)(i % depth) ? 1.0f : 0.0f;
}
