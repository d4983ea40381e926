// tc_epilogues.cuh — fused epilogues of the tcgen05 conv GEMM, TMA-staged variant.
//
// The accumulator lives in TMEM with one ROW per thread, but HBM wants whole rows per warp.
// So every epilogue tensor moves through shared memory as half-panels of 128 rows x 32 bf16
// columns (64-byte rows, 64B swizzle): inputs (residual, cached pre-activations, ...) arrive by
// TMA load, outputs leave by TMA store, and rows / columns outside the tensor are clipped by
// the tensor map (no per-thread bounds logic).  A functor only sees 16 columns of one row:
//
//   Epi::chunk(params, acc, b, acc_col, half, col, in_mask, in, out)
//     acc.load16(c, v)  accumulator columns [c, c+16) of this row, relative to the CTA tile
//     acc_col           first accumulator column of this chunk (gate: filter half; gate half at +half)
//     col               first output column of this chunk in the output tensors' own numbering
//     in[k][16]         staged inputs (fp32), valid when bit k of in_mask is set
//     out[k][16]        results (fp32; the kernel rounds to bf16 and stages them for the TMA store)
//     bs                per-tile bias table in shared memory (the kernel's L1 is carved down to a few KB by
//                       the operand ring, so per-chunk global bias loads would each pay an L2 round trip):
//                       Epi::bias_load() fetches this thread's entries at tile start (latency hidden behind
//                       the wait for the accumulator), the kernel stores them, chunk() reads them by broadcast
//   kBiasFloats(BN) table entries; each of the 256 epilogue threads loads entry `tid` (and tid+256 if needed)
#pragma once
#include "common.cuh"

__device__ __forceinline__ void ld_bias16(const float* p, float* v) {   // shared-memory broadcast read
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 q = reinterpret_cast<const float4*>(p)[i];
    v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
  }
}

// out = act(acc + bias[n] + cbias[b][n]) + res      (layers.py:66-74,213,222-223; model.py:105-119,236)
// (2 input half-panels: the skip sum and the head convs have no epilogue input at all and get 5 mainloop stages; the unfused
// conv1 with a residual input keeps a 2-slot ring.  C2: 6.10 -> 6.00 ms/step, same box)
template <bool FAST> struct TcEpiBiasActRes {
  static constexpr int NIN = 1, NOUT = 1;
  static constexpr int kInPanels = 2, kOutSlots = 4;
  static constexpr bool kGate = false;
  struct Params { const float* bias; const float* cbias; int ldcb; int act; int N; };
  static constexpr int kBiasFloats(int BN) { return BN; }
  // entry i of the tile's table: bias[n0+i] + cbias[b][n0+i]
  static __device__ __forceinline__ float bias_load(const Params& p, int b, int tile_col0, int BN, int i) {
    const int n = tile_col0 + i;
    float v = 0.f;
    if (n < p.N) {
      if (p.bias) v = __ldg(p.bias + n);
      if (p.cbias) v += __ldg(p.cbias + (long long)b * p.ldcb + n);
    }
    return v;
  }
  template <class Acc>
  static __device__ __forceinline__ void chunk(const Params& p, Acc& acc, int b, int acc_col, int half, int col, uint32_t in_mask,
                                               const float (*in)[16], float (*out)[16], const float* bs) {
    float v[16];
    acc.load16(acc_col, v);
    {
      float t[16];
      ld_bias16(bs + acc_col, t);
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] += t[i];
    }
    if (p.act != ACT_LINEAR) {
      wn_act16<FAST>(p.act, v);
    }
    if (in_mask & 1u) {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] += in[0][i];
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) out[0][i] = v[i];
  }
};

// gated activation (layers.py:203-210): tile = [filter half | gate half]; outputs P, Q, g.
// bf16 tier: the backward pass needs z only to evaluate the gate's derivative.  Instead of z the forward pass caches the
// two derivative coefficients themselves, computed from the un-rounded fp32 accumulator it holds anyway:
//   P = d g / d z_f = sigmoid(z_s) (1 - tanh(z_f)^2)        Q = d g / d z_s = tanh(z_f) sigmoid(z_s) (1 - sigmoid(z_s))
// (same bytes as z_f, z_s).  The gate adjoint becomes d z_f = d g * P, d z_s = d g * Q: no tanh / sigmoid recomputation
// (2 MUFU + ~20 issue slots per element: the stack-backward kernel's DG epilogue was instruction bound at 8.3 k cycles per
// 256-row tile, MUFU floor 4.1 k), and the coefficients carry bf16's 2^-9 relative error instead of the error of a derivative
// evaluated at a bf16-rounded z (up to 1.2 %).  The fp32 tier keeps z (csrc/epilogues.cuh).
template <bool FAST> struct TcEpiGate {
  static constexpr int NIN = 0, NOUT = 3;
  static constexpr int kInPanels = 0, kOutSlots = 3;
  static constexpr bool kGate = true;
  struct Params { const float* bias; const float* cbias; int D; };
  static constexpr int kBiasFloats(int BN) { return BN; }
  // table = [filter half (BN/2) | gate half (BN/2)], same order as the accumulator tile; tile_col0 = first channel
  static __device__ __forceinline__ float bias_load(const Params& p, int b, int tile_col0, int BN, int i) {
    const int half = BN >> 1;
    const int ch = tile_col0 + (i < half ? i : i - half);
    float v = 0.f;
    if (ch < p.D) {
      const int n = i < half ? ch : p.D + ch;
      v = __ldg(p.bias + n);
      if (p.cbias) v += __ldg(p.cbias + (long long)b * 2 * p.D + n);
    }
    return v;
  }
  template <class Acc>
  static __device__ __forceinline__ void chunk(const Params& p, Acc& acc, int b, int acc_col, int half, int col, uint32_t in_mask,
                                               const float (*in)[16], float (*out)[16], const float* bs) {
    float f[16], s[16];
    acc.load16(acc_col, f);
    acc.load16(half + acc_col, s);
    {
      float t[16];
      ld_bias16(bs + acc_col, t);
#pragma unroll
      for (int i = 0; i < 16; ++i) f[i] += t[i];
      ld_bias16(bs + half + acc_col, t);
#pragma unroll
      for (int i = 0; i < 16; ++i) s[i] += t[i];
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float th = wn_tanh<FAST>(f[i]), sg = wn_sigmoid<FAST>(s[i]);
      const float g = th * sg;
      out[0][i] = fmaf(-sg * th, th, sg);      // P = sg (1 - th^2)
      out[1][i] = fmaf(-g, sg, g);             // Q = th sg (1 - sg)
      out[2][i] = g;
    }
  }
};

// adjoint of the gate: acc = dg; inputs the cached derivative coefficients P, Q (see TcEpiGate); outputs dz_f, dz_s
// Ring depths trade against mainloop stages (every 4 half-panels = one 32 KB operand stage).  Measured on C2 (same box, ms/step):
// dgrad with 4 input half-panels (4 mainloop stages instead of 3) 6.10 vs 6.25; gate adjoint with 4 instead of 8: 6.36 (its
// epilogue streams z from HBM and wants the deep ring).
template <bool FAST> struct TcEpiGateBwd {
  static constexpr int NIN = 2, NOUT = 2;
  static constexpr int kInPanels = 8, kOutSlots = 2;
  static constexpr bool kGate = false;
  struct Params { int D; };
  static constexpr int kBiasFloats(int BN) { return 0; }
  static __device__ __forceinline__ float bias_load(const Params& p, int b, int tile_col0, int BN, int i) { return 0.f; }
  template <class Acc>
  static __device__ __forceinline__ void chunk(const Params& p, Acc& acc, int b, int acc_col, int half, int col, uint32_t in_mask,
                                               const float (*in)[16], float (*out)[16], const float* bs) {
    float dg[16];
    acc.load16(acc_col, dg);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      out[0][i] = dg[i] * in[0][i];
      out[1][i] = dg[i] * in[1][i];
    }
  }
};

// dgrad: out = (acc + add) * act'(y)    (residual pass-through; activation adjoint from its cached output)
struct TcEpiActBwd {
  static constexpr int NIN = 2, NOUT = 1;
  static constexpr int kInPanels = 4, kOutSlots = 4;
  static constexpr bool kGate = false;
  struct Params { int act; };
  static constexpr int kBiasFloats(int BN) { return 0; }
  static __device__ __forceinline__ float bias_load(const Params& p, int b, int tile_col0, int BN, int i) { return 0.f; }
  template <class Acc>
  static __device__ __forceinline__ void chunk(const Params& p, Acc& acc, int b, int acc_col, int half, int col, uint32_t in_mask,
                                               const float (*in)[16], float (*out)[16], const float* bs) {
    float v[16];
    acc.load16(acc_col, v);
    if (in_mask & 1u) {
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] += in[0][i];
    }
    if (in_mask & 2u) {
      wn_act_grad16(p.act, in[1], v);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) out[0][i] = v[i];
  }
};
