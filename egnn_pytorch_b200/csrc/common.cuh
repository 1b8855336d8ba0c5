// Shared helpers for libegnn_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stddef.h>
#include <math.h>

#include "../../include/egnn_b200.h"

namespace egnn {

// ------------------------------------------------------------------ error plumbing
#define EGNN_CUDA_TRY(expr)                                         \
  do {                                                              \
    cudaError_t _e = (expr);                                        \
    if (_e != cudaSuccess) return EGNN_ERR_CUDA - (int)_e;          \
  } while (0)

#define EGNN_TRY(expr)                                              \
  do {                                                              \
    int _r = (expr);                                                \
    if (_r != EGNN_OK) return _r;                                   \
  } while (0)

__host__ __device__ inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ inline size_t round_up(size_t a, size_t b) { return (a + b - 1) / b * b; }
__host__ __device__ inline int round_up_i(int a, int b) { return (a + b - 1) / b * b; }

// Lays blocks out back to back in one buffer: take() returns the offset of the next block, and each block's size is
// rounded up to `align` so the one after it starts aligned.
struct BumpAlloc {
  size_t total = 0;
  size_t take(size_t n, size_t align = 256) { const size_t r = total; total += round_up(n, align); return r; }
};

// ------------------------------------------------------------------ derived sizes
struct Dims {
  int B, N, C, dim, edge_dim, label_dim, num_labels, m, F, k;
  int Qd;      // distance feature channels 2F+1            (egnn_pytorch.py:34-41)
  int Q;       // per-pair scalar channels Qd + edge_dim
  int E;       // edge_input_dim                             (egnn_pytorch.py:175)
  int H;       // hidden width 2E                            (egnn_pytorch.py:179)
  int Hp;      // H rounded up to 8 (zero padded)
  int M;       // B*N rows
  int row0, row1;
};

inline Dims make_dims(const EgnnLayerDesc& d) {
  Dims s;
  s.B = d.B; s.N = d.N; s.C = d.C; s.dim = d.dim; s.edge_dim = d.edge_dim;
  s.label_dim = d.label_dim; s.num_labels = d.num_labels; s.m = d.m_dim; s.F = d.fourier; s.k = d.k;
  s.Qd = 2 * d.fourier + 1;
  s.Q = s.Qd + d.edge_dim;
  s.E = 2 * d.dim + s.Q + d.label_dim;
  s.H = 2 * s.E;
  s.Hp = round_up_i(s.H, 8);
  s.M = d.B * d.N;
  s.row0 = d.row_begin; s.row1 = d.row_end;
  if (s.row0 == 0 && s.row1 == 0) s.row1 = d.N;
  return s;
}

// ------------------------------------------------------------------ dropout (training mode, egnn_pytorch.py:176-208)
// nn.Dropout(p) sits between Linear-1 and SiLU of edge_mlp / node_mlp / coors_mlp.  The masks are never stored: every
// kernel (forward, recompute, backward) regenerates the keep/drop decision of an element from a counter hash of
// (seed, stream, element index) -- stream 0: edge hidden (pair, channel), 1: coors hidden (pair, unit), 2: node hidden
// (node, channel).  Statistically equivalent to the reference's Philox masks, not bit-equal (nothing could be).
struct DropCfg {
  unsigned int thr;            // drop when hash < thr;  0 = dropout off
  float inv_keep;              // 1 / (1 - p)
  unsigned long long seed;
};
__host__ __device__ inline DropCfg make_drop(double p, unsigned long long seed) {
  DropCfg d;
  d.thr = p > 0.0 ? (unsigned int)(p * 4294967296.0 > 4294967295.0 ? 4294967295.0 : p * 4294967296.0) : 0u;
  d.inv_keep = p > 0.0 && p < 1.0 ? (float)(1.0 / (1.0 - p)) : 1.f;
  d.seed = seed;
  return d;
}
// multiplier of the pre-activation: 0 (dropped) or 1/(1-p) (kept)
__device__ __forceinline__ float drop_mul(const DropCfg& d, unsigned int stream, unsigned long long idx) {
  unsigned long long z = idx * 0x9E3779B97F4A7C15ull + d.seed + (unsigned long long)stream * 0xD1B54A32D192ED03ull;
  z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27; z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (unsigned int)(z >> 32) < d.thr ? 0.f : d.inv_keep;
}

// ------------------------------------------------------------------ scalar math
template <typename T> __device__ __forceinline__ T silu_acc(T x);
template <> __device__ __forceinline__ float silu_acc<float>(float x) {
  // x * sigmoid(x): ex2.approx-based __expf (2 ulp) and rcp.approx-based __fdividef (2 ulp); for x < -88 the
  // denominator overflows to +inf and the quotient is -0, which is the correct limit.
  return __fdividef(x, 1.0f + __expf(-x));
}
template <> __device__ __forceinline__ double silu_acc<double>(double x) {
  return x / (1.0 + exp(-x));
}
// nn.GELU() (exact): 0.5 x (1 + erf(x / sqrt 2))   (GlobalLinearAttention's feed-forward, egnn_pytorch.py:127)
template <typename T> __device__ __forceinline__ T gelu_acc(T x);
template <> __device__ __forceinline__ float gelu_acc<float>(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
template <> __device__ __forceinline__ double gelu_acc<double>(double x) { return 0.5 * x * (1.0 + erf(x * 0.70710678118654752440)); }
template <typename T> __device__ __forceinline__ T sigmoid_acc(T x);
template <> __device__ __forceinline__ float sigmoid_acc<float>(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
template <> __device__ __forceinline__ double sigmoid_acc<double>(double x) { return 1.0 / (1.0 + exp(-x)); }

template <typename T> __device__ __forceinline__ T fma_t(T a, T b, T c);
template <> __device__ __forceinline__ float fma_t<float>(float a, float b, float c) { return fmaf(a, b, c); }
template <> __device__ __forceinline__ double fma_t<double>(double a, double b, double c) { return fma(a, b, c); }

// a*a + acc WITHOUT fma contraction: the reference forms (rel ** 2).sum(-1) (egnn_pytorch.py:233) with separate
// multiplies and adds, and neighbour ranking is sensitive to the last bit near the k-th boundary.
template <typename T> __device__ __forceinline__ T sq_acc(T a, T acc);
template <> __device__ __forceinline__ float sq_acc<float>(float a, float acc) { return __fadd_rn(acc, __fmul_rn(a, a)); }
template <> __device__ __forceinline__ double sq_acc<double>(double a, double acc) { return __dadd_rn(acc, __dmul_rn(a, a)); }

// Two values that travel together through a contraction.  fp32: one 64-bit register pair and one packed FFMA2
// (fma.rn.f32x2, the same IEEE fma per lane, so results are bit-identical to scalar code) per update -- the SIMT pair
// kernels are issue-bound and most of their instructions are these contractions; fp64: two DFMAs.
template <typename T> struct Pk2;
template <> struct Pk2<float> {
  unsigned long long v;
  __device__ __forceinline__ static Pk2 make(float lo, float hi) {
    Pk2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
    return r;
  }
  __device__ __forceinline__ void fma(const Pk2& a, const Pk2& b) {       // this += a * b
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(v) : "l"(a.v), "l"(b.v));
  }
  __device__ __forceinline__ float lo() const { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); return x; }
  __device__ __forceinline__ float hi() const { float x, y; asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v)); return y; }
};
template <> struct Pk2<double> {
  double x, y;
  __device__ __forceinline__ static Pk2 make(double lo, double hi) { Pk2 r; r.x = lo; r.y = hi; return r; }
  __device__ __forceinline__ void fma(const Pk2& a, const Pk2& b) { x = ::fma(a.x, b.x, x); y = ::fma(a.y, b.y, y); }
  __device__ __forceinline__ double lo() const { return x; }
  __device__ __forceinline__ double hi() const { return y; }
};

// 4 consecutive elements, 4-element aligned.
template <typename T> struct Vec4;
template <> struct Vec4<float> {
  float v[4];
  __device__ __forceinline__ void load(const float* p) {
    float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  __device__ __forceinline__ void load_g(const float* p) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
};
template <> struct Vec4<double> {
  double v[4];
  __device__ __forceinline__ void load(const double* p) {
    double2 a = *reinterpret_cast<const double2*>(p);
    double2 b = *reinterpret_cast<const double2*>(p + 2);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
  __device__ __forceinline__ void load_g(const double* p) {
    double2 a = __ldg(reinterpret_cast<const double2*>(p));
    double2 b = __ldg(reinterpret_cast<const double2*>(p + 2));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
};

template <typename T> __device__ __forceinline__ T shfl_xor_t(T v, int m);
template <> __device__ __forceinline__ float shfl_xor_t<float>(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <> __device__ __forceinline__ double shfl_xor_t<double>(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
template <typename T> __device__ __forceinline__ T shfl_idx_t(T v, int l);
template <> __device__ __forceinline__ float shfl_idx_t<float>(float v, int l) { return __shfl_sync(0xffffffffu, v, l); }
template <> __device__ __forceinline__ double shfl_idx_t<double>(double v, int l) { return __shfl_sync(0xffffffffu, v, l); }

// ------------------------------------------------------------------ packed parameter layout (SIMT path)
// All offsets in elements of T; every block is 4-element aligned.
struct SimtPackLayout {
  size_t w2t;     // [Hp][MP]     W2 transposed, zero padded (MP = 16 or 32)
  size_t wq;      // [Q][Hp]      per-pair scalar columns of W1: distance features then edges
  size_t tab;     // [num_labels][Hp]  label_emb @ W1[:, label cols]^T
  size_t w3;      // [4m][MP]     coors_mlp.0.weight, padded
  size_t b3;      // [4m]
  size_t w4;      // [4m]
  size_t misc;    // b2[MP] | gate_w[MP] | gate_b | b4 | coors_scale | pad
  size_t total;
  int MP;
};

inline SimtPackLayout simt_pack_layout(const Dims& s) {
  SimtPackLayout L;
  L.MP = s.m <= 16 ? 16 : 32;
  BumpAlloc o;
  L.w2t = o.take((size_t)s.Hp * L.MP, 4);
  L.wq = o.take((size_t)s.Q * s.Hp, 4);
  L.tab = o.take((size_t)(s.label_dim > 0 ? s.num_labels : 0) * s.Hp, 4);
  L.w3 = o.take((size_t)4 * s.m * L.MP, 4);
  L.b3 = o.take((size_t)4 * s.m, 4);
  L.w4 = o.take((size_t)4 * s.m, 4);
  L.misc = o.take((size_t)2 * L.MP + 4, 4);
  L.total = o.total;
  return L;
}

}  // namespace egnn
