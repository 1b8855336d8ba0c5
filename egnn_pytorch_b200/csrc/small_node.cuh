// Per-node stages of the bf16 path for narrow layers (dim <= 64): one WARP per node, weights staged once per CTA in
// shared memory (transposed, bf16), fp32 arithmetic.
//
// Why: with dim = 32 the per-node GEMMs of a layer are 9 k and 5 k FMAs per node -- the tcgen05 GEMM (TMEM allocation,
// cp.async ring, 128-row tiles) spends 10-11 us of fixed latency on each of them, and the node update needs three
// launches (LayerNorm+concat, Linear+SiLU, Linear+residual).  BASELINE configs 3 and 5 (EGNN_Network, dim 32) are made
// of exactly these launches.  Here:
//   tables_small_kernel      A' = 0.5 (h W1_i^T + b1) (fp32), B' = 0.5 h W1_j^T (bf16)            (egnn_pytorch.py:283-287,
//                            Linear 1 of edge_mlp split over its inputs, DESIGN.md section 2)        one launch
//   node_update_small_kernel h' = node_mlp([LN(h) | m_i]) + h                                      (egnn_pytorch.py:335-340)
//                            LayerNorm, concat, Linear+SiLU, Linear, residual                        one launch
// Intermediates stay in fp32 (the GEMM path rounds LN(h) and the hidden layer to bf16), so results are at least as close
// to the fp32 reference; per-node results do not depend on the launch partition (row ranges stay bit-identical).
#pragma once

#include <cuda_bf16.h>
#include "common.cuh"

namespace egnn {

constexpr int SN_WARPS = 8;
constexpr int SN_DIM_MAX = 64;
constexpr size_t SMALL_NODE_SMEM_MAX = 160 * 1024;   // staged weights beyond this: the GEMM path
constexpr int SN_TABLES_M_MAX = 4096;                // the table kernel re-reads its weights per node (28 % FMA density): measured
                                                     // faster than the GEMMs at 1024 nodes (12 vs 20 us), slower at 8192 (35 vs 21 us)

struct TablesSmallArgs {
  const __nv_bfloat16* feats;      // [M][dim]
  const __nv_bfloat16* w1i;        // [Hp][dim]
  const __nv_bfloat16* w1j;        // [Hp][dim]
  const float* b1;                 // [Hp]
  float* Atab;                     // [M][Hp]
  __nv_bfloat16* Btab;             // [M][Hp]
  int M, N, dim, Hp, row0, row1;   // A' only for rows [row0, row1) of every graph; B' for all nodes
};

inline size_t tables_small_smem(int dim, int Hp) { return (size_t)2 * dim * Hp * 2 + (size_t)Hp * 4 + (size_t)SN_WARPS * SN_DIM_MAX * 4; }

static __global__ void __launch_bounds__(SN_WARPS * 32) tables_small_kernel(const TablesSmallArgs a) {
  extern __shared__ __align__(16) unsigned char sn_sm[];
  const int dim = a.dim, Hp = a.Hp;
  __nv_bfloat16* wi = reinterpret_cast<__nv_bfloat16*>(sn_sm);          // [dim][Hp]  (transposed)
  __nv_bfloat16* wj = wi + (size_t)dim * Hp;                             // [dim][Hp]
  float* b1 = reinterpret_cast<float*>(wj + (size_t)dim * Hp);           // [Hp]
  float* xs = b1 + Hp;                                                   // [WARPS][DIM_MAX]
  for (int e = threadIdx.x; e < Hp * dim; e += SN_WARPS * 32) {
    const int c = e / dim, k = e - c * dim;
    wi[k * Hp + c] = a.w1i[e];
    wj[k * Hp + c] = a.w1j[e];
  }
  for (int c = threadIdx.x; c < Hp; c += SN_WARPS * 32) b1[c] = a.b1[c];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* x = xs + warp * SN_DIM_MAX;
  for (int node = blockIdx.x * SN_WARPS + warp; node < a.M; node += gridDim.x * SN_WARPS) {
    const int i = node % a.N;
    const bool do_a = i >= a.row0 && i < a.row1;
    __syncwarp();
    for (int k = lane; k < dim; k += 32) x[k] = __bfloat162float(a.feats[(size_t)node * dim + k]);
    __syncwarp();
    for (int c = 2 * lane; c < Hp; c += 64) {                            // Hp is a multiple of 16: pairs never straddle the end
      float ai0 = 0.f, ai1 = 0.f, aj0 = 0.f, aj1 = 0.f;
#pragma unroll 8
      for (int k = 0; k < dim; ++k) {
        const float xv = x[k];
        const float2 w_i = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(wi + k * Hp + c));
        const float2 w_j = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(wj + k * Hp + c));
        ai0 = fmaf(xv, w_i.x, ai0); ai1 = fmaf(xv, w_i.y, ai1);
        aj0 = fmaf(xv, w_j.x, aj0); aj1 = fmaf(xv, w_j.y, aj1);
      }
      if (do_a) *reinterpret_cast<float2*>(a.Atab + (size_t)node * Hp + c) = make_float2(0.5f * (ai0 + b1[c]), 0.5f * (ai1 + b1[c + 1]));
      *reinterpret_cast<__nv_bfloat162*>(a.Btab + (size_t)node * Hp + c) = __floats2bfloat162_rn(0.5f * aj0, 0.5f * aj1);
    }
  }
}

struct NodeSmallArgs {
  const __nv_bfloat16* feats;      // [M][dim]
  const __nv_bfloat16* node_in;    // [M][Kn]: columns [dim, dim + m) hold m_i (written by the fused edge kernel)
  const __nv_bfloat16* wn1;        // [2 dim][Kn]
  const float* bn1;                // [2 dim]
  const __nv_bfloat16* wn2;        // [dim][2 dim]
  const float* bn2;                // [dim]
  const float* lng; const float* lnb;
  __nv_bfloat16* out;              // [M][dim]  (may alias feats: a warp reads its row before it writes it)
  int B, N, dim, Kn, m, row0, row1, do_norm;
};

inline size_t node_small_smem(int dim, int Kn) {
  return (size_t)Kn * 2 * dim * 2 + (size_t)2 * dim * dim * 2 + (size_t)3 * dim * 4 + (size_t)SN_WARPS * (Kn + 2 * dim) * 4;
}

static __global__ void __launch_bounds__(SN_WARPS * 32) node_update_small_kernel(const NodeSmallArgs a) {
  extern __shared__ __align__(16) unsigned char sn_sm[];
  const int dim = a.dim, Kn = a.Kn, H2 = 2 * a.dim;
  __nv_bfloat16* w1 = reinterpret_cast<__nv_bfloat16*>(sn_sm);          // [Kn][2 dim]   (transposed)
  __nv_bfloat16* w2 = w1 + (size_t)Kn * H2;                              // [2 dim][dim]  (transposed)
  float* bn1 = reinterpret_cast<float*>(w2 + (size_t)H2 * dim);          // [2 dim]
  float* bn2 = bn1 + H2;                                                 // [dim]
  float* bufs = bn2 + dim;                                               // [WARPS][Kn + 2 dim]
  for (int e = threadIdx.x; e < H2 * Kn; e += SN_WARPS * 32) {
    const int o = e / Kn, k = e - o * Kn;
    w1[k * H2 + o] = a.wn1[e];
  }
  for (int e = threadIdx.x; e < dim * H2; e += SN_WARPS * 32) {
    const int o = e / H2, k = e - o * H2;
    w2[k * dim + o] = a.wn2[e];
  }
  for (int c = threadIdx.x; c < H2; c += SN_WARPS * 32) bn1[c] = a.bn1[c];
  for (int c = threadIdx.x; c < dim; c += SN_WARPS * 32) bn2[c] = a.bn2[c];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* x = bufs + warp * (Kn + H2);                                    // [Kn]   LN(h) | m_i | 0
  float* hid = x + Kn;                                                   // [2 dim]
  const int R = a.row1 - a.row0, rows = a.B * R;
  for (int r = blockIdx.x * SN_WARPS + warp; r < rows; r += gridDim.x * SN_WARPS) {
    const size_t node = (size_t)(r / R) * a.N + a.row0 + r % R;
    const __nv_bfloat16* h = a.feats + node * dim;
    // dim <= 64: lane holds channels lane and lane + 32
    const float h0 = lane < dim ? __bfloat162float(h[lane]) : 0.f;
    const float h1 = lane + 32 < dim ? __bfloat162float(h[lane + 32]) : 0.f;
    float y0 = h0, y1 = h1;
    if (a.do_norm) {                                                     // nn.LayerNorm(dim), eps 1e-5, biased variance
      float s = h0 + h1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const float mu = s / dim;
      const float t0 = lane < dim ? h0 - mu : 0.f, t1 = lane + 32 < dim ? h1 - mu : 0.f;
      float v = t0 * t0 + t1 * t1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      const float rstd = rsqrtf(v / dim + 1e-5f);
      if (lane < dim) y0 = t0 * rstd * a.lng[lane] + a.lnb[lane];
      if (lane + 32 < dim) y1 = t1 * rstd * a.lng[lane + 32] + a.lnb[lane + 32];
    }
    __syncwarp();
    if (lane < dim) x[lane] = y0;
    if (lane + 32 < dim) x[lane + 32] = y1;
    for (int c = dim + lane; c < Kn; c += 32) x[c] = c < dim + a.m ? __bfloat162float(a.node_in[node * Kn + c]) : 0.f;
    __syncwarp();
    for (int o = 2 * lane; o < H2; o += 64) {                            // Linear(dim + m, 2 dim) + SiLU
      float a0 = bn1[o], a1 = bn1[o + 1];
#pragma unroll 8
      for (int k = 0; k < Kn; ++k) {
        const float2 w = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(w1 + k * H2 + o));
        a0 = fmaf(x[k], w.x, a0); a1 = fmaf(x[k], w.y, a1);
      }
      hid[o] = silu_acc(a0); hid[o + 1] = silu_acc(a1);
    }
    __syncwarp();
    const int o = 2 * lane;
    if (o < dim) {                                                       // Linear(2 dim, dim) + residual
      float a0 = bn2[o], a1 = bn2[o + 1];
#pragma unroll 8
      for (int k = 0; k < H2; ++k) {
        const float2 w = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(w2 + k * dim + o));
        a0 = fmaf(hid[k], w.x, a0); a1 = fmaf(hid[k], w.y, a1);
      }
      const float2 res = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(h + o));
      *reinterpret_cast<__nv_bfloat162*>(a.out + node * dim + o) = __floats2bfloat162_rn(a0 + res.x, a1 + res.y);
    }
  }
}

// ---- the same two stages for the fp32 / fp64 SIMT path (weights in their natural layout, tables as P = [A | B]) ----
// node_in (LN(h) part) and h1 are still written: the backward reads them from the forward workspace.

template <typename T>
struct TablesSmallSimtArgs {
  const T* feats;                  // [M][dim]
  const T* W1;                     // edge_mlp.0.weight [H][E]: columns [0, dim) multiply h_i, [dim, 2 dim) multiply h_j
  const T* b1;                     // [H]
  T* P;                            // [M][2 Hp]: A at columns [0, Hp), B at [Hp, 2 Hp); columns >= H are zero
  int M, dim, H, Hp, E;
};

template <typename T>
inline size_t tables_small_simt_smem(int dim, int Hp) { return ((size_t)2 * dim * Hp + Hp + (size_t)SN_WARPS * SN_DIM_MAX) * sizeof(T); }

template <typename T>
__global__ void __launch_bounds__(SN_WARPS * 32) tables_small_simt_kernel(const TablesSmallSimtArgs<T> a) {
  extern __shared__ __align__(16) unsigned char sn_sm[];
  const int dim = a.dim, Hp = a.Hp;
  T* wi = reinterpret_cast<T*>(sn_sm);                                   // [dim][Hp]  (transposed, zero beyond H)
  T* wj = wi + (size_t)dim * Hp;
  T* b1 = wj + (size_t)dim * Hp;                                         // [Hp]
  T* xs = b1 + Hp;                                                       // [WARPS][DIM_MAX]
  for (int e = threadIdx.x; e < Hp * dim; e += SN_WARPS * 32) {
    const int c = e / dim, k = e - c * dim;
    wi[k * Hp + c] = c < a.H ? a.W1[(size_t)c * a.E + k] : T(0);
    wj[k * Hp + c] = c < a.H ? a.W1[(size_t)c * a.E + dim + k] : T(0);
  }
  for (int c = threadIdx.x; c < Hp; c += SN_WARPS * 32) b1[c] = c < a.H ? a.b1[c] : T(0);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  T* x = xs + warp * SN_DIM_MAX;
  for (int node = blockIdx.x * SN_WARPS + warp; node < a.M; node += gridDim.x * SN_WARPS) {
    __syncwarp();
    for (int k = lane; k < dim; k += 32) x[k] = a.feats[(size_t)node * dim + k];
    __syncwarp();
    for (int c = lane; c < Hp; c += 32) {
      T ai = b1[c], aj = T(0);
#pragma unroll 8
      for (int k = 0; k < dim; ++k) {
        ai = fma(x[k], wi[k * Hp + c], ai);
        aj = fma(x[k], wj[k * Hp + c], aj);
      }
      a.P[(size_t)node * 2 * Hp + c] = ai;
      a.P[(size_t)node * 2 * Hp + Hp + c] = aj;
    }
  }
}

template <typename T>
struct NodeSmallSimtArgs {
  const T* feats;                  // [M][dim]
  T* node_in;                      // [M][dim + m]: LN(h) written here, m_i read from columns [dim, dim + m)
  T* h1;                           // [M][2 dim]   silu(Linear 1), kept for the backward
  const T* wn1; const T* bn1;      // node_mlp.0  [2 dim][dim + m]
  const T* wn2; const T* bn2;      // node_mlp.3  [dim][2 dim]
  const T* lng; const T* lnb;
  T* out;                          // [M][dim]
  int B, N, dim, m, row0, row1, do_norm;
};

template <typename T>
inline size_t node_small_simt_smem(int dim, int m) {
  return ((size_t)(dim + m) * 2 * dim + (size_t)2 * dim * dim + 3 * dim + (size_t)SN_WARPS * (dim + m + 2 * dim)) * sizeof(T);
}

template <typename T>
__global__ void __launch_bounds__(SN_WARPS * 32) node_update_small_simt_kernel(const NodeSmallSimtArgs<T> a) {
  extern __shared__ __align__(16) unsigned char sn_sm[];
  const int dim = a.dim, Kn = a.dim + a.m, H2 = 2 * a.dim;
  T* w1 = reinterpret_cast<T*>(sn_sm);                                   // [Kn][2 dim]   (transposed)
  T* w2 = w1 + (size_t)Kn * H2;                                          // [2 dim][dim]  (transposed)
  T* bn1 = w2 + (size_t)H2 * dim;
  T* bn2 = bn1 + H2;
  T* bufs = bn2 + dim;                                                   // [WARPS][Kn + 2 dim]
  for (int e = threadIdx.x; e < H2 * Kn; e += SN_WARPS * 32) {
    const int o = e / Kn, k = e - o * Kn;
    w1[k * H2 + o] = a.wn1[e];
  }
  for (int e = threadIdx.x; e < dim * H2; e += SN_WARPS * 32) {
    const int o = e / H2, k = e - o * H2;
    w2[k * dim + o] = a.wn2[e];
  }
  for (int c = threadIdx.x; c < H2; c += SN_WARPS * 32) bn1[c] = a.bn1[c];
  for (int c = threadIdx.x; c < dim; c += SN_WARPS * 32) bn2[c] = a.bn2[c];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  T* x = bufs + warp * (Kn + H2);
  T* hid = x + Kn;
  const int R = a.row1 - a.row0, rows = a.B * R;
  for (int r = blockIdx.x * SN_WARPS + warp; r < rows; r += gridDim.x * SN_WARPS) {
    const size_t node = (size_t)(r / R) * a.N + a.row0 + r % R;
    const T* h = a.feats + node * dim;
    const T h0 = lane < dim ? h[lane] : T(0);
    const T h1v = lane + 32 < dim ? h[lane + 32] : T(0);
    T y0 = h0, y1 = h1v;
    if (a.do_norm) {
      T s = h0 + h1v;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += shfl_xor_t<T>(s, o);
      const T mu = s / T(dim);
      const T t0 = lane < dim ? h0 - mu : T(0), t1 = lane + 32 < dim ? h1v - mu : T(0);
      T v = t0 * t0 + t1 * t1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += shfl_xor_t<T>(v, o);
      const T rstd = T(1) / sqrt(v / T(dim) + T(1e-5));
      if (lane < dim) y0 = t0 * rstd * a.lng[lane] + a.lnb[lane];
      if (lane + 32 < dim) y1 = t1 * rstd * a.lng[lane + 32] + a.lnb[lane + 32];
    }
    __syncwarp();
    T* nin = a.node_in + node * Kn;
    if (lane < dim) { x[lane] = y0; nin[lane] = y0; }
    if (lane + 32 < dim) { x[lane + 32] = y1; nin[lane + 32] = y1; }
    for (int c = dim + lane; c < Kn; c += 32) x[c] = nin[c];
    __syncwarp();
    for (int o = lane; o < H2; o += 32) {
      T acc = bn1[o];
#pragma unroll 8
      for (int k = 0; k < Kn; ++k) acc = fma(x[k], w1[k * H2 + o], acc);
      const T hv = silu_acc<T>(acc);
      hid[o] = hv;
      a.h1[node * H2 + o] = hv;
    }
    __syncwarp();
    for (int o = lane; o < dim; o += 32) {
      T acc = bn2[o];
#pragma unroll 8
      for (int k = 0; k < H2; ++k) acc = fma(hid[k], w2[k * dim + o], acc);
      a.out[node * dim + o] = acc + (o == lane ? h0 : h1v);
    }
  }
}

}  // namespace egnn
