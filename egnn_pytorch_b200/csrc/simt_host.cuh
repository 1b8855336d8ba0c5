// Host-side helpers shared by the forward (egnn_api.cu) and backward (egnn_backward.cu) orchestration:
// descriptor validation, the forward workspace layout and the GEMM launcher.
#pragma once
#include "common.cuh"
#include "simt_kernels.cuh"
#include "launch.cuh"
#include <algorithm>

namespace egnn {

// ------------------------------------------------------------------ validation
static int validate_desc(const EgnnLayerDesc* d) {
  if (!d) return EGNN_ERR_NULL;
  if (d->abi_version != EGNN_ABI_VERSION) return EGNN_ERR_ABI;
  if (d->dtype != EGNN_DTYPE_F32 && d->dtype != EGNN_DTYPE_F64 && d->dtype != EGNN_DTYPE_BF16)
    return EGNN_ERR_UNSUPPORTED;
  if (d->B <= 0 || d->N <= 0 || d->dim <= 0 || d->C <= 0 || d->edge_dim < 0 || d->label_dim < 0 ||
      d->fourier < 0 || d->m_dim <= 0 || d->k < 0)
    return EGNN_ERR_SHAPE;
  if (d->B > 65535) return EGNN_ERR_SHAPE;
  if (d->C > PAIR_CMAX) return EGNN_ERR_UNSUPPORTED;
  if (d->m_dim > 32) return EGNN_ERR_UNSUPPORTED;
  if (d->fourier > 30) return EGNN_ERR_UNSUPPORTED;
  if (d->k > d->N) return EGNN_ERR_SHAPE;                 // torch.topk raises too (:258)
  if (d->label_dim > 0 && (d->num_labels <= 0 || d->num_labels > 255)) return EGNN_ERR_SHAPE;
  if (!(d->flags & (EGNN_FLAG_UPDATE_FEATS | EGNN_FLAG_UPDATE_COORS))) return EGNN_ERR_SHAPE;   // :171
  if (d->reserved != 0) return EGNN_ERR_SHAPE;
  if (!(d->dropout_p >= 0.0 && d->dropout_p < 1.0)) return EGNN_ERR_SHAPE;
  if (d->dropout_p > 0.0 && d->dtype == EGNN_DTYPE_BF16) return EGNN_ERR_UNSUPPORTED;     // training runs the fp32 / fp64 kernels
  if (d->row_begin < 0 || d->row_end < 0 || d->row_end > d->N || d->row_begin > d->row_end) return EGNN_ERR_SHAPE;
  return EGNN_OK;
}

static inline size_t elem_size(int dtype) { return dtype == EGNN_DTYPE_F64 ? 8 : (dtype == EGNN_DTYPE_F32 ? 4 : 2); }

// ------------------------------------------------------------------ SIMT workspace
struct SimtWs {
  size_t P, node_in, h1, nbr_idx, nbr_ok, hpart, total;
  int hsplit;
};
// Tiny dense graphs (the README example, BASELINE config 1): too few (row, neighbour) tiles to fill the GPU, so the
// hidden axis is split over CTAs and the partial sums take one trip through the workspace.
static int simt_hsplit(const Dims& s) {
  if (s.k != 0 || (long long)s.B * s.N * s.N > 4096 || s.Hp < 512 || s.row0 != 0 || s.row1 != s.N) return 1;
  return std::min(32, ceil_div(s.Hp, PAIR_CH));
}
static SimtWs simt_ws_layout(const Dims& s, size_t es, uint32_t flags) {
  SimtWs w;
  BumpAlloc o;
  w.P = o.take((size_t)s.M * 2 * s.Hp * es);
  const bool uf = flags & EGNN_FLAG_UPDATE_FEATS;
  w.node_in = o.take(uf ? (size_t)s.M * (s.dim + s.m) * es : 0);
  w.h1 = o.take(uf ? (size_t)s.M * 2 * s.dim * es : 0);
  w.nbr_idx = o.take((size_t)s.M * s.k * sizeof(int32_t));
  w.nbr_ok = o.take((size_t)s.M * s.k);
  w.hsplit = simt_hsplit(s);
  w.hpart = o.take(w.hsplit > 1 ? (size_t)w.hsplit * s.B * s.N * s.N * 32 * es : 0);
  w.total = o.total;
  return w;
}

template <typename T, int ACT, bool RES>
static int launch_gemm(const T* A, int lda, const T* W, int ldw, const T* bias, const T* R, int ldr, T* C,
                       int ldo, int Mr, int Nv, int Nout, int K, RowMap map, cudaStream_t st, DropCfg drop = DropCfg{0u, 1.f, 0ull}) {
  constexpr int V = 16 / (int)sizeof(T);
  const size_t skinny_smem = (size_t)16 * ((K + V - 1) / V * V) * sizeof(T);
  if (Mr <= 16 && skinny_smem <= 96 * 1024) {
    // columns per warp: as many as still give about one CTA per SM (the kernel is bound by weight streaming)
    const int cols = Nout >= 148 * SKINNY_WARPS * 4 ? 4 : (Nout >= 148 * SKINNY_WARPS * 2 ? 2 : 1);
    auto kernel = cols == 4 ? gemm_skinny_kernel<T, ACT, RES, 4> : cols == 2 ? gemm_skinny_kernel<T, ACT, RES, 2> : gemm_skinny_kernel<T, ACT, RES, 1>;
    return launch(kernel, ceil_div(Nout, SKINNY_WARPS * cols), SKINNY_WARPS * 32, skinny_smem, st, A, lda, W, ldw, bias, R, ldr, C, ldo, Mr,
                  Nv, Nout, K, map, drop);
  }
  return launch(gemm_nt_kernel<T, ACT, RES>, dim3(ceil_div(Nout, 64), ceil_div(Mr, 64)), 256, 0, st, A, lda, W, ldw, bias, R, ldr, C, ldo,
                Mr, Nv, Nout, K, map, drop);
}

static int check_ptrs(const EgnnLayerDesc& d, const EgnnLayerWeights* w, const EgnnLayerIO* io) {
  if (!w || !w->edge_w1 || !w->edge_b1 || !w->edge_w2 || !w->edge_b2) return EGNN_ERR_NULL;
  if ((d.flags & EGNN_FLAG_SOFT_EDGES) && (!w->gate_w || !w->gate_b)) return EGNN_ERR_NULL;
  if ((d.flags & EGNN_FLAG_NORM_FEATS) && (d.flags & EGNN_FLAG_UPDATE_FEATS) && (!w->norm_g || !w->norm_b)) return EGNN_ERR_NULL;
  if ((d.flags & EGNN_FLAG_NORM_COORS) && !w->coors_scale) return EGNN_ERR_NULL;
  if ((d.flags & EGNN_FLAG_UPDATE_FEATS) && (!w->node_w1 || !w->node_b1 || !w->node_w2 || !w->node_b2)) return EGNN_ERR_NULL;
  if ((d.flags & EGNN_FLAG_UPDATE_COORS) && (!w->coors_w1 || !w->coors_b1 || !w->coors_w2 || !w->coors_b2)) return EGNN_ERR_NULL;
  if (d.label_dim > 0 && !w->label_emb) return EGNN_ERR_NULL;
  if (io) {
    if (!io->feats || !io->coors || !io->feats_out || !io->coors_out) return EGNN_ERR_NULL;
    if (d.edge_dim > 0 && !io->edges) return EGNN_ERR_NULL;
    if (d.label_dim > 0 && !io->edge_labels) return EGNN_ERR_NULL;
    const uintptr_t all = (uintptr_t)io->feats | (uintptr_t)io->feats_out | (uintptr_t)io->edges;
    if (all & 0xF) return EGNN_ERR_ALIGN;
  }
  return EGNN_OK;
}

}  // namespace egnn
