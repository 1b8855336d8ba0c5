#pragma once
// Per-layer backward orchestration (templated on the element type; instantiated once per type in
// egnn_backward.cu (fp32) and egnn_backward_f64.cu (fp64) so the two compile concurrently):
//   node update reversed -> bwd1 / bwd2 / bwd3 (simt_backward.cuh) -> per-node tables reversed -> unpack.
#include "common.cuh"
#include "simt_kernels.cuh"
#include "simt_backward.cuh"
#include "simt_host.cuh"

namespace egnn {

struct BwdWs {
  size_t gP, gpk, rec, pre2, h1pre, ga, g_node_in, gyx, total;
};

inline BwdWs bwd_ws_layout(const Dims& s, const SimtPackLayout& L, size_t es, uint32_t flags) {
  BwdWs w;
  BumpAlloc o;
  const size_t J = s.k > 0 ? s.k : s.N;
  const bool uf = flags & EGNN_FLAG_UPDATE_FEATS;
  w.gP = o.take((size_t)s.M * 2 * s.Hp * es);
  w.gpk = o.take(L.total * es);
  w.rec = o.take((size_t)s.M * J * rec_layout(s, L.MP).R * es);
  w.pre2 = o.take(s.k == 0 ? (size_t)s.M * s.N * L.MP * es : 0);
  w.h1pre = o.take(uf ? (size_t)s.M * 2 * s.dim * es : 0);
  w.ga = o.take(uf ? (size_t)s.M * 2 * s.dim * es : 0);
  w.g_node_in = o.take(uf ? (size_t)s.M * (s.dim + s.m) * es : 0);
  w.gyx = o.take((uf && (flags & EGNN_FLAG_NORM_FEATS)) ? (size_t)s.M * s.dim * es : 0);
  w.total = o.total;
  return w;
}

// Dynamic shared memory of the larger of bwd1 and the bwd2 variant launch_pair_bwd picks (the same size functions
// the launches use).  The dense recompute (launch_tiled_recompute) is left out: it falls back by itself.
template <typename T>
inline size_t backward_smem_bytes(const Dims& s, uint32_t flags) {
  const SimtPackLayout L = simt_pack_layout(s);
  const bool knn = s.k > 0;
  const int R = rec_layout(s, L.MP).R;
  const size_t b1 = bwd1_smem_bytes<T>(s, L, knn, (flags & EGNN_FLAG_SOFT_EDGES) != 0);
  const size_t b2 = knn ? bwd2_knn_smem_bytes<T>(s, R) : bwd2_dense_smem_bytes<T>(s, R);
  return std::max(b1, b2);
}

inline int backward_supported(const EgnnLayerDesc& d) {
  if (d.dtype != EGNN_DTYPE_F32 && d.dtype != EGNN_DTYPE_F64) return EGNN_ERR_UNSUPPORTED;
  if (!(d.row_begin == 0 && (d.row_end == 0 || d.row_end == d.N))) return EGNN_ERR_UNSUPPORTED;
  if (d.label_dim > 0 && d.num_labels > BW2_MAXLAB) return EGNN_ERR_UNSUPPORTED;
  const Dims s = make_dims(d);
  const size_t smem = d.dtype == EGNN_DTYPE_F64 ? backward_smem_bytes<double>(s, d.flags) : backward_smem_bytes<float>(s, d.flags);
  if (smem > DYN_SMEM_MAX) return EGNN_ERR_UNSUPPORTED;     // launch() would refuse it
  return EGNN_OK;
}

// C[r,c] += sum_k A(r,k) B(k,c); K is split so that small outputs with a long reduction still fill the GPU.
template <typename T>
static int launch_gemm_acc(const T* A, long ars, long aks, const T* B, long bks, long bcs, T* C, long ldc, int Mr,
                           int Nc, int K, cudaStream_t st) {
  if (Mr <= 0 || Nc <= 0 || K <= 0) return EGNN_OK;
  const int tiles = ceil_div(Mr, 64) * ceil_div(Nc, 64);
  int splits = std::max(1, std::min(ceil_div(296, tiles), ceil_div(K, 64)));
  splits = std::min(splits, 65535);
  const int kper = round_up_i(ceil_div(K, splits), 16);
  splits = ceil_div(K, kper);
  return launch(gemm_acc_kernel<T>, dim3(ceil_div(Nc, 64), ceil_div(Mr, 64), splits), 256, 0, st, A, ars, aks, B, bks, bcs, C, ldc, Mr, Nc,
                K, kper);
}

template <typename T>
static int launch_colsum(const T* X, long ld, int rows, int cols, T* out, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return EGNN_OK;
  dim3 grid(ceil_div(cols, 32), std::max(1, std::min(64, ceil_div(rows, 64))));
  return launch(colsum_acc_kernel<T>, grid, dim3(32, 8), 0, st, X, ld, rows, cols, out);
}

// Dense: W2 silu(pre1) for every pair with the register-tiled forward kernel (its split-H "phase 1" stores exactly
// that); returns EGNN_ERR_UNSUPPORTED when its shared memory does not fit, and bwd1 then recomputes by itself.
template <typename T, int MP, int PP>
static int launch_tiled_recompute(const BwdArgs<T>& a, T* pre2, cudaStream_t st) {
  PairArgs<T> f;
  f.s = a.s; f.L = a.L; f.flags = a.flags; f.has_mask = a.has_mask; f.TS = 32; f.clamp = a.clamp;
  f.P = a.P; f.ldP = a.ldP; f.coors = a.coors; f.edges = a.edges; f.labels = a.labels; f.mask = a.mask;
  f.nbr_idx = nullptr; f.nbr_ok = nullptr; f.packed = a.packed;
  f.m_out = nullptr; f.ld_m = 0; f.coors_out = nullptr;
  f.hpart = pre2; f.hsplit = 1; f.phase = 1;
  f.pre2_out = nullptr;
  f.drop = a.drop;                                    // the recompute must draw the forward's masks
  return launch(pair_dense_tiled_kernel<T, MP, PP>, dim3(ceil_div(a.s.N, 4 * PP), a.s.B, 1), PAIR_THREADS,
                pair_tiled_smem_bytes<T>(a.s, a.L, PP), st, f);
}

template <typename T, int MP, bool KNN>
static int launch_pair_bwd(BwdArgs<T>& a, bool saved_pre2, cudaStream_t st) {
  const Dims& s = a.s;
  if constexpr (!KNN) {
    if (!saved_pre2) {
    T* pre2 = const_cast<T*>(a.pre2);
    const int rc = launch_tiled_recompute<T, MP, (MP == 32 && sizeof(T) == 8) ? 1 : 2>(a, pre2, st);
    if (rc == EGNN_ERR_UNSUPPORTED) a.pre2 = nullptr;
    else EGNN_TRY(rc);
    }
  }
  const int TI = PAIR_THREADS / a.TS;
  dim3 g1(ceil_div(s.N, TI), s.B);
  EGNN_TRY(launch(pair_bwd1_kernel<T, MP, KNN>, g1, PAIR_THREADS,
                  bwd1_smem_bytes<T>(s, a.L, KNN, (a.flags & EGNN_FLAG_SOFT_EDGES) != 0), st, a));
  const bool q1 = s.Q == 1 && s.label_dim == 0, drop = a.drop.thr != 0;
  if constexpr (KNN) {
    auto bwd2 = q1 ? (drop ? pair_bwd2_knn_kernel<T, MP, 1, true> : pair_bwd2_knn_kernel<T, MP, 1, false>)
              : s.Q <= 8 ? (drop ? pair_bwd2_knn_kernel<T, MP, 8, true> : pair_bwd2_knn_kernel<T, MP, 8, false>)
                         : (drop ? pair_bwd2_knn_kernel<T, MP, 0, true> : pair_bwd2_knn_kernel<T, MP, 0, false>);
    EGNN_TRY(launch(bwd2, dim3(ceil_div(s.N, a.TI2), ceil_div(s.Hp, BW2_TH), s.B), BW2_TH, bwd2_knn_smem_bytes<T>(s, a.rl.R), st, a));
  } else {
    auto bwd2 = q1 ? (drop ? pair_bwd2_dense_kernel<T, MP, 1, true> : pair_bwd2_dense_kernel<T, MP, 1, false>)
                   : (drop ? pair_bwd2_dense_kernel<T, MP, 0, true> : pair_bwd2_dense_kernel<T, MP, 0, false>);
    EGNN_TRY(launch(bwd2, dim3(ceil_div(s.N, BW2_ROWS), ceil_div(s.Hp, BW2_TH), s.B), BW2_TH, bwd2_dense_smem_bytes<T>(s, a.rl.R), st, a));
  }
  return launch(pair_bwd3_kernel<T, KNN>, g1, PAIR_THREADS, 0, st, a);
}

template <typename T>
int simt_backward(const EgnnLayerDesc& d, const EgnnLayerWeights& w, const void* packed, const EgnnLayerIO& io,
                         const void* fwd_ws, const EgnnLayerGrads& gr, void* ws, size_t ws_bytes, cudaStream_t st) {
  const Dims s = make_dims(d);
  const SimtPackLayout L = simt_pack_layout(s);
  const SimtWs fl = simt_ws_layout(s, sizeof(T), d.flags);
  const BwdWs bl = bwd_ws_layout(s, L, sizeof(T), d.flags);
  if (ws_bytes < bl.total) return EGNN_ERR_WORKSPACE;
  const bool uf = d.flags & EGNN_FLAG_UPDATE_FEATS, uc = d.flags & EGNN_FLAG_UPDATE_COORS;
  const bool nf = d.flags & EGNN_FLAG_NORM_FEATS;
  const char* fbase = static_cast<const char*>(fwd_ws);
  char* base = static_cast<char*>(ws);
  const T* P = reinterpret_cast<const T*>(fbase + fl.P);
  const T* node_in = reinterpret_cast<const T*>(fbase + fl.node_in);
  const T* h1 = reinterpret_cast<const T*>(fbase + fl.h1);
  const int32_t* nbr_idx = reinterpret_cast<const int32_t*>(fbase + fl.nbr_idx);
  const uint8_t* nbr_ok = reinterpret_cast<const uint8_t*>(fbase + fl.nbr_ok);
  if (s.k > 0 && io.nbr_idx) { nbr_idx = io.nbr_idx; nbr_ok = nullptr; }
  T* gP = reinterpret_cast<T*>(base + bl.gP);
  T* gpk = reinterpret_cast<T*>(base + bl.gpk);
  T* rec = reinterpret_cast<T*>(base + bl.rec);
  T* h1pre = reinterpret_cast<T*>(base + bl.h1pre);
  T* ga = reinterpret_cast<T*>(base + bl.ga);
  T* g_node_in = reinterpret_cast<T*>(base + bl.g_node_in);
  T* gyx = reinterpret_cast<T*>(base + bl.gyx);
  const T* feats = static_cast<const T*>(io.feats);
  const T* W1 = static_cast<const T*>(w.edge_w1);
  const T* go = static_cast<const T*>(gr.g_feats_out);
  T* g_feats = static_cast<T*>(gr.g_feats);
  T* g_coors = static_cast<T*>(gr.g_coors);
  const int M = s.M, dim = s.dim, m = s.m, dn = s.dim + s.m, d2 = 2 * s.dim;
  const RowMap ident{s.N, s.N, 0};
  const size_t J = s.k > 0 ? s.k : s.N;

  // ---- zero the accumulators and the parameter-gradient outputs
  auto zero = [&](void* p, size_t bytes) -> int {
    if (p && bytes) EGNN_CUDA_TRY(cudaMemsetAsync(p, 0, bytes, st));
    return EGNN_OK;
  };
  const size_t es = sizeof(T);
  EGNN_TRY(zero(gP, (size_t)M * 2 * s.Hp * es));
  EGNN_TRY(zero(gpk, L.total * es));
  EGNN_TRY(zero(rec, (size_t)M * J * rec_layout(s, L.MP).R * es));
  EGNN_TRY(zero(gr.w.edge_w1, (size_t)s.H * s.E * es));
  EGNN_TRY(zero(gr.w.edge_b1, (size_t)s.H * es));
  EGNN_TRY(zero(gr.w.edge_w2, (size_t)m * s.H * es));
  EGNN_TRY(zero(gr.w.edge_b2, (size_t)m * es));
  EGNN_TRY(zero(gr.w.gate_w, (size_t)m * es));
  EGNN_TRY(zero(gr.w.gate_b, es));
  EGNN_TRY(zero(gr.w.norm_g, (size_t)dim * es));
  EGNN_TRY(zero(gr.w.norm_b, (size_t)dim * es));
  EGNN_TRY(zero(gr.w.coors_scale, es));
  EGNN_TRY(zero(gr.w.node_w1, (size_t)d2 * dn * es));
  EGNN_TRY(zero(gr.w.node_b1, (size_t)d2 * es));
  EGNN_TRY(zero(gr.w.node_w2, (size_t)dim * d2 * es));
  EGNN_TRY(zero(gr.w.node_b2, (size_t)dim * es));
  EGNN_TRY(zero(gr.w.coors_w1, (size_t)4 * m * m * es));
  EGNN_TRY(zero(gr.w.coors_b1, (size_t)4 * m * es));
  EGNN_TRY(zero(gr.w.coors_w2, (size_t)4 * m * es));
  EGNN_TRY(zero(gr.w.coors_b2, es));
  EGNN_TRY(zero(gr.w.label_emb, (size_t)s.num_labels * s.label_dim * es));
  if (gr.g_edges && s.k > 0) EGNN_TRY(zero(gr.g_edges, (size_t)M * s.N * s.edge_dim * es));
  // residual / identity paths: h' = ... + h (:337, :339), x' = x + ... (:315, :317)
  EGNN_CUDA_TRY(cudaMemcpyAsync(g_feats, go, (size_t)M * dim * es, cudaMemcpyDeviceToDevice, st));
  EGNN_CUDA_TRY(cudaMemcpyAsync(g_coors, gr.g_coors_out, (size_t)M * s.C * es, cudaMemcpyDeviceToDevice, st));

  // ---- node update reversed (egnn_pytorch.py:335-337)
  if (uf) {
    const T* Wn1 = static_cast<const T*>(w.node_w1);
    const T* Wn2 = static_cast<const T*>(w.node_w2);
    EGNN_TRY(zero(ga, (size_t)M * d2 * es));
    EGNN_TRY(zero(g_node_in, (size_t)M * dn * es));
    EGNN_TRY((launch_gemm<T, 0, false>(node_in, dn, Wn1, dn, static_cast<const T*>(w.node_b1), nullptr, 0, h1pre, d2, M,
                                       d2, d2, dn, ident, st)));
    // dWn2[n][k] = sum_r go[r][n] h1[r][k];  db2 = colsum(go);  ga = go Wn2
    EGNN_TRY(launch_gemm_acc<T>(go, 1, dim, h1, d2, 1, static_cast<T*>(gr.w.node_w2), d2, dim, d2, M, st));
    EGNN_TRY(launch_colsum<T>(go, dim, M, dim, static_cast<T*>(gr.w.node_b2), st));
    EGNN_TRY(launch_gemm_acc<T>(go, dim, 1, Wn2, d2, 1, ga, d2, M, d2, dim, st));
    EGNN_TRY(launch(dsilu_mul_kernel<T>, (int)std::min<size_t>(2048, ((size_t)M * d2 + 255) / 256), 256, 0, st, ga, h1pre,
                    (size_t)M * d2, make_drop(d.dropout_p, d.dropout_seed)));
    // dWn1[k][c] = sum_r gh1[r][k] node_in[r][c];  db1 = colsum(gh1);  g_node_in = gh1 Wn1
    EGNN_TRY(launch_gemm_acc<T>(ga, 1, d2, node_in, dn, 1, static_cast<T*>(gr.w.node_w1), dn, d2, dn, M, st));
    EGNN_TRY(launch_colsum<T>(ga, d2, M, d2, static_cast<T*>(gr.w.node_b1), st));
    EGNN_TRY(launch_gemm_acc<T>(ga, d2, 1, Wn1, dn, 1, g_node_in, dn, M, dn, d2, st));
    EGNN_TRY(launch(ln_bwd_kernel<T>, ceil_div(M * 32, 256), 256, 0, st, feats, static_cast<const T*>(w.norm_g), g_node_in, dn,
                    g_feats, gyx, dim, M, nf ? 1 : 0));
    if (nf) {
      EGNN_TRY(launch_colsum<T>(gyx, dim, M, dim, static_cast<T*>(gr.w.norm_g), st));
      EGNN_TRY(launch_colsum<T>(g_node_in, dn, M, dim, static_cast<T*>(gr.w.norm_b), st));
    }
  }

  // ---- the edge step reversed
  BwdArgs<T> a;
  a.s = s; a.L = L; a.rl = rec_layout(s, L.MP); a.flags = d.flags; a.has_mask = io.mask != nullptr;
  a.clamp = (T)d.clamp;
  a.P = P; a.ldP = 2 * s.Hp;
  a.coors = static_cast<const T*>(io.coors);
  a.edges = static_cast<const T*>(io.edges);
  a.labels = s.label_dim > 0 ? io.edge_labels : nullptr;
  a.mask = io.mask;
  a.nbr_idx = nbr_idx; a.nbr_ok = nbr_ok;
  a.packed = static_cast<const T*>(packed);
  a.g_node_in = uf ? g_node_in : nullptr; a.ld_g = dn;
  a.g_coors_out = static_cast<const T*>(gr.g_coors_out);
  a.drop = make_drop(d.dropout_p, d.dropout_seed);
  const bool saved = io.pre2_out != nullptr;                 // the forward kept W2 silu(pre1) per pair
  a.pre2 = saved ? static_cast<const T*>(io.pre2_out)
                 : (s.k == 0 ? reinterpret_cast<const T*>(base + bl.pre2) : nullptr);
  a.rec = rec; a.gpk = gpk; a.gP = gP; a.g_coors = g_coors;
  a.g_edges = (s.edge_dim > 0) ? static_cast<T*>(gr.g_edges) : nullptr;
  if (s.k > 0) {
    int TS = 1;
    while (TS < s.k && TS < 32) TS <<= 1;
    a.TS = TS; a.TI2 = 16;
    if (L.MP == 16) EGNN_TRY((launch_pair_bwd<T, 16, true>(a, false, st)));
    else EGNN_TRY((launch_pair_bwd<T, 32, true>(a, false, st)));
  } else {
    a.TS = 32; a.TI2 = 32;
    if (L.MP == 16) EGNN_TRY((launch_pair_bwd<T, 16, false>(a, saved, st)));
    else EGNN_TRY((launch_pair_bwd<T, 32, false>(a, saved, st)));
  }

  // ---- per-node tables reversed: A = h W1[:, :dim]^T + b1, B = h W1[:, dim:2dim]^T
  T* gW1 = static_cast<T*>(gr.w.edge_w1);
  const int ldP = 2 * s.Hp;
  EGNN_TRY(launch_gemm_acc<T>(gP, ldP, 1, W1, s.E, 1, g_feats, dim, M, dim, s.H, st));                 // g_h += gA W1_i
  EGNN_TRY(launch_gemm_acc<T>(gP + s.Hp, ldP, 1, W1 + dim, s.E, 1, g_feats, dim, M, dim, s.H, st));    // g_h += gB W1_j
  EGNN_TRY(launch_gemm_acc<T>(gP, 1, ldP, feats, dim, 1, gW1, s.E, s.H, dim, M, st));                   // dW1_i = gA^T h
  EGNN_TRY(launch_gemm_acc<T>(gP + s.Hp, 1, ldP, feats, dim, 1, gW1 + dim, s.E, s.H, dim, M, st));      // dW1_j = gB^T h
  EGNN_TRY(launch_colsum<T>(gP, ldP, M, s.H, static_cast<T*>(gr.w.edge_b1), st));                       // db1

  (void)uc; (void)h1;
  return launch(unpack_grads_kernel<T>, 148, 256, 0, st, s, L, d.flags, gpk, W1, static_cast<const T*>(w.label_emb), gr.w);
}

}  // namespace egnn
