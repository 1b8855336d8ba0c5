// extern "C" entry points of libegnn_b200.so (see include/egnn_b200.h) and the per-layer
// orchestration: [neighbour select] -> per-node tables -> fused edge kernel -> node update.
#include "common.cuh"
#include "simt_kernels.cuh"
#include "fast_path.h"
#include "knn_select.h"
#include "simt_host.cuh"
#include "small_node.cuh"
#include <algorithm>

namespace egnn {

template <typename T, int MP, bool KNN>
static int launch_pair(const PairArgs<T>& a, cudaStream_t st) {
  dim3 grid(ceil_div(a.s.row1 - a.s.row0, PAIR_THREADS / a.TS), a.s.B);
  return launch(pair_kernel<T, MP, KNN>, grid, PAIR_THREADS, pair_smem_bytes<T>(a.s, a.L, KNN), st, a);
}

template <typename T, int MP, int PP>
static int launch_pair_tiled(const PairArgs<T>& a, cudaStream_t st) {
  const size_t smem = pair_tiled_smem_bytes<T>(a.s, a.L, PP);
  dim3 grid(ceil_div(a.s.row1 - a.s.row0, 4 * PP), a.s.B);
  if (a.hsplit > 1) {
    PairArgs<T> a1 = a, a2 = a;
    a1.phase = 1; a2.phase = 2;
    a1.pre2_out = nullptr;                            // partial sums; phase 2 holds the full ones
    EGNN_TRY(launch(pair_dense_tiled_kernel<T, MP, PP>, dim3(grid.x, grid.y, a.hsplit), PAIR_THREADS, smem, st, a1));
    return launch(pair_dense_tiled_kernel<T, MP, PP>, grid, PAIR_THREADS, smem, st, a2);
  }
  return launch(pair_dense_tiled_kernel<T, MP, PP>, grid, PAIR_THREADS, smem, st, a);
}

template <typename T>
static int simt_forward(const EgnnLayerDesc& d, const EgnnLayerWeights& w, const void* packed,
                        const EgnnLayerIO& io, void* ws, size_t ws_bytes, cudaStream_t st) {
  const Dims s = make_dims(d);
  const SimtPackLayout L = simt_pack_layout(s);
  const SimtWs wl = simt_ws_layout(s, sizeof(T), d.flags);
  if (ws_bytes < wl.total) return EGNN_ERR_WORKSPACE;
  if (s.row1 <= s.row0) return EGNN_OK;
  char* base = static_cast<char*>(ws);
  T* P = reinterpret_cast<T*>(base + wl.P);
  T* node_in = reinterpret_cast<T*>(base + wl.node_in);
  T* h1 = reinterpret_cast<T*>(base + wl.h1);
  int32_t* nbr_idx = reinterpret_cast<int32_t*>(base + wl.nbr_idx);
  uint8_t* nbr_ok = reinterpret_cast<uint8_t*>(base + wl.nbr_ok);
  const T* feats = static_cast<const T*>(io.feats);
  const T* W1 = static_cast<const T*>(w.edge_w1);
  const bool uf = d.flags & EGNN_FLAG_UPDATE_FEATS, uc = d.flags & EGNN_FLAG_UPDATE_COORS;
  const RowMap ident{s.N, s.N, 0};

  // 1. neighbour lists (egnn_pytorch.py:237-260)
  if (s.k > 0) EGNN_TRY(select_neighbours(d, s, io, d.dtype, nbr_idx, nbr_ok, st));
  // 2. per-node tables  A = h W1[:, :dim]^T + b1,  B = h W1[:, dim:2dim]^T   (split of :287's Linear-1)
  {
    StageTimer tm(st, STAGE_NODE_PRE);
    if (s.dim <= SN_DIM_MAX && s.M <= SN_TABLES_M_MAX && tables_small_simt_smem<T>(s.dim, s.Hp) <= SMALL_NODE_SMEM_MAX) {   // narrow layer, few nodes: one launch
      TablesSmallSimtArgs<T> t;
      t.feats = feats; t.W1 = W1; t.b1 = static_cast<const T*>(w.edge_b1); t.P = P;
      t.M = s.M; t.dim = s.dim; t.H = s.H; t.Hp = s.Hp; t.E = s.E;
      int sms = 0;
      EGNN_TRY(device_sm_count(&sms));
      EGNN_TRY(launch(tables_small_simt_kernel<T>, std::min(ceil_div(s.M, SN_WARPS), 4 * sms), SN_WARPS * 32,
                      tables_small_simt_smem<T>(s.dim, s.Hp), st, t));
    } else {
      EGNN_TRY((launch_gemm<T, 0, false>(feats, s.dim, W1, s.E, static_cast<const T*>(w.edge_b1), nullptr, 0, P,
                                          2 * s.Hp, s.M, s.H, s.Hp, s.dim, ident, st)));
      EGNN_TRY((launch_gemm<T, 0, false>(feats, s.dim, W1 + s.dim, s.E, nullptr, nullptr, 0, P + s.Hp, 2 * s.Hp,
                                          s.M, s.H, s.Hp, s.dim, ident, st)));
    }
  }
  // 3. fused edge step
  PairArgs<T> a;
  a.s = s; a.L = L; a.flags = d.flags; a.has_mask = io.mask != nullptr;
  a.clamp = (T)d.clamp;
  a.P = P; a.ldP = 2 * s.Hp;
  a.coors = static_cast<const T*>(io.coors);
  a.edges = static_cast<const T*>(io.edges);
  a.labels = s.label_dim > 0 ? io.edge_labels : nullptr;
  a.mask = io.mask;
  a.nbr_idx = nbr_idx; a.nbr_ok = nbr_ok;
  a.packed = static_cast<const T*>(packed);
  a.m_out = uf ? node_in + s.dim : nullptr;
  a.ld_m = s.dim + s.m;
  a.coors_out = uc ? static_cast<T*>(io.coors_out) : nullptr;
  a.hpart = reinterpret_cast<T*>(base + wl.hpart); a.hsplit = wl.hsplit; a.phase = 0;
  a.pre2_out = static_cast<T*>(io.pre2_out);
  a.drop = make_drop(d.dropout_p, d.dropout_seed);
  {
    StageTimer tm(st, STAGE_PAIR);
    if (s.k > 0) {
      int TS = 1;
      while (TS < s.k && TS < 32) TS <<= 1;
      a.TS = TS;
      if (L.MP == 16) EGNN_TRY((launch_pair<T, 16, true>(a, st)));
      else EGNN_TRY((launch_pair<T, 32, true>(a, st)));
    } else {
      a.TS = 32;
      constexpr int PP = 2;                                // rows per thread of the register-tiled dense kernel
      int rc;
      if (L.MP == 16) rc = launch_pair_tiled<T, 16, PP>(a, st);
      else rc = launch_pair_tiled<T, 32, sizeof(T) == 4 ? 2 : 1>(a, st);
      if (rc == EGNN_ERR_UNSUPPORTED) {                   // shared memory budget: thread-per-pair kernel
        if (L.MP == 16) rc = launch_pair<T, 16, false>(a, st);
        else rc = launch_pair<T, 32, false>(a, st);
      }
      EGNN_TRY(rc);
    }
  }
  // 4. node update  h' = node_mlp([LN(h) | m_i]) + h   (egnn_pytorch.py:335-337)
  StageTimer post_tm(st, STAGE_NODE_POST);
  const int Rr = s.row1 - s.row0, Mr = s.B * Rr;
  const RowMap map{Rr, s.N, s.row0};
  if (uf && d.dropout_p == 0.0 && s.dim <= SN_DIM_MAX && node_small_simt_smem<T>(s.dim, s.m) <= SMALL_NODE_SMEM_MAX) {
    // narrow layer: LayerNorm, concat, both Linear layers and the residual in one launch (node_in / h1 still written)
    NodeSmallSimtArgs<T> n;
    n.feats = feats; n.node_in = node_in; n.h1 = h1;
    n.wn1 = static_cast<const T*>(w.node_w1); n.bn1 = static_cast<const T*>(w.node_b1);
    n.wn2 = static_cast<const T*>(w.node_w2); n.bn2 = static_cast<const T*>(w.node_b2);
    n.lng = static_cast<const T*>(w.norm_g); n.lnb = static_cast<const T*>(w.norm_b);
    n.out = static_cast<T*>(io.feats_out);
    n.B = s.B; n.N = s.N; n.dim = s.dim; n.m = s.m; n.row0 = s.row0; n.row1 = s.row1;
    n.do_norm = (d.flags & EGNN_FLAG_NORM_FEATS) ? 1 : 0;
    int sms = 0;
    EGNN_TRY(device_sm_count(&sms));
    EGNN_TRY(launch(node_update_small_simt_kernel<T>, std::min(ceil_div(Mr, SN_WARPS), 4 * sms), SN_WARPS * 32,
                    node_small_simt_smem<T>(s.dim, s.m), st, n));
  } else if (uf) {
    EGNN_TRY(launch(ln_concat_kernel<T>, ceil_div(Mr * 32, 256), 256, 0, st, feats, static_cast<const T*>(w.norm_g),
                    static_cast<const T*>(w.norm_b), node_in, s.dim + s.m, s.dim, Mr, map, (d.flags & EGNN_FLAG_NORM_FEATS) ? 1 : 0));
    EGNN_TRY((launch_gemm<T, 1, false>(node_in, s.dim + s.m, static_cast<const T*>(w.node_w1), s.dim + s.m,
                                       static_cast<const T*>(w.node_b1), nullptr, 0, h1, 2 * s.dim, Mr, 2 * s.dim,
                                       2 * s.dim, s.dim + s.m, map, st, make_drop(d.dropout_p, d.dropout_seed))));
    EGNN_TRY((launch_gemm<T, 0, true>(h1, 2 * s.dim, static_cast<const T*>(w.node_w2), 2 * s.dim,
                                      static_cast<const T*>(w.node_b2), feats, s.dim, static_cast<T*>(io.feats_out),
                                      s.dim, Mr, s.dim, s.dim, 2 * s.dim, map, st)));
  } else if (io.feats_out != io.feats) {
    EGNN_CUDA_TRY(cudaMemcpyAsync(io.feats_out, io.feats, (size_t)s.M * s.dim * sizeof(T), cudaMemcpyDeviceToDevice, st));
  }
  if (!uc && io.coors_out != io.coors)
    EGNN_CUDA_TRY(cudaMemcpyAsync(io.coors_out, io.coors, (size_t)s.M * s.C * sizeof(T), cudaMemcpyDeviceToDevice, st));
  return EGNN_OK;
}

}  // namespace egnn

using namespace egnn;

extern "C" int egnn_abi_version(void) { return EGNN_ABI_VERSION; }

extern "C" const char* egnn_strerror(int code) {
  switch (code) {
    case EGNN_OK: return "ok";
    case EGNN_ERR_NULL: return "required pointer is NULL";
    case EGNN_ERR_SHAPE: return "inconsistent or out-of-range sizes";
    case EGNN_ERR_UNSUPPORTED: return "option combination not supported by this build";
    case EGNN_ERR_ALIGN: return "pointer not 16-byte aligned";
    case EGNN_ERR_WORKSPACE: return "workspace or packed-parameter buffer too small";
    case EGNN_ERR_ABI: return "ABI version mismatch";
    default: break;
  }
  if (code <= EGNN_ERR_CUDA) return cudaGetErrorString((cudaError_t)(EGNN_ERR_CUDA - code));
  return "unknown error";
}

extern "C" int egnn_layer_packed_bytes(const EgnnLayerDesc* desc, size_t* out_bytes) {
  if (!out_bytes) return EGNN_ERR_NULL;
  EGNN_TRY(validate_desc(desc));
  const Dims s = make_dims(*desc);
  if (desc->dtype == EGNN_DTYPE_BF16) return fast_packed_bytes(*desc, out_bytes);
  *out_bytes = round_up(simt_pack_layout(s).total * elem_size(desc->dtype), 256);
  return EGNN_OK;
}

extern "C" int egnn_layer_pack_weights(const EgnnLayerDesc* desc, const EgnnLayerWeights* w, void* packed,
                                       size_t packed_bytes, void* stream) {
  EGNN_TRY(validate_desc(desc));
  if (!packed) return EGNN_ERR_NULL;
  EGNN_TRY(check_ptrs(*desc, w, nullptr));
  size_t need = 0;
  EGNN_TRY(egnn_layer_packed_bytes(desc, &need));
  if (packed_bytes < need) return EGNN_ERR_WORKSPACE;
  if ((uintptr_t)packed & 0xF) return EGNN_ERR_ALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Dims s = make_dims(*desc);
  if (desc->dtype == EGNN_DTYPE_BF16) return fast_pack_weights(*desc, *w, packed, packed_bytes, st);
  const SimtPackLayout L = simt_pack_layout(s);
  if (desc->dtype == EGNN_DTYPE_F64) return launch(simt_pack_kernel<double>, 148, 256, 0, st, s, L, *w, desc->flags, static_cast<double*>(packed));
  return launch(simt_pack_kernel<float>, 148, 256, 0, st, s, L, *w, desc->flags, static_cast<float*>(packed));
}

extern "C" int egnn_layer_workspace_bytes(const EgnnLayerDesc* desc, size_t* out_bytes) {
  if (!out_bytes) return EGNN_ERR_NULL;
  EGNN_TRY(validate_desc(desc));
  const Dims s = make_dims(*desc);
  if (desc->dtype == EGNN_DTYPE_BF16) return fast_workspace_bytes(*desc, out_bytes);
  *out_bytes = simt_ws_layout(s, elem_size(desc->dtype), desc->flags).total + 256;
  return EGNN_OK;
}

extern "C" int egnn_layer_forward(const EgnnLayerDesc* desc, const EgnnLayerWeights* w, const void* packed,
                                  const EgnnLayerIO* io, void* workspace, size_t workspace_bytes, void* stream) {
  EGNN_TRY(validate_desc(desc));
  if (!io || !packed || !workspace) return EGNN_ERR_NULL;
  EGNN_TRY(check_ptrs(*desc, w, io));
  if ((uintptr_t)workspace & 0xFF) return EGNN_ERR_ALIGN;
  if ((uintptr_t)packed & 0xF) return EGNN_ERR_ALIGN;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (desc->dtype) {
    case EGNN_DTYPE_F64: return simt_forward<double>(*desc, *w, packed, *io, workspace, workspace_bytes, st);
    case EGNN_DTYPE_F32: return simt_forward<float>(*desc, *w, packed, *io, workspace, workspace_bytes, st);
    case EGNN_DTYPE_BF16: return fast_forward(*desc, *w, packed, *io, workspace, workspace_bytes, st);
    default: return EGNN_ERR_UNSUPPORTED;
  }
}

extern "C" int egnn_layer_forward_host(const EgnnLayerDesc* desc, const EgnnLayerWeights* w, const void* packed,
                                       const EgnnLayerIO* hio, void* stream) {
  EGNN_TRY(validate_desc(desc));
  if (!hio || !packed) return EGNN_ERR_NULL;
  if (!hio->feats || !hio->coors || !hio->feats_out || !hio->coors_out) return EGNN_ERR_NULL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Dims s = make_dims(*desc);
  const size_t es = elem_size(desc->dtype);
  const size_t cs = desc->dtype == EGNN_DTYPE_F64 ? 8 : 4;
  const size_t nf = (size_t)s.M * s.dim * es, nc = (size_t)s.M * s.C * cs;
  const size_t ne = hio->edges ? (size_t)s.M * s.N * s.edge_dim * es : 0;
  const size_t nl = hio->edge_labels ? (size_t)s.M * s.N : 0;
  const size_t nm = hio->mask ? (size_t)s.M : 0;
  const size_t na = hio->adj ? (size_t)((desc->flags & EGNN_FLAG_ADJ_BATCHED) ? s.B : 1) * s.N * s.N : 0;
  const size_t nn = hio->nbr_idx ? (size_t)s.M * s.k * sizeof(int32_t) : 0;
  size_t wsb = 0;
  EGNN_TRY(egnn_layer_workspace_bytes(desc, &wsb));
  // one device arena: [feats | feats_out | coors | coors_out | edges | labels | mask | adj | workspace]
  size_t off[10];
  size_t o = 0;
  const size_t sizes[10] = {nf, nf, nc, nc, ne, nl, nm, na, wsb, nn};
  for (int i = 0; i < 10; ++i) { off[i] = o; o += round_up(sizes[i], 256); }
  char* arena = nullptr;
  EGNN_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&arena), o + 256, st));
  int rc = EGNN_OK;
  auto h2d = [&](int slot, const void* src, size_t n) {
    if (n && rc == EGNN_OK) {
      cudaError_t e = cudaMemcpyAsync(arena + off[slot], src, n, cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) rc = EGNN_ERR_CUDA - (int)e;
    }
  };
  h2d(0, hio->feats, nf); h2d(2, hio->coors, nc); h2d(4, hio->edges, ne); h2d(5, hio->edge_labels, nl);
  h2d(6, hio->mask, nm); h2d(7, hio->adj, na); h2d(9, hio->nbr_idx, nn);
  if (rc == EGNN_OK) {
    EgnnLayerIO dio;
    dio.feats = arena + off[0]; dio.feats_out = arena + off[1];
    dio.coors = arena + off[2]; dio.coors_out = arena + off[3];
    dio.edges = ne ? arena + off[4] : nullptr;
    dio.edge_labels = nl ? reinterpret_cast<uint8_t*>(arena + off[5]) : nullptr;
    dio.mask = nm ? reinterpret_cast<uint8_t*>(arena + off[6]) : nullptr;
    dio.adj = na ? reinterpret_cast<uint8_t*>(arena + off[7]) : nullptr;
    dio.nbr_idx = nn ? reinterpret_cast<int32_t*>(arena + off[9]) : nullptr;
    dio.pre2_out = nullptr;
    rc = egnn_layer_forward(desc, w, packed, &dio, arena + off[8], wsb, stream);
  }
  if (rc == EGNN_OK) {
    cudaError_t e = cudaMemcpyAsync(hio->feats_out, arena + off[1], nf, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hio->coors_out, arena + off[3], nc, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) rc = EGNN_ERR_CUDA - (int)e;
  }
  cudaFreeAsync(arena, st);
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc == EGNN_OK && e != cudaSuccess) rc = EGNN_ERR_CUDA - (int)e;
  return rc;
}

extern "C" int egnn_gemm_bf16(int32_t M, int32_t N, int32_t K, const void* A, const void* W, const float* bias,
                              float scale, int32_t act, void* out, int32_t out_f32, void* stream) {
  return debug_gemm_bf16(M, N, K, A, W, bias, scale, act, out, out_f32, static_cast<cudaStream_t>(stream));
}

// ---- diagnostics (see profile.h): per-stage CUDA-event timing on the launch stream ----------
extern "C" int egnn_profile_enable(int on) {
  Profiler& p = Profiler::get();
  std::lock_guard<std::mutex> g(p.mu);
  p.on = on != 0;
  return EGNN_OK;
}

extern "C" int egnn_profile_read(float* ms_out, int32_t* spans_out, int64_t* launches_out, int reset) {
  Profiler& p = Profiler::get();
  std::lock_guard<std::mutex> g(p.mu);
  float ms[STAGE_COUNT] = {0, 0, 0, 0};
  int32_t n[STAGE_COUNT] = {0, 0, 0, 0};
  for (auto& sp : p.spans) {
    EGNN_CUDA_TRY(cudaEventSynchronize(sp.b));
    float t = 0.f;
    EGNN_CUDA_TRY(cudaEventElapsedTime(&t, sp.a, sp.b));
    ms[sp.stage] += t;
    n[sp.stage] += 1;
  }
  for (int i = 0; i < STAGE_COUNT; ++i) {
    if (ms_out) ms_out[i] = ms[i];
    if (spans_out) spans_out[i] = n[i];
  }
  if (launches_out) *launches_out = p.launches;
  if (reset) {
    for (auto& sp : p.spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    p.spans.clear();
    p.launches = 0;
  }
  return EGNN_OK;
}
