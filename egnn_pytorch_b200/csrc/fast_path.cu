// bf16 tensor-core path of the layer (EGNN_DTYPE_BF16): parameter packing, workspace layout and the
// per-layer launch sequence   node tables (tcgen05 GEMM x2) -> fused edge kernel (tc_pair.cuh)
//                             -> LayerNorm/concat -> node MLP (tcgen05 GEMM x2).
// Option sets the tensor-core kernels do not cover return EGNN_ERR_UNSUPPORTED; the binding then runs
// the fp32 SIMT kernels (never a CPU path).
#include <stdlib.h>
#include "fast_path.h"
#include "knn_select.h"
#include "launch.cuh"
#include "tc_gemm.cuh"
#include "tc_pair.cuh"
#include "tc_knn.cuh"
#include "small_node.cuh"

namespace egnn {
namespace {

struct FastDims {
  Dims s;
  int Hp;      // H rounded up to 16 (one K step of the fused kernels' MMA)
  int Kn;      // dim + m rounded up to 8 (K of the first node GEMM)
  int L;       // one-hot label channels (num_labels when the layer has a label embedding)
  int QT;      // per-pair scalar channels: d | sin | cos | continuous edges | one-hot labels
  int QR;      // rows of the packed Wq table (>= 1 + TK_QE so that the neighbour-list kernel can view rows 1..4)
};

// layout of the packed-parameter buffer (byte offsets, 256-aligned)
struct FastPack {
  size_t w1i, w1j, b1, wq, w2p, epi, wn1, bn1, wn2, bn2, lng, lnb, total;
};

FastDims fast_dims(const EgnnLayerDesc& d) {
  FastDims f;
  f.s = make_dims(d);
  f.Hp = round_up_i(f.s.H, 16);
  f.Kn = round_up_i(f.s.dim + f.s.m, 8);
  f.L = d.label_dim > 0 ? d.num_labels : 0;
  f.QT = 1 + 2 * d.fourier + d.edge_dim + f.L;
  f.QR = f.QT > 1 + TK_QE ? f.QT : 1 + TK_QE;
  return f;
}

// neighbour-list kernel: lean (distance only), edges (<= 4 continuous channels in registers), generic (everything else)
int knn_mode(const FastDims& f) {
  if (f.s.C == 3 && f.s.F == 0 && f.L == 0) return f.s.edge_dim == 0 ? TK_LEAN : (f.s.edge_dim <= TK_QE ? TK_EDGES : TK_GEN);
  return TK_GEN;
}

// the lean instantiation of the dense kernel covers 3-D coordinates with the distance as the only per-pair channel
bool pair_is_lean(const FastDims& f) { return f.s.C == 3 && f.QT == 1; }

FastPack fast_pack_layout(const FastDims& f) {
  FastPack p;
  BumpAlloc o;
  const int d = f.s.dim;
  p.w1i = o.take((size_t)f.Hp * d * 2);
  p.w1j = o.take((size_t)f.Hp * d * 2);
  p.b1 = o.take((size_t)f.Hp * 4);
  p.wq = o.take((size_t)f.QR * f.Hp * 4);
  p.w2p = o.take((size_t)f.Hp * 32);
  p.epi = o.take((size_t)TP_EPI_FLOATS * 4);
  p.wn1 = o.take((size_t)2 * d * f.Kn * 2);
  p.bn1 = o.take((size_t)2 * d * 4);
  p.wn2 = o.take((size_t)d * 2 * d * 2);
  p.bn2 = o.take((size_t)d * 4);
  p.lng = o.take((size_t)d * 4);
  p.lnb = o.take((size_t)d * 4);
  p.total = o.total;
  return p;
}

int fast_supported(const EgnnLayerDesc& d) {
  const FastDims f = fast_dims(d);
  if (d.m_dim != 16) return EGNN_ERR_UNSUPPORTED;                  // one 16-column accumulator per (row, warpgroup)
  if (d.dim % 8 != 0) return EGNN_ERR_UNSUPPORTED;                 // 16-byte rows for cp.async
  if (d.C < 1 || d.C > TP_CMAX) return EGNN_ERR_UNSUPPORTED;
  if (d.k == 0) {                                                  // dense all-pairs: tc_pair_kernel<lean | generic>
    if (f.QT > TP_QMAX) return EGNN_ERR_UNSUPPORTED;
    const size_t smem = pair_is_lean(f) ? tc_pair_smem_bytes<false>(f.Hp, 1) : tc_pair_smem_bytes<true>(f.Hp, f.QT, 1 + 2 * f.s.F);
    if (smem > TC_SMEM_MAX) return EGNN_ERR_UNSUPPORTED;
  } else {                                                         // neighbour lists: tc_knn_kernel<lean | edges | generic>
    if (d.k > 32) return EGNN_ERR_UNSUPPORTED;
    const int mode = knn_mode(f);
    if (mode == TK_GEN && f.QT > TP_QMAX) return EGNN_ERR_UNSUPPORTED;
    if (tc_knn_smem_bytes(f.Hp, mode, f.QT) > TC_SMEM_MAX) return EGNN_ERR_UNSUPPORTED;
  }
  return EGNN_OK;
}

__device__ __forceinline__ float bf(const void* p, size_t i) { return __bfloat162float(static_cast<const __nv_bfloat16*>(p)[i]); }

__global__ void fast_pack_kernel(FastDims f, FastPack L, EgnnLayerWeights w, uint32_t flags, unsigned char* out) {
  const Dims& s = f.s;
  const size_t stride = (size_t)gridDim.x * blockDim.x, t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int d = s.dim, H = s.H, E = s.E, Hp = f.Hp;
  __nv_bfloat16* w1i = reinterpret_cast<__nv_bfloat16*>(out + L.w1i);
  __nv_bfloat16* w1j = reinterpret_cast<__nv_bfloat16*>(out + L.w1j);
  for (size_t x = t0; x < (size_t)Hp * d; x += stride) {
    const int c = (int)(x / d), k = (int)(x % d);
    const __nv_bfloat16 z = __float2bfloat16(0.f);
    w1i[x] = c < H ? static_cast<const __nv_bfloat16*>(w.edge_w1)[(size_t)c * E + k] : z;
    w1j[x] = c < H ? static_cast<const __nv_bfloat16*>(w.edge_w1)[(size_t)c * E + d + k] : z;
  }
  float* b1 = reinterpret_cast<float*>(out + L.b1);
  for (size_t c = t0; c < (size_t)Hp; c += stride) b1[c] = c < (size_t)H ? bf(w.edge_b1, c) : 0.f;
  // Per-pair scalar columns of W1, pre-halved, in the kernels' channel order:
  //   row 0: d_ij (W1 column 2d + 2F, the LAST of the fourier block, egnn_pytorch.py:34-41) | rows 1..F: sin(d / 2^k)
  //   | rows F+1..2F: cos(d / 2^k) | edge_dim rows: continuous edge channels | L rows: label table
  //   Tab[l] = label_emb[l] @ W1[:, label columns]^T  (the embedding of :430-432 folded through Linear-1).
  float* wq = reinterpret_cast<float*>(out + L.wq);
  const int F = s.F, ed = s.edge_dim, ld = s.label_dim;
  for (size_t x = t0; x < (size_t)f.QR * Hp; x += stride) {
    const int q = (int)(x / Hp);
    const size_t c = x % Hp;
    float v = 0.f;
    if (c < (size_t)H) {
      const size_t row = c * E + 2 * d;
      if (q == 0) v = bf(w.edge_w1, row + 2 * F);
      else if (q <= 2 * F) v = bf(w.edge_w1, row + (q - 1));
      else if (q < 1 + 2 * F + ed) v = bf(w.edge_w1, row + 2 * F + 1 + (q - 1 - 2 * F));
      else if (q < 1 + 2 * F + ed + f.L) {
        const int l = q - 1 - 2 * F - ed;
        for (int t = 0; t < ld; ++t) v += bf(w.label_emb, (size_t)l * ld + t) * bf(w.edge_w1, row + 2 * F + 1 + ed + t);
      }
    }
    wq[x] = 0.5f * v;
  }
  // W2 [16][H] -> UMMA K-major core matrices: [slab = c/16][kc = (c%16)/8][nc = n/8][r = n%8][e = c%8]
  __nv_bfloat16* w2p = reinterpret_cast<__nv_bfloat16*>(out + L.w2p);
  for (size_t x = t0; x < (size_t)Hp * 16; x += stride) {
    const int e = (int)(x & 7), r = (int)((x >> 3) & 7), nc = (int)((x >> 6) & 1), kc = (int)((x >> 7) & 1);
    const int slab = (int)(x >> 8);
    const int n = nc * 8 + r, c = slab * 16 + kc * 8 + e;
    w2p[x] = c < H ? static_cast<const __nv_bfloat16*>(w.edge_w2)[(size_t)n * H + c] : __float2bfloat16(0.f);
  }
  // epilogue constants (fp32): W3[64][16] | b3[64] | w4[64] | b2[16] | gate_w[16] | gate_b, b4, scale, 0
  float* epi = reinterpret_cast<float*>(out + L.epi);
  const bool uc = flags & EGNN_FLAG_UPDATE_COORS, soft = flags & EGNN_FLAG_SOFT_EDGES;
  for (size_t x = t0; x < (size_t)TP_EPI_FLOATS; x += stride) {
    float v = 0.f;
    if (x < 1024) v = uc ? bf(w.coors_w1, x) : 0.f;
    else if (x < 1088) v = uc ? bf(w.coors_b1, x - 1024) : 0.f;
    else if (x < 1152) v = uc ? bf(w.coors_w2, x - 1088) : 0.f;
    else if (x < 1168) v = bf(w.edge_b2, x - 1152);
    else if (x < 1184) v = soft ? bf(w.gate_w, x - 1168) : 0.f;
    else if (x == 1184) v = soft ? bf(w.gate_b, 0) : 0.f;
    else if (x == 1185) v = uc ? bf(w.coors_b2, 0) : 0.f;
    else if (x == 1186) v = (flags & EGNN_FLAG_NORM_COORS) ? bf(w.coors_scale, 0) : 1.f;
    epi[x] = v;
  }
  if (flags & EGNN_FLAG_UPDATE_FEATS) {
    __nv_bfloat16* wn1 = reinterpret_cast<__nv_bfloat16*>(out + L.wn1);
    const int Kin = d + s.m;
    for (size_t x = t0; x < (size_t)2 * d * f.Kn; x += stride) {
      const int n = (int)(x / f.Kn), k = (int)(x % f.Kn);
      wn1[x] = k < Kin ? static_cast<const __nv_bfloat16*>(w.node_w1)[(size_t)n * Kin + k] : __float2bfloat16(0.f);
    }
    __nv_bfloat16* wn2 = reinterpret_cast<__nv_bfloat16*>(out + L.wn2);
    for (size_t x = t0; x < (size_t)d * 2 * d; x += stride) wn2[x] = static_cast<const __nv_bfloat16*>(w.node_w2)[x];
    float* bn1 = reinterpret_cast<float*>(out + L.bn1);
    for (size_t x = t0; x < (size_t)2 * d; x += stride) bn1[x] = bf(w.node_b1, x);
    float* bn2 = reinterpret_cast<float*>(out + L.bn2);
    float* lng = reinterpret_cast<float*>(out + L.lng);
    float* lnb = reinterpret_cast<float*>(out + L.lnb);
    const bool nf = flags & EGNN_FLAG_NORM_FEATS;
    for (size_t x = t0; x < (size_t)d; x += stride) {
      bn2[x] = bf(w.node_b2, x);
      lng[x] = nf ? bf(w.norm_g, x) : 1.f;
      lnb[x] = nf ? bf(w.norm_b, x) : 0.f;
    }
  }
}

// node_in[row, 0:dim] = LayerNorm(h[row]) | h[row] (bf16), pad columns [dim+m, Kn) = 0; one warp per row.
__global__ void ln_concat_bf16_kernel(const __nv_bfloat16* __restrict__ h, const float* __restrict__ g,
                                      const float* __restrict__ bta, __nv_bfloat16* __restrict__ node_in, int Kn, int dim,
                                      int m, int M, int do_norm) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = threadIdx.x % 32;
  if (row >= M) return;
  const __nv_bfloat16* x = h + (size_t)row * dim;
  __nv_bfloat16* y = node_in + (size_t)row * Kn;
  for (int c = dim + m + lane; c < Kn; c += 32) y[c] = __float2bfloat16(0.f);
  if (!do_norm) {
    for (int c = lane; c < dim; c += 32) y[c] = x[c];
    return;
  }
  float s = 0.f;
  for (int c = lane; c < dim; c += 32) s += __bfloat162float(x[c]);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mu = s / dim;
  float v = 0.f;
  for (int c = lane; c < dim; c += 32) { const float t = __bfloat162float(x[c]) - mu; v += t * t; }
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const float rstd = rsqrtf(v / dim + 1e-5f);
  for (int c = lane; c < dim; c += 32) y[c] = __float2bfloat16((__bfloat162float(x[c]) - mu) * rstd * g[c] + bta[c]);
}

struct FastWs { size_t Atab, Btab, node_in, h1, nbr_idx, nbr_ok, gpart, gcount, total; };
constexpr int TP_JSPLIT_MAX = 8;
FastWs fast_ws_layout(const FastDims& f, uint32_t flags) {
  FastWs w;
  BumpAlloc o;
  const bool uf = flags & EGNN_FLAG_UPDATE_FEATS;
  w.Atab = o.take((size_t)f.s.M * f.Hp * 4);
  w.Btab = o.take(((size_t)f.s.M + 128) * f.Hp * 2);    // +128 rows: the dense kernel reads (and discards) up to a tile past the end
  w.node_in = o.take(uf ? (size_t)f.s.M * f.Kn * 2 : 0);
  w.h1 = o.take(uf ? (size_t)f.s.M * 2 * f.s.dim * 2 : 0);
  w.nbr_idx = o.take((size_t)f.s.M * f.s.k * sizeof(int32_t));
  w.nbr_ok = o.take((size_t)f.s.M * f.s.k);
  // dense kernel, j-split mode: partial sums and arrival counters per row group (the counters are kept zero between calls)
  const size_t rgs = f.s.k == 0 ? (size_t)f.s.B * ceil_div(f.s.row1 - f.s.row0, TP_TI) : 0;
  w.gpart = o.take(rgs * TP_JSPLIT_MAX * TP_TI * TpCfg<true>::PW * 8);
  w.gcount = o.take(rgs * 4);
  w.total = o.total;
  return w;
}

// Optional start-up delay between the warpgroups of the persistent dense kernel (tc_pair.cuh), EGNN_B200_SKEW_NS.
// Default 0: measured on B200 (profiles/r02_tc_pair_skew_sweep.txt) de-phasing the warpgroups' epilogues buys nothing --
// the kernel is bound by per-warp latency (1/2/3/4 warps per sub-partition reach 0.28/0.47/0.58/0.67 of the MUFU
// roofline), not by the pipe idling during the epilogues.
uint32_t pair_skew_ns() {
  static const uint32_t v = [] {
    const char* e = getenv("EGNN_B200_SKEW_NS");
    return e ? (uint32_t)strtoul(e, nullptr, 10) : 0u;
  }();
  return v;
}

// one launch for one (g2 == nullptr) or two problems over the same rows
int launch_tc_gemm(const TcGemmArgs& g, cudaStream_t st, const TcGemmArgs* g2 = nullptr) {
  if (g.M <= 0) return EGNN_OK;
  TcGemmPair gp;
  gp.p[0] = g;
  gp.p[1] = g2 ? *g2 : g;
  gp.nt0 = ceil_div(g.Nout, GEMM_BN);
  const int nt1 = g2 ? ceil_div(g2->Nout, GEMM_BN) : 0;
  return launch_upto(TC_SMEM_MAX, tc_gemm_kernel, dim3(gp.nt0 + nt1, ceil_div(g.M, GEMM_BM)), 128, GEMM_SMEM_BYTES, st, gp);
}

}  // namespace

int debug_gemm_bf16(int M, int N, int K, const void* A, const void* W, const float* bias, float scale, int act,
                    void* out, int out_f32, cudaStream_t st) {
  if (!A || !W || !out) return EGNN_ERR_NULL;
  if (M <= 0 || N <= 0 || K <= 0 || K % 8 != 0 || N % 8 != 0) return EGNN_ERR_SHAPE;
  TcGemmArgs g{};
  g.A = static_cast<const __nv_bfloat16*>(A); g.lda = K; g.W = static_cast<const __nv_bfloat16*>(W); g.ldw = K;
  g.bias = bias; g.R = nullptr; g.ldr = 0; g.out = out; g.ldo = N; g.out_f32 = out_f32;
  g.M = M; g.Nv = N; g.Nout = N; g.K = K; g.scale = scale; g.act = act;
  return launch_tc_gemm(g, st);
}

int fast_packed_bytes(const EgnnLayerDesc& d, size_t* out) {
  EGNN_TRY(fast_supported(d));
  *out = fast_pack_layout(fast_dims(d)).total;
  return EGNN_OK;
}

int fast_pack_weights(const EgnnLayerDesc& d, const EgnnLayerWeights& w, void* packed, size_t bytes, cudaStream_t st) {
  EGNN_TRY(fast_supported(d));
  const FastDims f = fast_dims(d);
  const FastPack L = fast_pack_layout(f);
  if (bytes < L.total) return EGNN_ERR_WORKSPACE;
  return launch(fast_pack_kernel, 296, 256, 0, st, f, L, w, d.flags, static_cast<unsigned char*>(packed));
}

int fast_workspace_bytes(const EgnnLayerDesc& d, size_t* out) {
  EGNN_TRY(fast_supported(d));
  *out = fast_ws_layout(fast_dims(d), d.flags).total + 256;
  return EGNN_OK;
}

int fast_forward(const EgnnLayerDesc& d, const EgnnLayerWeights& w, const void* packed, const EgnnLayerIO& io,
                 void* ws, size_t ws_bytes, cudaStream_t st) {
  (void)w;
  EGNN_TRY(fast_supported(d));
  const FastDims f = fast_dims(d);
  const Dims& s = f.s;
  const FastPack L = fast_pack_layout(f);
  const FastWs wl = fast_ws_layout(f, d.flags);
  if (ws_bytes < wl.total) return EGNN_ERR_WORKSPACE;
  const unsigned char* pk = static_cast<const unsigned char*>(packed);
  unsigned char* base = static_cast<unsigned char*>(ws);
  float* Atab = reinterpret_cast<float*>(base + wl.Atab);
  __nv_bfloat16* Btab = reinterpret_cast<__nv_bfloat16*>(base + wl.Btab);
  __nv_bfloat16* node_in = reinterpret_cast<__nv_bfloat16*>(base + wl.node_in);
  __nv_bfloat16* h1 = reinterpret_cast<__nv_bfloat16*>(base + wl.h1);
  const __nv_bfloat16* feats = static_cast<const __nv_bfloat16*>(io.feats);
  const bool uf = d.flags & EGNN_FLAG_UPDATE_FEATS, uc = d.flags & EGNN_FLAG_UPDATE_COORS;

  // Row range (row-sharded single graph, SURVEY.md section 8(e)): the j side (B') always covers all nodes, the i side
  // (A', the fused kernel's row groups, the node update) only rows [row0, row1) of every graph.
  const int r0 = s.row0, r1 = s.row1, R = r1 - r0;
  const bool all_rows = (r0 == 0 && r1 == s.N);
  const int nseg = all_rows ? 1 : s.B;                        // contiguous row segments for the per-node GEMMs
  auto seg_begin = [&](int sg) { return all_rows ? (size_t)0 : (size_t)sg * s.N + r0; };
  const int seg_rows = all_rows ? s.M : R;

  {  // per-node tables, pre-halved for the tanh form of SiLU:  A' = 0.5 (h W1_i^T + b1),  B' = 0.5 h W1_j^T
    StageTimer tm(st, STAGE_NODE_PRE);
    if (s.dim <= SN_DIM_MAX && s.M <= SN_TABLES_M_MAX) {  // narrow layer, few nodes: one warp per node, one launch (small_node.cuh)
      TablesSmallArgs t{};
      t.feats = feats; t.w1i = reinterpret_cast<const __nv_bfloat16*>(pk + L.w1i); t.w1j = reinterpret_cast<const __nv_bfloat16*>(pk + L.w1j);
      t.b1 = reinterpret_cast<const float*>(pk + L.b1); t.Atab = Atab; t.Btab = Btab;
      t.M = s.M; t.N = s.N; t.dim = s.dim; t.Hp = f.Hp; t.row0 = r0; t.row1 = r1;
      int sms = 0;
      EGNN_TRY(device_sm_count(&sms));
      EGNN_TRY(launch_upto(TC_SMEM_MAX, tables_small_kernel, std::min(ceil_div(s.M, SN_WARPS), 4 * sms), SN_WARPS * 32,
                           tables_small_smem(s.dim, f.Hp), st, t));
    } else {
      TcGemmArgs g{};
      g.lda = s.dim; g.K = s.dim; g.Nv = f.Hp; g.Nout = f.Hp; g.scale = 0.5f; g.act = 0; g.R = nullptr; g.ldr = 0; g.ldo = f.Hp;
      g.W = reinterpret_cast<const __nv_bfloat16*>(pk + L.w1i); g.ldw = s.dim;
      g.bias = reinterpret_cast<const float*>(pk + L.b1);
      g.out_f32 = 1;
      TcGemmArgs gb = g;                                    // B' = 0.5 h W1_j^T over ALL rows
      gb.A = feats; gb.M = s.M;
      gb.W = reinterpret_cast<const __nv_bfloat16*>(pk + L.w1j); gb.bias = nullptr;
      gb.out = Btab; gb.out_f32 = 0;
      if (all_rows) {                                       // both tables in one launch (same rows, same activations)
        g.A = feats; g.M = s.M; g.out = Atab;
        EGNN_TRY(launch_tc_gemm(g, st, &gb));
      } else {
        for (int sg = 0; sg < nseg; ++sg) {
          g.A = feats + seg_begin(sg) * s.dim; g.M = seg_rows; g.out = Atab + seg_begin(sg) * f.Hp;
          EGNN_TRY(launch_tc_gemm(g, st));
        }
        EGNN_TRY(launch_tc_gemm(gb, st));
      }
    }
  }
  if (s.k == 0) {  // fused edge kernel, dense all-pairs (persistent: one CTA per SM walks the row groups)
    StageTimer tm(st, STAGE_PAIR);
    TcPairArgs a{};
    a.B = s.B; a.N = s.N; a.Hp = f.Hp; a.ldn = f.Kn;
    a.C = s.C; a.Q = f.QT; a.F = s.F; a.edge_dim = s.edge_dim; a.num_labels = f.L;
    a.row0 = r0; a.row1 = r1;
    a.flags = d.flags; a.has_mask = io.mask != nullptr; a.clamp = (float)d.clamp;
    a.skew_ns = pair_skew_ns();
    a.Atab = Atab; a.Btab = Btab;
    a.wq = reinterpret_cast<const float*>(pk + L.wq);
    a.w2p = reinterpret_cast<const __nv_bfloat16*>(pk + L.w2p);
    a.epi = reinterpret_cast<const float*>(pk + L.epi);
    a.coors = static_cast<const float*>(io.coors);
    a.edges = static_cast<const __nv_bfloat16*>(io.edges);
    a.labels = f.L > 0 ? io.edge_labels : nullptr;
    a.mask = io.mask;
    a.m_out = uf ? node_in + s.dim : nullptr;
    a.coors_out = uc ? static_cast<float*>(io.coors_out) : nullptr;
    if (f.L > 0 && !io.edge_labels) return EGNN_ERR_NULL;
    if (s.edge_dim > 0 && !io.edges) return EGNN_ERR_NULL;
    int sms = 0;
    EGNN_TRY(device_sm_count(&sms));
    int items = s.B * ceil_div(R, TP_TI);
    if (items > 0) {
      // too few row groups to balance one CTA per SM: deal the j-blocks of every row group to 2 / 4 / 8 items
      const int njb = ceil_div(s.N, TP_JB);
      int js = 1;
      while (js < TP_JSPLIT_MAX && items * js < 6 * sms && js * 2 <= njb) js *= 2;
      a.jsplit = js;
      a.gpart = reinterpret_cast<double*>(base + wl.gpart);
      a.gcount = reinterpret_cast<unsigned int*>(base + wl.gcount);
      if (js > 1) {
        // the counters must be zero on entry; the kernel leaves them zero, so only a workspace that was never used in
        // this mode (or was used for something else) needs the memset -- it is cheap enough to do always
        EGNN_CUDA_TRY(cudaMemsetAsync(a.gcount, 0, (size_t)items * 4, st));
        items *= js;
      }
      const int grid = items < sms ? items : sms;
      if (items < 2 * sms) a.skew_ns = 0;                      // too few row groups per CTA for the de-phasing to pay
      if (pair_is_lean(f))
        EGNN_TRY(launch_upto(TC_SMEM_MAX, tc_pair_kernel<false>, grid, TP_THREADS, tc_pair_smem_bytes<false>(f.Hp, 1), st, a));
      else
        EGNN_TRY(launch_upto(TC_SMEM_MAX, tc_pair_kernel<true>, grid, TP_THREADS, tc_pair_smem_bytes<true>(f.Hp, f.QT, 1 + 2 * f.s.F), st, a));
    }
  } else {         // neighbour lists: distance + top-k select, then the gathered fused edge kernel
    int32_t* nbr_idx = reinterpret_cast<int32_t*>(base + wl.nbr_idx);
    uint8_t* nbr_ok = base + wl.nbr_ok;
    EGNN_TRY(select_neighbours(d, s, io, EGNN_DTYPE_F32, nbr_idx, nbr_ok, st));
    StageTimer tm(st, STAGE_PAIR);
    TcKnnArgs a{};
    a.B = s.B; a.N = s.N; a.Hp = f.Hp; a.ldn = f.Kn; a.dim = s.dim; a.k = s.k; a.edge_dim = s.edge_dim;
    a.C = s.C; a.Q = f.QT; a.F = s.F; a.num_labels = f.L; a.row0 = r0; a.row1 = r1;
    a.labels = f.L > 0 ? io.edge_labels : nullptr;
    if (f.L > 0 && !io.edge_labels) return EGNN_ERR_NULL;
    if (s.edge_dim > 0 && !io.edges) return EGNN_ERR_NULL;
    a.flags = d.flags; a.has_mask = io.mask != nullptr; a.clamp = (float)d.clamp;
    a.Atab = Atab; a.Btab = Btab;
    a.wdh = reinterpret_cast<const float*>(pk + L.wq);                       // row 0 of the Wq table (no fourier here)
    a.weh = reinterpret_cast<const float*>(pk + L.wq) + f.Hp;                // rows 1..4: edge channels (zero beyond edge_dim)
    a.w2p = reinterpret_cast<const __nv_bfloat16*>(pk + L.w2p);
    a.epi = reinterpret_cast<const float*>(pk + L.epi);
    a.coors = static_cast<const float*>(io.coors);
    a.edges = static_cast<const __nv_bfloat16*>(io.edges);
    a.mask = io.mask;
    a.nbr_idx = nbr_idx; a.nbr_ok = nbr_ok;
    a.m_out = uf ? node_in + s.dim : nullptr;
    a.coors_out = uc ? static_cast<float*>(io.coors_out) : nullptr;
    const int mode = knn_mode(f);
    const int rows = tc_knn_rows_per_cta(f.Hp, mode, f.QT);         // 8 (two CTAs per SM) when shared memory allows
    const size_t smem = tc_knn_smem_bytes(f.Hp, mode, f.QT, rows);
    const bool r8 = rows == 8;
    auto kernel = mode == TK_LEAN ? (r8 ? tc_knn_kernel<TK_LEAN, 8> : tc_knn_kernel<TK_LEAN, 16>)
                : mode == TK_EDGES ? (r8 ? tc_knn_kernel<TK_EDGES, 8> : tc_knn_kernel<TK_EDGES, 16>)
                                   : (r8 ? tc_knn_kernel<TK_GEN, 8> : tc_knn_kernel<TK_GEN, 16>);
    if (R > 0) EGNN_TRY(launch_upto(TC_SMEM_MAX, kernel, dim3(ceil_div(R, rows), s.B), rows * 32, smem, st, a));
  }
  StageTimer post(st, STAGE_NODE_POST);
  __nv_bfloat16* fout = static_cast<__nv_bfloat16*>(io.feats_out);
  if (uf) {  // h' = node_mlp([LN(h) | m_i]) + h
    if (s.dim <= SN_DIM_MAX && R > 0) {                   // narrow layer: LayerNorm, concat, both Linear layers and the residual in one launch
      NodeSmallArgs n{};
      n.feats = feats; n.node_in = node_in; n.wn1 = reinterpret_cast<const __nv_bfloat16*>(pk + L.wn1);
      n.bn1 = reinterpret_cast<const float*>(pk + L.bn1); n.wn2 = reinterpret_cast<const __nv_bfloat16*>(pk + L.wn2);
      n.bn2 = reinterpret_cast<const float*>(pk + L.bn2); n.lng = reinterpret_cast<const float*>(pk + L.lng);
      n.lnb = reinterpret_cast<const float*>(pk + L.lnb); n.out = fout;
      n.B = s.B; n.N = s.N; n.dim = s.dim; n.Kn = f.Kn; n.m = s.m; n.row0 = r0; n.row1 = r1; n.do_norm = (d.flags & EGNN_FLAG_NORM_FEATS) ? 1 : 0;
      int sms = 0;
      EGNN_TRY(device_sm_count(&sms));
      EGNN_TRY(launch_upto(TC_SMEM_MAX, node_update_small_kernel, std::min(ceil_div(s.B * R, SN_WARPS), 4 * sms), SN_WARPS * 32,
                           node_small_smem(s.dim, f.Kn), st, n));
    } else
    for (int sg = 0; sg < nseg; ++sg) {
      const size_t o = seg_begin(sg);
      EGNN_TRY(launch(ln_concat_bf16_kernel, ceil_div(seg_rows * 32, 256), 256, 0, st, feats + o * s.dim,
                      reinterpret_cast<const float*>(pk + L.lng), reinterpret_cast<const float*>(pk + L.lnb), node_in + o * f.Kn,
                      f.Kn, s.dim, s.m, seg_rows, (d.flags & EGNN_FLAG_NORM_FEATS) ? 1 : 0));
      TcGemmArgs g{};
      g.A = node_in + o * f.Kn; g.lda = f.Kn; g.K = f.Kn; g.M = seg_rows; g.Nv = 2 * s.dim; g.Nout = 2 * s.dim; g.scale = 1.f; g.act = 1;
      g.W = reinterpret_cast<const __nv_bfloat16*>(pk + L.wn1); g.ldw = f.Kn;
      g.bias = reinterpret_cast<const float*>(pk + L.bn1);
      g.out = h1 + o * 2 * s.dim; g.ldo = 2 * s.dim; g.out_f32 = 0;
      EGNN_TRY(launch_tc_gemm(g, st));
      g.A = h1 + o * 2 * s.dim; g.lda = 2 * s.dim; g.K = 2 * s.dim; g.Nv = s.dim; g.Nout = s.dim; g.act = 0;
      g.W = reinterpret_cast<const __nv_bfloat16*>(pk + L.wn2); g.ldw = 2 * s.dim;
      g.bias = reinterpret_cast<const float*>(pk + L.bn2);
      g.R = feats + o * s.dim; g.ldr = s.dim;
      g.out = fout + o * s.dim; g.ldo = s.dim; g.out_f32 = 0;
      EGNN_TRY(launch_tc_gemm(g, st));
    }
  } else if (io.feats_out != io.feats) {
    for (int sg = 0; sg < nseg; ++sg)
      EGNN_CUDA_TRY(cudaMemcpyAsync(fout + seg_begin(sg) * s.dim, feats + seg_begin(sg) * s.dim, (size_t)seg_rows * s.dim * 2,
                                    cudaMemcpyDeviceToDevice, st));
  }
  if (!uc && io.coors_out != io.coors)
    for (int sg = 0; sg < nseg; ++sg)
      EGNN_CUDA_TRY(cudaMemcpyAsync(static_cast<float*>(io.coors_out) + seg_begin(sg) * s.C,
                                    static_cast<const float*>(io.coors) + seg_begin(sg) * s.C, (size_t)seg_rows * s.C * 4,
                                    cudaMemcpyDeviceToDevice, st));
  return EGNN_OK;
}

}  // namespace egnn
