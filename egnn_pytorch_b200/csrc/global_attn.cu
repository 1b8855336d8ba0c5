// GlobalLinearAttention of EGNN_Network on the device (SURVEY.md section 8(f) rank 4; reference egnn_pytorch.py:81-144,
// used between layers at :445-446): a few global tokens attend over the (masked) nodes, the nodes attend over the
// induced tokens, residuals, then a pre-norm GELU feed-forward on the nodes.  fp32 / fp64 SIMT kernels; the nine Linear
// layers go through the same tiled GEMM as the layer's per-node contractions, the two softmax cores are their own
// small kernels (scores over N nodes for T <= 32 tokens; T scores per node).
#include "common.cuh"
#include "simt_kernels.cuh"
#include "simt_host.cuh"
#include <float.h>

namespace egnn {
namespace {

template <typename T> __device__ __forceinline__ T neg_max();
template <> __device__ __forceinline__ float neg_max<float>() { return -FLT_MAX; }        // -torch.finfo(dtype).max, :102
template <> __device__ __forceinline__ double neg_max<double>() { return -DBL_MAX; }
template <typename T> __device__ __forceinline__ T exp_t(T x);
template <> __device__ __forceinline__ float exp_t<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ double exp_t<double>(double x) { return exp(x); }

// y = LayerNorm(x) * g + b, one warp per row (eps 1e-5, biased variance)
template <typename T>
__global__ void ga_layernorm_kernel(const T* __restrict__ x, const T* __restrict__ g, const T* __restrict__ b, T* __restrict__ y,
                                    int rows, int dim) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = threadIdx.x % 32;
  if (row >= rows) return;
  const T* xr = x + (size_t)row * dim;
  T s = T(0);
  for (int c = lane; c < dim; c += 32) s += xr[c];
  for (int o = 16; o > 0; o >>= 1) s += shfl_xor_t<T>(s, o);
  const T mu = s / T(dim);
  T v = T(0);
  for (int c = lane; c < dim; c += 32) { const T t = xr[c] - mu; v += t * t; }
  for (int o = 16; o > 0; o >>= 1) v += shfl_xor_t<T>(v, o);
  const T rstd = T(1) / sqrt(v / T(dim) + T(1e-5));
  for (int c = lane; c < dim; c += 32) y[(size_t)row * dim + c] = (xr[c] - mu) * rstd * g[c] + b[c];
}

// attn1 scores: S[b,h,t,n] = scale * q[b,t,h,:] . k[b,n,h,:], masked keys -> -max (:99-104).  kv rows are [k | v].
template <typename T>
__global__ void ga_scores_kernel(const T* __restrict__ q, const T* __restrict__ kv, const uint8_t* __restrict__ mask,
                                 T* __restrict__ S, int B, int N, int Tk, int heads, int dh, T scale) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)B * heads * Tk * N;
  if (idx >= total) return;
  const int n = (int)(idx % N);
  const int t = (int)((idx / N) % Tk);
  const int h = (int)((idx / ((size_t)N * Tk)) % heads);
  const int b = (int)(idx / ((size_t)N * Tk * heads));
  const int inner = heads * dh;
  const T* qp = q + ((size_t)b * Tk + t) * inner + h * dh;
  const T* kp = kv + ((size_t)b * N + n) * 2 * inner + h * dh;
  T acc = T(0);
  for (int d = 0; d < dh; ++d) acc = fma_t<T>(qp[d], kp[d], acc);
  acc *= scale;
  if (mask && !mask[(size_t)b * N + n]) acc = neg_max<T>();
  S[idx] = acc;
}

// attn1: softmax over n of S[b,h,t,:] and o[b,t,h,:] = sum_n p_n v[b,n,h,:]; one CTA per (t, h, b)
template <typename T>
__global__ void __launch_bounds__(256) ga_softmax_av_kernel(const T* __restrict__ S, const T* __restrict__ kv, T* __restrict__ o,
                                                            int N, int Tk, int heads, int dh) {
  __shared__ T red[256];
  __shared__ T stat[2];
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
  const int inner = heads * dh;
  const T* s = S + (((size_t)b * heads + h) * Tk + t) * N;
  T mx = neg_max<T>();
  for (int n = tid; n < N; n += 256) mx = s[n] > mx ? s[n] : mx;
  red[tid] = mx;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) { if (tid < w) red[tid] = red[tid + w] > red[tid] ? red[tid + w] : red[tid]; __syncthreads(); }
  if (tid == 0) stat[0] = red[0];
  __syncthreads();
  mx = stat[0];
  T sum = T(0);
  for (int n = tid; n < N; n += 256) sum += exp_t<T>(s[n] - mx);
  red[tid] = sum;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) { if (tid < w) red[tid] += red[tid + w]; __syncthreads(); }
  if (tid == 0) stat[1] = red[0];
  __syncthreads();
  const T inv = T(1) / stat[1];
  // weighted sum of the value rows: thread = (channel d, n-group); groups reduced through shared memory, fixed order
  const int groups = 256 / dh > 0 ? 256 / dh : 1;
  for (int d0 = 0; d0 < dh; d0 += 256) {
    const int d = d0 + (dh <= 256 ? tid % dh : tid), grp = dh <= 256 ? tid / dh : 0;
    T acc = T(0);
    if (d < dh && grp < groups)
      for (int n = grp; n < N; n += groups)
        acc = fma_t<T>(exp_t<T>(s[n] - mx) * inv, kv[((size_t)b * N + n) * 2 * inner + inner + h * dh + d], acc);
    red[tid] = acc;
    __syncthreads();
    if (d < dh && grp == 0) {
      T tot = T(0);
      for (int gq = 0; gq < groups; ++gq) tot += red[gq * dh + (d - d0)];
      o[((size_t)b * Tk + t) * inner + h * dh + d] = tot;
    }
    __syncthreads();
  }
}

// attn2: per (b, n, h): Tk scores against the induced tokens, softmax over them (no mask, :137), weighted value sum.
// One warp per (b, n, h); lanes stride the head channels.
template <typename T>
__global__ void ga_attn2_kernel(const T* __restrict__ q, const T* __restrict__ kv, T* __restrict__ o, int B, int N, int Tk,
                                int heads, int dh, T scale) {
  const size_t wid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (wid >= (size_t)B * N * heads) return;
  const int h = (int)(wid % heads);
  const size_t bn = wid / heads;
  const int b = (int)(bn / N);
  const int inner = heads * dh;
  const T* qp = q + bn * inner + h * dh;
  T sc[32];
  T mx = neg_max<T>();
  for (int t = 0; t < Tk; ++t) {
    const T* kp = kv + ((size_t)b * Tk + t) * 2 * inner + h * dh;
    T acc = T(0);
    for (int d = lane; d < dh; d += 32) acc = fma_t<T>(qp[d], kp[d], acc);
    for (int off = 16; off > 0; off >>= 1) acc += shfl_xor_t<T>(acc, off);
    sc[t] = acc * scale;
    mx = sc[t] > mx ? sc[t] : mx;
  }
  T sum = T(0);
  for (int t = 0; t < Tk; ++t) { sc[t] = exp_t<T>(sc[t] - mx); sum += sc[t]; }
  const T inv = T(1) / sum;
  for (int d = lane; d < dh; d += 32) {
    T acc = T(0);
    for (int t = 0; t < Tk; ++t) acc = fma_t<T>(sc[t] * inv, kv[((size_t)b * Tk + t) * 2 * inner + inner + h * dh + d], acc);
    o[bn * inner + h * dh + d] = acc;
  }
}

template <typename T>
__global__ void ga_add_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}

struct GaWs { size_t xn, qn, q1, kv1, S, o1, induced, q2, kv2, o2, x1, hff, total; };
GaWs ga_layout(const EgnnGlobalAttnDesc& d, size_t es) {
  GaWs w;
  BumpAlloc o;
  auto take = [&](size_t elems) { return o.take(elems * es); };
  const size_t BN = (size_t)d.B * d.N, BT = (size_t)d.B * d.T, inner = (size_t)d.heads * d.dim_head;
  w.xn = take(BN * d.dim); w.qn = take(BT * d.dim); w.q1 = take(BT * inner); w.kv1 = take(BN * 2 * inner);
  w.S = take((size_t)d.B * d.heads * d.T * d.N); w.o1 = take(BT * inner); w.induced = take(BT * d.dim);
  w.q2 = take(BN * inner); w.kv2 = take(BT * 2 * inner); w.o2 = take(BN * inner); w.x1 = take(BN * d.dim);
  w.hff = take(BN * 4 * d.dim);
  w.total = o.total;
  return w;
}

int ga_validate(const EgnnGlobalAttnDesc* d) {
  if (!d) return EGNN_ERR_NULL;
  if (d->abi_version != EGNN_ABI_VERSION) return EGNN_ERR_ABI;
  if (d->dtype != EGNN_DTYPE_F32 && d->dtype != EGNN_DTYPE_F64) return EGNN_ERR_UNSUPPORTED;
  if (d->B <= 0 || d->N <= 0 || d->T <= 0 || d->dim <= 0 || d->heads <= 0 || d->dim_head <= 0) return EGNN_ERR_SHAPE;
  if (d->T > 32) return EGNN_ERR_UNSUPPORTED;
  if (d->B > 65535 || d->heads > 65535) return EGNN_ERR_SHAPE;
  return EGNN_OK;
}

template <typename T>
int ga_forward(const EgnnGlobalAttnDesc& d, const EgnnGlobalAttnWeights& w, const EgnnGlobalAttnIO& io, void* ws, cudaStream_t st) {
  const GaWs L = ga_layout(d, sizeof(T));
  char* base = static_cast<char*>(ws);
  auto P = [&](size_t off) { return reinterpret_cast<T*>(base + off); };
  auto W = [](const void* p) { return static_cast<const T*>(p); };
  const int BN = d.B * d.N, BT = d.B * d.T, inner = d.heads * d.dim_head, dim = d.dim;
  const T scale = T(1) / sqrt(T(d.dim_head));                                     // dim_head ** -0.5, :86
  const T* x = W(io.x);
  const T* qs = W(io.queries);
  const RowMap idn{BN, BN, 0}, idt{BT, BT, 0};
  // x, queries = norm_seq(x), norm_queries(queries)                              :134
  EGNN_TRY(launch(ga_layernorm_kernel<T>, ceil_div(BN * 32, 256), 256, 0, st, x, W(w.norm_seq_g), W(w.norm_seq_b), P(L.xn), BN, dim));
  EGNN_TRY(launch(ga_layernorm_kernel<T>, ceil_div(BT * 32, 256), 256, 0, st, qs, W(w.norm_q_g), W(w.norm_q_b), P(L.qn), BT, dim));
  // induced = attn1(queries, x, mask)                                            :136
  EGNN_TRY((launch_gemm<T, 0, false>(P(L.qn), dim, W(w.a1_wq), dim, nullptr, nullptr, 0, P(L.q1), inner, BT, inner, inner, dim, idt, st)));
  EGNN_TRY((launch_gemm<T, 0, false>(P(L.xn), dim, W(w.a1_wkv), dim, nullptr, nullptr, 0, P(L.kv1), 2 * inner, BN, 2 * inner, 2 * inner, dim, idn, st)));
  const size_t scores = (size_t)d.B * d.heads * d.T * d.N;
  EGNN_TRY(launch(ga_scores_kernel<T>, (unsigned)((scores + 255) / 256), 256, 0, st, P(L.q1), P(L.kv1), io.mask, P(L.S), d.B, d.N, d.T,
                  d.heads, d.dim_head, scale));
  EGNN_TRY(launch(ga_softmax_av_kernel<T>, dim3(d.T, d.heads, d.B), 256, 0, st, P(L.S), P(L.kv1), P(L.o1), d.N, d.T, d.heads, d.dim_head));
  EGNN_TRY((launch_gemm<T, 0, false>(P(L.o1), inner, W(w.a1_wo), inner, W(w.a1_bo), nullptr, 0, P(L.induced), dim, BT, dim, dim, inner, idt, st)));
  // out = attn2(x, induced);  x = out + res_x                                     :137, :139
  EGNN_TRY((launch_gemm<T, 0, false>(P(L.xn), dim, W(w.a2_wq), dim, nullptr, nullptr, 0, P(L.q2), inner, BN, inner, inner, dim, idn, st)));
  EGNN_TRY((launch_gemm<T, 0, false>(P(L.induced), dim, W(w.a2_wkv), dim, nullptr, nullptr, 0, P(L.kv2), 2 * inner, BT, 2 * inner, 2 * inner, dim, idt, st)));
  const size_t warps = (size_t)BN * d.heads;
  EGNN_TRY(launch(ga_attn2_kernel<T>, (unsigned)((warps * 32 + 255) / 256), 256, 0, st, P(L.q2), P(L.kv2), P(L.o2), d.B, d.N, d.T, d.heads,
                  d.dim_head, scale));
  EGNN_TRY((launch_gemm<T, 0, true>(P(L.o2), inner, W(w.a2_wo), inner, W(w.a2_bo), x, dim, P(L.x1), dim, BN, dim, dim, inner, idn, st)));
  // queries = induced + res_queries                                              :140
  EGNN_TRY(launch(ga_add_kernel<T>, ceil_div(BT * dim, 256), 256, 0, st, P(L.induced), qs, static_cast<T*>(io.queries_out), (size_t)BT * dim));
  // x = ff(x) + x                                                                :142
  EGNN_TRY(launch(ga_layernorm_kernel<T>, ceil_div(BN * 32, 256), 256, 0, st, P(L.x1), W(w.ff_ln_g), W(w.ff_ln_b), P(L.xn), BN, dim));
  EGNN_TRY((launch_gemm<T, 2, false>(P(L.xn), dim, W(w.ff_w1), dim, W(w.ff_b1), nullptr, 0, P(L.hff), 4 * dim, BN, 4 * dim, 4 * dim, dim, idn, st)));
  EGNN_TRY((launch_gemm<T, 0, true>(P(L.hff), 4 * dim, W(w.ff_w2), 4 * dim, W(w.ff_b2), P(L.x1), dim, static_cast<T*>(io.x_out), dim, BN, dim, dim,
                                    4 * dim, idn, st)));
  return EGNN_OK;
}

}  // namespace
}  // namespace egnn

extern "C" int egnn_global_attn_workspace_bytes(const EgnnGlobalAttnDesc* d, size_t* out) {
  EGNN_TRY(egnn::ga_validate(d));
  if (!out) return EGNN_ERR_NULL;
  *out = egnn::ga_layout(*d, d->dtype == EGNN_DTYPE_F64 ? 8 : 4).total + 256;
  return EGNN_OK;
}

extern "C" int egnn_global_attn_forward(const EgnnGlobalAttnDesc* d, const EgnnGlobalAttnWeights* w, const EgnnGlobalAttnIO* io,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  EGNN_TRY(egnn::ga_validate(d));
  if (!w || !io || !workspace || !io->x || !io->queries || !io->x_out || !io->queries_out) return EGNN_ERR_NULL;
  const void* const* wp = reinterpret_cast<const void* const*>(w);
  for (size_t i = 0; i < sizeof(EgnnGlobalAttnWeights) / sizeof(void*); ++i)
    if (!wp[i]) return EGNN_ERR_NULL;
  if (workspace_bytes < egnn::ga_layout(*d, d->dtype == EGNN_DTYPE_F64 ? 8 : 4).total) return EGNN_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return d->dtype == EGNN_DTYPE_F64 ? egnn::ga_forward<double>(*d, *w, *io, workspace, st)
                                    : egnn::ga_forward<float>(*d, *w, *io, workspace, st);
}
