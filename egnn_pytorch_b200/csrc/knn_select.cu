// Neighbour ranking + top-k select fused into the distance pass
// (reference egnn_pytorch.py:232-233 all-pairs distance, :237-260 ranking and topk).
//
//   rank(i,j) = ||x_i - x_j||^2
//             = 1e5   if a mask is given and either end is padded            (:240-242)
//             = -1    if an adjacency is given and i == j                      (:255)
//             = 0     if an adjacency is given and adj[i,j], i != j            (:256)
//   keep the k smallest (rank, j) pairs in ascending lexicographic order -> deterministic
//   "lowest index wins" tie rule (torch.topk leaves ties unspecified).
//
// k <= 32: one warp per row keeps the running top-32 sorted across its lanes; candidates that
// beat the current k-th entry are queued in shared memory and merged 32 at a time with a
// warp-bitonic sort + merge, so the O(N^2) ranking matrix is never written.
// k  > 32: one block per row sorts all N (rank, j) pairs in shared memory (bitonic).
#include "knn_select.h"
#include "launch.cuh"

namespace egnn {

template <typename T>
struct SelArgs {
  int B, N, C, k;
  const T* coors;
  const uint8_t* mask;
  const uint8_t* adj;
  int adj_batched;
  T valid_radius;
  int32_t* out_idx;
  uint8_t* out_ok;
};

template <typename T>
__device__ __forceinline__ T rank_of(const SelArgs<T>& a, int b, int i, int j, const T* xi, bool mask_i) {
  const T* xj = a.coors + ((size_t)b * a.N + j) * a.C;
  T d = T(0);
  for (int c = 0; c < a.C; ++c) d = sq_acc<T>(xi[c] - xj[c], d);
  if (a.mask && !(mask_i && a.mask[(size_t)b * a.N + j])) d = T(1e5);
  if (a.adj) {
    if (i == j) d = T(-1);
    else if (a.adj[((size_t)(a.adj_batched ? b : 0) * a.N + i) * a.N + j]) d = T(0);
  }
  return d;
}

template <typename T>
__device__ __forceinline__ bool lex_less(T ka, int ia, T kb, int ib) {
  return ka < kb || (ka == kb && ia < ib);
}

// One compare-exchange step of a warp bitonic network on (key, idx) pairs.
template <typename T>
__device__ __forceinline__ void cmpex(T& key, int& idx, int lane, int partner_xor, bool ascending_block) {
  T ok = shfl_xor_t<T>(key, partner_xor);
  int oi = __shfl_xor_sync(0xffffffffu, idx, partner_xor);
  const bool lower = (lane & partner_xor) == 0;
  const bool other_less = lex_less<T>(ok, oi, key, idx);
  // in an ascending block the lower lane keeps the min
  const bool take_other = (lower == ascending_block) ? other_less : !other_less && !(ok == key && oi == idx);
  if (take_other) { key = ok; idx = oi; }
}

template <typename T>
__device__ __forceinline__ void warp_sort_asc(T& key, int& idx, int lane) {
#pragma unroll
  for (int size = 2; size <= 32; size <<= 1) {
    const bool asc = (lane & size) == 0 || size == 32;
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) cmpex<T>(key, idx, lane, stride, asc);
  }
}

// best (sorted ascending across lanes) <- the 32 smallest of best U cand.
template <typename T>
__device__ __forceinline__ void warp_merge(T& bkey, int& bidx, T ckey, int cidx, int lane) {
  warp_sort_asc<T>(ckey, cidx, lane);
  // reverse the candidates so that best ++ reversed(cand) is bitonic; lane l meets cand[31-l]
  T rk = shfl_idx_t<T>(ckey, 31 - lane);
  int ri = __shfl_sync(0xffffffffu, cidx, 31 - lane);
  if (lex_less<T>(rk, ri, bkey, bidx)) { bkey = rk; bidx = ri; }
  // the kept 32 form a bitonic sequence: finish with the 5 merge steps
#pragma unroll
  for (int stride = 16; stride > 0; stride >>= 1) cmpex<T>(bkey, bidx, lane, stride, true);
}

constexpr int SEL_WARPS_MAX = 16;   // rows per CTA (one warp each, all of the same graph): 16, or 8 for grids that would not fill the GPU
constexpr int SEL_JC = 1024;        // candidates staged per pass: coordinates as SoA + mask bytes in shared memory

template <typename T>
inline size_t sel_smem_bytes(int C, int warps = SEL_WARPS_MAX) {
  return (size_t)C * SEL_JC * sizeof(T) + SEL_JC + (size_t)warps * 64 * (sizeof(T) + sizeof(int)) + 64;
}

// CDIM = 3: the coordinate loops are exactly three steps (the generic instantiation, CDIM = 0, issues all eight predicated
// steps per candidate -- 125 instead of ~55 instructions per trip of the scan, which is 63 % of the kernel; ncu source page)
template <typename T, int SEL_WARPS, int CDIM>
__global__ void __launch_bounds__(SEL_WARPS * 32)
knn_warp_select_kernel(const SelArgs<T> a) {
  constexpr int NC = CDIM ? CDIM : 8;
  extern __shared__ __align__(16) unsigned char sel_sm[];
  T* xs = reinterpret_cast<T*>(sel_sm);                                   // [C][JC]
  T* qkey = xs + (size_t)a.C * SEL_JC;                                    // [WARPS][64]
  int* qidx = reinterpret_cast<int*>(qkey + SEL_WARPS * 64);              // [WARPS][64]
  uint8_t* ms = reinterpret_cast<uint8_t*>(qidx + SEL_WARPS * 64);        // [JC]
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int b = blockIdx.y;
  const int iraw = blockIdx.x * SEL_WARPS + warp;
  const bool rv = iraw < a.N;
  const int i = rv ? iraw : a.N - 1;
  const size_t row = (size_t)b * a.N + i;
  T xi[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) xi[c] = (CDIM || c < a.C) ? a.coors[row * a.C + c] : T(0);
  const bool mask_i = a.mask ? a.mask[row] != 0 : true;
  const uint8_t* adjrow = a.adj ? a.adj + ((size_t)(a.adj_batched ? b : 0) * a.N + i) * a.N : nullptr;
  const T INF = T(INFINITY);
  const int IMAX = 0x7fffffff;
  T* myqk = qkey + warp * 64;
  int* myqi = qidx + warp * 64;

  T bkey = INF; int bidx = IMAX;       // lane l: l-th smallest so far
  T thr_key = INF; int thr_idx = IMAX; // the k-th smallest so far
  int count = 0;                       // queued candidates (warp-uniform)

  for (int jc0 = 0; jc0 < a.N; jc0 += SEL_JC) {
    const int jn = min(SEL_JC, a.N - jc0);
    __syncthreads();                   // previous pass fully consumed
    for (int jj = threadIdx.x; jj < jn; jj += SEL_WARPS * 32) {          // one candidate per thread: no index division
      const T* src = a.coors + ((size_t)b * a.N + jc0 + jj) * a.C;
#pragma unroll
      for (int c = 0; c < NC; ++c)
        if (CDIM || c < a.C) xs[c * SEL_JC + jj] = src[c];
      if (a.mask) ms[jj] = a.mask[(size_t)b * a.N + jc0 + jj];
    }
    __syncthreads();

    // two groups of 32 candidates per trip: their distance chains overlap; each group is then filtered against the
    // current k-th entry and queued (the second group may see a threshold one merge old -- it only queues a few more)
    for (int j0 = 0; j0 < jn; j0 += 64) {
      T key[2];
      bool pass[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int jj = j0 + 32 * u + lane, j = jc0 + jj;
        const bool jvalid = jj < jn;
        key[u] = INF;
        if (jvalid) {
          T d = T(0);
#pragma unroll
          for (int c = 0; c < NC; ++c)
            if (CDIM || c < a.C) d = sq_acc<T>(xi[c] - xs[c * SEL_JC + jj], d);
          if (a.mask && !(mask_i && ms[jj])) d = T(1e5);
          if (adjrow) {
            if (i == j) d = T(-1);
            else if (adjrow[j]) d = T(0);
          }
          key[u] = d;
        }
        pass[u] = jvalid && lex_less<T>(key[u], j, thr_key, thr_idx);
      }
      if (!__any_sync(0xffffffffu, pass[0] || pass[1])) continue;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const unsigned bal = __ballot_sync(0xffffffffu, pass[u]);
        if (bal == 0) continue;
        if (pass[u]) {
          const int pos = count + __popc(bal & ((1u << lane) - 1));
          myqk[pos] = key[u];
          myqi[pos] = jc0 + j0 + 32 * u + lane;
        }
        count += __popc(bal);
        __syncwarp();
        if (count >= 32) {
          T ckey = myqk[lane];
          int cidx = myqi[lane];
          __syncwarp();
          if (lane + 32 < count) {         // shift the tail of the queue down
            T tk = myqk[lane + 32]; int ti = myqi[lane + 32];
            myqk[lane] = tk; myqi[lane] = ti;
          }
          count -= 32;
          __syncwarp();
          warp_merge<T>(bkey, bidx, ckey, cidx, lane);
          thr_key = shfl_idx_t<T>(bkey, a.k - 1);
          thr_idx = __shfl_sync(0xffffffffu, bidx, a.k - 1);
        }
      }
    }
  }
  if (count > 0) {
    T ckey = lane < count ? myqk[lane] : INF;
    int cidx = lane < count ? myqi[lane] : IMAX;
    warp_merge<T>(bkey, bidx, ckey, cidx, lane);
  }
  if (rv && lane < a.k) {
    const size_t o = row * a.k + lane;
    a.out_idx[o] = bidx;
    if (a.out_ok) a.out_ok[o] = bkey <= a.valid_radius ? 1 : 0;
  }
}

// k > 32: block-wide bitonic sort of all N candidates in shared memory.
template <typename T>
__global__ void __launch_bounds__(256)
knn_block_sort_kernel(const SelArgs<T> a, int Npad) {
  extern __shared__ __align__(16) unsigned char sel_smem[];
  T* keys = reinterpret_cast<T*>(sel_smem);
  int* idxs = reinterpret_cast<int*>(keys + Npad);
  const int row = blockIdx.x;
  const int b = row / a.N, i = row % a.N;
  const T* xi = a.coors + (size_t)row * a.C;
  const bool mask_i = a.mask ? a.mask[row] != 0 : true;
  for (int j = threadIdx.x; j < Npad; j += blockDim.x) {
    keys[j] = j < a.N ? rank_of<T>(a, b, i, j, xi, mask_i) : T(INFINITY);
    idxs[j] = j < a.N ? j : 0x7fffffff;
  }
  __syncthreads();
  for (int size = 2; size <= Npad; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < Npad / 2; t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));     // index with the `stride` bit clear
        const int hi = lo + stride;
        const bool asc = (lo & size) == 0;
        const bool hi_less = lex_less<T>(keys[hi], idxs[hi], keys[lo], idxs[lo]);
        if (hi_less == asc) {
          T tk = keys[lo]; keys[lo] = keys[hi]; keys[hi] = tk;
          int ti = idxs[lo]; idxs[lo] = idxs[hi]; idxs[hi] = ti;
        }
      }
      __syncthreads();
    }
  }
  for (int s = threadIdx.x; s < a.k; s += blockDim.x) {
    const size_t o = (size_t)row * a.k + s;
    a.out_idx[o] = idxs[s];
    if (a.out_ok) a.out_ok[o] = keys[s] <= a.valid_radius ? 1 : 0;
  }
}

template <typename T>
static int launch_select(int B, int N, int C, int k, const void* coors, const uint8_t* mask, const uint8_t* adj,
                         int adj_batched, double valid_radius, int32_t* out_idx, uint8_t* out_ok, cudaStream_t st) {
  SelArgs<T> a;
  a.B = B; a.N = N; a.C = C; a.k = k;
  a.coors = static_cast<const T*>(coors);
  a.mask = mask; a.adj = adj; a.adj_batched = adj_batched;
  a.valid_radius = (T)valid_radius;
  a.out_idx = out_idx; a.out_ok = out_ok;
  if (k <= 32) {
    // 16 rows per CTA halve the staging work per row; small problems keep 8 so that more SMs take part
    const bool wide = (long)B * ceil_div(N, 16) >= 296;
    const int warps = wide ? 16 : 8;
    auto kernel = C == 3 ? (wide ? knn_warp_select_kernel<T, 16, 3> : knn_warp_select_kernel<T, 8, 3>)
                         : (wide ? knn_warp_select_kernel<T, 16, 0> : knn_warp_select_kernel<T, 8, 0>);
    return launch(kernel, dim3(ceil_div(N, warps), B), warps * 32, sel_smem_bytes<T>(C, warps), st, a);
  }
  int Npad = 1;
  while (Npad < N) Npad <<= 1;
  const size_t smem = (size_t)Npad * (sizeof(T) + sizeof(int));
  if (smem > 200 * 1024) return EGNN_ERR_UNSUPPORTED;     // N too large for the k>32 path
  return launch(knn_block_sort_kernel<T>, B * N, 256, smem, st, a, Npad);
}

static int knn_select_dispatch(int32_t dtype, int B, int N, int C, int k, const void* coors, const uint8_t* mask,
                               const uint8_t* adj, int adj_batched, double valid_radius, int32_t* out_idx,
                               uint8_t* out_ok, cudaStream_t st) {
  if (!coors || !out_idx) return EGNN_ERR_NULL;
  if (B <= 0 || B > 65535 || N <= 0 || C <= 0 || C > 8 || k <= 0 || k > N) return EGNN_ERR_SHAPE;
  if (dtype == EGNN_DTYPE_F64)
    return launch_select<double>(B, N, C, k, coors, mask, adj, adj_batched, valid_radius, out_idx, out_ok, st);
  return launch_select<float>(B, N, C, k, coors, mask, adj, adj_batched, valid_radius, out_idx, out_ok, st);
}

// only_sparse_neighbors WITH a node mask (egnn_pytorch.py:249-260, :296): valid_radius is 0, so the only slots whose
// pair mask can be true are the node itself (rank -1) and its adjacent nodes (rank 0, ties to the lowest index) --
// whatever top-k fills the remaining slots with is masked out (nbhd_mask = rank <= 0).  Those lists need no distance
// ranking at all: one warp scans the node's adjacency row in index order.  Slot 0 = self, then the adjacent nodes
// ascending (exactly the top-k order of the valid slots, truncated at k like top-k); unused slots point at the node
// itself with ok = 0.  Replaces an O(N^2) ranking pass (295 us per layer at N = 8192, BASELINE config 5) by a row scan.
__global__ void __launch_bounds__(256) adj_neighbors_kernel(int B, int N, int k, const uint8_t* __restrict__ adj, int adj_batched,
                                                            int32_t* __restrict__ out_idx, uint8_t* __restrict__ out_ok) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = threadIdx.x % 32;
  if (row >= B * N) return;
  const int b = row / N, i = row % N;
  const uint8_t* a = adj + ((size_t)(adj_batched ? b : 0) * N + i) * N;
  int32_t* oi = out_idx + (size_t)row * k;
  uint8_t* ok = out_ok ? out_ok + (size_t)row * k : nullptr;
  if (lane == 0) { oi[0] = i; if (ok) ok[0] = 1; }
  int pos = 1;
  const bool wide = (N % 4 == 0) && ((reinterpret_cast<uintptr_t>(adj) & 3) == 0);
  if (wide) {
    const uint32_t* a4 = reinterpret_cast<const uint32_t*>(a);
    for (int j0 = 0; j0 < N && pos < k; j0 += 128) {
      const int j = j0 + lane * 4;
      uint32_t w = j < N ? __ldg(a4 + j / 4) : 0u;
      // clear the node's own entry; count and place this lane's up to four hits
      uint32_t bits = 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) if (((w >> (8 * t)) & 0xffu) && j + t != i) bits |= 1u << t;
      const int cnt = __popc(bits);
      int pre = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, pre, o); if (lane >= o) pre += v; }
      const int total = __shfl_sync(0xffffffffu, pre, 31);
      int p = pos + pre - cnt;
#pragma unroll
      for (int t = 0; t < 4; ++t)
        if (bits & (1u << t)) { if (p < k) { oi[p] = j + t; if (ok) ok[p] = 1; } ++p; }
      pos += total;
    }
  } else {
    for (int j0 = 0; j0 < N && pos < k; j0 += 32) {
      const int j = j0 + lane;
      const bool hit = j < N && a[j] != 0 && j != i;
      const uint32_t m = __ballot_sync(0xffffffffu, hit);
      const int p = pos + __popc(m & ((1u << lane) - 1u));
      if (hit && p < k) { oi[p] = j; if (ok) ok[p] = 1; }
      pos += __popc(m);
    }
  }
  pos = pos < k ? pos : k;
  // unused slots: the node itself with ok = 0, or -1 (the edge-list convention of EgnnLayerIO.nbr_idx) when no ok array is kept
  for (int p = pos + lane; p < k; p += 32) { oi[p] = ok ? i : -1; if (ok) ok[p] = 0; }
}

static int adj_neighbors_dispatch(int B, int N, int k, const uint8_t* adj, int adj_batched, int32_t* out_idx,
                                  uint8_t* out_ok, cudaStream_t st) {
  if (!adj || !out_idx) return EGNN_ERR_NULL;
  if (B <= 0 || N <= 0 || k <= 0 || k > N) return EGNN_ERR_SHAPE;
  const long long threads = (long long)B * N * 32;
  return launch(adj_neighbors_kernel, (unsigned)((threads + 255) / 256), 256, 0, st, B, N, k, adj, adj_batched, out_idx, out_ok);
}

int select_neighbours(const EgnnLayerDesc& d, const Dims& s, const EgnnLayerIO& io, int32_t coors_dtype, int32_t*& idx,
                      uint8_t*& ok, cudaStream_t st) {
  if (io.nbr_idx) {                                  // edge-list mode: the caller's lists, no ranking
    idx = const_cast<int32_t*>(io.nbr_idx);
    ok = nullptr;
    return EGNN_OK;
  }
  StageTimer tm(st, STAGE_SELECT);
  const int adj_batched = (d.flags & EGNN_FLAG_ADJ_BATCHED) ? 1 : 0;
  if ((d.flags & EGNN_FLAG_ONLY_SPARSE) && io.mask && io.adj)      // every slot top-k could add is masked out: row scan
    return adj_neighbors_dispatch(s.B, s.N, s.k, io.adj, adj_batched, idx, ok, st);
  const double vr = (d.flags & EGNN_FLAG_ONLY_SPARSE) ? 0.0 : d.valid_radius;     // :250
  return knn_select_dispatch(coors_dtype, s.B, s.N, s.C, s.k, io.coors, io.mask, io.adj, adj_batched, vr, idx, ok, st);
}

}  // namespace egnn

extern "C" int egnn_knn_select(int32_t dtype, int32_t B, int32_t N, int32_t C, int32_t k, const void* coors,
                               const uint8_t* mask, const uint8_t* adj, int32_t adj_batched,
                               double valid_radius, int32_t* out_idx, uint8_t* out_ok, void* stream) {
  return egnn::knn_select_dispatch(dtype, B, N, C, k, coors, mask, adj, adj_batched, valid_radius, out_idx,
                                   out_ok, static_cast<cudaStream_t>(stream));
}

extern "C" int egnn_adj_neighbors(int32_t B, int32_t N, int32_t k, const uint8_t* adj, int32_t adj_batched, int32_t* out_idx,
                                  uint8_t* out_ok, void* stream) {
  return egnn::adj_neighbors_dispatch(B, N, k, adj, adj_batched, out_idx, out_ok, static_cast<cudaStream_t>(stream));
}
