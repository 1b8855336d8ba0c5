// N-th degree adjacency of EGNN_Network (reference egnn_pytorch.py:414-428) on bit-packed rows.
//
// The reference squares the dense float adjacency (`adj.float() @ adj.float() > 0`, :425), an
// O(N^3) bmm that is 37 % of its CPU time at N=8192 (SURVEY.md section 3.2).  Here a row of the
// next adjacency is the OR of the current rows of its neighbours:
//     next[i] = OR_{j : adj[i][j]} adj[j]            (boolean matrix square)
//     newly   = next XOR adj   -> labels := degree   (:426-427: "(next.float() - adj.float()).bool()")
//     adj     = next                                 (:428; the EXPANDED matrix is squared again)
#include "launch.cuh"

namespace egnn {

__global__ void adj_pack_kernel(const uint8_t* __restrict__ adj_in, int adj_batched, int B, int N, int W,
                                uint32_t* __restrict__ bits, uint8_t* __restrict__ labels) {
  // one warp per (row, word)
  const size_t gw = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (gw >= (size_t)B * N * W) return;
  const int w = (int)(gw % W);
  const size_t row = gw / W;                  // b*N + i
  const int b = (int)(row / N), i = (int)(row % N);
  const int j = w * 32 + lane;
  uint8_t v = 0;
  if (j < N) {
    v = adj_in[((size_t)(adj_batched ? b : 0) * N + i) * N + j] ? 1 : 0;
    labels[row * N + j] = v;                  // :420 adj_indices = adj.long()
  }
  const unsigned word = __ballot_sync(0xffffffffu, v != 0);
  if (lane == 0) bits[row * W + w] = word;
}

// one block per row (b, i)
__global__ void __launch_bounds__(128)
adj_square_kernel(const uint32_t* __restrict__ bin, uint32_t* __restrict__ bout, uint8_t* __restrict__ labels,
                  int N, int W, int degree) {
  extern __shared__ int nbrs[];               // neighbour list of this row (at most N entries)
  __shared__ int n_nbrs;
  const size_t row = blockIdx.x;
  const int b = (int)(row / N);
  const uint32_t* myrow = bin + row * W;
  if (threadIdx.x == 0) n_nbrs = 0;
  __syncthreads();
  for (int w = threadIdx.x; w < W; w += blockDim.x) {
    uint32_t word = myrow[w];
    if (word) {
      int base = atomicAdd(&n_nbrs, __popc(word));
      while (word) {
        int bit = __ffs(word) - 1;
        word &= word - 1;
        nbrs[base++] = w * 32 + bit;
      }
    }
  }
  __syncthreads();
  const int cnt = n_nbrs;
  for (int w = threadIdx.x; w < W; w += blockDim.x) {
    uint32_t acc = 0;
    for (int t = 0; t < cnt; ++t) acc |= bin[((size_t)b * N + nbrs[t]) * W + w];
    uint32_t newly = acc ^ myrow[w];
    bout[row * W + w] = acc;
    while (newly) {
      int bit = __ffs(newly) - 1;
      newly &= newly - 1;
      labels[row * N + w * 32 + bit] = (uint8_t)degree;
    }
  }
}

__global__ void adj_unpack_kernel(const uint32_t* __restrict__ bits, int B, int N, int W,
                                  uint8_t* __restrict__ adj_out, int32_t* __restrict__ max_row_sum) {
  const size_t gw = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (gw >= (size_t)B * N) return;
  const size_t row = gw;
  int cnt = 0;
  for (int w = 0; w < W; ++w) {
    const uint32_t word = bits[row * W + w];
    cnt += __popc(word);
    const int j = w * 32 + lane;
    if (j < N) adj_out[row * N + j] = (word >> lane) & 1u;
  }
  if (lane == 0 && max_row_sum) atomicMax(max_row_sum, cnt);
}

}  // namespace egnn

extern "C" int egnn_adj_workspace_bytes(int32_t B, int32_t N, size_t* out_bytes) {
  if (!out_bytes) return EGNN_ERR_NULL;
  if (B <= 0 || N <= 0) return EGNN_ERR_SHAPE;
  const size_t W = (size_t)egnn::ceil_div(N, 32);
  *out_bytes = 2 * egnn::round_up((size_t)B * N * W * 4, 256);
  return EGNN_OK;
}

extern "C" int egnn_adj_expand(int32_t B, int32_t N, int32_t num_degrees, const uint8_t* adj_in,
                               int32_t adj_batched, uint8_t* adj_out, uint8_t* labels_out,
                               int32_t* max_row_sum, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace egnn;
  if (!adj_in || !adj_out || !labels_out || !workspace) return EGNN_ERR_NULL;
  if (B <= 0 || N <= 0 || num_degrees < 1 || num_degrees > 255) return EGNN_ERR_SHAPE;
  size_t need = 0;
  EGNN_TRY(egnn_adj_workspace_bytes(B, N, &need));
  if (workspace_bytes < need) return EGNN_ERR_WORKSPACE;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int W = ceil_div(N, 32);
  uint32_t* b0 = static_cast<uint32_t*>(workspace);
  uint32_t* b1 = reinterpret_cast<uint32_t*>(static_cast<char*>(workspace) + need / 2);
  const size_t warps = (size_t)B * N * W;
  EGNN_TRY(launch(adj_pack_kernel, (unsigned)((warps * 32 + 255) / 256), 256, 0, st, adj_in, adj_batched, B, N, W, b0, labels_out));
  const size_t nb_smem = (size_t)N * sizeof(int);
  if (nb_smem > 200 * 1024) return EGNN_ERR_UNSUPPORTED;
  for (int degree = 2; degree <= num_degrees; ++degree) {
    EGNN_TRY(launch(adj_square_kernel, B * N, 128, nb_smem, st, b0, b1, labels_out, N, W, degree));
    uint32_t* t = b0; b0 = b1; b1 = t;
  }
  if (max_row_sum) EGNN_CUDA_TRY(cudaMemsetAsync(max_row_sum, 0, sizeof(int32_t), st));
  return launch(adj_unpack_kernel, (unsigned)(((size_t)B * N * 32 + 255) / 256), 256, 0, st, b0, B, N, W, adj_out, max_row_sum);
}

// ------------------------------------------------------------------------------------------------------------------
// Node embedding of EGNN_Network (reference egnn_pytorch.py:401-408) in one launch:
//     feats[b, n, :] = token_emb[tokens[b, n], :] (+ pos_emb[n, :])
// (the reference runs nn.Embedding, an arange + nn.Embedding for the positions and an in-place add).  Element type T for
// tables and output; tokens int64.  One warp per node row.
namespace egnn {
template <typename T>
__global__ void embed_nodes_kernel(const int64_t* __restrict__ tokens, const T* __restrict__ tok_emb, const T* __restrict__ pos_emb,
                                   T* __restrict__ out, int B, int N, int dim, int num_tokens) {
  const size_t row = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (row >= (size_t)B * N) return;
  const int n = (int)(row % N);
  long long t = tokens[row];
  t = t < 0 ? 0 : (t >= num_tokens ? num_tokens - 1 : t);            // nn.Embedding would raise; never read out of bounds
  const T* te = tok_emb + (size_t)t * dim;
  const T* pe = pos_emb ? pos_emb + (size_t)n * dim : nullptr;
  for (int c = lane; c < dim; c += 32) {
    if constexpr (sizeof(T) == 2) {
      const float v = __bfloat162float(te[c]) + (pe ? __bfloat162float(pe[c]) : 0.f);     // one rounding, like bf16 add
      out[row * dim + c] = __float2bfloat16(v);
    } else {
      out[row * dim + c] = te[c] + (pe ? pe[c] : T(0));
    }
  }
}
}  // namespace egnn

extern "C" int egnn_embed_nodes(int32_t dtype, int32_t B, int32_t N, int32_t dim, int32_t num_tokens, const int64_t* tokens,
                                const void* token_emb, const void* pos_emb, void* out, void* stream) {
  if (!tokens || !token_emb || !out) return EGNN_ERR_NULL;
  if (B <= 0 || N <= 0 || dim <= 0 || num_tokens <= 0) return EGNN_ERR_SHAPE;
  const unsigned grid = (unsigned)(((size_t)B * N * 32 + 255) / 256);
  auto run = [&](auto elem) {
    using T = decltype(elem);
    return egnn::launch(egnn::embed_nodes_kernel<T>, grid, 256, 0, static_cast<cudaStream_t>(stream), tokens,
                        static_cast<const T*>(token_emb), static_cast<const T*>(pos_emb), static_cast<T*>(out), B, N, dim, num_tokens);
  };
  if (dtype == EGNN_DTYPE_F64) return run(double{});
  if (dtype == EGNN_DTYPE_F32) return run(float{});
  return run(__nv_bfloat16{});
}
