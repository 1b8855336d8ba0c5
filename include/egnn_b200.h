/*
 * egnn_b200.h -- C ABI of libegnn_b200.so, the B200 (sm_100a) implementation of the
 * E(n)-equivariant message-passing layer of lucidrains/egnn-pytorch.
 *
 * The reference has no FFI: its boundary is the Python nn.Module API
 * (reference egnn_pytorch/__init__.py:1, EGNN.forward egnn_pytorch/egnn_pytorch.py:224-341,
 * EGNN_Network.forward :390-454).  This header is the boundary a binding for that path
 * would target; `egnn_pytorch_b200/egnn.py` is such a binding (ctypes), keeping the
 * reference's module names, constructor arguments, forward signatures and state-dict keys.
 *
 * Conventions
 *  - plain C, no CUDA or torch types: device pointers are `void*` / `const void*`,
 *    the stream is the `cudaStream_t` handle passed as `void*` (NULL = default stream);
 *  - the library BORROWS every pointer for the duration of the call, allocates nothing that
 *    outlives the call and never synchronises the stream (HOST-buffer entry excepted);
 *  - every entry returns 0 on success or a negative EGNN_ERR_* code and never throws;
 *  - all tensors are contiguous, row-major, in the layouts written next to each field;
 *  - re-entrant across streams and devices; the only mutable global state is one mutex-guarded per-device cache of
 *    kernel shared-memory opt-ins (only ever raised) and SM counts, and the opt-in profiler below.
 */
#ifndef EGNN_B200_H_
#define EGNN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EGNN_ABI_VERSION 3   /* 2: EgnnLayerIO grew nbr_idx + pre2_out; backward entry points added
                                3: peer-memory all-gather communicator (egnn_comm_*), egnn_global_attn_* */

/* ---- error codes ------------------------------------------------------------------- */
#define EGNN_OK                 0
#define EGNN_ERR_NULL          -1   /* required pointer is NULL                           */
#define EGNN_ERR_SHAPE         -2   /* inconsistent / out-of-range sizes                  */
#define EGNN_ERR_UNSUPPORTED   -3   /* option combination this build has no kernel for    */
#define EGNN_ERR_ALIGN         -4   /* pointer not aligned as documented (16 bytes)       */
#define EGNN_ERR_WORKSPACE     -5   /* workspace / packed buffer too small                */
#define EGNN_ERR_ABI           -6   /* desc.abi_version != EGNN_ABI_VERSION               */
#define EGNN_ERR_CUDA       -1000   /* -(1000 + cudaError_t) for CUDA runtime failures    */

/* ---- element types of feats / edges / weights / outputs ---------------------------- */
#define EGNN_DTYPE_F32   0   /* SIMT fp32 kernels ("accurate" path)                       */
#define EGNN_DTYPE_F64   1   /* SIMT fp64 kernels (the reference's tests run in fp64)     */
#define EGNN_DTYPE_BF16  2   /* tcgen05 bf16 tensor-core kernels, fp32 accumulation       */

/* ---- flags (EgnnLayerDesc.flags) ---------------------------------------------------- */
#define EGNN_FLAG_NORM_FEATS    (1u << 0)   /* node_norm = LayerNorm  (egnn_pytorch.py:191)   */
#define EGNN_FLAG_NORM_COORS    (1u << 1)   /* coors_norm = CoorsNorm (:192, :67-77)          */
#define EGNN_FLAG_UPDATE_FEATS  (1u << 2)   /* node_mlp present       (:196-201)              */
#define EGNN_FLAG_UPDATE_COORS  (1u << 3)   /* coors_mlp present      (:203-208)              */
#define EGNN_FLAG_SOFT_EDGES    (1u << 4)   /* edge_gate present      (:186-189)              */
#define EGNN_FLAG_POOL_MEAN     (1u << 5)   /* m_pool_method == 'mean' (:325-330)             */
#define EGNN_FLAG_CLAMP         (1u << 6)   /* coor_weights_clamp_value is set (:311-313)     */
#define EGNN_FLAG_ONLY_SPARSE   (1u << 7)   /* only_sparse_neighbors: valid_radius := 0 (:250);
                                               the caller passes k = max adjacency row sum   */
#define EGNN_FLAG_ADJ_BATCHED   (1u << 8)   /* io.adj is [B,N,N] instead of [N,N] (:245)      */

/*
 * Static description of one layer call.  E = 2*dim + 2*fourier + 1 + edge_dim + label_dim
 * is the reference's edge_input_dim (egnn_pytorch.py:175); H = 2*E.
 */
typedef struct EgnnLayerDesc {
  int32_t  abi_version;   /* EGNN_ABI_VERSION                                             */
  int32_t  dtype;         /* EGNN_DTYPE_*                                                 */
  int32_t  B, N;          /* graphs, nodes per graph                                      */
  int32_t  C;             /* coordinate dimension, 1..8 (tests/test_equivariance.py:40 uses 5) */
  int32_t  dim;           /* node feature width                                           */
  int32_t  edge_dim;      /* continuous edge channels read from io.edges (0 = none)       */
  int32_t  label_dim;     /* columns of edge_mlp.0.weight fed by the label embedding (adj_dim,
                             egnn_pytorch.py:430-432), 0 = none                           */
  int32_t  num_labels;    /* rows of weights.label_emb                                    */
  int32_t  m_dim;         /* message width (default 16), <= 32                            */
  int32_t  fourier;       /* fourier_features                                             */
  int32_t  k;             /* 0 = dense all-pairs; >0 = neighbours per node, i.e. the reference's
                             use_nearest branch (:237-268) with num_nearest = k           */
  uint32_t flags;         /* EGNN_FLAG_*                                                  */
  int32_t  row_begin;     /* evaluate i-rows [row_begin, row_end) only (row-sharded multi-GPU); */
  int32_t  row_end;       /*   0,0 = all rows.  Outputs keep their full [B,N,*] layout.   */
  int32_t  reserved;      /* must be 0                                                    */
  double   valid_radius;  /* used only when k>0 AND io.mask != NULL (:260, :296); +inf ok */
  double   clamp;         /* coor_weights_clamp_value when EGNN_FLAG_CLAMP                */
  double   dropout_p;     /* training-mode dropout probability of edge_mlp / node_mlp / coors_mlp (egnn_pytorch.py:176-208);
                             0 = off (eval mode).  fp32 / fp64 kernels only.                */
  uint64_t dropout_seed;  /* masks are regenerated from (seed, element index) in forward AND backward: pass the SAME
                             desc to egnn_layer_backward; draw a fresh seed per training step */
} EgnnLayerDesc;

/*
 * Device pointers to the layer's parameters, each exactly as nn.Linear / nn.LayerNorm stores it
 * (row-major [out, in]) under the state-dict key named on the right.  Element type = desc.dtype.
 * Pointers for modules the flags disable may be NULL.
 */
typedef struct EgnnLayerWeights {
  const void* edge_w1;    /* [H, E]      edge_mlp.0.weight   */
  const void* edge_b1;    /* [H]         edge_mlp.0.bias     */
  const void* edge_w2;    /* [m, H]      edge_mlp.3.weight   */
  const void* edge_b2;    /* [m]         edge_mlp.3.bias     */
  const void* gate_w;     /* [1, m]      edge_gate.0.weight  */
  const void* gate_b;     /* [1]         edge_gate.0.bias    */
  const void* norm_g;     /* [dim]       node_norm.weight    */
  const void* norm_b;     /* [dim]       node_norm.bias      */
  const void* coors_scale;/* [1]         coors_norm.scale    */
  const void* node_w1;    /* [2dim, dim+m]  node_mlp.0.weight */
  const void* node_b1;    /* [2dim]      node_mlp.0.bias     */
  const void* node_w2;    /* [dim, 2dim] node_mlp.3.weight   */
  const void* node_b2;    /* [dim]       node_mlp.3.bias     */
  const void* coors_w1;   /* [4m, m]     coors_mlp.0.weight  */
  const void* coors_b1;   /* [4m]        coors_mlp.0.bias    */
  const void* coors_w2;   /* [1, 4m]     coors_mlp.3.weight  */
  const void* coors_b2;   /* [1]         coors_mlp.3.bias    */
  const void* label_emb;  /* [num_labels, label_dim]  EGNN_Network.adj_emb.weight (or NULL) */
} EgnnLayerWeights;

/*
 * Per-call tensors (device memory).  feats/edges/feats_out have element type desc.dtype;
 * coors/coors_out are float64 when desc.dtype == F64 and float32 otherwise.
 */
typedef struct EgnnLayerIO {
  const void*    feats;      /* [B, N, dim]                                               */
  const void*    coors;      /* [B, N, C]                                                 */
  const void*    edges;      /* [B, N, N, edge_dim] or NULL when edge_dim == 0            */
  const uint8_t* edge_labels;/* [B, N, N] label index per pair, or NULL when label_dim == 0 */
  const uint8_t* mask;       /* [B, N] 0/1, or NULL (= the reference's mask=None)         */
  const uint8_t* adj;        /* [N, N] or [B, N, N] 0/1 (EGNN_FLAG_ADJ_BATCHED), or NULL;
                                only read when k > 0                                      */
  void*          feats_out;  /* [B, N, dim]                                               */
  void*          coors_out;  /* [B, N, C]                                                 */
  const int32_t* nbr_idx;    /* optional, k > 0 only: caller-supplied neighbour lists [B, N, k] (edge-list
                                mode, SURVEY.md section 8(f) rank 3): the distance/top-k pass is skipped.  An entry
                                < 0 is an empty slot and never contributes.  NULL = select as the reference does. */
  void*          pre2_out;   /* optional, fp32/fp64 training only: [B, N, J, MP] with J = N (dense) or k (neighbour lists)
                                and MP = 16 when m_dim <= 16, else 32.  egnn_layer_forward stores the per-pair
                                pre-activation of edge_mlp's second SiLU there; egnn_layer_backward, given the same
                                pointer, skips recomputing it -- a speed / memory trade (64 B per pair in fp32).
                                NULL = nothing stored, backward recomputes. */
} EgnnLayerIO;

int         egnn_abi_version(void);
const char* egnn_strerror(int code);

/* Bytes of the packed-parameter buffer for `desc` (depends on dtype and sizes only). */
int egnn_layer_packed_bytes(const EgnnLayerDesc* desc, size_t* out_bytes);

/* Re-layout the parameters for the kernels (split W1 into per-node and per-pair parts,
 * transpose W2, fold the label embedding into a [num_labels, H] table, bf16 copies for the
 * tensor-core path).  Enqueued on `stream`; call again whenever a parameter changes. */
int egnn_layer_pack_weights(const EgnnLayerDesc* desc, const EgnnLayerWeights* w,
                            void* packed, size_t packed_bytes, void* stream);

/* Bytes of scratch `egnn_layer_forward` needs for `desc` (per-node tables, neighbour lists). */
int egnn_layer_workspace_bytes(const EgnnLayerDesc* desc, size_t* out_bytes);

/* One EGNN layer forward == reference EGNN.forward (egnn_pytorch.py:224-341), enqueued on
 * `stream`.  `packed` comes from egnn_layer_pack_weights with an identical desc (B, N, k,
 * flags and the row range may differ).  `workspace` must be 256-byte aligned. */
int egnn_layer_forward(const EgnnLayerDesc* desc, const EgnnLayerWeights* w, const void* packed,
                       const EgnnLayerIO* io, void* workspace, size_t workspace_bytes,
                       void* stream);

/* Same call with HOST buffers for io.* (pinned or pageable): allocates device staging,
 * copies in, runs, copies feats_out / coors_out back and synchronises.  Parameters (`w`,
 * `packed`) stay device-resident.  This is the end-to-end entry `bench.py` times as `e2e`. */
int egnn_layer_forward_host(const EgnnLayerDesc* desc, const EgnnLayerWeights* w,
                            const void* packed, const EgnnLayerIO* host_io, void* stream);

/*
 * Backward of one layer (SURVEY.md section 8(f) rank 1): what autograd computes through the reference's
 * EGNN.forward (egnn_pytorch.py:224-341).  fp32 / fp64 kernels only (EGNN_ERR_UNSUPPORTED for bf16 and for a row
 * range).  The edge step is recomputed pair by pair, so the only saved state is the forward WORKSPACE:
 * `fwd_workspace` must be the buffer egnn_layer_forward ran on with the same desc / io, unmodified since.
 * Gradient buffers are OVERWRITTEN (not accumulated into).  Neighbour selection contributes no gradient.
 */
typedef struct EgnnLayerWeightGrads {   /* one buffer per EgnnLayerWeights field, same shape and dtype; NULL for
                                           modules the flags disable */
  void* edge_w1; void* edge_b1; void* edge_w2; void* edge_b2; void* gate_w; void* gate_b;
  void* norm_g; void* norm_b; void* coors_scale;
  void* node_w1; void* node_b1; void* node_w2; void* node_b2;
  void* coors_w1; void* coors_b1; void* coors_w2; void* coors_b2; void* label_emb;
} EgnnLayerWeightGrads;

typedef struct EgnnLayerGrads {
  const void* g_feats_out;   /* [B, N, dim]  dL/d feats_out (input)                         */
  const void* g_coors_out;   /* [B, N, C]    dL/d coors_out (input)                         */
  void*       g_feats;       /* [B, N, dim]  dL/d feats                                     */
  void*       g_coors;       /* [B, N, C]    dL/d coors                                     */
  void*       g_edges;       /* [B, N, N, edge_dim] dL/d edges, or NULL (not wanted / edge_dim == 0) */
  EgnnLayerWeightGrads w;
} EgnnLayerGrads;

int egnn_layer_backward_workspace_bytes(const EgnnLayerDesc* desc, size_t* out_bytes);
int egnn_layer_backward(const EgnnLayerDesc* desc, const EgnnLayerWeights* w, const void* packed,
                        const EgnnLayerIO* io, const void* fwd_workspace, const EgnnLayerGrads* grads,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Neighbour selection alone == ranking + topk of egnn_pytorch.py:237-260: for every node the k
 * lowest-ranked nodes (rank = squared distance; 1e5 if either end is masked out; -1 self and 0
 * adjacent when `adj` is given), ascending, ties to the lowest index.
 * coors [B,N,C] (float32, or float64 when dtype == EGNN_DTYPE_F64); mask/adj as in EgnnLayerIO;
 * out_idx int32 [B,N,k]; out_ok uint8 [B,N,k] = (rank <= valid_radius), may be NULL. */
int egnn_knn_select(int32_t dtype, int32_t B, int32_t N, int32_t C, int32_t k,
                    const void* coors, const uint8_t* mask, const uint8_t* adj, int32_t adj_batched,
                    double valid_radius, int32_t* out_idx, uint8_t* out_ok, void* stream);

/* Neighbour lists from an adjacency alone: slot 0 = the node itself, then its adjacent nodes in ascending index order,
 * truncated at k -- exactly the slots of egnn_knn_select whose rank is <= 0 (egnn_pytorch.py:255-256), i.e. every slot that
 * survives `only_sparse_neighbors` with a node mask (valid_radius = 0, :250, :296).  They do not depend on the coordinates,
 * so EGNN_Network builds them once per adjacency and hands them to every layer (EgnnLayerIO.nbr_idx).
 * adj [N,N] or [B,N,N] 0/1 bytes; out_idx int32 [B,N,k]; out_ok uint8 [B,N,k] or NULL.  Unused slots: the node itself with
 * ok = 0, or -1 when out_ok is NULL. */
int egnn_adj_neighbors(int32_t B, int32_t N, int32_t k, const uint8_t* adj, int32_t adj_batched, int32_t* out_idx,
                       uint8_t* out_ok, void* stream);

/* N-th degree adjacency of EGNN_Network (egnn_pytorch.py:414-428) without the dense A@A:
 * adj_in [N,N] or [B,N,N] 0/1; writes the expanded adjacency adj_out [B,N,N] 0/1, the degree
 * labels labels_out [B,N,N] (0 = not connected, d = first reached in round d) and
 * max_row_sum[0] = max over rows of sum_j adj_out (the reference's `num_nearest` under
 * only_sparse_neighbors, :249).  workspace: egnn_adj_workspace_bytes(B, N). */
int egnn_adj_workspace_bytes(int32_t B, int32_t N, size_t* out_bytes);
int egnn_adj_expand(int32_t B, int32_t N, int32_t num_degrees, const uint8_t* adj_in,
                    int32_t adj_batched, uint8_t* adj_out, uint8_t* labels_out,
                    int32_t* max_row_sum, void* workspace, size_t workspace_bytes, void* stream);

/* Node embedding of EGNN_Network (egnn_pytorch.py:401-408) in one launch: out[b,n,:] = token_emb[tokens[b,n],:] +
 * pos_emb[n,:] (pos_emb may be NULL).  Tables and output have element type `dtype`; tokens are int64 [B,N]. */
int egnn_embed_nodes(int32_t dtype, int32_t B, int32_t N, int32_t dim, int32_t num_tokens, const int64_t* tokens,
                     const void* token_emb, const void* pos_emb, void* out, void* stream);

/* The tcgen05 GEMM the bf16 path uses for its per-node contractions, exposed for unit tests:
 * out[M,N] = act(scale * (A[M,K] W[N,K]^T + bias[N])), A/W bf16 row-major, K and N multiples of 8,
 * act 0 = none / 1 = SiLU, out fp32 (out_f32 = 1) or bf16. */
int egnn_gemm_bf16(int32_t M, int32_t N, int32_t K, const void* A, const void* W, const float* bias,
                   float scale, int32_t act, void* out, int32_t out_f32, void* stream);

/*
 * GlobalLinearAttention of EGNN_Network (reference egnn_pytorch.py:81-144, applied between layers at :445-446): the
 * T global tokens attend over the (masked) nodes, the nodes attend over the induced tokens, residuals, pre-norm GELU
 * feed-forward.  Forward only, fp32 / fp64 (a bf16 module passes fp32 copies).  Weights exactly as the reference's
 * state dict stores them (row-major [out, in]); all pointers device memory, contiguous.
 */
typedef struct EgnnGlobalAttnDesc {
  int32_t abi_version;    /* EGNN_ABI_VERSION */
  int32_t dtype;          /* EGNN_DTYPE_F32 | EGNN_DTYPE_F64 */
  int32_t B, N, T;        /* graphs, nodes, global tokens (T <= 32) */
  int32_t dim, heads, dim_head;
} EgnnGlobalAttnDesc;

typedef struct EgnnGlobalAttnWeights {
  const void* norm_seq_g; const void* norm_seq_b;      /* [dim]  norm_seq.weight / .bias        */
  const void* norm_q_g;   const void* norm_q_b;        /* [dim]  norm_queries.weight / .bias    */
  const void* a1_wq;  const void* a1_wkv;              /* [inner, dim], [2 inner, dim]  attn1.to_q / to_kv.weight (inner = heads * dim_head) */
  const void* a1_wo;  const void* a1_bo;               /* [dim, inner], [dim]           attn1.to_out.weight / .bias */
  const void* a2_wq;  const void* a2_wkv; const void* a2_wo; const void* a2_bo;   /* attn2, same shapes */
  const void* ff_ln_g; const void* ff_ln_b;            /* [dim]          ff.0.weight / .bias    */
  const void* ff_w1;  const void* ff_b1;               /* [4 dim, dim], [4 dim]   ff.1          */
  const void* ff_w2;  const void* ff_b2;               /* [dim, 4 dim], [dim]     ff.3          */
} EgnnGlobalAttnWeights;

typedef struct EgnnGlobalAttnIO {
  const void*    x;            /* [B, N, dim] node features                         */
  const void*    queries;      /* [B, T, dim] global tokens                         */
  const uint8_t* mask;         /* [B, N] 0/1 or NULL; a fully masked graph attends uniformly (:101-104) */
  void*          x_out;        /* [B, N, dim]                                       */
  void*          queries_out;  /* [B, T, dim]                                       */
} EgnnGlobalAttnIO;

int egnn_global_attn_workspace_bytes(const EgnnGlobalAttnDesc* desc, size_t* out_bytes);
int egnn_global_attn_forward(const EgnnGlobalAttnDesc* desc, const EgnnGlobalAttnWeights* w, const EgnnGlobalAttnIO* io,
                             void* workspace, size_t workspace_bytes, void* stream);

/*
 * Peer-memory all-gather over NVLink for the ROW-SHARDED single graph (SURVEY.md section 8(e) row 2; reference
 * semantics: the all-pairs pass of egnn_pytorch.py:232-233 runs over ALL nodes, so every rank needs every rank's
 * coordinates and features on the j side).  One process per GPU.  The communicator is the one object of this library
 * that owns device memory beyond a call: a gather buffer (2 x payload_bytes, double-buffered by call parity) that the
 * peers map with CUDA IPC.
 *   egnn_comm_create   -> allocates the buffer on the current device, returns the communicator and a 64-byte IPC handle;
 *                         exchange the handles of all ranks out of band (torch.distributed.all_gather_object) ...
 *   egnn_comm_connect  -> ... and pass all of them (world x 64 bytes, rank order) to map the peers' buffers.
 *   egnn_comm_allgather-> ONE kernel on `stream`: copies this rank's `nseg` segments src[s] (bytes[s], multiples of 4)
 *                         to byte offset dst_off[s] of EVERY rank's buffer with P2P stores over NVLink, raises this rank's
 *                         epoch flag in every peer and waits (on the device) for every peer's flag.  Kernels enqueued
 *                         after it on the same stream see the complete buffer at *gathered_out (valid until the call
 *                         after next).  Every rank must make the same sequence of calls.  No host synchronisation.
 *   egnn_comm_status   -> 0, or 1 if a wait timed out (a peer never arrived); synchronises.
 */
#define EGNN_IPC_HANDLE_BYTES 64
int egnn_comm_create(int32_t world, int32_t rank, size_t payload_bytes, void** comm_out, void* ipc_handle_out);
int egnn_comm_connect(void* comm, const void* all_handles);
int egnn_comm_allgather(void* comm, int32_t nseg, const void* const* src, const size_t* dst_off, const size_t* bytes,
                        void** gathered_out, void* stream);
int egnn_comm_status(void* comm, int32_t* status_out);
int egnn_comm_destroy(void* comm);

/* Diagnostics for benchmarks: when enabled, every egnn_layer_forward brackets its stages
 * (0 neighbour select, 1 per-node tables, 2 fused edge kernel, 3 node update) with CUDA events
 * on the launch stream, and the library counts every kernel it launches, from any entry point
 * (forward, backward, weight packing, adjacency, embedding, global attention, all-gather).
 * egnn_profile_read synchronises those events and returns the accumulated milliseconds / span
 * counts per stage (arrays of 4) and the launch count.  Off by default. */
int egnn_profile_enable(int on);
int egnn_profile_read(float* ms_out, int32_t* spans_out, int64_t* launches_out, int reset);

#ifdef __cplusplus
}
#endif
#endif  /* EGNN_B200_H_ */
