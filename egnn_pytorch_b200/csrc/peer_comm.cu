// Peer-memory all-gather over NVLink for the row-sharded single graph (SURVEY.md section 8(e) row 2):
// every rank owns a contiguous block of i-rows; a layer needs ALL coordinates and ALL node features on the j side
// (reference semantics: the all-pairs pass of egnn_pytorch.py:232-233 over the gathered nodes).  Instead of a
// host-driven collective, ONE kernel per rank pushes the rank's rows straight into every peer's gather buffer
// with P2P stores over NVLink (the buffers are cudaMalloc'ed here and mapped into the peers with CUDA IPC), then
// raises an epoch flag in each peer and waits for the flags the peers raise here.  The kernel is enqueued on the
// caller's stream, so the layer's kernels that follow see the complete [coors | feats] arrays -- no host sync.
//
// Buffers are double-buffered by epoch parity: a rank that is one call ahead writes the OTHER half, and it cannot be
// two calls ahead because call n+1 waits for every peer's epoch-(n+1) flag, which a peer only raises after it
// finished (stream order) everything that read the epoch-(n-1) half.
#include "launch.cuh"
#include <string.h>
#include <new>

namespace egnn {
namespace {

constexpr int COMM_MAX_RANKS = 8;
constexpr int COMM_MAX_SEGS = 16;
constexpr unsigned long long COMM_TIMEOUT_NS = 20ull * 1000 * 1000 * 1000;      // a lost peer must not hang the GPU

// header at the start of every rank's buffer (device memory, written by peers over NVLink)
struct CommHeader {
  uint32_t flags[2][COMM_MAX_RANKS];   // [parity][source rank] = epoch of the last completed push
  uint32_t done_ctas;                  // local: CTAs of the running push that finished copying
  uint32_t status;                     // local: 0 ok, 1 = timed out waiting for a peer
  uint32_t pad[46];
};
static_assert(sizeof(CommHeader) == 256, "header layout");

}  // namespace

struct Comm {
  int world = 0, rank = 0, device = 0;
  size_t half_bytes = 0;               // payload bytes of one parity half
  unsigned char* local = nullptr;      // header | half 0 | half 1
  unsigned char* peer[COMM_MAX_RANKS] = {nullptr};
  uint32_t epoch = 0;
  bool connected = false;
};

namespace {

struct PushArgs {
  int world, rank, nseg;
  uint32_t epoch;
  unsigned char* peer[COMM_MAX_RANKS];       // base of every rank's buffer as mapped in this process
  size_t half_off;                           // byte offset of this epoch's half from the base
  const unsigned char* src[COMM_MAX_SEGS];
  size_t dst_off[COMM_MAX_SEGS];
  size_t bytes[COMM_MAX_SEGS];
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// grid.x CTAs share the copy; blockIdx.y = destination rank (including this one).  Payload segments are pushed with
// 16-byte stores when source, destination and size allow it, 4-byte stores otherwise.
__global__ void __launch_bounds__(256) peer_push_kernel(const PushArgs a) {
  const int dst_rank = blockIdx.y;
  unsigned char* dst_base = a.peer[dst_rank] + a.half_off;
  for (int sg = 0; sg < a.nseg; ++sg) {
    const unsigned char* src = a.src[sg];
    unsigned char* dst = dst_base + a.dst_off[sg];
    const size_t n = a.bytes[sg];
    if (((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) | n) & 15) == 0) {
      const uint4* s4 = reinterpret_cast<const uint4*>(src);
      uint4* d4 = reinterpret_cast<uint4*>(dst);
      for (size_t x = (size_t)blockIdx.x * blockDim.x + threadIdx.x; x < n / 16; x += (size_t)gridDim.x * blockDim.x) d4[x] = s4[x];
    } else {
      const uint32_t* s1 = reinterpret_cast<const uint32_t*>(src);
      uint32_t* d1 = reinterpret_cast<uint32_t*>(dst);
      for (size_t x = (size_t)blockIdx.x * blockDim.x + threadIdx.x; x < n / 4; x += (size_t)gridDim.x * blockDim.x) d1[x] = s1[x];
    }
  }
  // the last CTA to finish (of all destinations) raises this rank's flag everywhere and waits for the peers' flags
  __threadfence_system();
  __syncthreads();
  __shared__ bool last;
  CommHeader* me = reinterpret_cast<CommHeader*>(a.peer[a.rank]);
  if (threadIdx.x == 0) {
    const uint32_t total = gridDim.x * gridDim.y;
    last = atomicAdd(&me->done_ctas, 1u) == total - 1;
  }
  __syncthreads();
  if (!last) return;
  if (threadIdx.x == 0) me->done_ctas = 0;
  const int par = a.epoch & 1;
  if ((int)threadIdx.x < a.world) {
    __threadfence_system();
    CommHeader* ph = reinterpret_cast<CommHeader*>(a.peer[threadIdx.x]);
    st_release_sys(&ph->flags[par][a.rank], a.epoch);                      // "rank's rows of this epoch have landed in your buffer"
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(&me->flags[par][threadIdx.x]) != a.epoch) {       // rows of rank threadIdx.x have landed here
      __nanosleep(200);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > COMM_TIMEOUT_NS) { me->status = 1; break; }
    }
  }
}

}  // namespace
}  // namespace egnn

using egnn::Comm;

extern "C" {

int egnn_comm_create(int32_t world, int32_t rank, size_t payload_bytes, void** comm_out, void* ipc_handle_out) {
  if (!comm_out || !ipc_handle_out) return EGNN_ERR_NULL;
  if (world < 1 || world > egnn::COMM_MAX_RANKS || rank < 0 || rank >= world) return EGNN_ERR_SHAPE;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "EGNN_IPC_HANDLE_BYTES");
  Comm* c = new (std::nothrow) Comm();
  if (!c) return EGNN_ERR_CUDA;
  c->world = world; c->rank = rank;
  c->half_bytes = egnn::round_up(payload_bytes, 256);
  EGNN_CUDA_TRY(cudaGetDevice(&c->device));
  const size_t total = sizeof(egnn::CommHeader) + 2 * c->half_bytes;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&c->local), total);
  if (e != cudaSuccess) { delete c; return EGNN_ERR_CUDA - (int)e; }
  e = cudaMemset(c->local, 0, sizeof(egnn::CommHeader));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, c->local);
  if (e != cudaSuccess) { cudaFree(c->local); delete c; return EGNN_ERR_CUDA - (int)e; }
  memcpy(ipc_handle_out, &h, sizeof(h));
  c->peer[rank] = c->local;
  *comm_out = c;
  return EGNN_OK;
}

int egnn_comm_connect(void* comm, const void* all_handles) {
  if (!comm || !all_handles) return EGNN_ERR_NULL;
  Comm* c = static_cast<Comm*>(comm);
  const unsigned char* hs = static_cast<const unsigned char*>(all_handles);
  for (int r = 0; r < c->world; ++r) {
    if (r == c->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, hs + (size_t)r * sizeof(h), sizeof(h));
    void* p = nullptr;
    EGNN_CUDA_TRY(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    c->peer[r] = static_cast<unsigned char*>(p);
  }
  c->connected = true;
  return EGNN_OK;
}

int egnn_comm_allgather(void* comm, int32_t nseg, const void* const* src, const size_t* dst_off, const size_t* bytes,
                        void** gathered_out, void* stream) {
  if (!comm || !src || !dst_off || !bytes || !gathered_out) return EGNN_ERR_NULL;
  Comm* c = static_cast<Comm*>(comm);
  if (!c->connected && c->world > 1) return EGNN_ERR_UNSUPPORTED;
  if (nseg < 1 || nseg > egnn::COMM_MAX_SEGS) return EGNN_ERR_SHAPE;
  egnn::PushArgs a{};
  a.world = c->world; a.rank = c->rank; a.nseg = nseg;
  a.epoch = ++c->epoch;
  a.half_off = sizeof(egnn::CommHeader) + (size_t)(a.epoch & 1) * c->half_bytes;
  size_t most = 0;
  for (int r = 0; r < c->world; ++r) a.peer[r] = c->peer[r];
  for (int s = 0; s < nseg; ++s) {
    if (bytes[s] % 4 != 0 || dst_off[s] % 4 != 0 || (reinterpret_cast<uintptr_t>(src[s]) & 3)) return EGNN_ERR_ALIGN;
    if (dst_off[s] + bytes[s] > c->half_bytes) return EGNN_ERR_WORKSPACE;
    a.src[s] = static_cast<const unsigned char*>(src[s]); a.dst_off[s] = dst_off[s]; a.bytes[s] = bytes[s];
    most = bytes[s] > most ? bytes[s] : most;
  }
  int ctas = (int)((most / 16 + 255) / 256);
  ctas = ctas < 1 ? 1 : (ctas > 16 ? 16 : ctas);                 // NVLink is saturated by a handful of CTAs per peer
  EGNN_TRY(egnn::launch(egnn::peer_push_kernel, dim3(ctas, c->world), 256, 0, static_cast<cudaStream_t>(stream), a));
  *gathered_out = c->local + a.half_off;
  return EGNN_OK;
}

int egnn_comm_status(void* comm, int32_t* status_out) {
  if (!comm || !status_out) return EGNN_ERR_NULL;
  Comm* c = static_cast<Comm*>(comm);
  uint32_t v = 0;
  EGNN_CUDA_TRY(cudaMemcpy(&v, &reinterpret_cast<egnn::CommHeader*>(c->local)->status, 4, cudaMemcpyDeviceToHost));
  *status_out = (int32_t)v;
  return EGNN_OK;
}

int egnn_comm_destroy(void* comm) {
  if (!comm) return EGNN_OK;
  Comm* c = static_cast<Comm*>(comm);
  for (int r = 0; r < c->world; ++r)
    if (r != c->rank && c->peer[r]) cudaIpcCloseMemHandle(c->peer[r]);
  if (c->local) cudaFree(c->local);
  delete c;
  return EGNN_OK;
}

}  // extern "C"
