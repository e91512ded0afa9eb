// HP-A: gradient allreduce over NVLink/NVSwitch peer memory -- no NCCL, no serialisation, no host staging.
//
//   K-A1  ar_stage_kernel    : pack (=) or accumulate (+=) a tensor list into the rank's symmetric staging buffer and
//                              optionally zero the sources, one launch for the whole list.
//   K-A2  ar_oneshot_kernel  : per-block flag barrier with every peer (st.release.sys into the peer's flag row /
//                              ld.acquire.sys on the local row), then each rank pulls all peers' staging with 16 B P2P
//                              loads, sums in ascending rank order in fp32, multiplies by 1.0f/sum(num_gradients) and
//                              scatters straight into the destination tensors.  (N-1)*S bytes in per GPU, one barrier.
//         ar_twoshot_kernel  : reduce-scatter by P2P loads (rank r reduces slice r), all-gather by P2P stores into
//                              every peer's staging, second flag barrier, local scatter.  2(N-1)/N*S per direction.
// Both give bit-identical results on every rank and identical to each other (same summation order).
//   K-A0  ar_gate_kernel     : ONE 32-thread CTA.  Pushes this rank's {numGradients,numSkipped,batchSize,has_grads}
//                              into every peer's sync block, waits for theirs, sums them and decides whether the
//                              virtual-batch gate is open (sum(batchSize) >= min_batch).  The reduce kernel that
//                              follows on the stream reads the decision: closed -> it returns at once, open -> it needs
//                              no start barrier (every peer's staging is complete once its header has arrived).
//                              Replaces the count allreduce over RPC (src/accumulator.cc:1035-1078).
//
// Reference semantics being replaced: src/accumulator.cc:941-980 (stage), src/group.h:195-212 (add),
// src/group.h:570-654,687-787 (tree reduce + share), src/accumulator.cc:425-452 (copy_ + mul_(1.0f/numGradients)).
#include "mb_common.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <unistd.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

namespace mb {
namespace {

constexpr int kArThreads = 512;
constexpr int kArMaxBlocks = 1024;
constexpr int kArMaxTensors = 4096;
constexpr uint32_t kHandleMagic = 0x4d423230u;  // "MB20"

struct TensorEnt {
  uint64_t ptr;    // device address of the tensor's first float
  uint64_t off;    // first float in the flat layout (multiple of 4)
  uint64_t numel;  // floats
};

// Lives in device memory of its owner, mapped by every peer.  Zero-initialised.
struct SyncBlock {
  mb_ar_hdr hdr[2];                                 // [epoch parity], written by the owner before it signals
  uint32_t flagsA[kArMaxBlocks][MB_AR_MAX_WORLD];   // [block][source rank] = epoch: "my data for this round is staged"
  uint32_t flagsB[kArMaxBlocks][MB_AR_MAX_WORLD];   // two-shot: "my reduced slice is written to your staging"
  // gated rounds (K-A0): headers are PUSHED by their owner into every peer's block, then the flag is released
  mb_ar_hdr ghdr[2][MB_AR_MAX_WORLD];               // [epoch parity][source rank]
  uint32_t gate[MB_AR_MAX_WORLD];                   // [source rank] = epoch: "my header is in, my staging is complete"
};

// Written by the gate kernel, read by the reduce kernel that follows it on the stream (device-local).
struct GateOut {
  mb_ar_hdr tot;
  uint32_t mask;      // ranks with has_grads
  int32_t decision;   // 1 = reduce, 0 = gate closed (short batch) or barrier failure: the reduce kernel returns
  uint32_t epoch;
  uint32_t pad;
};

struct HostResult {
  mb_ar_hdr sum;
  int32_t status;
  uint32_t epoch;
};

// One rank's symmetric memory is ONE cudaMalloc block whose size is a multiple of 2 MiB: [staging | SyncBlock].  CUDA IPC
// shares whole 2 MiB-granular blocks and cudaIpcOpenMemHandle returns the BASE of the block a pointer lives in, so a
// small allocation that the driver sub-allocated next to others would be opened at the wrong address; owning whole
// blocks (and carrying the offset from the block base, measured with cuMemGetAddressRange) rules that out.
struct HandleImpl {
  uint32_t magic;
  int32_t pid;
  int32_t device;
  int32_t rank;
  uint64_t block_ptr;     // owner's virtual address of the block (same-process peers use it directly)
  uint64_t base_offset;   // block_ptr - base of the driver allocation that the IPC handle maps
  uint64_t sync_offset;   // SyncBlock offset inside the block
  uint64_t xfer_offset;   // publish region offset inside the block
  uint64_t max_bytes;
  int32_t nslots;
  int32_t ipc_ok;
  cudaIpcMemHandle_t h_block;
};
static_assert(sizeof(HandleImpl) <= MB_AR_HANDLE_BYTES, "mb_ar_handle too small");

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

}  // namespace
}  // namespace mb

struct mb_ar_ctx {
  int rank = 0, world = 1, device = 0, nslots = 1;
  uint64_t max_bytes = 0;  // per staging buffer, multiple of 16
  void* block = nullptr;             // the one IPC-exported allocation: [staging | SyncBlock], multiple of 2 MiB
  uint64_t block_bytes = 0, sync_offset = 0;
  float* staging = nullptr;          // nslots * MB_AR_BUFS_PER_SLOT buffers (ring, see mb_ar_allreduce)
  uint64_t xfer_offset = 0;          // the publish region (max_bytes) behind the ring: mb_ar_xfer_pack / _unpack
  mb::SyncBlock* sync = nullptr;
  void* peer_block[MB_AR_MAX_WORLD] = {};  // IPC-opened base of each peer's block (what must be closed)
  float* peer_staging[MB_AR_MAX_WORLD] = {};
  mb::SyncBlock* peer_sync[MB_AR_MAX_WORLD] = {};
  bool imported[MB_AR_MAX_WORLD] = {};
  bool ipc_opened[MB_AR_MAX_WORLD] = {};
  uint32_t epoch = 0;
  int parity[MB_AR_MAX_SLOTS] = {};
  mb::HostResult* result_host = nullptr;  // pinned + mapped, one per slot
  mb::HostResult* result_dev = nullptr;
  uint32_t* abort_host = nullptr;
  uint32_t* abort_dev = nullptr;
  mb::GateOut* gate_out = nullptr;   // device, one per slot
  cudaEvent_t ev[MB_AR_MAX_SLOTS][3] = {};  // gated rounds: before K-A0 / between K-A0 and K-A2 / after K-A2 (timing)
  bool ev_valid[MB_AR_MAX_SLOTS] = {};
  mb::TensorEnt* tab_dev[2] = {nullptr, nullptr};  // 0: stage sources, 1: allreduce destinations
  std::vector<mb::TensorEnt> tab_host[2];
  bool tab_bytes[2] = {false, false};  // the table holds byte entries (mixed-dtype lists), see SegInfo
  std::mutex mu;
};

namespace mb {
namespace {

struct ArParams {
  float* stage[MB_AR_MAX_WORLD];     // every rank's staging buffer for this slot/ring position ([rank] = own)
  SyncBlock* sync[MB_AR_MAX_WORLD];  // every rank's sync block
  const TensorEnt* dst_tab;          // ntensors entries; ignored when ntensors == 0 (flat destination)
  float* flat_dst;                   // ntensors == 0: result goes to flat_dst[v*4..], same layout as the staging
  const GateOut* gate;               // non-null: gated round (K-A0 ran before this kernel on the stream)
  uint32_t ntensors;
  uint32_t epoch;
  uint64_t total_vec;  // flat length in float4 units
  uint64_t slice_vec;  // two-shot: ceil(total_vec / world)
  mb_ar_hdr my_hdr;
  int32_t rank;
  int32_t world;
  int32_t scale;
  int32_t force_u1;  // tuning aid: disable the U-way unrolled path
  int32_t inplace;   // two-shot: the destination IS this rank's staging buffer (the all-gather already put it there)
  HostResult* result;
  const uint32_t* abort_flag;
  uint64_t timeout_ns;
};

struct StageParams {
  float* staging;
  const TensorEnt* tab;
  uint32_t ntensors;
  int32_t accumulate;
  int32_t zero_src;
  uint64_t total_vec;
};

struct GateParams {
  SyncBlock* sync[MB_AR_MAX_WORLD];
  GateOut* out;
  HostResult* result;
  const uint32_t* abort_flag;
  mb_ar_hdr my_hdr;
  uint64_t min_batch;
  uint64_t timeout_ns;
  uint32_t epoch;
  int32_t rank;
  int32_t world;
};

// ---- flat layout <-> tensor list ---------------------------------------------------------------------------------

// The tensor table lives in dynamic shared memory as three arrays (pointers, numel, first float4).  A thread's flat
// index only ever grows inside a kernel, so the owning tensor is found by walking a per-thread cursor forward: no
// per-vector search and no dependent global load (round 1 did a 6-step binary search + a 24 B global load per 16 B of
// payload -- 0.15 of HBM).
struct TensorTable {
  const uint64_t* ptr;
  const uint64_t* numel;
  const uint32_t* off;  // first float4 of tensor i
  uint32_t n;
};

__device__ __forceinline__ TensorTable load_table(uint8_t* smem, const TensorEnt* tab, uint32_t n) {
  uint64_t* s_ptr = reinterpret_cast<uint64_t*>(smem);
  uint64_t* s_numel = s_ptr + n;
  uint32_t* s_off = reinterpret_cast<uint32_t*>(s_numel + n);
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    const TensorEnt e = tab[i];
    s_ptr[i] = e.ptr;
    s_numel[i] = e.numel;
    s_off[i] = (uint32_t)(e.off >> 2);
  }
  TensorTable t;
  t.ptr = s_ptr;
  t.numel = s_numel;
  t.off = s_off;
  t.n = n;
  return t;
}

// Advance `cur` to the tensor that owns float4 index v (v never decreases between calls with the same cursor).
__device__ __forceinline__ void seek_tensor(const TensorTable& tb, uint32_t v, uint32_t& cur) {
  if (cur + 1 < tb.n && tb.off[cur + 1] <= v) {
    // jump: binary search over (cur, n) -- taken once per tensor boundary, not once per vector
    uint32_t lo = cur + 1, hi = tb.n;
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (tb.off[mid] <= v) lo = mid; else hi = mid;
    }
    cur = lo;
  }
}

__device__ __forceinline__ void store_vec(float* d, uint64_t valid, const float4& r) {
  if (valid >= 4 && (reinterpret_cast<uintptr_t>(d) & 15u) == 0) {
    st_f4(d, r);
  } else {
    d[0] = r.x;
    if (valid > 1) d[1] = r.y;
    if (valid > 2) d[2] = r.z;
    if (valid > 3) d[3] = r.w;
  }
}

__device__ __forceinline__ void scatter_vec(const TensorTable& tb, uint64_t v, const float4& r, uint32_t& cur) {
  seek_tensor(tb, (uint32_t)v, cur);
  const uint64_t within = (v - tb.off[cur]) * 4;
  const uint64_t numel = tb.numel[cur];
  if (within >= numel) return;  // padding-only vector (empty tensor)
  store_vec(reinterpret_cast<float*>(tb.ptr[cur]) + within, numel - within, r);
}

// ---- K-A1 --------------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(kArThreads) ar_stage_kernel(const __grid_constant__ StageParams p) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  const TensorTable tb = load_table(dyn_smem, p.tab, p.ntensors);
  __syncthreads();
  // each block owns a contiguous span of the flat layout: consecutive iterations touch consecutive 8 KiB chunks
  const uint64_t per_block = (p.total_vec + gridDim.x - 1) / gridDim.x;
  const uint64_t begin = (uint64_t)blockIdx.x * per_block;
  const uint64_t end = min(begin + per_block, p.total_vec);
  uint32_t cur = 0;
  for (uint64_t v = begin + threadIdx.x; v < end; v += kArThreads) {
    seek_tensor(tb, (uint32_t)v, cur);
    const uint64_t within = (v - tb.off[cur]) * 4;
    const uint64_t numel = tb.numel[cur];
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (within < numel) {
      float* s = reinterpret_cast<float*>(tb.ptr[cur]) + within;
      const uint64_t valid = numel - within;
      const bool vec = valid >= 4 && (reinterpret_cast<uintptr_t>(s) & 15u) == 0;
      if (vec) {
        g = *reinterpret_cast<const float4*>(s);
      } else {
        g.x = s[0];
        if (valid > 1) g.y = s[1];
        if (valid > 2) g.z = s[2];
        if (valid > 3) g.w = s[3];
      }
      if (p.zero_src) store_vec(s, valid, make_float4(0.f, 0.f, 0.f, 0.f));
    }
    float4* d = reinterpret_cast<float4*>(p.staging) + v;
    if (p.accumulate) {
      // staged += new  (src/accumulator.cc:975 targetGradients[i].add_(addGrads[i]))
      const float4 a = *d;
      g = make_float4(__fadd_rn(a.x, g.x), __fadd_rn(a.y, g.y), __fadd_rn(a.z, g.z), __fadd_rn(a.w, g.w));
    }
    *d = g;
  }
}

// ---- publish region: one-way bulk transfer of a tensor list between members (late-joiner model sync) -------------

struct UnpackParams {
  const float* src;  // the source rank's publish region (peer memory)
  const TensorEnt* tab;
  uint32_t ntensors;
  uint64_t total_vec;
};

// dst tensors <- flat layout in `src`, 4 x 16 B peer loads in flight per thread
__global__ void __launch_bounds__(kArThreads) ar_unpack_kernel(const __grid_constant__ UnpackParams p) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  const TensorTable tb = load_table(dyn_smem, p.tab, p.ntensors);
  __syncthreads();
  const uint64_t per_block = (p.total_vec + gridDim.x - 1) / gridDim.x;
  const uint64_t begin = (uint64_t)blockIdx.x * per_block;
  const uint64_t end = min(begin + per_block, p.total_vec);
  uint32_t cur = 0;
  for (uint64_t base = begin; base < end; base += 4ull * kArThreads) {
    float4 x[4];
    uint64_t v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[k] = base + (uint64_t)k * kArThreads + threadIdx.x;
      if (v[k] < end) x[k] = ld_peer_f4(p.src + v[k] * 4);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (v[k] < end) scatter_vec(tb, v[k], x[k], cur);
  }
}

// ---- barrier ----------------------------------------------------------------------------------------------------

// Bounded wait until *local >= epoch (relaxed system-scope polling; the caller fences).  Returns false on timeout/abort.
__device__ __forceinline__ bool wait_flag(const uint32_t* local, uint32_t epoch, uint64_t timeout_ns,
                                          const uint32_t* abort_flag) {
  // Poll with RELAXED system-scope loads and fence once after the flag is seen (relaxed load + acquire fence is an
  // acquire pattern).  An acquire load per poll is a system-scope fence per poll: hundreds of spinning threads doing
  // that slowed the peers' NVLink reads of this GPU's memory (bimodal 40 us / 150 us rounds at N=4).
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while ((int32_t)(ld_relaxed_sys_u32(local) - epoch) < 0) {
    __nanosleep(32);
    if ((++spins & 255u) == 0) {
      const uint64_t now = globaltimer_ns();
      if (t0 == 0) t0 = now;
      if (now - t0 > timeout_ns || ld_volatile_u32(abort_flag) != 0) return false;
    }
  }
  return true;
}

// Every block pairs with the same-numbered block on every peer.  Returns false on timeout / abort.
__device__ __forceinline__ bool block_barrier(const ArParams& p, bool second) {
  __syncthreads();  // the block's earlier writes happen-before the release below (cumulativity through bar.sync)
  const int t = threadIdx.x;
  int fail = 0;
  if (t < p.world && t != p.rank) {
    SyncBlock* peer = p.sync[t];
    uint32_t* remote = second ? &peer->flagsB[blockIdx.x][p.rank] : &peer->flagsA[blockIdx.x][p.rank];
    st_release_sys_u32(remote, p.epoch);
    SyncBlock* me = p.sync[p.rank];
    const uint32_t* local = second ? &me->flagsB[blockIdx.x][t] : &me->flagsA[blockIdx.x][t];
    if (!wait_flag(local, p.epoch, p.timeout_ns, p.abort_flag)) fail = 1;
    fence_acq_rel_sys();
  }
  return __syncthreads_or(fail) == 0;
}

__device__ __forceinline__ void report_failure(const ArParams& p) {
  if (threadIdx.x == 0) {
    p.result->status = MB_ETIMEOUT;
    p.result->epoch = p.epoch;
    __threadfence_system();
  }
}

// ---- K-A0 gate ---------------------------------------------------------------------------------------------------

// One warp.  Lane t handles peer t: push my header into its block, release my flag there, wait for its flag here.
__global__ void __launch_bounds__(32) ar_gate_kernel(const __grid_constant__ GateParams p) {
  const int t = threadIdx.x;
  const uint32_t par = p.epoch & 1u;
  int fail = 0;
  if (t < p.world && t != p.rank) {
    volatile mb_ar_hdr* h = &p.sync[t]->ghdr[par][p.rank];
    h->num_gradients = p.my_hdr.num_gradients;
    h->num_skipped = p.my_hdr.num_skipped;
    h->batch_size = p.my_hdr.batch_size;
    h->has_grads = p.my_hdr.has_grads;
    // release: the header stores above AND this stream's earlier kernels (the staged gradients) are visible to a
    // peer that acquires the flag
    st_release_sys_u32(&p.sync[t]->gate[p.rank], p.epoch);
    if (!wait_flag(&p.sync[p.rank]->gate[t], p.epoch, p.timeout_ns, p.abort_flag)) fail = 1;
    fence_acq_rel_sys();
  }
  fail = __any_sync(0xffffffffu, fail);
  if (t != 0) return;
  GateOut o;
  o.tot = mb_ar_hdr{0, 0, 0, 0};
  o.mask = 0;
  o.epoch = p.epoch;
  o.pad = 0;
  if (fail) {
    o.decision = 0;
    *p.out = o;
    p.result->status = MB_ETIMEOUT;
    p.result->epoch = p.epoch;
    __threadfence_system();
    return;
  }
  for (int r = 0; r < p.world; ++r) {
    uint64_t ng, ns, bs, hg;
    if (r == p.rank) {
      ng = p.my_hdr.num_gradients, ns = p.my_hdr.num_skipped, bs = p.my_hdr.batch_size, hg = p.my_hdr.has_grads;
    } else {
      const volatile mb_ar_hdr* ph = &p.sync[p.rank]->ghdr[par][r];
      ng = ph->num_gradients, ns = ph->num_skipped, bs = ph->batch_size, hg = ph->has_grads;
    }
    o.tot.num_gradients += ng;
    o.tot.num_skipped += ns;
    o.tot.batch_size += bs;
    if (hg) {
      o.mask |= 1u << r;
      o.tot.has_grads += 1;
    }
  }
  o.decision = o.tot.batch_size >= p.min_batch ? 1 : 0;
  *p.out = o;
  if (!o.decision) {
    // gate closed (src/accumulator.cc:1051: size < virtualBatchSize): nothing is reduced, the host counts again later
    p.result->sum = o.tot;
    p.result->status = MB_AR_SHORT;
    p.result->epoch = p.epoch;
  }
}

// After the first barrier: sum the peers' headers (u64 adds, src/group.h:209-211) and build the has-gradients mask.
__device__ __forceinline__ void gather_headers(const ArParams& p, mb_ar_hdr* s_total, uint32_t* s_mask) {
  if (threadIdx.x == 0) {
    mb_ar_hdr tot = {0, 0, 0, 0};
    uint32_t mask = 0;
    for (int r = 0; r < p.world; ++r) {
      uint64_t ng, ns, bs, hg;
      if (r == p.rank) {
        ng = p.my_hdr.num_gradients, ns = p.my_hdr.num_skipped, bs = p.my_hdr.batch_size, hg = p.my_hdr.has_grads;
      } else {
        const volatile mb_ar_hdr* ph = &p.sync[r]->hdr[p.epoch & 1u];
        ng = ph->num_gradients, ns = ph->num_skipped, bs = ph->batch_size, hg = ph->has_grads;
      }
      tot.num_gradients += ng;
      tot.num_skipped += ns;
      tot.batch_size += bs;
      if (hg) {
        mask |= 1u << r;
        tot.has_grads += 1;
      }
    }
    *s_total = tot;
    *s_mask = mask;
  }
  __syncthreads();
}

__device__ __forceinline__ void publish_header(const ArParams& p) {
  // every block writes the same value; the block's own release (block_barrier) orders it before its flag
  if (threadIdx.x == 0) {
    volatile mb_ar_hdr* h = &p.sync[p.rank]->hdr[p.epoch & 1u];
    h->num_gradients = p.my_hdr.num_gradients;
    h->num_skipped = p.my_hdr.num_skipped;
    h->batch_size = p.my_hdr.batch_size;
    h->has_grads = p.my_hdr.has_grads;
  }
}

// Common prologue of the reduce kernels.  Ungated: publish header, per-block barrier with every peer, sum headers.
// Gated: K-A0 already did all of that once for the whole GPU; read its verdict.  Returns false when the kernel must
// return (barrier failure, or gate closed).
__device__ __forceinline__ bool reduce_prologue(const ArParams& p, mb_ar_hdr* s_total, uint32_t* s_mask) {
  if (p.gate) {
    __shared__ int s_go;
    if (threadIdx.x == 0) {
      const GateOut g = *p.gate;
      s_go = g.decision && g.epoch == p.epoch;
      *s_total = g.tot;
      *s_mask = g.mask;
    }
    __syncthreads();
    return s_go != 0;
  }
  publish_header(p);
  if (!block_barrier(p, false)) {
    report_failure(p);
    return false;
  }
  gather_headers(p, s_total, s_mask);
  return true;
}

__device__ __forceinline__ float reduce_scale(const ArParams& p, const mb_ar_hdr& tot) {
  // fp32 reciprocal then fp32 multiply, exactly as grad.mul_(1.0f / data.numGradients) (src/accumulator.cc:442)
  if (!p.scale || tot.num_gradients == 0) return 1.0f;
  return __fdiv_rn(1.0f, (float)tot.num_gradients);
}

__device__ __forceinline__ void add4(float4& a, const float4& b) {
  a.x = __fadd_rn(a.x, b.x);
  a.y = __fadd_rn(a.y, b.y);
  a.z = __fadd_rn(a.z, b.z);
  a.w = __fadd_rn(a.w, b.w);
}

// Sum of element v over the ranks in `mask`, ascending rank order, fp32, for U vectors at once (v[k], k < U).  Fast
// path (every rank contributes): all U*NR loads are issued before the first add, so U*NR*16 B are in flight per thread
// -- NVLink latency is ~2 us, bandwidth needs megabytes in flight (B300_MICROARCH "NVLink").
template <int NR, int U>
__device__ __forceinline__ void reduce_vecs(float* const* stage, uint32_t mask, const uint64_t (&v)[U],
                                            float4 (&acc)[U]) {
  if (mask == (1u << NR) - 1u) {
    float4 x[U][NR];
#pragma unroll
    for (int k = 0; k < U; ++k)
#pragma unroll
      for (int r = 0; r < NR; ++r) x[k][r] = ld_peer_f4(stage[r] + v[k] * 4);
#pragma unroll
    for (int k = 0; k < U; ++k) {
      acc[k] = x[k][0];
#pragma unroll
      for (int r = 1; r < NR; ++r) add4(acc[k], x[k][r]);
    }
    return;
  }
  // some ranks skipped (src/group.h:206-208: the side without gradients adopts the other's): sequential, rare
#pragma unroll
  for (int k = 0; k < U; ++k) {
    acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    bool first = true;
#pragma unroll 1
    for (int r = 0; r < NR; ++r) {
      if (!(mask & (1u << r))) continue;
      const float4 x = ld_peer_f4(stage[r] + v[k] * 4);
      if (first) {
        acc[k] = x;
        first = false;
      } else {
        add4(acc[k], x);
      }
    }
  }
}

// Default unroll: U*NR = 16 loads of 16 B in flight per thread.
constexpr int default_unroll(int nr) { return nr >= 8 ? 2 : nr >= 4 ? 4 : 8; }

__device__ __forceinline__ float4 scale_vec(const float4& a, float s, bool do_scale) {
  if (!do_scale) return a;
  return make_float4(__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s), __fmul_rn(a.w, s));
}

__device__ __forceinline__ void write_result(const ArParams& p, const mb_ar_hdr& tot) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    // plain stores to the host-mapped result block: the host reads it only after an event behind this kernel has
    // completed, and kernel completion makes them visible -- a system fence here costs ~2 us of a ~8 us kernel
    p.result->sum = tot;
    p.result->status = MB_OK;
    p.result->epoch = p.epoch;
  }
}

// Destination of the reduced vectors: the flat result buffer (ntensors == 0) or the tensor list.
struct Sink {
  TensorTable tb;
  float* flat;
  uint32_t cur;
  __device__ __forceinline__ void put(uint64_t v, const float4& r) {
    if (flat) st_f4(flat + v * 4, r);
    else scatter_vec(tb, v, r, cur);
  }
};

__device__ __forceinline__ Sink make_sink(const ArParams& p, uint8_t* smem) {
  Sink s;
  s.cur = 0;
  if (p.ntensors == 0) {
    s.flat = p.flat_dst;
    s.tb = TensorTable{nullptr, nullptr, nullptr, 0};
  } else {
    s.flat = nullptr;
    s.tb = load_table(smem, p.dst_tab, p.ntensors);
  }
  return s;
}

// ---- K-A2 one-shot ----------------------------------------------------------------------------------------------

template <int NR, int U>
__global__ void __launch_bounds__(kArThreads, 1) ar_oneshot_kernel(const __grid_constant__ ArParams p) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  __shared__ mb_ar_hdr s_total;
  __shared__ uint32_t s_mask;
  Sink sink = make_sink(p, dyn_smem);
  if (!reduce_prologue(p, &s_total, &s_mask)) return;
  const uint32_t mask = s_mask;
  const mb_ar_hdr tot = s_total;
  const bool do_scale = p.scale && tot.num_gradients != 0;
  const float s = reduce_scale(p, tot);
  // Each block-iteration owns a contiguous chunk of U*512 vectors (U*8 KiB): thread t handles chunk[k*512 + t],
  // k < U, all U*NR peer loads in flight before the first add.  (Lanes must never be clamped to a common address:
  // thousands of threads loading one peer line serialise on NVLink -- measured 10x slowdowns.)
  const uint32_t nthr = blockDim.x;  // 512, or 256 / 128 for small messages so that every SM gets a chunk
  const uint64_t kChunk = (uint64_t)U * nthr;
  for (uint64_t base = (uint64_t)blockIdx.x * kChunk; base < p.total_vec; base += (uint64_t)gridDim.x * kChunk) {
    if (base + kChunk <= p.total_vec && !p.force_u1) {
      uint64_t v[U];
      float4 r[U];
#pragma unroll
      for (int k = 0; k < U; ++k) v[k] = base + (uint64_t)k * nthr + threadIdx.x;
      reduce_vecs<NR, U>(p.stage, mask, v, r);  // mask == 0 -> zeros (src/accumulator.cc:426-428)
#pragma unroll
      for (int k = 0; k < U; ++k) sink.put(v[k], scale_vec(r[k], s, do_scale));
    } else {
      const uint64_t cend = min(base + kChunk, p.total_vec);
      for (uint64_t v0 = base + threadIdx.x; v0 < cend; v0 += nthr) {
        uint64_t v[1] = {v0};
        float4 r[1];
        reduce_vecs<NR, 1>(p.stage, mask, v, r);
        sink.put(v0, scale_vec(r[0], s, do_scale));
      }
    }
  }
  write_result(p, tot);
}

// ---- K-A2 two-shot ----------------------------------------------------------------------------------------------

template <int NR, int U>
__global__ void __launch_bounds__(kArThreads, 1) ar_twoshot_kernel(const __grid_constant__ ArParams p) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  __shared__ mb_ar_hdr s_total;
  __shared__ uint32_t s_mask;
  Sink sink = make_sink(p, dyn_smem);
  if (!reduce_prologue(p, &s_total, &s_mask)) return;
  const uint32_t mask = s_mask;
  const mb_ar_hdr tot = s_total;
  const bool do_scale = p.scale && tot.num_gradients != 0;
  const float s = reduce_scale(p, tot);
  const uint32_t nthr = blockDim.x;
  const uint64_t kChunk = (uint64_t)U * nthr;
  const uint64_t gstride = (uint64_t)gridDim.x * kChunk;
  // phase 1: reduce my slice and write it into every peer's staging (in place: slice `rank` of a peer's staging is
  // read only by me, and I overwrite an element only after I have loaded it) and into my own.  Chunks are relative
  // to the slice start so that block b touches the same relative ranges of every slice on every rank.
  {
    const uint64_t sbase = (uint64_t)p.rank * p.slice_vec;
    const uint64_t slen = sbase < p.total_vec ? min(p.slice_vec, p.total_vec - sbase) : 0;
    auto emit = [&](uint64_t v, const float4& red) {
      const float4 o = scale_vec(red, s, do_scale);
#pragma unroll
      for (int q = 0; q < NR; ++q) st_f4(p.stage[q] + v * 4, o);
    };
    for (uint64_t cb = (uint64_t)blockIdx.x * kChunk; cb < slen; cb += gstride) {
      if (cb + kChunk <= slen && !p.force_u1) {
        uint64_t v[U];
        float4 r[U];
#pragma unroll
        for (int k = 0; k < U; ++k) v[k] = sbase + cb + (uint64_t)k * nthr + threadIdx.x;
        reduce_vecs<NR, U>(p.stage, mask, v, r);
#pragma unroll
        for (int k = 0; k < U; ++k) emit(v[k], r[k]);
      } else {
        const uint64_t cend = min(cb + kChunk, slen);
        for (uint64_t j = cb + threadIdx.x; j < cend; j += nthr) {
          uint64_t v[1] = {sbase + j};
          float4 r[1];
          reduce_vecs<NR, 1>(p.stage, mask, v, r);
          emit(v[0], r[0]);
        }
      }
    }
  }
  if (!block_barrier(p, true)) {
    report_failure(p);
    return;
  }
  if (p.inplace) {
    // the caller consumes the result from this rank's staging buffer itself: nothing left to move
    write_result(p, tot);
    return;
  }
  // phase 2: every slice is now complete in my own staging (mine included, written by this same block before the
  // barrier); block b reads exactly what the peers' block b wrote.  Slices ascend, so the sink's cursor only moves
  // forward.
  float* mine = p.stage[p.rank];
#pragma unroll 1
  for (int q = 0; q < NR; ++q) {
    const uint64_t sbase = (uint64_t)q * p.slice_vec;
    const uint64_t slen = sbase < p.total_vec ? min(p.slice_vec, p.total_vec - sbase) : 0;
    for (uint64_t cb = (uint64_t)blockIdx.x * kChunk; cb < slen; cb += gstride) {
      const uint64_t cend = min(cb + kChunk, slen);
      if (cb + kChunk <= slen) {
        float4 x[U];
#pragma unroll
        for (int k = 0; k < U; ++k) x[k] = ld_peer_f4(mine + (sbase + cb + (uint64_t)k * nthr + threadIdx.x) * 4);
#pragma unroll
        for (int k = 0; k < U; ++k) sink.put(sbase + cb + (uint64_t)k * nthr + threadIdx.x, x[k]);
      } else {
        for (uint64_t j = cb + threadIdx.x; j < cend; j += nthr) sink.put(sbase + j, ld_peer_f4(mine + (sbase + j) * 4));
      }
    }
  }
  write_result(p, tot);
}

using ArKernel = void (*)(const ArParams);

template <int NR, int U>
ArKernel pick(bool twoshot) {
  return twoshot ? (ArKernel)ar_twoshot_kernel<NR, U> : (ArKernel)ar_oneshot_kernel<NR, U>;
}

template <int NR>
ArKernel pick_unroll(bool twoshot, int unroll) {
  // U*NR <= 16 keeps the kernels under 128 registers at 512 threads
  if (unroll >= 8 && NR <= 2) return pick<NR, 8>(twoshot);
  if (unroll >= 4 && NR <= 4) return pick<NR, 4>(twoshot);
  if (unroll >= 2) return pick<NR, 2>(twoshot);
  return pick<NR, 1>(twoshot);
}

// Returns the kernel and the unroll it was instantiated with.
ArKernel kernel_for(int world, bool twoshot, int want_unroll, int* unroll_out) {
  int u = want_unroll >= 8 && world <= 2 ? 8 : want_unroll >= 4 && world <= 4 ? 4 : want_unroll >= 2 ? 2 : 1;
  *unroll_out = u;
  switch (world) {
    case 1: return pick_unroll<1>(twoshot, u);
    case 2: return pick_unroll<2>(twoshot, u);
    case 3: return pick_unroll<3>(twoshot, u);
    case 4: return pick_unroll<4>(twoshot, u);
    case 5: return pick_unroll<5>(twoshot, u);
    case 6: return pick_unroll<6>(twoshot, u);
    case 7: return pick_unroll<7>(twoshot, u);
    case 8: return pick_unroll<8>(twoshot, u);
  }
  return nullptr;
}

// ---- mixed-dtype lists (bf16 / fp16 segments) ---------------------------------------------------------------------
// The 16 B vector stays the unit of every load and store; only the arithmetic on a vector depends on the dtype run
// (segment) it lies in.  fp32 vectors are reduced exactly as above; a half-width vector is widened to 8 fp32 lanes,
// summed with __fadd_rn in rank order, scaled with __fmul_rn and rounded once (cvt.rn.{bf16,f16}x2.f32).  The tensor
// table of these kernels is in BYTES: TensorEnt.off = byte offset / 4 (so load_table's >> 2 still yields the first
// vector) and TensorEnt.numel = byte length.  All-fp32 lists never reach them (the _ex entry points route those to the
// kernels above).

struct SegInfo {
  uint64_t end[3];  // cumulative end of each segment in 16 B vectors (unused: ~0)
  int32_t dt[3];
};

struct ArSegParams {
  ArParams b;
  SegInfo seg;
};

struct StageSegParams {
  StageParams b;
  SegInfo seg;
};

__device__ __forceinline__ int seg_dtype(const SegInfo& s, uint64_t v) {
  return v < s.end[0] ? s.dt[0] : v < s.end[1] ? s.dt[1] : s.dt[2];
}

__device__ __forceinline__ uint4 ld_peer_u4(const uint4* p) {
  const float4 f = ld_peer_f4(reinterpret_cast<const float*>(p));
  return make_uint4(__float_as_uint(f.x), __float_as_uint(f.y), __float_as_uint(f.z), __float_as_uint(f.w));
}
__device__ __forceinline__ void st_u4(uint4* p, const uint4& v) {
  st_f4(reinterpret_cast<float*>(p),
        make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w)));
}

// 16 B <-> 8 fp32 lanes (half-width dtypes): bf16 widens with a shift, fp16 with cvt.f32.f16 (both exact)
__device__ __forceinline__ void widen8(int dt, const uint4& x, float (&f)[8]) {
  const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (dt == MB_DT_BF16) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    } else {
      __half2_raw r;
      r.x = (unsigned short)(w[i] & 0xffffu);
      r.y = (unsigned short)(w[i] >> 16);
      const float2 t = __half22float2(__half2(r));
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
}
__device__ __forceinline__ uint4 narrow8(int dt, const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (dt == MB_DT_BF16) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);  // cvt.rn.bf16x2.f32
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    } else {
      const __half2 h = __floats2half2_rn(f[2 * i], f[2 * i + 1]);  // cvt.rn.f16x2.f32
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// Sum of the NR vectors x[r] (ranks in `mask`, ascending), scaled, in the vector's dtype.  mask == 0 -> zeros.
template <int NR>
__device__ __forceinline__ uint4 combine_vec(int dt, const uint4 (&x)[NR], uint32_t mask, float s, bool do_scale) {
  const bool all = mask == (1u << NR) - 1u;
  if (dt == MB_DT_F32) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    bool first = true;
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      if (!all && !(mask & (1u << r))) continue;
      const float4 y = make_float4(__uint_as_float(x[r].x), __uint_as_float(x[r].y), __uint_as_float(x[r].z),
                                   __uint_as_float(x[r].w));
      if (first) acc = y;
      else add4(acc, y);
      first = false;
    }
    acc = scale_vec(acc, s, do_scale);
    return make_uint4(__float_as_uint(acc.x), __float_as_uint(acc.y), __float_as_uint(acc.z), __float_as_uint(acc.w));
  }
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  bool first = true;
#pragma unroll
  for (int r = 0; r < NR; ++r) {
    if (!all && !(mask & (1u << r))) continue;
    float y[8];
    widen8(dt, x[r], y);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = first ? y[j] : __fadd_rn(acc[j], y[j]);
    first = false;
  }
  if (do_scale) {
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = __fmul_rn(acc[j], s);
  }
  return narrow8(dt, acc);
}

// Reduce U vectors: all U*NR peer loads in flight before the first add (every rank contributes), or only the loads of
// the ranks in `mask` (skipping ranks: rare).  Results are already scaled and rounded to the vector's dtype.
template <int NR, int U>
__device__ __forceinline__ void reduce_vecs_seg(const ArSegParams& p, uint32_t mask, const uint64_t (&v)[U],
                                                float s, bool do_scale, uint4 (&out)[U]) {
  const uint4* const* stage = reinterpret_cast<const uint4* const*>(p.b.stage);
  uint4 x[U][NR];
  const bool all = mask == (1u << NR) - 1u;
#pragma unroll
  for (int k = 0; k < U; ++k)
#pragma unroll
    for (int r = 0; r < NR; ++r) x[k][r] = (all || (mask & (1u << r))) ? ld_peer_u4(stage[r] + v[k]) : make_uint4(0, 0, 0, 0);
#pragma unroll
  for (int k = 0; k < U; ++k) out[k] = combine_vec<NR>(seg_dtype(p.seg, v[k]), x[k], mask, s, do_scale);
}

// Byte-table destination: 16 B stores, or 2 B stores for a tensor's tail / an unaligned tensor.
__device__ __forceinline__ void scatter_bytes(const TensorTable& tb, uint64_t v, const uint4& r, uint32_t& cur) {
  seek_tensor(tb, (uint32_t)v, cur);
  const uint64_t within = (v - tb.off[cur]) * 16;
  const uint64_t nbytes = tb.numel[cur];
  if (within >= nbytes) return;  // padding-only vector (empty tensor)
  const uint64_t valid = nbytes - within;
  char* d = reinterpret_cast<char*>(tb.ptr[cur]) + within;
  if (valid >= 16 && (reinterpret_cast<uintptr_t>(d) & 15u) == 0) {
    st_u4(reinterpret_cast<uint4*>(d), r);
  } else {
    const uint16_t* h = reinterpret_cast<const uint16_t*>(&r);
    const int nh = valid >= 16 ? 8 : (int)(valid >> 1);
    for (int i = 0; i < nh; ++i) reinterpret_cast<uint16_t*>(d)[i] = h[i];
  }
}

struct SinkB {
  TensorTable tb;
  uint4* flat;
  uint32_t cur;
  __device__ __forceinline__ void put(uint64_t v, const uint4& r) {
    if (flat) st_u4(flat + v, r);
    else scatter_bytes(tb, v, r, cur);
  }
};

__device__ __forceinline__ SinkB make_sink_b(const ArParams& p, uint8_t* smem) {
  SinkB s;
  s.cur = 0;
  if (p.ntensors == 0) {
    s.flat = reinterpret_cast<uint4*>(p.flat_dst);
    s.tb = TensorTable{nullptr, nullptr, nullptr, 0};
  } else {
    s.flat = nullptr;
    s.tb = load_table(smem, p.dst_tab, p.ntensors);
  }
  return s;
}

template <int NR, int U>
__global__ void __launch_bounds__(kArThreads, 1) ar_oneshot_seg_kernel(const __grid_constant__ ArSegParams sp) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  __shared__ mb_ar_hdr s_total;
  __shared__ uint32_t s_mask;
  const ArParams& p = sp.b;
  SinkB sink = make_sink_b(p, dyn_smem);
  if (!reduce_prologue(p, &s_total, &s_mask)) return;
  const uint32_t mask = s_mask;
  const mb_ar_hdr tot = s_total;
  const bool do_scale = p.scale && tot.num_gradients != 0;
  const float s = reduce_scale(p, tot);
  const uint32_t nthr = blockDim.x;
  const uint64_t kChunk = (uint64_t)U * nthr;
  for (uint64_t base = (uint64_t)blockIdx.x * kChunk; base < p.total_vec; base += (uint64_t)gridDim.x * kChunk) {
    if (base + kChunk <= p.total_vec && !p.force_u1) {
      uint64_t v[U];
      uint4 r[U];
#pragma unroll
      for (int k = 0; k < U; ++k) v[k] = base + (uint64_t)k * nthr + threadIdx.x;
      reduce_vecs_seg<NR, U>(sp, mask, v, s, do_scale, r);
#pragma unroll
      for (int k = 0; k < U; ++k) sink.put(v[k], r[k]);
    } else {
      const uint64_t cend = min(base + kChunk, p.total_vec);
      for (uint64_t v0 = base + threadIdx.x; v0 < cend; v0 += nthr) {
        uint64_t v[1] = {v0};
        uint4 r[1];
        reduce_vecs_seg<NR, 1>(sp, mask, v, s, do_scale, r);
        sink.put(v0, r[0]);
      }
    }
  }
  write_result(p, tot);
}

// Same phases as ar_twoshot_kernel: the reduce-scatter stores the ROUNDED values, the all-gather and the local copy
// move bytes.
template <int NR, int U>
__global__ void __launch_bounds__(kArThreads, 1) ar_twoshot_seg_kernel(const __grid_constant__ ArSegParams sp) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  __shared__ mb_ar_hdr s_total;
  __shared__ uint32_t s_mask;
  const ArParams& p = sp.b;
  SinkB sink = make_sink_b(p, dyn_smem);
  if (!reduce_prologue(p, &s_total, &s_mask)) return;
  const uint32_t mask = s_mask;
  const mb_ar_hdr tot = s_total;
  const bool do_scale = p.scale && tot.num_gradients != 0;
  const float s = reduce_scale(p, tot);
  const uint32_t nthr = blockDim.x;
  const uint64_t kChunk = (uint64_t)U * nthr;
  const uint64_t gstride = (uint64_t)gridDim.x * kChunk;
  uint4* const* stage = reinterpret_cast<uint4* const*>(p.stage);
  {
    const uint64_t sbase = (uint64_t)p.rank * p.slice_vec;
    const uint64_t slen = sbase < p.total_vec ? min(p.slice_vec, p.total_vec - sbase) : 0;
    for (uint64_t cb = (uint64_t)blockIdx.x * kChunk; cb < slen; cb += gstride) {
      if (cb + kChunk <= slen && !p.force_u1) {
        uint64_t v[U];
        uint4 r[U];
#pragma unroll
        for (int k = 0; k < U; ++k) v[k] = sbase + cb + (uint64_t)k * nthr + threadIdx.x;
        reduce_vecs_seg<NR, U>(sp, mask, v, s, do_scale, r);
#pragma unroll
        for (int k = 0; k < U; ++k)
#pragma unroll
          for (int q = 0; q < NR; ++q) st_u4(stage[q] + v[k], r[k]);
      } else {
        const uint64_t cend = min(cb + kChunk, slen);
        for (uint64_t j = cb + threadIdx.x; j < cend; j += nthr) {
          uint64_t v[1] = {sbase + j};
          uint4 r[1];
          reduce_vecs_seg<NR, 1>(sp, mask, v, s, do_scale, r);
#pragma unroll
          for (int q = 0; q < NR; ++q) st_u4(stage[q] + v[0], r[0]);
        }
      }
    }
  }
  if (!block_barrier(p, true)) {
    report_failure(p);
    return;
  }
  if (p.inplace) {
    write_result(p, tot);
    return;
  }
  const uint4* mine = stage[p.rank];
#pragma unroll 1
  for (int q = 0; q < NR; ++q) {
    const uint64_t sbase = (uint64_t)q * p.slice_vec;
    const uint64_t slen = sbase < p.total_vec ? min(p.slice_vec, p.total_vec - sbase) : 0;
    for (uint64_t cb = (uint64_t)blockIdx.x * kChunk; cb < slen; cb += gstride) {
      const uint64_t cend = min(cb + kChunk, slen);
      if (cb + kChunk <= slen) {
        uint4 x[U];
#pragma unroll
        for (int k = 0; k < U; ++k) x[k] = ld_peer_u4(mine + sbase + cb + (uint64_t)k * nthr + threadIdx.x);
#pragma unroll
        for (int k = 0; k < U; ++k) sink.put(sbase + cb + (uint64_t)k * nthr + threadIdx.x, x[k]);
      } else {
        for (uint64_t j = cb + threadIdx.x; j < cend; j += nthr) sink.put(sbase + j, ld_peer_u4(mine + sbase + j));
      }
    }
  }
  write_result(p, tot);
}

using ArSegKernel = void (*)(const ArSegParams);

template <int NR, int U>
ArSegKernel pick_seg(bool twoshot) {
  return twoshot ? (ArSegKernel)ar_twoshot_seg_kernel<NR, U> : (ArSegKernel)ar_oneshot_seg_kernel<NR, U>;
}

// Same U x NR table as pick_unroll, but only the reachable pairs are instantiated: eight fp32 accumulators per
// half-width vector make the unreachable ones (e.g. U=8 at NR=8) spill at 512 threads.
template <int NR>
ArSegKernel pick_unroll_seg(bool twoshot, int unroll) {
  if constexpr (NR <= 2) {
    if (unroll >= 8) return pick_seg<NR, 8>(twoshot);
  }
  if constexpr (NR <= 4) {
    if (unroll >= 4) return pick_seg<NR, 4>(twoshot);
  }
  if (unroll >= 2) return pick_seg<NR, 2>(twoshot);
  return pick_seg<NR, 1>(twoshot);
}

ArSegKernel kernel_for_seg(int world, bool twoshot, int want_unroll, int* unroll_out) {
  int u = want_unroll >= 8 && world <= 2 ? 8 : want_unroll >= 4 && world <= 4 ? 4 : want_unroll >= 2 ? 2 : 1;
  *unroll_out = u;
  switch (world) {
    case 1: return pick_unroll_seg<1>(twoshot, u);
    case 2: return pick_unroll_seg<2>(twoshot, u);
    case 3: return pick_unroll_seg<3>(twoshot, u);
    case 4: return pick_unroll_seg<4>(twoshot, u);
    case 5: return pick_unroll_seg<5>(twoshot, u);
    case 6: return pick_unroll_seg<6>(twoshot, u);
    case 7: return pick_unroll_seg<7>(twoshot, u);
    case 8: return pick_unroll_seg<8>(twoshot, u);
  }
  return nullptr;
}

// K-A1 for mixed lists: staging (=|+=) sources, per 16 B vector; += rounds in the dtype (ATen's add_ on bf16 / fp16
// computes in fp32 and rounds once).
__global__ void __launch_bounds__(kArThreads) ar_stage_seg_kernel(const __grid_constant__ StageSegParams sp) {
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  const StageParams& p = sp.b;
  const TensorTable tb = load_table(dyn_smem, p.tab, p.ntensors);
  __syncthreads();
  const uint64_t per_block = (p.total_vec + gridDim.x - 1) / gridDim.x;
  const uint64_t begin = (uint64_t)blockIdx.x * per_block;
  const uint64_t end = min(begin + per_block, p.total_vec);
  uint32_t cur = 0;
  for (uint64_t v = begin + threadIdx.x; v < end; v += kArThreads) {
    seek_tensor(tb, (uint32_t)v, cur);
    const uint64_t within = (v - tb.off[cur]) * 16;
    const uint64_t nbytes = tb.numel[cur];
    uint4 g = make_uint4(0, 0, 0, 0);
    if (within < nbytes) {
      char* s = reinterpret_cast<char*>(tb.ptr[cur]) + within;
      const uint64_t valid = nbytes - within;
      if (valid >= 16 && (reinterpret_cast<uintptr_t>(s) & 15u) == 0) {
        g = *reinterpret_cast<const uint4*>(s);
        if (p.zero_src) *reinterpret_cast<uint4*>(s) = make_uint4(0, 0, 0, 0);
      } else {
        uint16_t* h = reinterpret_cast<uint16_t*>(&g);
        const int nh = valid >= 16 ? 8 : (int)(valid >> 1);
        for (int i = 0; i < nh; ++i) {
          h[i] = reinterpret_cast<const uint16_t*>(s)[i];
          if (p.zero_src) reinterpret_cast<uint16_t*>(s)[i] = 0;
        }
      }
    }
    uint4* d = reinterpret_cast<uint4*>(p.staging) + v;
    if (p.accumulate) {
      const uint4 a = *d;
      const int dt = seg_dtype(sp.seg, v);
      if (dt == MB_DT_F32) {
        g = make_uint4(__float_as_uint(__fadd_rn(__uint_as_float(a.x), __uint_as_float(g.x))),
                       __float_as_uint(__fadd_rn(__uint_as_float(a.y), __uint_as_float(g.y))),
                       __float_as_uint(__fadd_rn(__uint_as_float(a.z), __uint_as_float(g.z))),
                       __float_as_uint(__fadd_rn(__uint_as_float(a.w), __uint_as_float(g.w))));
      } else {
        float fa[8], fg[8];
        widen8(dt, a, fa);
        widen8(dt, g, fg);
#pragma unroll
        for (int j = 0; j < 8; ++j) fa[j] = __fadd_rn(fa[j], fg[j]);
        g = narrow8(dt, fa);
      }
    }
    *d = g;
  }
}

// ---- host helpers ------------------------------------------------------------------------------------------------

constexpr int kBufs = MB_AR_BUFS_PER_SLOT;

uint64_t flat_layout(const uint64_t* numel, int n) {
  uint64_t off = 0;
  for (int i = 0; i < n; ++i) off += (numel[i] + 3) & ~3ull;
  return off;
}

// Bring the device copy of tensor table `which` up to date with (ptrs, numel).  The cached host copy is compared in
// place (no allocation when nothing changed -- the steady state: the same .grad tensors every step).
int sync_table(mb_ar_ctx* ctx, int which, const void* const* ptrs, const uint64_t* numel, int n, uint64_t* total_out,
               cudaStream_t stream) {
  auto& cache = ctx->tab_host[which];
  bool same = cache.size() == (size_t)n && !ctx->tab_bytes[which];
  uint64_t off = 0;
  for (int i = 0; i < n; ++i) {
    if (same) {
      const TensorEnt& e = cache[i];
      same = e.ptr == reinterpret_cast<uint64_t>(ptrs[i]) && e.numel == numel[i] && e.off == off;
    }
    off += (numel[i] + 3) & ~3ull;
  }
  *total_out = off;
  if (same) return MB_OK;
  ctx->tab_bytes[which] = false;
  cache.resize(n);
  off = 0;
  for (int i = 0; i < n; ++i) {
    cache[i] = TensorEnt{reinterpret_cast<uint64_t>(ptrs[i]), off, numel[i]};
    off += (numel[i] + 3) & ~3ull;
  }
  if (n > 0) {
    // pageable source: the runtime stages it before returning, and the copy is ordered on `stream` after any kernel
    // still reading the previous table
    MB_CUDA(cudaMemcpyAsync(ctx->tab_dev[which], cache.data(), (size_t)n * sizeof(TensorEnt), cudaMemcpyHostToDevice,
                            stream));
  }
  return MB_OK;
}

// mb_ar_layout: dtype runs in the order fp32, bf16, fp16, list order inside a run, every tensor 16 B aligned.
int layout_ex(const uint64_t* numel, const int32_t* dtype, int n, uint64_t* off, uint64_t* total, mb_ar_segment* segs) {
  static const int32_t kOrder[3] = {MB_DT_F32, MB_DT_BF16, MB_DT_F16};
  uint64_t at = 0;
  int nseg = 0;
  for (int32_t d : kOrder) {
    const uint64_t begin = at, esize = d == MB_DT_F32 ? 4 : 2;
    for (int i = 0; i < n; ++i) {
      if (dtype[i] != d) continue;
      if (off) off[i] = at;
      at += (numel[i] * esize + 15) & ~15ull;
    }
    if (at > begin) {
      if (segs) segs[nseg] = mb_ar_segment{begin, at, d, 0};
      ++nseg;
    }
  }
  if (total) *total = at;
  return nseg;
}

SegInfo seg_info(const mb_ar_segment* segs, int nseg) {
  SegInfo si;
  for (int k = 0; k < 3; ++k) {
    si.end[k] = k < nseg ? segs[k].end / 16 : ~0ull;
    si.dt[k] = k < nseg ? segs[k].dtype : (nseg ? segs[nseg - 1].dtype : MB_DT_F32);
  }
  return si;
}

// Validates a dtype array; *all_f32 = every tensor is fp32 (the list then runs the fp32 entry points unchanged).
int check_dtypes(const char* fn, const int32_t* dtype, int n, bool* all_f32) {
  *all_f32 = true;
  for (int i = 0; i < n; ++i) {
    MB_CHECK_ARG(dtype[i] == MB_DT_F32 || dtype[i] == MB_DT_BF16 || dtype[i] == MB_DT_F16,
                 "%s: tensor %d has dtype %d; supported: MB_DT_F32, MB_DT_BF16, MB_DT_F16", fn, i, (int)dtype[i]);
    if (dtype[i] != MB_DT_F32) *all_f32 = false;
  }
  return MB_OK;
}

// Byte-table variant of sync_table for mixed lists: entries in layout (offset) order, {ptr, byte offset / 4, bytes}.
int sync_table_bytes(mb_ar_ctx* ctx, int which, const void* const* ptrs, const uint64_t* numel, const int32_t* dtype,
                     int n, const uint64_t* off, cudaStream_t stream) {
  std::vector<TensorEnt> ents;
  ents.reserve(n);
  for (int32_t d : {MB_DT_F32, MB_DT_BF16, MB_DT_F16})
    for (int i = 0; i < n; ++i)
      if (dtype[i] == d)
        ents.push_back(TensorEnt{reinterpret_cast<uint64_t>(ptrs[i]), off[i] / 4, numel[i] * (d == MB_DT_F32 ? 4 : 2)});
  auto& cache = ctx->tab_host[which];
  bool same = ctx->tab_bytes[which] && cache.size() == ents.size();
  for (size_t i = 0; same && i < ents.size(); ++i)
    same = cache[i].ptr == ents[i].ptr && cache[i].off == ents[i].off && cache[i].numel == ents[i].numel;
  if (same) return MB_OK;
  cache.swap(ents);
  ctx->tab_bytes[which] = true;
  if (n > 0)
    MB_CUDA(cudaMemcpyAsync(ctx->tab_dev[which], cache.data(), (size_t)n * sizeof(TensorEnt), cudaMemcpyHostToDevice,
                            stream));
  return MB_OK;
}

float* ring_buffer(mb_ar_ctx* ctx, float* base, int slot, int ahead) {
  const uint64_t floats = ctx->max_bytes / 4;
  return base + ((uint64_t)slot * kBufs + (uint64_t)((ctx->parity[slot] + ahead) % kBufs)) * floats;
}

uint64_t env_u64(const char* name, uint64_t dflt) {
  const char* e = std::getenv(name);
  if (!e || !*e) return dflt;
  return std::strtoull(e, nullptr, 0);
}

uint64_t twoshot_min_bytes(int world) {
  // below this the one-shot kernel (no mid barrier) wins; above it the (N-1)x ingress dominates.
  // MB_AR_TWOSHOT_MIN_BYTES overrides (measured crossovers are recorded in DESIGN.md).
  static const uint64_t forced = env_u64("MB_AR_TWOSHOT_MIN_BYTES", 0);
  if (forced) return forced;
  if (world <= 2) return ~0ull;  // two-shot moves the same bytes as one-shot at N=2
  if (world <= 4) return 4ull << 20;  // measured on 4 B200: 1 MB 32 vs 36 us, 4.4 MB 51 vs 50 us, 16 MB 114 vs 80 us
  return 1ull << 20;
}

std::mutex g_smem_mu;

int ensure_dyn_smem(const void* fn, size_t bytes) {
  if (bytes <= 48 * 1024) return MB_OK;
  std::lock_guard<std::mutex> l(g_smem_mu);
  MB_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return MB_OK;
}

size_t table_bytes(uint32_t n) { return (size_t)n * (8 + 8 + 4); }

// A mixed-dtype round whose byte table (tab_dev[1]) is already uploaded: see launch_reduce.
struct SegLaunch {
  uint64_t total_vec;
  uint32_t ntab;  // 0: the result goes to `flat`
  void* flat;
  SegInfo info;
};

// Shared by mb_ar_allreduce (ungated: in-kernel per-block barrier) and mb_ar_reduce_gated (K-A0 + barrier-free reduce),
// and by their _ex variants for lists with bf16 / fp16 segments (seg != nullptr: dst / numel / flat_* are unused).
int launch_reduce(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, float* const* dst, const uint64_t* numel,
                  int ntensors, float* flat_dst, uint64_t flat_numel, int scale, int algo, uint32_t timeout_ms,
                  bool gated, uint64_t min_batch, cudaStream_t stream, const SegLaunch* seg = nullptr) {
  uint64_t total = 0;
  uint32_t ntab = 0;
  float* flat_sink = nullptr;
  const bool timed_round = gated;
  if (seg) {
    total = seg->total_vec * 4;
    ntab = seg->ntab;
    flat_sink = static_cast<float*>(seg->flat);
  } else if (dst) {
    MB_CHECK_ARG(numel != nullptr, "mb_ar_allreduce: numel is null");
    MB_CHECK_ARG(ntensors >= 1 && ntensors <= kArMaxTensors, "mb_ar_allreduce: ntensors %d not in [1,%d]", ntensors,
                 kArMaxTensors);
    int rc = sync_table(ctx, 1, reinterpret_cast<const void* const*>(dst), numel, ntensors, &total, stream);
    if (rc) return rc;
    ntab = (uint32_t)ntensors;
  } else {
    MB_CHECK_ARG(flat_dst != nullptr, "mb_ar_allreduce: neither dst nor flat_dst given");
    if ((flat_numel & 3u) == 0 && (reinterpret_cast<uintptr_t>(flat_dst) & 15u) == 0) {
      // whole float4 vectors, vector-aligned: the kernel stores straight into it, no table
      total = flat_numel;
      flat_sink = flat_dst;
    } else {
      const void* ptr = flat_dst;
      int rc = sync_table(ctx, 1, &ptr, &flat_numel, 1, &total, stream);
      if (rc) return rc;
      ntab = 1;
    }
  }
  MB_CHECK_ARG(total * 4 <= ctx->max_bytes, "mb_ar_allreduce: %llu bytes exceed the context's max_bytes %llu",
               (unsigned long long)(total * 4), (unsigned long long)ctx->max_bytes);
  MB_CHECK_ARG(total < (1ull << 33), "mb_ar_allreduce: tensor list too large");
  for (int r = 0; r < ctx->world; ++r) {
    if (!ctx->imported[r]) {
      set_error("mb_ar_allreduce: peer %d has not been imported", r);
      return MB_ESTATE;
    }
  }
  const uint64_t timeout_ns = (uint64_t)(timeout_ms ? timeout_ms : 30000u) * 1000000ull;
  const uint32_t epoch = ++ctx->epoch;
  int launches = 0;

  if (gated && ctx->world == 1) {
    // single member (src/group.h:738-741 short-circuit): the gate is a host-side comparison
    if (my_hdr->batch_size < min_batch) {
      HostResult* r = ctx->result_host + slot;
      r->sum = *my_hdr;
      r->sum.has_grads = my_hdr->has_grads ? 1 : 0;
      r->status = MB_AR_SHORT;
      r->epoch = epoch;
      ctx->ev_valid[slot] = false;
      return 0;
    }
    gated = false;  // the N=1 reduce kernel has no barrier to skip
  }
  // the context's own events bracket the two launches of a gated round (mb_ar_round_times): the wait for the slowest
  // peer (K-A0) and the data movement (K-A2) are told apart without the host handing event handles across the ABI
  const bool timed = timed_round;
  if (timed) MB_CUDA(cudaEventRecord(ctx->ev[slot][0], stream));
  if (gated) {
    GateParams g;
    std::memset(&g, 0, sizeof(g));
    for (int r = 0; r < ctx->world; ++r) g.sync[r] = ctx->peer_sync[r];
    g.out = ctx->gate_out + slot;
    g.result = ctx->result_dev + slot;
    g.abort_flag = ctx->abort_dev;
    g.my_hdr = *my_hdr;
    g.my_hdr.has_grads = my_hdr->has_grads ? 1 : 0;
    g.min_batch = min_batch;
    g.timeout_ns = timeout_ns;
    g.epoch = epoch;
    g.rank = ctx->rank;
    g.world = ctx->world;
    ar_gate_kernel<<<1, 32, 0, stream>>>(g);
    MB_CUDA(cudaGetLastError());
    ++launches;
  }
  if (timed) MB_CUDA(cudaEventRecord(ctx->ev[slot][1], stream));

  ArParams p;
  std::memset(&p, 0, sizeof(p));
  for (int r = 0; r < ctx->world; ++r) {
    p.stage[r] = ring_buffer(ctx, ctx->peer_staging[r], slot, 0);
    p.sync[r] = ctx->peer_sync[r];
  }
  p.dst_tab = ctx->tab_dev[1];
  p.flat_dst = flat_sink;
  p.gate = gated ? ctx->gate_out + slot : nullptr;
  p.ntensors = ntab;
  p.epoch = epoch;
  p.total_vec = total / 4;
  p.slice_vec = (p.total_vec + ctx->world - 1) / ctx->world;
  p.my_hdr = *my_hdr;
  p.my_hdr.has_grads = my_hdr->has_grads ? 1 : 0;
  p.rank = ctx->rank;
  p.world = ctx->world;
  p.scale = scale ? 1 : 0;
  p.result = ctx->result_dev + slot;
  p.abort_flag = ctx->abort_dev;
  p.timeout_ns = timeout_ns;

  bool twoshot = false;
  if (ctx->world > 1) {
    if (algo == MB_AR_ALGO_TWOSHOT) twoshot = true;
    else if (algo == MB_AR_ALGO_AUTO) twoshot = total * 4 >= twoshot_min_bytes(ctx->world);
  }
  if (!twoshot && ctx->world > 1 && flat_sink != nullptr && flat_sink == p.stage[ctx->rank]) {
    set_error("mb_ar_allreduce: an in-place destination (this rank's staging) needs the two-shot algorithm");
    return MB_EINVAL;
  }
  const int sms = sm_count(ctx->device);
  if (sms <= 0) return MB_ECUDA;
  const uint64_t work_vec = twoshot ? p.slice_vec : p.total_vec;
  // One CTA per SM: with two, the per-block barrier pairs (block b <-> block b on every peer) run in two waves that start
  // at different times on different GPUs; measured on 2 B200: 8-64 MB rounds became bimodal (43 us vs 370 us).
  static const uint64_t blocks_per_sm = env_u64("MB_AR_BLOCKS_PER_SM", 1);
  static const uint64_t force_u1 = env_u64("MB_AR_FORCE_U1", 0);
  static const uint64_t env_unroll = env_u64("MB_AR_UNROLL", 0);
  const uint64_t max_grid = std::min<uint64_t>((uint64_t)sms * blocks_per_sm, kArMaxBlocks);
  // Unroll: as many loads in flight per thread as fit (U*NR = 16), but never so coarse that SMs stay idle: a 4.4 MB
  // gradient set at U=8 is only 67 chunks -- 67 of 148 SMs pulling over NVLink.
  // Few chunks (a 4.4 MB gradient set is a 0.55 MB slice per rank at N=8): shrink the CTAs before giving up SMs --
  // 256- or 128-thread CTAs with one vector per thread keep all 148 SMs pulling over NVLink.
  static const uint64_t env_threads = env_u64("MB_AR_THREADS", 0);
  int want_unroll = env_unroll ? (int)env_unroll : default_unroll(ctx->world);
  uint32_t threads = env_threads ? (uint32_t)env_threads : (uint32_t)kArThreads;
  auto chunks = [&](uint32_t thr, int u) { return (work_vec + (uint64_t)thr * u - 1) / ((uint64_t)thr * u); };
  if (!env_unroll)
    while (want_unroll > 1 && chunks(threads, want_unroll) < max_grid) want_unroll >>= 1;
  if (!env_threads)
    while (threads > 128 && chunks(threads, want_unroll) < max_grid) threads >>= 1;
  int unroll = 1;
  ArKernel k = nullptr;
  ArSegKernel ks = nullptr;
  if (seg) ks = kernel_for_seg(ctx->world, twoshot, want_unroll, &unroll);
  else k = kernel_for(ctx->world, twoshot, want_unroll, &unroll);
  const uint64_t chunk = (uint64_t)threads * unroll;
  uint64_t want = (work_vec + chunk - 1) / chunk;
  if (want == 0) want = 1;
  p.force_u1 = (int32_t)force_u1;
  p.inplace = (twoshot && flat_sink != nullptr && flat_sink == p.stage[ctx->rank]) ? 1 : 0;
  const uint32_t grid = (uint32_t)std::min<uint64_t>(want, max_grid);
  const size_t smem = table_bytes(ntab);
  if (seg) {
    int rc = ensure_dyn_smem(reinterpret_cast<const void*>(ks), smem);
    if (rc) return rc;
    ArSegParams sp;
    sp.b = p;
    sp.seg = seg->info;
    ks<<<grid, threads, smem, stream>>>(sp);
  } else {
    int rc = ensure_dyn_smem(reinterpret_cast<const void*>(k), smem);
    if (rc) return rc;
    k<<<grid, threads, smem, stream>>>(p);
  }
  MB_CUDA(cudaGetLastError());
  if (timed) {
    MB_CUDA(cudaEventRecord(ctx->ev[slot][2], stream));
    ctx->ev_valid[slot] = true;
  }
  return launches + 1;
}

}  // namespace
}  // namespace mb

using namespace mb;

extern "C" {

uint64_t mb_ar_flat_numel(const uint64_t* numel, int ntensors) {
  if (!numel || ntensors <= 0) return 0;
  return flat_layout(numel, ntensors);
}

int mb_ar_ctx_create(int rank, int world, int device, uint64_t max_bytes, int nslots, mb_ar_ctx** out) {
  MB_CHECK_ARG(out != nullptr, "mb_ar_ctx_create: out is null");
  *out = nullptr;
  MB_CHECK_ARG(world >= 1 && world <= MB_AR_MAX_WORLD, "mb_ar_ctx_create: world %d not in [1,%d]", world,
               MB_AR_MAX_WORLD);
  MB_CHECK_ARG(rank >= 0 && rank < world, "mb_ar_ctx_create: rank %d not in [0,%d)", rank, world);
  MB_CHECK_ARG(nslots >= 1 && nslots <= MB_AR_MAX_SLOTS, "mb_ar_ctx_create: nslots %d not in [1,%d]", nslots,
               MB_AR_MAX_SLOTS);
  MB_CHECK_ARG(max_bytes > 0, "mb_ar_ctx_create: max_bytes is 0");
  DeviceGuard g(device);
  if (!g.ok) return cuda_fail(cudaGetLastError(), "cudaSetDevice", __FILE__, __LINE__);
  mb_ar_ctx* ctx = new (std::nothrow) mb_ar_ctx();
  if (!ctx) return MB_ENOMEM;
  ctx->rank = rank;
  ctx->world = world;
  ctx->device = device;
  ctx->nslots = nslots;
  ctx->max_bytes = (max_bytes + 15) & ~15ull;
  auto fail = [&](int rc) {
    mb_ar_ctx_destroy(ctx);
    return rc;
  };
#define MB_TRY(expr)                                                                  \
  do {                                                                                \
    cudaError_t e__ = (expr);                                                         \
    if (e__ != cudaSuccess) return fail(cuda_fail(e__, #expr, __FILE__, __LINE__));   \
  } while (0)
  ctx->xfer_offset = (ctx->max_bytes * kBufs * (uint64_t)nslots + 255) & ~255ull;
  const uint64_t staging_bytes = (ctx->xfer_offset + ctx->max_bytes + 255) & ~255ull;
  ctx->sync_offset = staging_bytes;
  ctx->block_bytes = (staging_bytes + sizeof(SyncBlock) + (2ull << 20) - 1) & ~((2ull << 20) - 1);
  MB_TRY(cudaMalloc(&ctx->block, ctx->block_bytes));
  MB_TRY(cudaMemset(ctx->block, 0, ctx->block_bytes));
  ctx->staging = static_cast<float*>(ctx->block);
  ctx->sync = reinterpret_cast<SyncBlock*>(static_cast<char*>(ctx->block) + ctx->sync_offset);
  MB_TRY(cudaHostAlloc(&ctx->result_host, sizeof(HostResult) * MB_AR_MAX_SLOTS, cudaHostAllocMapped));
  std::memset(ctx->result_host, 0, sizeof(HostResult) * MB_AR_MAX_SLOTS);
  MB_TRY(cudaHostGetDevicePointer(&ctx->result_dev, ctx->result_host, 0));
  MB_TRY(cudaHostAlloc(&ctx->abort_host, sizeof(uint32_t), cudaHostAllocMapped));
  *ctx->abort_host = 0;
  MB_TRY(cudaHostGetDevicePointer(&ctx->abort_dev, ctx->abort_host, 0));
  for (int w = 0; w < 2; ++w) MB_TRY(cudaMalloc(&ctx->tab_dev[w], sizeof(TensorEnt) * kArMaxTensors));
  for (int sl = 0; sl < MB_AR_MAX_SLOTS; ++sl)
    for (int k = 0; k < 3; ++k) MB_TRY(cudaEventCreate(&ctx->ev[sl][k]));
  MB_TRY(cudaMalloc(&ctx->gate_out, sizeof(GateOut) * MB_AR_MAX_SLOTS));
  MB_TRY(cudaMemset(ctx->gate_out, 0, sizeof(GateOut) * MB_AR_MAX_SLOTS));
  MB_TRY(cudaDeviceSynchronize());
#undef MB_TRY
  ctx->peer_staging[rank] = ctx->staging;
  ctx->peer_sync[rank] = ctx->sync;
  ctx->imported[rank] = true;
  *out = ctx;
  return MB_OK;
}

static void close_peers(mb_ar_ctx* ctx) {
  for (int r = 0; r < MB_AR_MAX_WORLD; ++r) {
    if (ctx->ipc_opened[r] && ctx->peer_block[r]) cudaIpcCloseMemHandle(ctx->peer_block[r]);
    ctx->ipc_opened[r] = false;
    ctx->imported[r] = false;
    ctx->peer_block[r] = nullptr;
    ctx->peer_staging[r] = nullptr;
    ctx->peer_sync[r] = nullptr;
  }
}

int mb_ar_ctx_destroy(mb_ar_ctx* ctx) {
  if (!ctx) return MB_OK;
  DeviceGuard g(ctx->device);
  cudaDeviceSynchronize();
  ctx->imported[ctx->rank] = false;
  ctx->peer_staging[ctx->rank] = nullptr;
  ctx->peer_sync[ctx->rank] = nullptr;
  close_peers(ctx);
  if (ctx->block) cudaFree(ctx->block);
  if (ctx->result_host) cudaFreeHost(ctx->result_host);
  if (ctx->abort_host) cudaFreeHost(ctx->abort_host);
  if (ctx->gate_out) cudaFree(ctx->gate_out);
  for (int sl = 0; sl < MB_AR_MAX_SLOTS; ++sl)
    for (int k = 0; k < 3; ++k)
      if (ctx->ev[sl][k]) cudaEventDestroy(ctx->ev[sl][k]);
  for (int w = 0; w < 2; ++w)
    if (ctx->tab_dev[w]) cudaFree(ctx->tab_dev[w]);
  delete ctx;
  return MB_OK;
}

int mb_ar_ctx_export(mb_ar_ctx* ctx, mb_ar_handle* out) {
  MB_CHECK_ARG(ctx && out, "mb_ar_ctx_export: null argument");
  DeviceGuard g(ctx->device);
  std::memset(out, 0, sizeof(*out));
  HandleImpl h;
  std::memset(&h, 0, sizeof(h));
  h.magic = kHandleMagic;
  h.pid = (int32_t)getpid();
  h.device = ctx->device;
  h.rank = ctx->rank;
  h.block_ptr = reinterpret_cast<uint64_t>(ctx->block);
  h.sync_offset = ctx->sync_offset;
  h.xfer_offset = ctx->xfer_offset;
  h.max_bytes = ctx->max_bytes;
  h.nslots = ctx->nslots;
  h.ipc_ok = 1;
  h.base_offset = 0;
  {
    // offset of our block inside the driver allocation the IPC handle maps (0 for a block-owning allocation)
    typedef int (*GetRangeFn)(unsigned long long*, size_t*, unsigned long long);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qr) == cudaSuccess && fn) {
      unsigned long long base = 0;
      size_t size = 0;
      if (reinterpret_cast<GetRangeFn>(fn)(&base, &size, (unsigned long long)h.block_ptr) == 0 && base)
        h.base_offset = h.block_ptr - base;
    } else {
      cudaGetLastError();
    }
  }
  if (cudaIpcGetMemHandle(&h.h_block, ctx->block) != cudaSuccess) {
    cudaGetLastError();  // same-process peers can still import by pointer
    h.ipc_ok = 0;
  }
  std::memcpy(out->bytes, &h, sizeof(h));
  return MB_OK;
}

int mb_ar_ctx_import(mb_ar_ctx* ctx, int peer_rank, const mb_ar_handle* handle) {
  MB_CHECK_ARG(ctx && handle, "mb_ar_ctx_import: null argument");
  MB_CHECK_ARG(peer_rank >= 0 && peer_rank < ctx->world, "mb_ar_ctx_import: peer rank %d not in [0,%d)", peer_rank,
               ctx->world);
  HandleImpl h;
  std::memcpy(&h, handle->bytes, sizeof(h));
  MB_CHECK_ARG(h.magic == kHandleMagic, "mb_ar_ctx_import: not an mb_ar_handle");
  MB_CHECK_ARG(h.max_bytes == ctx->max_bytes && h.nslots == ctx->nslots,
               "mb_ar_ctx_import: peer %d was created with max_bytes=%llu nslots=%d, local ctx has %llu/%d", peer_rank,
               (unsigned long long)h.max_bytes, h.nslots, (unsigned long long)ctx->max_bytes, ctx->nslots);
  std::lock_guard<std::mutex> l(ctx->mu);
  if (peer_rank == ctx->rank) return MB_OK;
  DeviceGuard g(ctx->device);
  if (ctx->imported[peer_rank]) {
    if (ctx->ipc_opened[peer_rank] && ctx->peer_block[peer_rank]) cudaIpcCloseMemHandle(ctx->peer_block[peer_rank]);
    ctx->peer_block[peer_rank] = nullptr;
    ctx->imported[peer_rank] = ctx->ipc_opened[peer_rank] = false;
  }
  if (h.pid == (int32_t)getpid()) {
    if (h.device != ctx->device) {
      int can = 0;
      MB_CUDA(cudaDeviceCanAccessPeer(&can, ctx->device, h.device));
      if (!can) {
        set_error("mb_ar_ctx_import: device %d cannot access peer device %d", ctx->device, h.device);
        return MB_ESTATE;
      }
      cudaError_t e = cudaDeviceEnablePeerAccess(h.device, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
    }
    ctx->peer_staging[peer_rank] = reinterpret_cast<float*>(h.block_ptr);
    ctx->peer_sync[peer_rank] = reinterpret_cast<SyncBlock*>(h.block_ptr + h.sync_offset);
    ctx->ipc_opened[peer_rank] = false;
  } else {
    if (!h.ipc_ok) {
      set_error("mb_ar_ctx_import: peer %d could not export CUDA IPC handles", peer_rank);
      return MB_ESTATE;
    }
    void* base = nullptr;
    MB_CUDA(cudaIpcOpenMemHandle(&base, h.h_block, cudaIpcMemLazyEnablePeerAccess));
    char* blk = static_cast<char*>(base) + h.base_offset;
    ctx->peer_block[peer_rank] = base;
    ctx->peer_staging[peer_rank] = reinterpret_cast<float*>(blk);
    ctx->peer_sync[peer_rank] = reinterpret_cast<SyncBlock*>(blk + h.sync_offset);
    ctx->ipc_opened[peer_rank] = true;
  }
  ctx->imported[peer_rank] = true;
  return MB_OK;
}

int mb_ar_ctx_reset(mb_ar_ctx* ctx, int new_rank, int new_world) {
  MB_CHECK_ARG(ctx != nullptr, "mb_ar_ctx_reset: null ctx");
  MB_CHECK_ARG(new_world >= 1 && new_world <= MB_AR_MAX_WORLD && new_rank >= 0 && new_rank < new_world,
               "mb_ar_ctx_reset: bad rank/world %d/%d", new_rank, new_world);
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  *ctx->abort_host = 1;  // release any kernel still spinning on a dead peer
  MB_CUDA(cudaDeviceSynchronize());
  ctx->imported[ctx->rank] = false;
  ctx->peer_staging[ctx->rank] = nullptr;
  ctx->peer_sync[ctx->rank] = nullptr;
  close_peers(ctx);
  MB_CUDA(cudaMemset(ctx->sync, 0, sizeof(SyncBlock)));
  MB_CUDA(cudaMemset(ctx->gate_out, 0, sizeof(GateOut) * MB_AR_MAX_SLOTS));
  MB_CUDA(cudaDeviceSynchronize());
  *ctx->abort_host = 0;
  ctx->epoch = 0;
  for (int s = 0; s < MB_AR_MAX_SLOTS; ++s) ctx->parity[s] = 0;
  ctx->rank = new_rank;
  ctx->world = new_world;
  ctx->peer_staging[new_rank] = ctx->staging;
  ctx->peer_sync[new_rank] = ctx->sync;
  ctx->imported[new_rank] = true;
  return MB_OK;
}

void* mb_ar_staging(mb_ar_ctx* ctx, int slot) { return mb_ar_buffer(ctx, slot, 0); }

void* mb_ar_buffer(mb_ar_ctx* ctx, int slot, int ahead) {
  if (!ctx || slot < 0 || slot >= ctx->nslots || ahead < 0 || ahead >= kBufs) return nullptr;
  return ring_buffer(ctx, ctx->staging, slot, ahead);
}

int mb_ar_slot_advance(mb_ar_ctx* ctx, int slot) {
  MB_CHECK_ARG(ctx != nullptr, "mb_ar_slot_advance: null ctx");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_slot_advance: slot %d out of range", slot);
  std::lock_guard<std::mutex> l(ctx->mu);
  ctx->parity[slot] = (ctx->parity[slot] + 1) % kBufs;
  return MB_OK;
}

int mb_ar_algo_for(mb_ar_ctx* ctx, uint64_t bytes) {
  if (!ctx) return MB_EINVAL;
  return (ctx->world > 1 && bytes >= twoshot_min_bytes(ctx->world)) ? MB_AR_ALGO_TWOSHOT : MB_AR_ALGO_ONESHOT;
}

int mb_ar_world(mb_ar_ctx* ctx) { return ctx ? ctx->world : MB_EINVAL; }
int mb_ar_rank(mb_ar_ctx* ctx) { return ctx ? ctx->rank : MB_EINVAL; }

int mb_ar_abort(mb_ar_ctx* ctx) {
  MB_CHECK_ARG(ctx != nullptr, "mb_ar_abort: null ctx");
  *reinterpret_cast<volatile uint32_t*>(ctx->abort_host) = 1;
  return MB_OK;
}

int mb_ar_stage(mb_ar_ctx* ctx, int slot, const float* const* grads, const uint64_t* numel, int ntensors,
                int accumulate, int zero_src, mb_stream_t stream_) {
  MB_CHECK_ARG(ctx && grads && numel, "mb_ar_stage: null argument");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_stage: slot %d out of range", slot);
  MB_CHECK_ARG(ntensors >= 1 && ntensors <= kArMaxTensors, "mb_ar_stage: ntensors %d not in [1,%d]", ntensors,
               kArMaxTensors);
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  uint64_t total = 0;
  int rc = sync_table(ctx, 0, reinterpret_cast<const void* const*>(grads), numel, ntensors, &total, stream);
  if (rc) return rc;
  MB_CHECK_ARG(total * 4 <= ctx->max_bytes, "mb_ar_stage: %llu bytes exceed the context's max_bytes %llu",
               (unsigned long long)(total * 4), (unsigned long long)ctx->max_bytes);
  if (total == 0) return 0;
  StageParams p;
  p.staging = ring_buffer(ctx, ctx->staging, slot, 0);
  p.tab = ctx->tab_dev[0];
  p.ntensors = (uint32_t)ntensors;
  p.accumulate = accumulate;
  p.zero_src = zero_src;
  p.total_vec = total / 4;
  const int sms = sm_count(ctx->device);
  if (sms <= 0) return MB_ECUDA;
  const uint64_t want = (p.total_vec + kArThreads - 1) / kArThreads;
  const uint32_t grid = (uint32_t)std::min<uint64_t>(want, (uint64_t)sms * 4);
  const size_t smem = table_bytes(p.ntensors);
  rc = ensure_dyn_smem(reinterpret_cast<const void*>(ar_stage_kernel), smem);
  if (rc) return rc;
  ar_stage_kernel<<<grid, kArThreads, smem, stream>>>(p);
  MB_CUDA(cudaGetLastError());
  return 1;
}

int mb_ar_allreduce(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, float* const* dst, const uint64_t* numel,
                    int ntensors, float* flat_dst, uint64_t flat_numel, int scale_by_num_gradients, int algo,
                    uint32_t timeout_ms, mb_stream_t stream_) {
  MB_CHECK_ARG(ctx && my_hdr, "mb_ar_allreduce: null argument");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_allreduce: slot %d out of range", slot);
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  int rc = launch_reduce(ctx, slot, my_hdr, dst, numel, ntensors, flat_dst, flat_numel, scale_by_num_gradients, algo,
                         timeout_ms, /*gated=*/false, 0, static_cast<cudaStream_t>(stream_));
  // the next round on this slot stages into the next ring buffer: peers may still be reading this one
  if (rc >= 0) ctx->parity[slot] = (ctx->parity[slot] + 1) % kBufs;
  return rc;
}

int mb_ar_reduce_gated(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, uint64_t min_batch_size, float* const* dst,
                       const uint64_t* numel, int ntensors, float* flat_dst, uint64_t flat_numel,
                       int scale_by_num_gradients, int algo, uint32_t timeout_ms, mb_stream_t stream_) {
  MB_CHECK_ARG(ctx && my_hdr, "mb_ar_reduce_gated: null argument");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_reduce_gated: slot %d out of range", slot);
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  return launch_reduce(ctx, slot, my_hdr, dst, numel, ntensors, flat_dst, flat_numel, scale_by_num_gradients, algo,
                       timeout_ms, /*gated=*/true, min_batch_size, static_cast<cudaStream_t>(stream_));
}

int mb_ar_layout(const uint64_t* numel, const int32_t* dtype, int ntensors, uint64_t* offset_bytes,
                 uint64_t* total_bytes, mb_ar_segment* segments) {
  MB_CHECK_ARG(ntensors >= 0 && (ntensors == 0 || (numel && dtype)), "mb_ar_layout: null argument");
  bool all_f32 = true;
  int rc = check_dtypes("mb_ar_layout", dtype, ntensors, &all_f32);
  if (rc) return rc;
  return layout_ex(numel, dtype, ntensors, offset_bytes, total_bytes, segments);
}

int mb_ar_stage_ex(mb_ar_ctx* ctx, int slot, const void* const* grads, const uint64_t* numel, const int32_t* dtype,
                   int ntensors, int accumulate, int zero_src, mb_stream_t stream_) {
  MB_CHECK_ARG(ctx && grads && numel && dtype, "mb_ar_stage_ex: null argument");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_stage_ex: slot %d out of range", slot);
  MB_CHECK_ARG(ntensors >= 1 && ntensors <= kArMaxTensors, "mb_ar_stage_ex: ntensors %d not in [1,%d]", ntensors,
               kArMaxTensors);
  bool all_f32 = true;
  int rc = check_dtypes("mb_ar_stage_ex", dtype, ntensors, &all_f32);
  if (rc) return rc;
  if (all_f32)
    return mb_ar_stage(ctx, slot, reinterpret_cast<const float* const*>(grads), numel, ntensors, accumulate, zero_src,
                       stream_);
  std::vector<uint64_t> off(ntensors);
  mb_ar_segment segs[3];
  uint64_t total = 0;
  const int nseg = layout_ex(numel, dtype, ntensors, off.data(), &total, segs);
  MB_CHECK_ARG(total <= ctx->max_bytes, "mb_ar_stage_ex: %llu bytes exceed the context's max_bytes %llu",
               (unsigned long long)total, (unsigned long long)ctx->max_bytes);
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  rc = sync_table_bytes(ctx, 0, grads, numel, dtype, ntensors, off.data(), stream);
  if (rc) return rc;
  if (total == 0) return 0;
  StageSegParams sp;
  sp.b.staging = ring_buffer(ctx, ctx->staging, slot, 0);
  sp.b.tab = ctx->tab_dev[0];
  sp.b.ntensors = (uint32_t)ntensors;
  sp.b.accumulate = accumulate;
  sp.b.zero_src = zero_src;
  sp.b.total_vec = total / 16;
  sp.seg = seg_info(segs, nseg);
  const int sms = sm_count(ctx->device);
  if (sms <= 0) return MB_ECUDA;
  const uint64_t want = (sp.b.total_vec + kArThreads - 1) / kArThreads;
  const uint32_t grid = (uint32_t)std::min<uint64_t>(want, (uint64_t)sms * 4);
  const size_t smem = table_bytes(sp.b.ntensors);
  rc = ensure_dyn_smem(reinterpret_cast<const void*>(ar_stage_seg_kernel), smem);
  if (rc) return rc;
  ar_stage_seg_kernel<<<grid, kArThreads, smem, stream>>>(sp);
  MB_CUDA(cudaGetLastError());
  return 1;
}

// mb_ar_allreduce_ex / mb_ar_reduce_gated_ex; the caller holds ctx->mu and the device guard.
static int reduce_ex_locked(const char* fn, mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, void* const* dst,
                            const uint64_t* numel, const int32_t* dtype, int ntensors, void* flat_dst,
                            uint64_t flat_bytes, int scale, int algo, uint32_t timeout_ms, bool gated,
                            uint64_t min_batch, cudaStream_t stream) {
  std::vector<uint64_t> off(ntensors);
  mb_ar_segment segs[3];
  uint64_t total = 0;
  const int nseg = layout_ex(numel, dtype, ntensors, off.data(), &total, segs);
  bool all_f32 = nseg == 0 || (nseg == 1 && segs[0].dtype == MB_DT_F32);
  for (int i = 0; i < ntensors; ++i) all_f32 = all_f32 && dtype[i] == MB_DT_F32;
  if (!dst) {
    MB_CHECK_ARG(flat_dst != nullptr, "%s: neither dst nor flat_dst given", fn);
    MB_CHECK_ARG(flat_bytes == total, "%s: flat_bytes %llu != layout size %llu", fn, (unsigned long long)flat_bytes,
                 (unsigned long long)total);
    MB_CHECK_ARG((reinterpret_cast<uintptr_t>(flat_dst) & 15u) == 0, "%s: flat_dst is not 16 B aligned", fn);
  }
  if (all_f32) {
    // exactly what mb_ar_allreduce / mb_ar_reduce_gated run for this list
    if (dst)
      return launch_reduce(ctx, slot, my_hdr, reinterpret_cast<float* const*>(dst), numel, ntensors, nullptr, 0, scale,
                           algo, timeout_ms, gated, min_batch, stream);
    return launch_reduce(ctx, slot, my_hdr, nullptr, nullptr, 0, static_cast<float*>(flat_dst), total / 4, scale, algo,
                         timeout_ms, gated, min_batch, stream);
  }
  MB_CHECK_ARG(total <= ctx->max_bytes, "%s: %llu bytes exceed the context's max_bytes %llu", fn,
               (unsigned long long)total, (unsigned long long)ctx->max_bytes);
  SegLaunch sl;
  sl.total_vec = total / 16;
  sl.ntab = 0;
  sl.flat = flat_dst;
  sl.info = seg_info(segs, nseg);
  if (dst) {
    int rc = sync_table_bytes(ctx, 1, dst, numel, dtype, ntensors, off.data(), stream);
    if (rc) return rc;
    sl.ntab = (uint32_t)ntensors;
    sl.flat = nullptr;
  }
  return launch_reduce(ctx, slot, my_hdr, nullptr, nullptr, 0, nullptr, 0, scale, algo, timeout_ms, gated, min_batch,
                       stream, &sl);
}

static int reduce_ex_args(const char* fn, mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, const uint64_t* numel,
                          const int32_t* dtype, int ntensors) {
  MB_CHECK_ARG(ctx && my_hdr && numel && dtype, "%s: null argument", fn);
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "%s: slot %d out of range", fn, slot);
  MB_CHECK_ARG(ntensors >= 1 && ntensors <= kArMaxTensors, "%s: ntensors %d not in [1,%d]", fn, ntensors,
               kArMaxTensors);
  bool all_f32 = true;
  return check_dtypes(fn, dtype, ntensors, &all_f32);
}

int mb_ar_allreduce_ex(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, void* const* dst, const uint64_t* numel,
                       const int32_t* dtype, int ntensors, void* flat_dst, uint64_t flat_bytes,
                       int scale_by_num_gradients, int algo, uint32_t timeout_ms, mb_stream_t stream_) {
  int rc = reduce_ex_args("mb_ar_allreduce_ex", ctx, slot, my_hdr, numel, dtype, ntensors);
  if (rc) return rc;
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  rc = reduce_ex_locked("mb_ar_allreduce_ex", ctx, slot, my_hdr, dst, numel, dtype, ntensors, flat_dst, flat_bytes,
                        scale_by_num_gradients, algo, timeout_ms, /*gated=*/false, 0, static_cast<cudaStream_t>(stream_));
  if (rc >= 0) ctx->parity[slot] = (ctx->parity[slot] + 1) % kBufs;
  return rc;
}

int mb_ar_reduce_gated_ex(mb_ar_ctx* ctx, int slot, const mb_ar_hdr* my_hdr, uint64_t min_batch_size, void* const* dst,
                          const uint64_t* numel, const int32_t* dtype, int ntensors, void* flat_dst,
                          uint64_t flat_bytes, int scale_by_num_gradients, int algo, uint32_t timeout_ms,
                          mb_stream_t stream_) {
  int rc = reduce_ex_args("mb_ar_reduce_gated_ex", ctx, slot, my_hdr, numel, dtype, ntensors);
  if (rc) return rc;
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  return reduce_ex_locked("mb_ar_reduce_gated_ex", ctx, slot, my_hdr, dst, numel, dtype, ntensors, flat_dst, flat_bytes,
                          scale_by_num_gradients, algo, timeout_ms, /*gated=*/true, min_batch_size,
                          static_cast<cudaStream_t>(stream_));
}

int mb_ar_round_times(mb_ar_ctx* ctx, int slot, float* gate_us, float* reduce_us) {
  MB_CHECK_ARG(ctx != nullptr, "mb_ar_round_times: null ctx");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_round_times: slot %d out of range", slot);
  std::lock_guard<std::mutex> l(ctx->mu);
  if (!ctx->ev_valid[slot]) {
    set_error("mb_ar_round_times: no timed round on slot %d", slot);
    return MB_ESTATE;
  }
  DeviceGuard g(ctx->device);
  float a = 0.f, b = 0.f;
  MB_CUDA(cudaEventElapsedTime(&a, ctx->ev[slot][0], ctx->ev[slot][1]));
  MB_CUDA(cudaEventElapsedTime(&b, ctx->ev[slot][1], ctx->ev[slot][2]));
  if (gate_us) *gate_us = a * 1e3f;
  if (reduce_us) *reduce_us = b * 1e3f;
  return MB_OK;
}

int mb_ar_xfer_pack(mb_ar_ctx* ctx, const float* const* tensors, const uint64_t* numel, int ntensors, mb_stream_t stream_) {
  MB_CHECK_ARG(ctx && tensors && numel, "mb_ar_xfer_pack: null argument");
  MB_CHECK_ARG(ntensors >= 1 && ntensors <= kArMaxTensors, "mb_ar_xfer_pack: ntensors %d not in [1,%d]", ntensors, kArMaxTensors);
  std::lock_guard<std::mutex> l(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  uint64_t total = 0;
  int rc = sync_table(ctx, 0, reinterpret_cast<const void* const*>(tensors), numel, ntensors, &total, stream);
  if (rc) return rc;
  MB_CHECK_ARG(total * 4 <= ctx->max_bytes, "mb_ar_xfer_pack: %llu bytes exceed the context's max_bytes %llu",
               (unsigned long long)(total * 4), (unsigned long long)ctx->max_bytes);
  if (total == 0) return 0;
  StageParams p;
  p.staging = reinterpret_cast<float*>(static_cast<char*>(ctx->block) + ctx->xfer_offset);
  p.tab = ctx->tab_dev[0];
  p.ntensors = (uint32_t)ntensors;
  p.accumulate = 0;
  p.zero_src = 0;
  p.total_vec = total / 4;
  const int sms = sm_count(ctx->device);
  if (sms <= 0) return MB_ECUDA;
  const uint32_t grid = (uint32_t)std::min<uint64_t>((p.total_vec + kArThreads - 1) / kArThreads, (uint64_t)sms * 4);
  const size_t smem = table_bytes(p.ntensors);
  rc = ensure_dyn_smem(reinterpret_cast<const void*>(ar_stage_kernel), smem);
  if (rc) return rc;
  ar_stage_kernel<<<grid, kArThreads, smem, stream>>>(p);
  MB_CUDA(cudaGetLastError());
  return 1;
}

int mb_ar_xfer_unpack(mb_ar_ctx* ctx, int src_rank, float* const* tensors, const uint64_t* numel, int ntensors,
                      mb_stream_t stream_) {
  MB_CHECK_ARG(ctx && tensors && numel, "mb_ar_xfer_unpack: null argument");
  MB_CHECK_ARG(ntensors >= 1 && ntensors <= kArMaxTensors, "mb_ar_xfer_unpack: ntensors %d not in [1,%d]", ntensors, kArMaxTensors);
  MB_CHECK_ARG(src_rank >= 0 && src_rank < ctx->world, "mb_ar_xfer_unpack: source rank %d not in [0,%d)", src_rank, ctx->world);
  std::lock_guard<std::mutex> l(ctx->mu);
  if (!ctx->imported[src_rank]) {
    set_error("mb_ar_xfer_unpack: peer %d has not been imported", src_rank);
    return MB_ESTATE;
  }
  DeviceGuard g(ctx->device);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  uint64_t total = 0;
  int rc = sync_table(ctx, 1, reinterpret_cast<const void* const*>(tensors), numel, ntensors, &total, stream);
  if (rc) return rc;
  MB_CHECK_ARG(total * 4 <= ctx->max_bytes, "mb_ar_xfer_unpack: %llu bytes exceed the context's max_bytes %llu",
               (unsigned long long)(total * 4), (unsigned long long)ctx->max_bytes);
  if (total == 0) return 0;
  UnpackParams p;
  // peer_staging[r] is the base of rank r's block (the ring starts there); the publish region sits at xfer_offset
  p.src = reinterpret_cast<const float*>(reinterpret_cast<const char*>(ctx->peer_staging[src_rank]) + ctx->xfer_offset);
  p.tab = ctx->tab_dev[1];
  p.ntensors = (uint32_t)ntensors;
  p.total_vec = total / 4;
  const int sms = sm_count(ctx->device);
  if (sms <= 0) return MB_ECUDA;
  const uint32_t grid = (uint32_t)std::min<uint64_t>((p.total_vec + 4ull * kArThreads - 1) / (4ull * kArThreads), (uint64_t)sms * 2);
  const size_t smem = table_bytes(p.ntensors);
  rc = ensure_dyn_smem(reinterpret_cast<const void*>(ar_unpack_kernel), smem);
  if (rc) return rc;
  ar_unpack_kernel<<<std::max<uint32_t>(grid, 1), kArThreads, smem, stream>>>(p);
  MB_CUDA(cudaGetLastError());
  return 1;
}

int mb_ar_result(mb_ar_ctx* ctx, int slot, mb_ar_hdr* sum_out, int* status_out) {
  MB_CHECK_ARG(ctx != nullptr, "mb_ar_result: null ctx");
  MB_CHECK_ARG(slot >= 0 && slot < ctx->nslots, "mb_ar_result: slot %d out of range", slot);
  const volatile HostResult* r = ctx->result_host + slot;
  if (sum_out) {
    sum_out->num_gradients = r->sum.num_gradients;
    sum_out->num_skipped = r->sum.num_skipped;
    sum_out->batch_size = r->sum.batch_size;
    sum_out->has_grads = r->sum.has_grads;
  }
  if (status_out) *status_out = r->status;
  return MB_OK;
}

}  // extern "C"
