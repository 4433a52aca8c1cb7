// Data-parallel gradient exchange over NVLink peer memory: the sum all-reduce of a range of the flat gradient arena
// (what DistributedDataParallel / dist.all_reduce would do for the reference's `loss.backward()`, train.py:66) as ONE
// kernel per bucket that reads and writes the peers' arenas directly.
//
// Every rank maps every rank's arena (cudaIpc handles exchanged once, rcv_peer_alloc / rcv_peer_open).  A launch on
// rank r:
//   1. ready barrier: posts "my gradients of this range are final" into every rank's flag block and waits for all
//      ranks' posts (the kernel boundary before it made its own gradients visible);
//   2. reduces ITS 1/N share of the range -- loads the N copies, adds them in rank order (the same bits on whichever
//      rank does it), stores the sum into all N arenas;
//   3. done barrier: the last CTA posts "my share is stored everywhere" and waits for all ranks' posts, so when the
//      kernel ends the whole range of the local arena holds the sums and no peer reads or writes it any more.
// Traffic per rank: (N-1)/N of the range in, (N-1)/N out, each element crossing NVLink once per direction (a two-shot
// all-reduce); latency: two flag round trips + one load round trip.  Flags carry a per-slot launch count (kept next
// to them, advanced by the kernel), so graph replays, warm-up runs and eager launches all line up as long as every
// rank issues the same launches per slot -- which SPMD training does.
// A peer that never arrives would leave the others spinning: after RCV_PEER_TIMEOUT_S (default 30 s) a launch gives
// up, sets *status and returns; the host checks it when it reads the step's loss.
#include "rcv_common.cuh"

#include <stdlib.h>

#include <type_traits>

namespace {

constexpr int NT = 256;
constexpr int PEER_MAX = 8;         // ranks (one NVSwitch node)
constexpr int SLOT_WORDS = 64;      // uint32 per slot: [0,8) ready, [16,24) done, 32 launch count, 33 CTA counter
constexpr int PEER_SLOTS = 16;

struct PeerArgs {
  float* arena[PEER_MAX];
  uint32_t* flags[PEER_MAX];
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer(const float4* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p)
               : "memory");
  return v;
}
__device__ __forceinline__ uint64_t now_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// spin until *flag has reached `epoch` (wrap-safe); false on time-out
__device__ __forceinline__ bool wait_flag(const uint32_t* flag, uint32_t epoch, uint64_t timeout_ns) {
  if ((int32_t)(ld_acquire_sys(flag) - epoch) >= 0) return true;
  const uint64_t t0 = now_ns();
  for (;;) {
    for (int i = 0; i < 64; ++i) {
      if ((int32_t)(ld_acquire_sys(flag) - epoch) >= 0) return true;
      __nanosleep(32);
    }
    if (now_ns() - t0 > timeout_ns) return false;
  }
}

template <int WORLD>
__global__ void __launch_bounds__(NT) peer_allreduce_kernel(PeerArgs pa, int rank, int slot, int64_t off4,
                                                            int64_t count4, uint64_t timeout_ns, int32_t* status) {
  rcv_pdl_enter();
  __shared__ uint32_t s_epoch;
  __shared__ int s_fail;
  uint32_t* mine = pa.flags[rank] + slot * SLOT_WORDS;
  if (threadIdx.x == 0) {
    s_epoch = *reinterpret_cast<volatile uint32_t*>(mine + 32) + 1;
    s_fail = 0;
  }
  __syncthreads();
  const uint32_t epoch = s_epoch;
  // 1. ready barrier
  if (blockIdx.x == 0 && threadIdx.x < WORLD)
    st_release_sys(pa.flags[threadIdx.x] + slot * SLOT_WORDS + rank, epoch);
  if (threadIdx.x < WORLD && !wait_flag(mine + threadIdx.x, epoch, timeout_ns)) s_fail = 1;
  __syncthreads();
  if (s_fail) {  // a peer never arrived: leave the arena alone, report, and do not wait again
    if (threadIdx.x == 0) atomicExch(status, 1);
    if (threadIdx.x == 0 && atomicAdd(mine + 33, 1u) == gridDim.x - 1) {
      mine[33] = 0;
      *reinterpret_cast<volatile uint32_t*>(mine + 32) = epoch;
    }
    return;
  }
  // 2. my share of the range: float4 [lo, hi)
  const int64_t per = (count4 + WORLD - 1) / WORLD;
  const int64_t lo = (int64_t)rank * per, hi = (lo + per < count4) ? lo + per : count4;
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t i = lo + (int64_t)blockIdx.x * NT + threadIdx.x; i < hi; i += stride) {
    float4 v[WORLD];
#pragma unroll
    for (int q = 0; q < WORLD; ++q) v[q] = ld_peer(reinterpret_cast<const float4*>(pa.arena[q]) + off4 + i);
    float4 s = v[0];
#pragma unroll
    for (int q = 1; q < WORLD; ++q) {
      s.x += v[q].x; s.y += v[q].y; s.z += v[q].z; s.w += v[q].w;
    }
#pragma unroll
    for (int q = 0; q < WORLD; ++q) reinterpret_cast<float4*>(pa.arena[q])[off4 + i] = s;
  }
  // 3. done barrier
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(mine + 33, 1u) == gridDim.x - 1) {
    __threadfence_system();
    mine[33] = 0;
    for (int q = 0; q < WORLD; ++q) st_release_sys(pa.flags[q] + slot * SLOT_WORDS + 16 + rank, epoch);
    bool ok = true;
    for (int q = 0; q < WORLD; ++q) ok = wait_flag(mine + 16 + q, epoch, timeout_ns) && ok;
    if (!ok) atomicExch(status, 1);
    *reinterpret_cast<volatile uint32_t*>(mine + 32) = epoch;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Small-vector exchange (TrainStep(global_batch=True)): buf[off, off+count) <- scale * sum over ranks, for the few
// hundred fp64 / int64 values of a BatchNorm layer's statistics or backward sums, a loss normaliser or a correct count.
// ONE CTA: every rank loads all N copies and writes only its own buffer, in place.  The order of the steps is what
// makes the in-place write safe:
//   1. ready barrier: "my values are final" (the kernel boundary before it made them visible);
//   2. load all N copies, add them in rank order (the same bits on every rank), keep the sums in shared memory;
//   3. done barrier: "I have read yours";
//   4. store the scaled sums into the local buffer.
// No peer can read a value after it was overwritten: a rank writes only after every peer has posted that its loads
// are done.  A rank's next write into the same buffer (the next step's memset, the next layer's statistics) follows
// its own launch in stream order, hence also every peer's loads.  Same flag words, launch counts and time-out as
// peer_allreduce_kernel: a slot must be used by one stream of each rank at a time.
constexpr int SMALL_MAX = 4096;  // elements per launch (32 KB of shared memory)

struct SmallArgs {
  void* buf[PEER_MAX];
  uint32_t* flags[PEER_MAX];
};

__device__ __forceinline__ double ld_peer_elem(const double* p) {
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ long long ld_peer_elem(const long long* p) {
  long long v;
  asm volatile("ld.relaxed.sys.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

template <typename T>
__global__ void __launch_bounds__(NT) peer_small_allreduce_kernel(SmallArgs pa, int world, int rank, int slot,
                                                                  int64_t off, int count, double scale,
                                                                  uint64_t timeout_ns, int32_t* status) {
  rcv_pdl_enter();
  __shared__ T s_sum[SMALL_MAX];
  __shared__ uint32_t s_epoch;
  __shared__ int s_fail;
  uint32_t* mine = pa.flags[rank] + slot * SLOT_WORDS;
  if (threadIdx.x == 0) {
    s_epoch = *reinterpret_cast<volatile uint32_t*>(mine + 32) + 1;
    s_fail = 0;
  }
  __syncthreads();
  const uint32_t epoch = s_epoch;
  // 1. ready barrier
  __threadfence_system();
  if (threadIdx.x < world) st_release_sys(pa.flags[threadIdx.x] + slot * SLOT_WORDS + rank, epoch);
  if (threadIdx.x < world && !wait_flag(mine + threadIdx.x, epoch, timeout_ns)) s_fail = 1;
  __syncthreads();
  const bool ok = !s_fail;
  // 2. every rank's copy, summed in rank order
  if (ok) {
    for (int i = threadIdx.x; i < count; i += NT) {
      T s = ld_peer_elem(reinterpret_cast<const T*>(pa.buf[0]) + off + i);
      for (int q = 1; q < world; ++q) s += ld_peer_elem(reinterpret_cast<const T*>(pa.buf[q]) + off + i);
      s_sum[i] = s;
    }
  }
  // 3. done barrier: the loads above are complete before any peer hears of it
  __threadfence_system();
  __syncthreads();
  if (ok) {
    if (threadIdx.x < world) st_release_sys(pa.flags[threadIdx.x] + slot * SLOT_WORDS + 16 + rank, epoch);
    if (threadIdx.x < world && !wait_flag(mine + 16 + threadIdx.x, epoch, timeout_ns)) s_fail = 1;
  }
  __syncthreads();
  if (s_fail) {  // a peer never arrived: leave the buffer alone and report
    if (threadIdx.x == 0) atomicExch(status, 1);
  } else {
    // 4. the local result, in place
    T* dst = reinterpret_cast<T*>(pa.buf[rank]) + off;
    for (int i = threadIdx.x; i < count; i += NT) {
      if constexpr (std::is_same<T, double>::value)
        dst[i] = s_sum[i] * scale;
      else
        dst[i] = s_sum[i];  // integer counts: exact sums, no scale
    }
  }
  if (threadIdx.x == 0) *reinterpret_cast<volatile uint32_t*>(mine + 32) = epoch;
}

uint64_t timeout_ns() {
  static uint64_t ns = [] {
    const char* e = getenv("RCV_PEER_TIMEOUT_S");
    double s = e ? atof(e) : 30.0;
    if (!(s > 0.0)) s = 30.0;
    return (uint64_t)(s * 1e9);
  }();
  return ns;
}

}  // namespace

extern "C" uint64_t rcv_peer_flag_bytes(void) { return (uint64_t)PEER_SLOTS * SLOT_WORDS * sizeof(uint32_t); }

extern "C" int rcv_peer_alloc(uint64_t bytes, void** ptr, void* handle64) {
  RCV_REQUIRE(bytes > 0 && ptr && handle64, RCV_ERR_BAD_ARG, "peer_alloc: bad arg");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  RCV_REQUIRE(e == cudaSuccess, RCV_ERR_CUDA, "peer_alloc: cudaMalloc(%llu): %s", (unsigned long long)bytes,
              cudaGetErrorString(e));
  e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), p);
  if (e != cudaSuccess) {
    cudaFree(p);
    RCV_REQUIRE(false, RCV_ERR_CUDA, "peer_alloc: %s", cudaGetErrorString(e));
  }
  *ptr = p;
  return RCV_OK;
}

extern "C" int rcv_peer_open(const void* handle64, void** ptr) {
  RCV_REQUIRE(handle64 && ptr, RCV_ERR_BAD_ARG, "peer_open: bad arg");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof(h));
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  RCV_REQUIRE(e == cudaSuccess, RCV_ERR_CUDA, "peer_open: cudaIpcOpenMemHandle: %s (peer-to-peer access between the "
              "ranks' GPUs is required)", cudaGetErrorString(e));
  *ptr = p;
  return RCV_OK;
}

extern "C" int rcv_peer_close(void* ptr) {
  RCV_REQUIRE(ptr, RCV_ERR_BAD_ARG, "peer_close: bad arg");
  cudaError_t e = cudaIpcCloseMemHandle(ptr);
  RCV_REQUIRE(e == cudaSuccess, RCV_ERR_CUDA, "peer_close: %s", cudaGetErrorString(e));
  return RCV_OK;
}

extern "C" int rcv_peer_free(void* ptr) {
  RCV_REQUIRE(ptr, RCV_ERR_BAD_ARG, "peer_free: bad arg");
  cudaError_t e = cudaFree(ptr);
  RCV_REQUIRE(e == cudaSuccess, RCV_ERR_CUDA, "peer_free: %s", cudaGetErrorString(e));
  return RCV_OK;
}

extern "C" int rcv_peer_allreduce(int32_t world, int32_t rank, int32_t slot, float* const* arenas,
                                  uint32_t* const* flags, int64_t offset, int64_t count, int32_t* status,
                                  void* stream) {
  RCV_REQUIRE(world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world && arenas && flags && status,
              RCV_ERR_BAD_ARG, "peer_allreduce: bad arg (world %d, rank %d)", world, rank);
  RCV_REQUIRE(slot >= 0 && slot < PEER_SLOTS, RCV_ERR_BAD_ARG, "peer_allreduce: slot %d of %d", slot, PEER_SLOTS);
  RCV_REQUIRE(offset >= 0 && count > 0 && offset % 4 == 0 && count % 4 == 0, RCV_ERR_BAD_ARG,
              "peer_allreduce: offset %lld / count %lld must be multiples of 4 floats", (long long)offset,
              (long long)count);
  PeerArgs pa;
  memset(&pa, 0, sizeof(pa));
  for (int q = 0; q < world; ++q) {
    RCV_REQUIRE(arenas[q] && flags[q] && ((uintptr_t)arenas[q] % 16 == 0), RCV_ERR_BAD_ARG,
                "peer_allreduce: arena / flags of rank %d", q);
    pa.arena[q] = arenas[q];
    pa.flags[q] = flags[q];
  }
  const int64_t count4 = count / 4, per = (count4 + world - 1) / world;
  int64_t nb = (per + NT * 2 - 1) / (NT * 2);  // ~2 float4 per thread per rank in flight
  if (nb > 64) nb = 64;
  if (nb < 1) nb = 1;
  const dim3 grid((unsigned)nb), block(NT);
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t tns = timeout_ns();
#define RCV_PEER_CASE(W)                                                                                            \
  case W:                                                                                                           \
    rcv_launch(peer_allreduce_kernel<W>, grid, block, 0, st, pa, rank, slot, offset / 4, count4, tns, status);     \
    break;
  switch (world) {
    RCV_PEER_CASE(1) RCV_PEER_CASE(2) RCV_PEER_CASE(3) RCV_PEER_CASE(4)
    RCV_PEER_CASE(5) RCV_PEER_CASE(6) RCV_PEER_CASE(7) RCV_PEER_CASE(8)
  }
#undef RCV_PEER_CASE
  RCV_CHECK_LAUNCH("peer_allreduce");
  return RCV_OK;
}

namespace {

template <typename T>
int peer_small_allreduce(const char* name, int32_t world, int32_t rank, int32_t slot, T* const* bufs,
                         uint32_t* const* flags, int64_t offset, int64_t count, double scale, int32_t* status,
                         void* stream) {
  RCV_REQUIRE(world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world && bufs && flags && status,
              RCV_ERR_BAD_ARG, "%s: bad arg (world %d, rank %d)", name, world, rank);
  RCV_REQUIRE(slot >= 0 && slot < PEER_SLOTS, RCV_ERR_BAD_ARG, "%s: slot %d of %d", name, slot, PEER_SLOTS);
  RCV_REQUIRE(offset >= 0 && count > 0 && count <= SMALL_MAX, RCV_ERR_BAD_ARG,
              "%s: offset %lld / count %lld (1..%d elements)", name, (long long)offset, (long long)count, SMALL_MAX);
  SmallArgs pa;
  memset(&pa, 0, sizeof(pa));
  for (int q = 0; q < world; ++q) {
    RCV_REQUIRE(bufs[q] && flags[q] && ((uintptr_t)bufs[q] % sizeof(T) == 0), RCV_ERR_BAD_ARG,
                "%s: buffer / flags of rank %d", name, q);
    pa.buf[q] = bufs[q];
    pa.flags[q] = flags[q];
  }
  rcv_launch(peer_small_allreduce_kernel<T>, dim3(1), dim3(NT), 0, (cudaStream_t)stream, pa, (int)world, (int)rank,
             (int)slot, offset, (int)count, scale, timeout_ns(), status);
  RCV_CHECK_LAUNCH(name);
  return RCV_OK;
}

}  // namespace

extern "C" int rcv_peer_allreduce_f64(int32_t world, int32_t rank, int32_t slot, double* const* bufs,
                                      uint32_t* const* flags, int64_t offset, int64_t count, double scale,
                                      int32_t* status, void* stream) {
  return peer_small_allreduce<double>("peer_allreduce_f64", world, rank, slot, bufs, flags, offset, count, scale,
                                      status, stream);
}

extern "C" int rcv_peer_allreduce_i64(int32_t world, int32_t rank, int32_t slot, int64_t* const* bufs,
                                      uint32_t* const* flags, int64_t offset, int64_t count, int32_t* status,
                                      void* stream) {
  return peer_small_allreduce<long long>("peer_allreduce_i64", world, rank, slot,
                                         reinterpret_cast<long long* const*>(bufs), flags, offset, count, 1.0, status,
                                         stream);
}
