// Shared internals of librcv_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "rcv_b200.h"

void rcv_set_error(const char* fmt, ...);

#define RCV_REQUIRE(cond, code, ...)      \
  do {                                    \
    if (!(cond)) {                        \
      rcv_set_error(__VA_ARGS__);         \
      return (code);                      \
    }                                     \
  } while (0)

// Check the launch that was just enqueued (no sync: only launch-config errors).
#define RCV_CHECK_LAUNCH(name)                                              \
  do {                                                                      \
    cudaError_t e__ = cudaGetLastError();                                   \
    if (e__ != cudaSuccess) {                                               \
      rcv_set_error("%s: %s", (name), cudaGetErrorString(e__));             \
      return RCV_ERR_CUDA;                                                  \
    }                                                                       \
  } while (0)

static inline int rcv_cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
// math modes that pick the engine per layer (tensor cores where the reduction pays): the fp32-parity mode and the
// two fast modes; RCV_MATH_FP32 / RCV_MATH_TF32X3 force one engine
static inline bool rcv_math_auto(int m) { return m == RCV_MATH_AUTO || m == RCV_MATH_TF32 || m == RCV_MATH_BF16; }

// ---------------------------------------------------------------------------
// Programmatic dependent launch.  A training step is ~100 short kernels back to back on one stream; with
// RCV_PDL=1 every kernel is launched with cudaLaunchAttributeProgrammaticStreamSerialization, so the next grid is
// rasterised and its CTAs become resident while the current one drains.  Every kernel of the library starts with
// rcv_pdl_enter(): it releases its dependents immediately (they only pre-stage) and then waits until all
// prerequisite grids have completed and flushed -- no kernel touches memory before that, so the data dependences
// are exactly those of plain stream order.  Both instructions are no-ops in a grid launched the ordinary way.
// ---------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ void rcv_pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
#endif

bool rcv_pdl_enabled();  // RCV_PDL (rcv_api.cu)

// ---------------------------------------------------------------------------
// Ordered flush: the fixed-order replacement of "every CTA atomically adds its partial vector into dst" used by the
// deterministic (_det) entry points.  Scratch layout (caller-owned, rcv_det_scratch_bytes): a uint32 arrival
// counter padded to RCV_DET_COUNTER_BYTES, then T partials[nslots][len].  128-byte aligned, zero-filled once by the
// caller, left with its counter zeroed again, one stream at a time -- the convention of rcv_conv_desc::workspace.
// ---------------------------------------------------------------------------
constexpr size_t RCV_DET_COUNTER_BYTES = 128;

static inline size_t rcv_det_bytes(long long nslots, long long len, size_t elem) {
  return RCV_DET_COUNTER_BYTES + (((size_t)nslots * (size_t)len * elem + 127) & ~(size_t)127);
}

// scratch each deterministic entry point needs (rcv_det_scratch_bytes)
size_t rcv_ce_fwd_det_bytes(int32_t N, int64_t HW);
size_t rcv_ce_weight_sum_det_bytes(int64_t count);
size_t rcv_dice_fwd_det_bytes(int32_t N, int32_t C, int64_t HW);
size_t rcv_l1_sum_det_bytes(int64_t n);

#ifdef __CUDACC__
// Called by every thread of the CTA (no early exits before it).  mine[0..len) (shared memory, or any memory every
// thread of the CTA can read) is this CTA's partial vector; slot comes from the launch geometry, never from the
// arrival order.  Each CTA parks its partial in its slot and takes a ticket; the one that arrives last adds up the
// slots and adds the total into dst (dst[i] += total, as the atomic form does), then resets the counter.  The order
// of the additions depends on nslots and blockDim.x only: thread t sums slots t, t + blockDim.x, ... in turn, the
// threads of a warp combine by a fixed butterfly, and thread 0 adds the warp sums in warp order -- the last CTA's
// whole block shares the work, so the tail stays short at a thousand slots.  No CTA waits for another, so CTAs that
// are not resident at the same time cannot deadlock it.  The memory ordering is that of the split reduction of the
// halo-staged tensor-core kernel (rcv_umma_halo.cu, split_exchange).  blockDim.x: a multiple of 32, at most 1024.
template <typename T>
__device__ __noinline__ void rcv_ordered_flush(void* scratch, int slot, int nslots, int len, const T* mine, T* dst) {
  __shared__ uint32_t s_ticket;
  __shared__ T s_warp[32];
  uint32_t* counter = reinterpret_cast<uint32_t*>(scratch);
  T* parts = reinterpret_cast<T*>(reinterpret_cast<unsigned char*>(scratch) + RCV_DET_COUNTER_BYTES);
  for (int i = threadIdx.x; i < len; i += blockDim.x) __stcg(parts + (size_t)slot * len + i, mine[i]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(counter, 1u);
  __syncthreads();
  if (s_ticket != (uint32_t)(nslots - 1)) return;
  __threadfence();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int i = 0; i < len; ++i) {
    T t = T(0);
    for (int s = threadIdx.x; s < nslots; s += blockDim.x) t += __ldcg(parts + (size_t)s * len + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) s_warp[warp] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
      T u = s_warp[0];
      for (int w = 1; w < nwarps; ++w) u += s_warp[w];
      dst[i] += u;
    }
    __syncthreads();  // s_warp is reused by the next element
  }
  if (threadIdx.x == 0) *counter = 0u;  // every slot has arrived: ready for the next launch
}
#endif

// The one way kernels are launched: plain stream order, or programmatic dependent launch when enabled.  Errors
// are picked up by RCV_CHECK_LAUNCH right after.
template <typename... KArgs, typename... Args>
inline void rcv_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                       Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr;
  memset(&attr, 0, sizeof(attr));
  if (rcv_pdl_enabled()) {
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
  }
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------------------
// Implicit-GEMM problem shared by conv forward, conv dgrad and the
// transposed-conv family.  out[n, cb, oy, ox] = sum_{ca, t} in[n, ca, iy, ix] *
// w[ca*wsA + cb*wsB + twi[t]] with (iy, ix) = (i*gs + tdy[t], j*gs + tdx[t])
// and (oy, ox) = (i*ostep + a, j*ostep + b) for pixel-grid point (i, j) of
// parity class (a, b) (ostep = 1: a single class).
// ---------------------------------------------------------------------------
struct RcvTapSet {
  int32_t n;
  int8_t dy[9], dx[9], wi[9];
};

struct RcvIgemm {
  const float* in;
  const float* w;
  const void* wpacked;  // rcv_conv_pack image of w for the tensor-core engine (may be NULL)
  float* out;
  const float* bias;
  const float* scale;
  const float* shift;
  const float* residual;
  double* stats;
  // normalise-on-load (forward, halo-staged tensor-core kernel only): the kernel reads in_scale[c]*x + in_shift[c]
  // (then ReLU if in_relu) in place of x -- the BatchNorm of the block that produced x, never materialised; the
  // zero padding applies to the transformed tensor.  NULL: x is read as it is.
  const float* in_scale;
  const float* in_shift;
  int32_t in_relu;
  // optional caller-owned scratch (rcv_conv_desc::workspace): split-reduction partial tiles + arrival counters
  void* ws;
  unsigned long long ws_bytes;
  int32_t res_C;  // channels of `residual` (== CB unless a partial skip: added to the first res_C channels only; narrow engine)
  int32_t N, CA, CB;
  int32_t Hin, Win, Hout, Wout, Hg, Wg;
  int32_t gs, ostep;
  int32_t wsA, wsB;
  int32_t epilogue;
  int32_t nclass;
  int32_t math;  // rcv_math
  int32_t debug; // timing experiments (RCV_UMMA_DEBUG), 0 in production
  long long* prof;  // per-phase clock64 samples of CTA 0 (rcv_debug_set_prof), NULL in production
  RcvTapSet taps[4];
};

// Weight-gradient problem: dw[cb*wsB + ca*wsA + twi[t]] += sum over pixel-grid
// points (n,i,j) of row[n,cb,i,j] * src[n,ca,i*gs+tdy[t], j*gs+tdx[t]].
struct RcvWgrad {
  const float* src;  // gathered (im2col) tensor [N, CA, Hin, Win]
  const float* row;  // dense tensor [N, CB, Hg, Wg]
  float* dw;
  float* dbias;      // += sum of row over pixels (NULL to skip)
  int32_t N, CA, CB;
  int32_t Hin, Win, Hg, Wg;
  int32_t gs;
  int32_t wsA, wsB;
  int32_t slab;      // pixels per split, multiple of 16
  int32_t qunits;    // tensor-core quad gather: (channel, tap-row) units per k tile
  int32_t math;      // rcv_math
  long long* prof;   // see RcvIgemm::prof
  // normalise-on-load (tensor-core quad gather only): the kernel reads in_scale[ca]*src + in_shift[ca] (then ReLU if
  // in_relu) in place of src at real pixels -- see RcvIgemm::in_scale; padding positions stay zero.  NULL: off.
  const float* in_scale;
  const float* in_shift;
  int32_t in_relu;
  RcvTapSet taps;
};

extern long long* g_rcv_prof;  // debug: phase-timing buffer (rcv_debug_set_prof)
// One entry of the batched weight-pack table (rcv_conv_pack_table_*).
constexpr int RCV_PACK_MAX_JOBS = 128;
struct RcvPackJob {
  RcvIgemm p;
  unsigned char* packed;
  long long chunk_begin, chunks;  // 16-byte chunks: prefix sum over the table, count of this job
  int32_t BN, ntiles, kbmax, kb;  // kb = fp32 elements per K block of the layer's configuration
};
int rcv_umma_pack_job(const RcvIgemm& p, void* packed, long long chunk_begin, RcvPackJob* job);
int rcv_launch_umma_pack_multi(const RcvPackJob* dev_jobs, int njobs, long long total_chunks, cudaStream_t st);

int rcv_launch_igemm(const RcvIgemm& p, cudaStream_t st);       // dispatch on p.math
int rcv_launch_igemm_simt(const RcvIgemm& p, cudaStream_t st);  // fp32 FFMA, CUDA cores
int rcv_launch_direct(const RcvIgemm& p, cudaStream_t st);      // fp32 direct conv, <= 16 output channels
bool rcv_direct_supported(const RcvIgemm& p);
int rcv_launch_narrow(const RcvIgemm& p, cudaStream_t st);      // fp32 FFMA2 direct conv, TMA halo staging, <= 16 output channels
bool rcv_narrow_supported(const RcvIgemm& p);
int rcv_pick_engine(const RcvIgemm& p, bool have_packed);      // rcv_engine that rcv_launch_igemm dispatches to
int rcv_launch_igemm_umma(const RcvIgemm& p, cudaStream_t st);  // tcgen05 3xTF32, TMEM accumulators
bool rcv_umma_halo_ok(const RcvIgemm& p, int bn, int kbb);    // stride-1 3x3, halo-staged A operand (rcv_umma_halo.cu)
int rcv_launch_igemm_umma_halo(const RcvIgemm& p, int bn, int kbb, cudaStream_t st);
size_t rcv_umma_workspace_bytes(const RcvIgemm& p);          // scratch the tensor-core engine can use for this problem (0: none)
size_t rcv_umma_halo_workspace_bytes(const RcvIgemm& p, int bn);
bool rcv_umma_c16_ok(const RcvIgemm& p);                       // 16 -> <= 16 stride-1 3x3: persistent tensor-core kernel (KB = 16 panel)
int rcv_launch_igemm_umma_c16(const RcvIgemm& p, cudaStream_t st);
bool rcv_umma_halo_bf16_ok(const RcvIgemm& p, int bn);        // RCV_MATH_BF16: would that kernel take bf16 operands (bf16 panel layout)
bool rcv_umma_takes_input_transform(const RcvIgemm& p);      // would rcv_launch_igemm_umma run the halo-staged kernel
bool rcv_umma_wgrad_takes_input_transform(const RcvWgrad& p);  // tensor-core weight gradient with the quad gather
bool rcv_umma_pays(const RcvIgemm& p);  // RCV_MATH_AUTO: is the reduction long enough for tensor cores
bool rcv_umma_supported(const RcvIgemm& p);  // geometry within the tensor-core engine's limits
size_t rcv_umma_packed_bytes(const RcvIgemm& p);
int rcv_launch_umma_pack(const RcvIgemm& p, void* packed, cudaStream_t st);
int rcv_launch_wgrad(const RcvWgrad& p, cudaStream_t st);       // dispatch on p.math
int rcv_launch_wgrad_umma(RcvWgrad p, cudaStream_t st);         // tcgen05 3xTF32
bool rcv_umma_wgrad_pays(const RcvWgrad& p);
int rcv_launch_narrow_wgrad(const RcvWgrad& p, cudaStream_t st);  // fp32 FFMA, TMA-staged, few row channels
bool rcv_narrow_wgrad_supported(const RcvWgrad& p);
int rcv_pick_wgrad_engine(const RcvWgrad& p);                  // rcv_engine that rcv_launch_wgrad dispatches to
