// MaxPool2d(2,2) with indices, weighted softmax cross-entropy fused with argmax
// and the per-image confusion matrix, and the label-map confusion kernel.
#include <math.h>

#include "rcv_common.cuh"

namespace {

constexpr int NT = 256;

// ---- max pool --------------------------------------------------------------
// Window scan order and comparison follow ATen's max_pool2d kernel: start at
// -inf with the first element's index, take v if (v > max) || isnan(v).
__global__ void __launch_bounds__(NT) maxpool_fwd_kernel(int64_t total, int H, int W,
                                                          const float* __restrict__ x,
                                                          float* __restrict__ y, int64_t* idx,
                                                          uint8_t* code) {
  rcv_pdl_enter();
  const int Ho = H >> 1, Wo = W >> 1;
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t o = (int64_t)blockIdx.x * NT + threadIdx.x; o < total; o += stride) {
    const int ox = (int)(o % Wo);
    const int64_t t = o / Wo;
    const int oy = (int)(t % Ho);
    const int64_t plane = t / Ho;
    const float* xp = x + plane * (int64_t)H * W + (int64_t)(2 * oy) * W + 2 * ox;
    const float2 r0 = __ldg(reinterpret_cast<const float2*>(xp));
    const float2 r1 = __ldg(reinterpret_cast<const float2*>(xp + W));
    float best = -INFINITY;
    int bc = 0;
    const float v[4] = {r0.x, r0.y, r1.x, r1.y};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (v[k] > best || isnan(v[k])) { best = v[k]; bc = k; }
    y[o] = best;
    if (idx) idx[o] = (int64_t)(2 * oy + (bc >> 1)) * W + 2 * ox + (bc & 1);
    if (code) code[o] = (uint8_t)bc;
  }
}

__global__ void __launch_bounds__(NT) maxpool_bwd_kernel(int64_t total, int H, int W,
                                                          const float* __restrict__ dy,
                                                          const uint8_t* __restrict__ code,
                                                          float* __restrict__ dx) {
  rcv_pdl_enter();
  const int Ho = H >> 1, Wo = W >> 1;
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t o = (int64_t)blockIdx.x * NT + threadIdx.x; o < total; o += stride) {
    const int ox = (int)(o % Wo);
    const int64_t t = o / Wo;
    const int oy = (int)(t % Ho);
    const int64_t plane = t / Ho;
    const float g = __ldg(dy + o);
    const int bc = code[o];
    float* xp = dx + plane * (int64_t)H * W + (int64_t)(2 * oy) * W + 2 * ox;
    *reinterpret_cast<float2*>(xp) = make_float2(bc == 0 ? g : 0.f, bc == 1 ? g : 0.f);
    *reinterpret_cast<float2*>(xp + W) = make_float2(bc == 2 ? g : 0.f, bc == 3 ? g : 0.f);
  }
}

// ---- cross entropy ----------------------------------------------------------
constexpr int CMAX = 8;

template <int C>
__device__ __forceinline__ void load_logits(const float* __restrict__ lp, int64_t HW, float (&z)[CMAX]) {
#pragma unroll
  for (int c = 0; c < C; ++c) z[c] = __ldg(lp + (int64_t)c * HW);
}

// grid: (chunks, N).  One thread per pixel of image blockIdx.y.  DET: loss_sums through the ordered flush over det
// (slot = linear block index) instead of atomics.
template <int C, bool DET = false>
__global__ void __launch_bounds__(NT) ce_fwd_kernel(int64_t HW, const float* __restrict__ logits,
                                                     const int64_t* __restrict__ target,
                                                     const float* __restrict__ class_w,
                                                     double* loss_sums, int64_t* argmax_out,
                                                     unsigned long long* conf,
                                                     unsigned long long* correct, void* det) {
  rcv_pdl_enter();
  __shared__ int hist[CMAX * CMAX];
  __shared__ double red[2][NT / 32];
  __shared__ int ncorrect;
  const int n = blockIdx.y;
  if (threadIdx.x < CMAX * CMAX) hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) ncorrect = 0;
  __syncthreads();
  float w[CMAX];
#pragma unroll
  for (int c = 0; c < C; ++c) w[c] = class_w ? __ldg(class_w + c) : 1.f;
  double lsum = 0.0, wsum = 0.0;
  int corr = 0;
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t px = (int64_t)blockIdx.x * NT + threadIdx.x; px < HW; px += stride) {
    float z[CMAX];
    load_logits<C>(logits + (int64_t)n * C * HW + px, HW, z);
    const int y = (int)__ldg(target + (int64_t)n * HW + px);
    float mx = z[0];
    int am = 0;
#pragma unroll
    for (int c = 1; c < C; ++c)
      if (z[c] > mx) { mx = z[c]; am = c; }
    // torch.max propagates NaN: first NaN wins
#pragma unroll
    for (int c = C - 1; c >= 0; --c)
      if (isnan(z[c])) am = c;
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) se += expf(z[c] - mx);
    const float lse = mx + logf(se);
    float zy = 0.f, wy = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c)
      if (c == y) { zy = z[c]; wy = w[c]; }
    lsum += (double)(wy * (lse - zy));
    wsum += (double)wy;
    if (argmax_out) argmax_out[(int64_t)n * HW + px] = am;
    if (conf && y >= 0 && y < C) atomicAdd(&hist[am * C + y], 1);
    corr += (am == y);
  }
  // block reduction
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
    wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
    corr += __shfl_xor_sync(0xffffffffu, corr, o);
  }
  const int wi = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    red[0][wi] = lsum;
    red[1][wi] = wsum;
    if (corr) atomicAdd(&ncorrect, corr);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int i = 0; i < NT / 32; ++i) { a += red[0][i]; b += red[1][i]; }
    if constexpr (DET) {
      red[0][0] = a;
      red[0][1] = b;
    } else if (loss_sums) {
      atomicAdd(loss_sums, a);
      atomicAdd(loss_sums + 1, b);
    }
    if (correct && ncorrect) atomicAdd(correct, (unsigned long long)ncorrect);
  }
  if (conf && threadIdx.x < C * C) {
    const int h = hist[threadIdx.x];
    if (h) atomicAdd(conf + (int64_t)n * C * C + threadIdx.x, (unsigned long long)h);
  }
  if constexpr (DET) {
    if (loss_sums) {
      __syncthreads();
      rcv_ordered_flush(det, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y, 2, red[0], loss_sums);
    }
  }
}

template <int C>
__global__ void __launch_bounds__(NT) ce_bwd_kernel(int64_t HW, const float* __restrict__ logits,
                                                     const int64_t* __restrict__ target,
                                                     const float* __restrict__ class_w,
                                                     const double* __restrict__ loss_sums,
                                                     const float* __restrict__ gscale,
                                                     float* __restrict__ dlogits) {
  rcv_pdl_enter();
  const int n = blockIdx.y;
  float w[CMAX];
#pragma unroll
  for (int c = 0; c < C; ++c) w[c] = class_w ? __ldg(class_w + c) : 1.f;
  const float gs = (gscale ? __ldg(gscale) : 1.f) / (float)loss_sums[1];
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t px = (int64_t)blockIdx.x * NT + threadIdx.x; px < HW; px += stride) {
    float z[CMAX];
    const int64_t base = (int64_t)n * C * HW + px;
    load_logits<C>(logits + base, HW, z);
    const int y = (int)__ldg(target + (int64_t)n * HW + px);
    float mx = z[0];
#pragma unroll
    for (int c = 1; c < C; ++c) mx = fmaxf(mx, z[c]);
    float e[CMAX], se = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) { e[c] = expf(z[c] - mx); se += e[c]; }
    float wy = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c)
      if (c == y) wy = w[c];
    const float k = gs * wy, inv = 1.f / se;
#pragma unroll
    for (int c = 0; c < C; ++c)
      dlogits[base + (int64_t)c * HW] = k * (e[c] * inv - (c == y ? 1.f : 0.f));
  }
}

__global__ void __launch_bounds__(NT) confusion_kernel(int C, int64_t HW,
                                                        const int64_t* __restrict__ pred,
                                                        const int64_t* __restrict__ target,
                                                        unsigned long long* conf) {
  rcv_pdl_enter();
  __shared__ int hist[CMAX * CMAX];
  const int n = blockIdx.y;
  if (threadIdx.x < CMAX * CMAX) hist[threadIdx.x] = 0;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t px = (int64_t)blockIdx.x * NT + threadIdx.x; px < HW; px += stride) {
    const int64_t p = __ldg(pred + (int64_t)n * HW + px), y = __ldg(target + (int64_t)n * HW + px);
    if (p >= 0 && p < C && y >= 0 && y < C) atomicAdd(&hist[(int)p * C + (int)y], 1);
  }
  __syncthreads();
  if (threadIdx.x < C * C) {
    const int h = hist[threadIdx.x];
    if (h) atomicAdd(conf + (int64_t)n * C * C + threadIdx.x, (unsigned long long)h);
  }
}

int blocks_for(int64_t items, int cap) {
  int64_t b = (items + NT - 1) / NT;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace

extern "C" int rcv_maxpool2x2_fwd(int32_t N, int32_t C, int32_t H, int32_t W, const float* x, float* y,
                                  int64_t* idx, uint8_t* code, void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && H > 1 && W > 1 && x && y, RCV_ERR_BAD_ARG, "maxpool_fwd: bad arg");
  RCV_REQUIRE((H & 1) == 0 && (W & 1) == 0, RCV_ERR_UNSUPPORTED,
              "maxpool_fwd: H and W must be even (got %dx%d)", H, W);
  const int64_t total = (int64_t)N * C * (H / 2) * (W / 2);
  rcv_launch(maxpool_fwd_kernel, dim3(blocks_for(total, 148 * 16)), dim3(NT), 0, (cudaStream_t)stream, total, H, W,
             x, y, idx, code);
  RCV_CHECK_LAUNCH("maxpool_fwd");
  return RCV_OK;
}

extern "C" int rcv_maxpool2x2_bwd(int32_t N, int32_t C, int32_t H, int32_t W, const float* dy,
                                  const uint8_t* code, float* dx, void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && H > 1 && W > 1 && dy && code && dx, RCV_ERR_BAD_ARG,
              "maxpool_bwd: bad arg");
  RCV_REQUIRE((H & 1) == 0 && (W & 1) == 0, RCV_ERR_UNSUPPORTED, "maxpool_bwd: H, W must be even");
  const int64_t total = (int64_t)N * C * (H / 2) * (W / 2);
  rcv_launch(maxpool_bwd_kernel, dim3(blocks_for(total, 148 * 16)), dim3(NT), 0, (cudaStream_t)stream, total, H, W,
             dy, code, dx);
  RCV_CHECK_LAUNCH("maxpool_bwd");
  return RCV_OK;
}

#define RCV_CE_DISPATCH(C_, CALL)                 \
  switch (C_) {                                   \
    case 1: { constexpr int CC = 1; CALL; } break; \
    case 2: { constexpr int CC = 2; CALL; } break; \
    case 3: { constexpr int CC = 3; CALL; } break; \
    case 4: { constexpr int CC = 4; CALL; } break; \
    case 5: { constexpr int CC = 5; CALL; } break; \
    case 6: { constexpr int CC = 6; CALL; } break; \
    case 7: { constexpr int CC = 7; CALL; } break; \
    case 8: { constexpr int CC = 8; CALL; } break; \
    default: break;                               \
  }

namespace {
dim3 ce_grid(int32_t N, int64_t HW) {
  return dim3(blocks_for(HW, rcv_cdiv(148 * 8, N) < 1 ? 1 : rcv_cdiv(148 * 8, N)), N);
}

int ce_fwd_launch(bool det, int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                  const float* class_w, double* loss_sums, int64_t* argmax, int64_t* conf, int64_t* correct,
                  void* scratch, void* stream) {
  RCV_REQUIRE(N > 0 && HW > 0 && logits && target, RCV_ERR_BAD_ARG, "ce_fwd: bad arg");
  RCV_REQUIRE(C >= 1 && C <= CMAX, RCV_ERR_UNSUPPORTED, "ce_fwd: C=%d (supported 1..8)", C);
  RCV_REQUIRE(N <= 65535, RCV_ERR_UNSUPPORTED, "ce_fwd: N=%d > 65535", N);
  const dim3 grid = ce_grid(N, HW);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* cf = reinterpret_cast<unsigned long long*>(conf);
  unsigned long long* cr = reinterpret_cast<unsigned long long*>(correct);
  if (det) {
    RCV_CE_DISPATCH(C, (rcv_launch(ce_fwd_kernel<CC, true>, grid, dim3(NT), 0, st, HW, logits, target, class_w,
                                   loss_sums, argmax, cf, cr, scratch)));
  } else {
    RCV_CE_DISPATCH(C, (rcv_launch(ce_fwd_kernel<CC>, grid, dim3(NT), 0, st, HW, logits, target, class_w,
                                   loss_sums, argmax, cf, cr, scratch)));
  }
  RCV_CHECK_LAUNCH("ce_fwd");
  return RCV_OK;
}
}  // namespace

extern "C" int rcv_ce_fwd(int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                          const float* class_w, double* loss_sums, int64_t* argmax, int64_t* conf,
                          int64_t* correct, void* stream) {
  return ce_fwd_launch(false, N, C, HW, logits, target, class_w, loss_sums, argmax, conf, correct, nullptr, stream);
}

size_t rcv_ce_fwd_det_bytes(int32_t N, int64_t HW) {
  const dim3 g = ce_grid(N, HW);
  return rcv_det_bytes((long long)g.x * g.y, 2, sizeof(double));
}

extern "C" int rcv_ce_fwd_det(int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                              const float* class_w, double* loss_sums, int64_t* argmax, int64_t* conf,
                              int64_t* correct, void* scratch, uint64_t scratch_bytes, void* stream) {
  RCV_REQUIRE(N > 0 && N <= 65535 && HW > 0, RCV_ERR_BAD_ARG, "ce_fwd_det: bad arg");
  RCV_REQUIRE(!loss_sums || (scratch && scratch_bytes >= rcv_ce_fwd_det_bytes(N, HW)), RCV_ERR_WORKSPACE,
              "ce_fwd_det: scratch of %llu bytes, %zu needed", (unsigned long long)scratch_bytes,
              rcv_ce_fwd_det_bytes(N, HW));
  return ce_fwd_launch(true, N, C, HW, logits, target, class_w, loss_sums, argmax, conf, correct, scratch, stream);
}

extern "C" int rcv_ce_bwd(int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                          const float* class_w, const double* loss_sums, const float* gscale,
                          float* dlogits, void* stream) {
  RCV_REQUIRE(N > 0 && HW > 0 && logits && target && loss_sums && dlogits, RCV_ERR_BAD_ARG,
              "ce_bwd: bad arg");
  RCV_REQUIRE(C >= 1 && C <= CMAX, RCV_ERR_UNSUPPORTED, "ce_bwd: C=%d (supported 1..8)", C);
  RCV_REQUIRE(N <= 65535, RCV_ERR_UNSUPPORTED, "ce_bwd: N=%d > 65535", N);
  dim3 grid(blocks_for(HW, rcv_cdiv(148 * 8, N) < 1 ? 1 : rcv_cdiv(148 * 8, N)), N);
  cudaStream_t st = (cudaStream_t)stream;
  RCV_CE_DISPATCH(C, (rcv_launch(ce_bwd_kernel<CC>, dim3(grid), dim3(NT), 0, st, HW, logits, target, class_w,
                                 loss_sums, gscale, dlogits)));
  RCV_CHECK_LAUNCH("ce_bwd");
  return RCV_OK;
}

namespace {
// The per-image IoU rule of the validation loops (train.py:148-153) from per-image confusion counts, and the
// weighted mean loss, in one tiny launch: iou_sum[c] = sum over images of inter / union (1 where union == 0),
// union = row + column - diagonal; loss = loss_sums[0] / loss_sums[1].  One warp per class.
__global__ void __launch_bounds__(256) metric_tail_kernel(int N, int C, const long long* __restrict__ conf,
                                                         const double* __restrict__ loss_sums, double* iou_sum,
                                                         double* loss) {
  rcv_pdl_enter();
  const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (c < C) {
    double acc = 0.0;
    for (int n = lane; n < N; n += 32) {
      const long long* m = conf + (size_t)n * C * C;
      long long row = 0, col = 0;
      for (int k = 0; k < C; ++k) {
        row += m[c * C + k];
        col += m[k * C + c];
      }
      const long long inter = m[c * C + c], uni = row + col - inter;
      acc += uni == 0 ? 1.0 : (double)inter / (double)uni;
    }
    // fixed-order tree: the sum does not depend on scheduling
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) iou_sum[c] = acc;
  }
  if (threadIdx.x == 0 && loss && loss_sums) *loss = loss_sums[0] / loss_sums[1];
}
}  // namespace

extern "C" int rcv_metric_tail(int32_t N, int32_t C, const int64_t* conf, const double* loss_sums, double* iou_sum,
                               double* loss, void* stream) {
  RCV_REQUIRE(N > 0 && conf && iou_sum, RCV_ERR_BAD_ARG, "metric_tail: bad arg");
  RCV_REQUIRE(C >= 1 && C <= CMAX, RCV_ERR_UNSUPPORTED, "metric_tail: C=%d (supported 1..8)", C);
  rcv_launch(metric_tail_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, (int)N, (int)C,
             reinterpret_cast<const long long*>(conf), loss_sums, iou_sum, loss);
  RCV_CHECK_LAUNCH("metric_tail");
  return RCV_OK;
}

extern "C" int rcv_confusion(int32_t N, int32_t C, int64_t HW, const int64_t* pred,
                             const int64_t* target, int64_t* conf, void* stream) {
  RCV_REQUIRE(N > 0 && HW > 0 && pred && target && conf, RCV_ERR_BAD_ARG, "confusion: bad arg");
  RCV_REQUIRE(C >= 1 && C <= CMAX, RCV_ERR_UNSUPPORTED, "confusion: C=%d (supported 1..8)", C);
  RCV_REQUIRE(N <= 65535, RCV_ERR_UNSUPPORTED, "confusion: N=%d > 65535", N);
  dim3 grid(blocks_for(HW, rcv_cdiv(148 * 8, N) < 1 ? 1 : rcv_cdiv(148 * 8, N)), N);
  rcv_launch(confusion_kernel, dim3(grid), dim3(NT), 0, (cudaStream_t)stream, C, HW, pred, target,
             reinterpret_cast<unsigned long long*>(conf));
  RCV_CHECK_LAUNCH("confusion");
  return RCV_OK;
}
