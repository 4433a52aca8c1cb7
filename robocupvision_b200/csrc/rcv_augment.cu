// The step either side of the hot path, as device kernels (SURVEY.md section 8f, row N4):
//   rcv_augment   dataset.py:123-131 (SSYUVDataset.__getitem__, train split): Normalize(mean, std),
//                 horizontal flip of image and label, ColorJitter (dataset.py:19-39: brightness / contrast on Y,
//                 a 2x2 saturation-hue matrix on U, V) -- one pass over the batch with per-image parameters,
//                 so the host-side DataLoader workers only decode.
//   rcv_dice_fwd / rcv_dice_bwd   DiceLoss (model.py:5-43, the --useDice option): per-class soft intersection
//                 and cardinality over softmax(logits) in one pass; the backward pass through the softmax in one.
#include "rcv_common.cuh"

namespace {

constexpr int NT = 256;
constexpr int CMAX = 8;

inline int blocks_for(int64_t n, int cap = 148 * 8) {
  int64_t b = (n + NT - 1) / NT;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// params[n] = {flip, b, c, m00, m01, m10, m11, unused}
__global__ void __launch_bounds__(NT) augment_kernel(int H, int W, const float* __restrict__ x,
                                                      float* __restrict__ y, const long long* __restrict__ lab_in,
                                                      long long* __restrict__ lab_out,
                                                      const float* __restrict__ params, float m0, float m1, float m2,
                                                      float s0, float s1, float s2) {
  rcv_pdl_enter();
  const int n = blockIdx.y;
  const float* pr = params + (size_t)n * 8;
  const bool flip = pr[0] != 0.f;
  const float b = pr[1], c = pr[2], m00 = pr[3], m01 = pr[4], m10 = pr[5], m11 = pr[6];
  const int64_t HW = (int64_t)H * W;
  const float* xi = x + (size_t)n * 3 * HW;
  float* yo = y + (size_t)n * 3 * HW;
  for (int64_t p = (int64_t)blockIdx.x * NT + threadIdx.x; p < HW; p += (int64_t)gridDim.x * NT) {
    const int i = (int)(p / W), j = (int)(p - (int64_t)i * W);
    const int64_t src = flip ? (int64_t)i * W + (W - 1 - j) : p;  // img.flip(2): mirror the columns
    // Normalize: (x - mean) / std per channel, the operation order of torchvision's normalize
    const float yv = (__ldg(xi + src) - m0) / s0;
    const float u = (__ldg(xi + HW + src) - m1) / s1;
    const float v = (__ldg(xi + 2 * HW + src) - m2) / s2;
    yo[p] = (yv + b) * c;                    // img[0] = (img[0] + b_val) * c_val
    yo[HW + p] = m00 * u + m01 * v;          // img[1:] = mtx @ img[1:]
    yo[2 * HW + p] = m10 * u + m11 * v;
    if (lab_in) lab_out[(size_t)n * HW + p] = lab_in[(size_t)n * HW + src];
  }
}

template <int C>
__device__ __forceinline__ void softmax_px(const float* __restrict__ lp, int64_t HW, float (&s)[CMAX]) {
  float z[CMAX];
#pragma unroll
  for (int c = 0; c < C; ++c) z[c] = __ldg(lp + (int64_t)c * HW);
  float mx = z[0];
#pragma unroll
  for (int c = 1; c < C; ++c) mx = fmaxf(mx, z[c]);
  float se = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) { s[c] = expf(z[c] - mx); se += s[c]; }
  const float inv = 1.f / se;
#pragma unroll
  for (int c = 0; c < C; ++c) s[c] *= inv;
}

// sums[c] += sum_p softmax_c(p) * [y_p == c];  sums[C + c] += sum_p (softmax_c(p) + [y_p == c]).
// DET: added into sums through the ordered flush over det (slot = linear block index) instead of atomics.
template <int C, bool DET = false>
__global__ void __launch_bounds__(NT) dice_fwd_kernel(int64_t HW, const float* __restrict__ logits,
                                                       const long long* __restrict__ target, double* sums,
                                                       void* det) {
  rcv_pdl_enter();
  __shared__ double red[2 * CMAX][NT / 32];
  const int n = blockIdx.y;
  float inter[CMAX], card[CMAX];
#pragma unroll
  for (int c = 0; c < C; ++c) inter[c] = card[c] = 0.f;
  int iter = 0;
  double dint[CMAX], dcard[CMAX];
#pragma unroll
  for (int c = 0; c < C; ++c) dint[c] = dcard[c] = 0.0;
  for (int64_t px = (int64_t)blockIdx.x * NT + threadIdx.x; px < HW; px += (int64_t)gridDim.x * NT) {
    float s[CMAX];
    softmax_px<C>(logits + (int64_t)n * C * HW + px, HW, s);
    const int y = (int)__ldg(target + (int64_t)n * HW + px);
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const float oh = (c == y) ? 1.f : 0.f;
      inter[c] += s[c] * oh;
      card[c] += s[c] + oh;
    }
    if ((++iter & 63) == 0) {
#pragma unroll
      for (int c = 0; c < C; ++c) { dint[c] += inter[c]; dcard[c] += card[c]; inter[c] = card[c] = 0.f; }
    }
  }
  const int wi = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    double a = dint[c] + (double)inter[c], b = dcard[c] + (double)card[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (l == 0) { red[c][wi] = a; red[CMAX + c][wi] = b; }
  }
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 2 * C) {
    const int which = threadIdx.x / C, c = threadIdx.x - which * C;
    for (int w = 0; w < NT / 32; ++w) t += red[which * CMAX + c][w];
    if constexpr (!DET) atomicAdd(sums + which * C + c, t);
  }
  if constexpr (DET) {
    __syncthreads();  // every row of red is read before red holds this CTA's partial, sums[] order
    if (threadIdx.x < 2 * C) (&red[0][0])[threadIdx.x] = t;
    __syncthreads();
    rcv_ordered_flush(det, blockIdx.y * gridDim.x + blockIdx.x, gridDim.x * gridDim.y, 2 * C, &red[0][0], sums);
  }
}

// loss = 1 - mean_c(2 w_c I_c / (K_c + eps));  dloss/ds_c(p) = a_c [y_p == c] + b_c with
// a_c = -2 w_c / (C (K_c + eps)), b_c = 2 w_c I_c / (C (K_c + eps)^2);  dz_k = s_k (d_k - sum_c d_c s_c)
template <int C>
__global__ void __launch_bounds__(NT) dice_bwd_kernel(int64_t HW, const float* __restrict__ logits,
                                                       const long long* __restrict__ target,
                                                       const float* __restrict__ weights,
                                                       const double* __restrict__ sums, float eps,
                                                       const float* __restrict__ gscale, float* __restrict__ dlogits) {
  rcv_pdl_enter();
  const int n = blockIdx.y;
  float a[CMAX], b[CMAX];
  const float gs = gscale ? __ldg(gscale) : 1.f;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const double I = sums[c], K = sums[C + c] + (double)eps;
    const double w = weights ? (double)__ldg(weights + c) : 1.0;
    a[c] = (float)(-2.0 * w / ((double)C * K)) * gs;
    b[c] = (float)(2.0 * w * I / ((double)C * K * K)) * gs;
  }
  for (int64_t px = (int64_t)blockIdx.x * NT + threadIdx.x; px < HW; px += (int64_t)gridDim.x * NT) {
    float s[CMAX];
    softmax_px<C>(logits + (int64_t)n * C * HW + px, HW, s);
    const int y = (int)__ldg(target + (int64_t)n * HW + px);
    float d[CMAX], dot = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      d[c] = b[c] + ((c == y) ? a[c] : 0.f);
      dot += d[c] * s[c];
    }
    float* o = dlogits + (int64_t)n * C * HW + px;
#pragma unroll
    for (int c = 0; c < C; ++c) o[(int64_t)c * HW] = s[c] * (d[c] - dot);
  }
}

#define RCV_DICE_DISPATCH(C, CALL)                                                                \
  switch (C) {                                                                                    \
    case 2: { constexpr int CC = 2; CALL; } break;                                                \
    case 3: { constexpr int CC = 3; CALL; } break;                                                \
    case 4: { constexpr int CC = 4; CALL; } break;                                                \
    case 5: { constexpr int CC = 5; CALL; } break;                                                \
    case 6: { constexpr int CC = 6; CALL; } break;                                                \
    case 7: { constexpr int CC = 7; CALL; } break;                                                \
    default: { constexpr int CC = 8; CALL; } break;                                               \
  }

}  // namespace

extern "C" int rcv_augment(int32_t N, int32_t H, int32_t W, const float* x, float* y, const int64_t* labels_in,
                           int64_t* labels_out, const float* params, const float* mean, const float* std_,
                           void* stream) {
  RCV_REQUIRE(N > 0 && H > 0 && W > 0 && x && y && params && mean && std_, RCV_ERR_BAD_ARG, "augment: bad arg");
  RCV_REQUIRE(x != y, RCV_ERR_BAD_ARG, "augment: in-place operation is not supported (the flip reads mirrored columns)");
  RCV_REQUIRE((labels_in == nullptr) == (labels_out == nullptr) && (labels_in == nullptr || labels_in != labels_out),
              RCV_ERR_BAD_ARG, "augment: labels_in / labels_out must both be given (distinct) or both be NULL");
  RCV_REQUIRE(N <= 65535, RCV_ERR_UNSUPPORTED, "augment: N=%d > 65535", N);
  RCV_REQUIRE(std_[0] != 0.f && std_[1] != 0.f && std_[2] != 0.f, RCV_ERR_BAD_ARG, "augment: zero std");
  const int64_t HW = (int64_t)H * W;
  int bx = rcv_cdiv(148 * 8, N);
  dim3 grid(blocks_for(HW, bx < 1 ? 1 : bx), N);
  rcv_launch(augment_kernel, dim3(grid), dim3(NT), 0, (cudaStream_t)stream, H, W, x, y,
             reinterpret_cast<const long long*>(labels_in), reinterpret_cast<long long*>(labels_out), params,
             mean[0], mean[1], mean[2], std_[0], std_[1], std_[2]);
  RCV_CHECK_LAUNCH("augment");
  return RCV_OK;
}

namespace {
dim3 dice_grid(int32_t N, int64_t HW) {
  const int bx = rcv_cdiv(148 * 8, N);
  return dim3(blocks_for(HW, bx < 1 ? 1 : bx), N);
}

int dice_fwd_launch(bool det, int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                    double* sums, void* scratch, void* stream) {
  RCV_REQUIRE(N > 0 && HW > 0 && logits && target && sums, RCV_ERR_BAD_ARG, "dice_fwd: bad arg");
  RCV_REQUIRE(C >= 2 && C <= CMAX, RCV_ERR_UNSUPPORTED, "dice_fwd: C=%d (supported 2..8)", C);
  RCV_REQUIRE(N <= 65535, RCV_ERR_UNSUPPORTED, "dice_fwd: N=%d > 65535", N);
  const dim3 grid = dice_grid(N, HW);
  cudaStream_t st = (cudaStream_t)stream;
  const long long* tg = reinterpret_cast<const long long*>(target);
  if (det) {
    RCV_DICE_DISPATCH(C, (rcv_launch(dice_fwd_kernel<CC, true>, grid, dim3(NT), 0, st, HW, logits, tg, sums, scratch)));
  } else {
    RCV_DICE_DISPATCH(C, (rcv_launch(dice_fwd_kernel<CC>, grid, dim3(NT), 0, st, HW, logits, tg, sums, scratch)));
  }
  RCV_CHECK_LAUNCH("dice_fwd");
  return RCV_OK;
}
}  // namespace

extern "C" int rcv_dice_fwd(int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                            double* sums, void* stream) {
  return dice_fwd_launch(false, N, C, HW, logits, target, sums, nullptr, stream);
}

size_t rcv_dice_fwd_det_bytes(int32_t N, int32_t C, int64_t HW) {
  const dim3 g = dice_grid(N, HW);
  return rcv_det_bytes((long long)g.x * g.y, 2 * C, sizeof(double));
}

extern "C" int rcv_dice_fwd_det(int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                                double* sums, void* scratch, uint64_t scratch_bytes, void* stream) {
  RCV_REQUIRE(N > 0 && N <= 65535 && HW > 0 && C >= 2 && C <= CMAX, RCV_ERR_BAD_ARG, "dice_fwd_det: bad arg");
  RCV_REQUIRE(scratch && scratch_bytes >= rcv_dice_fwd_det_bytes(N, C, HW), RCV_ERR_WORKSPACE,
              "dice_fwd_det: scratch of %llu bytes, %zu needed", (unsigned long long)scratch_bytes,
              rcv_dice_fwd_det_bytes(N, C, HW));
  return dice_fwd_launch(true, N, C, HW, logits, target, sums, scratch, stream);
}

extern "C" int rcv_dice_bwd(int32_t N, int32_t C, int64_t HW, const float* logits, const int64_t* target,
                            const float* weights, const double* sums, float eps, const float* gscale,
                            float* dlogits, void* stream) {
  RCV_REQUIRE(N > 0 && HW > 0 && logits && target && sums && dlogits, RCV_ERR_BAD_ARG, "dice_bwd: bad arg");
  RCV_REQUIRE(C >= 2 && C <= CMAX, RCV_ERR_UNSUPPORTED, "dice_bwd: C=%d (supported 2..8)", C);
  RCV_REQUIRE(N <= 65535, RCV_ERR_UNSUPPORTED, "dice_bwd: N=%d > 65535", N);
  int bx = rcv_cdiv(148 * 8, N);
  dim3 grid(blocks_for(HW, bx < 1 ? 1 : bx), N);
  cudaStream_t st = (cudaStream_t)stream;
  RCV_DICE_DISPATCH(C, (rcv_launch(dice_bwd_kernel<CC>, dim3(grid), dim3(NT), 0, st, HW, logits,
                                   reinterpret_cast<const long long*>(target), weights, sums, eps, gscale,
                                   dlogits)));
  RCV_CHECK_LAUNCH("dice_bwd");
  return RCV_OK;
}
