// The classifier head of a TRAINING step in one pass over the decoder's last feature map:
//   logits = W f + b  (the 1x1 classifier conv, model.py:259 / :411 / :554)
//   loss terms, argmax, correct pixels  (CrossEntropyLoss2d model.py:76-82, torch.max train.py:70)
//   dlogits = w_y (softmax - onehot) / sum_p w_{y_p}   (the backward of the mean-reduced weighted NLL)
//   dfeat = W^T dlogits, dW += dlogits f^T, db += dlogits
// instead of conv forward -> ce_fwd -> ce_bwd -> conv dgrad (+ conv wgrad on the side stream): the logits and their
// gradient (2 x N x C x HW floats, written once and read two / three times) never exist in memory.  Algorithmic
// bytes per pixel = 4 Cin (features) + 8 (label) + 4 Cin (feature gradient).  Measured (ncu, ROBO_UNet batch 64):
// 28.6 us = 3.1 TB/s algorithmic, 0.47 of the HBM peak; issue-bound (62 % issue slots at 16 warps per SM: 128
// registers for the C x Cin weight-gradient sums), DRAM itself at 24 % -- the feature gradient stays in L2.
// The normaliser sum_p w_{y_p} depends on the labels only and is produced beforehand by rcv_ce_weight_sum into
// loss_sums[1] (the same cell ce_fwd accumulates it into), so one pass suffices.
#include <math.h>

#include "rcv_common.cuh"

namespace {

constexpr int NT = 256;
constexpr int CMAX = 8;

template <int VEC>
struct VecT;
template <>
struct VecT<1> { using F = float; };
template <>
struct VecT<2> { using F = float2; };

template <int VEC>
__device__ __forceinline__ void ldv(const float* p, float (&o)[VEC]) {
  const typename VecT<VEC>::F v = __ldg(reinterpret_cast<const typename VecT<VEC>::F*>(p));
  const float* s = reinterpret_cast<const float*>(&v);
#pragma unroll
  for (int i = 0; i < VEC; ++i) o[i] = s[i];
}
template <int VEC>
__device__ __forceinline__ void stv(float* p, const float (&o)[VEC]) {
  typename VecT<VEC>::F v;
  float* s = reinterpret_cast<float*>(&v);
#pragma unroll
  for (int i = 0; i < VEC; ++i) s[i] = o[i];
  *reinterpret_cast<typename VecT<VEC>::F*>(p) = v;
}

// sum over all pixels of class_w[target] (1 without weights): the normaliser of the mean-reduced weighted loss.
// DET: added into out through the ordered flush over det (slot = block index) instead of an atomic.
template <bool DET>
__global__ void __launch_bounds__(NT) ce_wsum_kernel(int64_t count, int C, const int64_t* __restrict__ target,
                                                     const float* __restrict__ class_w, double* out, void* det) {
  rcv_pdl_enter();
  __shared__ double sh[NT / 32];
  __shared__ float s_w[CMAX];
  if (threadIdx.x < CMAX) s_w[threadIdx.x] = (threadIdx.x < C) ? (class_w ? class_w[threadIdx.x] : 1.f) : 0.f;
  __syncthreads();
  double tot = 0.0;  // per pixel in double, as ce_fwd accumulates it
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < count; i += stride) {
    const long long y = __ldg(reinterpret_cast<const long long*>(target) + i);
    tot += (y >= 0 && y < C) ? (double)s_w[y] : 0.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = tot;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < NT / 32; ++i) t += sh[i];
    if constexpr (DET) sh[0] = t;
    else atomicAdd(out, t);
  }
  if constexpr (DET) {
    __syncthreads();
    rcv_ordered_flush(det, blockIdx.x, gridDim.x, 1, sh, out);
  }
}

// thread = VEC consecutive pixels of one image; persistent grid-stride over all (image, pixel group) pairs
template <int C, int CIN, int VEC>
__global__ void __launch_bounds__(NT, CIN <= 8 ? 2 : 1) head_ce_kernel(int64_t HW, int64_t groups, const float* __restrict__ feat,
                                                     const float* __restrict__ weight,
                                                     const float* __restrict__ bias,
                                                     const int64_t* __restrict__ target,
                                                     const float* __restrict__ class_w,
                                                     const float* __restrict__ gscale, double* loss_sums,
                                                     unsigned long long* correct, float* __restrict__ dfeat,
                                                     float* dweight, float* dbias) {
  rcv_pdl_enter();
  constexpr int NACC = C * CIN + C;
  __shared__ __align__(16) float s_w[C * CIN];
  __shared__ float s_b[C], s_cw[C];
  __shared__ float s_red[NT / 32][NACC];
  __shared__ double s_l[NT / 32];
  __shared__ int s_corr;
  for (int i = threadIdx.x; i < C * CIN; i += NT) s_w[i] = weight[i];
  if (threadIdx.x < C) {
    s_b[threadIdx.x] = bias ? bias[threadIdx.x] : 0.f;
    s_cw[threadIdx.x] = class_w ? class_w[threadIdx.x] : 1.f;
  }
  if (threadIdx.x == 0) s_corr = 0;
  __syncthreads();
  const float gs = (gscale ? __ldg(gscale) : 1.f) / (float)loss_sums[1];
  float acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.f;
  double lsum = 0.0;
  int corr = 0;
  const int64_t gpi = HW / VEC;  // groups per image
  const int64_t stride = (int64_t)gridDim.x * NT;
  for (int64_t g = (int64_t)blockIdx.x * NT + threadIdx.x; g < groups; g += stride) {
    const int64_t n = g / gpi, px = (g - n * gpi) * VEC;
    const float* fp = feat + (size_t)n * CIN * HW + px;
    float x[CIN][VEC];
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) ldv<VEC>(fp + (size_t)ci * HW, x[ci]);
    long long yv[VEC];
    {
      const long long* tp = reinterpret_cast<const long long*>(target) + (size_t)n * HW + px;
      if (VEC == 1) {
        yv[0] = __ldg(tp);
      } else {
#pragma unroll
        for (int v = 0; v < VEC; v += 2) {
          const longlong2 t2 = __ldg(reinterpret_cast<const longlong2*>(tp + v));
          yv[v] = t2.x;
          yv[v + 1 < VEC ? v + 1 : v] = t2.y;
        }
      }
    }
    // The weights are read from shared memory where they are used (volatile: the compiler would otherwise keep all
    // C x CIN of them in registers next to the C x CIN sums); every weight read serves the VEC pixels of the thread.
    const volatile float* vw = s_w;
    float z[C][VEC];
#pragma unroll
    for (int c = 0; c < C; ++c) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) z[c][v] = s_b[c];
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) {
        const float w = vw[c * CIN + ci];
#pragma unroll
        for (int v = 0; v < VEC; ++v) z[c][v] = fmaf(w, x[ci][v], z[c][v]);
      }
    }
    // z <- dlogits, pixel by pixel
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const int y = (yv[v] >= 0 && yv[v] < C) ? (int)yv[v] : -1;
      float mx = z[0][v];
      int am = 0;
#pragma unroll
      for (int c = 1; c < C; ++c)
        if (z[c][v] > mx) { mx = z[c][v]; am = c; }
#pragma unroll
      for (int c = C - 1; c >= 0; --c)  // torch.max propagates NaN: first NaN wins
        if (isnan(z[c][v])) am = c;
      float zy = 0.f, wy = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c)
        if (c == y) { zy = z[c][v]; wy = s_cw[c]; }
      float se = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) { z[c][v] = expf(z[c][v] - mx); se += z[c][v]; }
      const float lse = mx + logf(se);
      lsum += (double)(wy * (lse - zy));
      corr += (am == y);
      const float k = gs * wy, inv = 1.f / se;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        z[c][v] = k * (z[c][v] * inv - (c == y ? 1.f : 0.f));
        acc[C * CIN + c] += z[c][v];
      }
    }
    // feature gradient (written over x) and the weight-gradient sums
    float* dp = dfeat + (size_t)n * CIN * HW + px;
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) {
      float d[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) d[v] = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float w = vw[c * CIN + ci];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          d[v] = fmaf(w, z[c][v], d[v]);
          acc[c * CIN + ci] = fmaf(z[c][v], x[ci][v], acc[c * CIN + ci]);
        }
      }
      stv<VEC>(dp + (size_t)ci * HW, d);
    }
  }
  // block reduction: shuffles, then the warps' rows in shared memory, then one atomic per number per CTA
  const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < NACC; ++i) {
    float a = acc[i];
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) a += __shfl_xor_sync(0xffffffffu, a, s);
    if (lane == 0) s_red[wi][i] = a;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    lsum += __shfl_xor_sync(0xffffffffu, lsum, s);
    corr += __shfl_xor_sync(0xffffffffu, corr, s);
  }
  if (lane == 0) {
    s_l[wi] = lsum;
    if (corr) atomicAdd(&s_corr, corr);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NACC; i += NT) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) a += s_red[w][i];
    if (i < C * CIN) {
      atomicAdd(dweight + i, a);
    } else if (dbias) {
      atomicAdd(dbias + (i - C * CIN), a);
    }
  }
  if (threadIdx.x == 0) {
    double a = 0.0;
    for (int w = 0; w < NT / 32; ++w) a += s_l[w];
    atomicAdd(loss_sums, a);
    if (correct && s_corr) atomicAdd(correct, (unsigned long long)s_corr);
  }
}

int vec_for(int Cin, int64_t HW, const void* a, const void* b, const void* c) {
  const uintptr_t al = (uintptr_t)a | (uintptr_t)b | (uintptr_t)c;
  // registers: Cin x VEC features + C x VEC logits + C x Cin sums; 8 channels: two pixels per thread at two CTAs per
  // SM, 16 channels: one pixel per thread
  if (Cin <= 8 && HW % 2 == 0 && al % 16 == 0) return 2;
  return 1;
}

template <int C, int CIN>
void launch_head(int vec, dim3 grid, cudaStream_t st, int64_t HW, int64_t N, const float* feat, const float* weight,
                 const float* bias, const int64_t* target, const float* class_w, const float* gscale,
                 double* loss_sums, unsigned long long* correct, float* dfeat, float* dweight, float* dbias) {
  if (vec == 4) return;
  else if (vec == 2)
    rcv_launch(head_ce_kernel<C, CIN, 2>, grid, dim3(NT), 0, st, HW, N * (HW / 2), feat, weight, bias, target, class_w,
               gscale, loss_sums, correct, dfeat, dweight, dbias);
  else
    rcv_launch(head_ce_kernel<C, CIN, 1>, grid, dim3(NT), 0, st, HW, N * HW, feat, weight, bias, target, class_w, gscale,
               loss_sums, correct, dfeat, dweight, dbias);
}

}  // namespace

// 1 if rcv_head_ce_train has a kernel for this head (classes 2..8 over 8 or 16 feature channels), else 0
extern "C" int rcv_head_ce_supported(int32_t Cin, int32_t C) {
  return (Cin == 8 || Cin == 16) && C >= 2 && C <= CMAX ? 1 : 0;
}

namespace {
int ce_wsum_blocks(int64_t count) {
  int64_t nb = (count + NT * 8 - 1) / (NT * 8);
  if (nb > 148 * 4) nb = 148 * 4;
  if (nb < 1) nb = 1;
  return (int)nb;
}

int ce_wsum_launch(bool det, int32_t C, int64_t count, const int64_t* target, const float* class_w, double* out,
                   void* scratch, void* stream) {
  RCV_REQUIRE(count > 0 && target && out, RCV_ERR_BAD_ARG, "ce_weight_sum: bad arg");
  RCV_REQUIRE(C >= 1 && C <= CMAX, RCV_ERR_UNSUPPORTED, "ce_weight_sum: C=%d (supported 1..8)", C);
  rcv_launch(det ? ce_wsum_kernel<true> : ce_wsum_kernel<false>, dim3((unsigned)ce_wsum_blocks(count)), dim3(NT), 0,
             (cudaStream_t)stream, count, (int)C, target, class_w, out, scratch);
  RCV_CHECK_LAUNCH("ce_weight_sum");
  return RCV_OK;
}
}  // namespace

extern "C" int rcv_ce_weight_sum(int32_t C, int64_t count, const int64_t* target, const float* class_w, double* out,
                                 void* stream) {
  return ce_wsum_launch(false, C, count, target, class_w, out, nullptr, stream);
}

size_t rcv_ce_weight_sum_det_bytes(int64_t count) { return rcv_det_bytes(ce_wsum_blocks(count), 1, sizeof(double)); }

extern "C" int rcv_ce_weight_sum_det(int32_t C, int64_t count, const int64_t* target, const float* class_w,
                                     double* out, void* scratch, uint64_t scratch_bytes, void* stream) {
  RCV_REQUIRE(count > 0, RCV_ERR_BAD_ARG, "ce_weight_sum_det: bad arg");
  RCV_REQUIRE(scratch && scratch_bytes >= rcv_ce_weight_sum_det_bytes(count), RCV_ERR_WORKSPACE,
              "ce_weight_sum_det: scratch of %llu bytes, %zu needed", (unsigned long long)scratch_bytes,
              rcv_ce_weight_sum_det_bytes(count));
  return ce_wsum_launch(true, C, count, target, class_w, out, scratch, stream);
}

extern "C" int rcv_head_ce_train(int32_t N, int32_t Cin, int32_t C, int64_t HW, const float* feat, const float* weight,
                                 const float* bias, const int64_t* target, const float* class_w, const float* gscale,
                                 double* loss_sums, int64_t* correct, float* dfeat, float* dweight, float* dbias,
                                 void* stream) {
  RCV_REQUIRE(N > 0 && HW > 0 && feat && weight && target && loss_sums && dfeat && dweight, RCV_ERR_BAD_ARG,
              "head_ce_train: bad arg");
  RCV_REQUIRE(rcv_head_ce_supported(Cin, C), RCV_ERR_UNSUPPORTED,
              "head_ce_train: %d classes over %d channels (supported: 2..8 classes over 8 or 16 channels)", C, Cin);
  const int vec = vec_for(Cin, HW, feat, dfeat, target);
  const int64_t groups = (int64_t)N * (HW / vec);
  int64_t nb = (groups + NT - 1) / NT;
  if (nb > 148 * 2) nb = 148 * 2;  // persistent: the per-CTA reduction at the end costs C * Cin atomics
  if (nb < 1) nb = 1;
  const dim3 grid((unsigned)nb);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* corr = reinterpret_cast<unsigned long long*>(correct);
#define RCV_HEAD_CASE(CC)                                                                                          \
  case CC:                                                                                                          \
    if (Cin == 8)                                                                                                   \
      launch_head<CC, 8>(vec, grid, st, HW, N, feat, weight, bias, target, class_w, gscale, loss_sums, corr, dfeat, \
                         dweight, dbias);                                                                           \
    else                                                                                                            \
      launch_head<CC, 16>(vec, grid, st, HW, N, feat, weight, bias, target, class_w, gscale, loss_sums, corr,      \
                          dfeat, dweight, dbias);                                                                   \
    break;
  switch (C) {
    RCV_HEAD_CASE(2) RCV_HEAD_CASE(3) RCV_HEAD_CASE(4) RCV_HEAD_CASE(5)
    RCV_HEAD_CASE(6) RCV_HEAD_CASE(7) RCV_HEAD_CASE(8)
  }
#undef RCV_HEAD_CASE
  RCV_CHECK_LAUNCH("head_ce_train");
  return RCV_OK;
}
