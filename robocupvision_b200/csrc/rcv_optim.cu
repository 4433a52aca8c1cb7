// Train-step tail over a flat fp32 parameter range: L1-regulariser sub-gradient,
// pruning mask, Adam / SGD update, and the sum|p| the reference adds to the loss
// (train.py:23-27, 52-67).  One streaming pass: reads p,g,m,v (+mask), writes p,m,v.
#include "rcv_common.cuh"

namespace {

constexpr int NT = 256;

// DET (both kernels): l1_sum through the ordered flush over det (slot = block index) instead of an atomic.
template <bool DET>
__global__ void __launch_bounds__(NT) adam_l1_kernel(int64_t n, float* __restrict__ p,
                                                      const float* __restrict__ g,
                                                      float* __restrict__ m, float* __restrict__ v,
                                                      const uint8_t* __restrict__ mask, float lr,
                                                      float b1, float b2, float eps, float bc1,
                                                      float bc2_sqrt, float l1_decay, float grad_scale,
                                                      double* l1_sum,
                                                      const int32_t* __restrict__ step_dev,
                                                      const float* __restrict__ lr_dev, void* det) {
  rcv_pdl_enter();
  __shared__ double sh[NT / 32];
  const int64_t stride = (int64_t)gridDim.x * NT;
  if (step_dev) {  // graph-replayable form: step count and lr live in device memory
    const double t = (double)__ldg(step_dev);
    bc1 = (float)(1.0 - pow((double)b1, t));
    bc2_sqrt = (float)sqrt(1.0 - pow((double)b2, t));
  }
  if (lr_dev) lr = __ldg(lr_dev);
  const float step_size = lr / bc1;
  float l1 = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < n; i += stride) {
    const float pv = p[i];
    l1 += fabsf(pv);
    float gv = grad_scale * g[i];
    if (l1_decay != 0.f) gv += l1_decay * (pv > 0.f ? 1.f : (pv < 0.f ? -1.f : 0.f));
    if (mask && mask[i]) gv = 0.f;
    // torch.optim.Adam (single-tensor path): exp_avg.lerp_(grad, 1-b1);
    // exp_avg_sq = b2*v + (1-b2)*g*g; denom = sqrt(v)/sqrt(bc2) + eps
    const float mv = m[i] + (gv - m[i]) * (1.f - b1);
    const float vv = b2 * v[i] + (1.f - b2) * gv * gv;
    m[i] = mv;
    v[i] = vv;
    const float denom = sqrtf(vv) / bc2_sqrt + eps;
    p[i] = pv - step_size * (mv / denom);
  }
  if (l1_sum) {
    double s = (double)l1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < NT / 32; ++i) t += sh[i];
      if constexpr (DET) sh[0] = t;
      else atomicAdd(l1_sum, t);
    }
    if constexpr (DET) {
      __syncthreads();
      rcv_ordered_flush(det, blockIdx.x, gridDim.x, 1, sh, l1_sum);
    }
  }
}

template <bool DET>
__global__ void __launch_bounds__(NT) sgd_kernel(int64_t n, float* __restrict__ p,
                                                  const float* __restrict__ g, float* __restrict__ buf,
                                                  const uint8_t* __restrict__ mask, float lr,
                                                  float momentum, float wd, float grad_scale,
                                                  int first_step, float l1_decay, double* l1_sum,
                                                  const float* __restrict__ lr_dev, void* det) {
  rcv_pdl_enter();
  __shared__ double sh[NT / 32];
  const int64_t stride = (int64_t)gridDim.x * NT;
  if (lr_dev) lr = __ldg(lr_dev);
  float l1 = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < n; i += stride) {
    const float pv = p[i];
    l1 += fabsf(pv);
    float gv = grad_scale * g[i];
    if (l1_decay != 0.f) gv += l1_decay * (pv > 0.f ? 1.f : (pv < 0.f ? -1.f : 0.f));
    if (mask && mask[i]) gv = 0.f;
    if (wd != 0.f) gv += wd * pv;
    if (momentum != 0.f) {
      const float b = first_step ? gv : momentum * buf[i] + gv;
      buf[i] = b;
      gv = b;
    }
    p[i] = pv - lr * gv;
  }
  if (l1_sum) {
    double s = (double)l1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < NT / 32; ++i) t += sh[i];
      if constexpr (DET) sh[0] = t;
      else atomicAdd(l1_sum, t);
    }
    if constexpr (DET) {
      __syncthreads();
      rcv_ordered_flush(det, blockIdx.x, gridDim.x, 1, sh, l1_sum);
    }
  }
}

int blocks_for(int64_t n) {
  int64_t b = (n + NT - 1) / NT;
  if (b > 148 * 8) b = 148 * 8;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace

namespace {
int adam_launch(bool det, int64_t n, float* p, const float* g, float* m, float* v, const uint8_t* mask, float lr,
                float beta1, float beta2, float eps, int32_t step, float l1_decay, float grad_scale, double* l1_sum,
                const int32_t* step_dev, const float* lr_dev, void* scratch, void* stream) {
  RCV_REQUIRE(n > 0 && p && g && m && v && (step >= 1 || step_dev), RCV_ERR_BAD_ARG,
              "adam_l1_step: bad arg");
  if (step < 1) step = 1;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  rcv_launch(det ? adam_l1_kernel<true> : adam_l1_kernel<false>, dim3(blocks_for(n)), dim3(NT), 0,
             (cudaStream_t)stream, n, p, g, m, v, mask, lr, beta1, beta2, eps, (float)bc1, (float)sqrt(bc2), l1_decay,
             grad_scale, l1_sum, step_dev, lr_dev, scratch);
  RCV_CHECK_LAUNCH("adam_l1_step");
  return RCV_OK;
}
}  // namespace

extern "C" int rcv_adam_l1_step(int64_t n, float* p, const float* g, float* m, float* v,
                                const uint8_t* mask, float lr, float beta1, float beta2, float eps,
                                int32_t step, float l1_decay, float grad_scale, double* l1_sum,
                                const int32_t* step_dev, const float* lr_dev, void* stream) {
  return adam_launch(false, n, p, g, m, v, mask, lr, beta1, beta2, eps, step, l1_decay, grad_scale, l1_sum, step_dev,
                     lr_dev, nullptr, stream);
}

size_t rcv_l1_sum_det_bytes(int64_t n) { return rcv_det_bytes(blocks_for(n), 1, sizeof(double)); }

#define RCV_L1_SCRATCH_CHECK(name)                                                                                 \
  RCV_REQUIRE(n > 0, RCV_ERR_BAD_ARG, name ": bad arg");                                                           \
  RCV_REQUIRE(!l1_sum || (scratch && scratch_bytes >= rcv_l1_sum_det_bytes(n)), RCV_ERR_WORKSPACE,                 \
              name ": scratch of %llu bytes, %zu needed", (unsigned long long)scratch_bytes, rcv_l1_sum_det_bytes(n))

extern "C" int rcv_adam_l1_step_det(int64_t n, float* p, const float* g, float* m, float* v,
                                    const uint8_t* mask, float lr, float beta1, float beta2, float eps,
                                    int32_t step, float l1_decay, float grad_scale, double* l1_sum,
                                    const int32_t* step_dev, const float* lr_dev, void* scratch,
                                    uint64_t scratch_bytes, void* stream) {
  RCV_L1_SCRATCH_CHECK("adam_l1_step_det");
  return adam_launch(true, n, p, g, m, v, mask, lr, beta1, beta2, eps, step, l1_decay, grad_scale, l1_sum, step_dev,
                     lr_dev, scratch, stream);
}

__global__ void counter_add_kernel(int32_t* c, int32_t inc) { rcv_pdl_enter(); *c += inc; }

extern "C" int rcv_counter_add(int32_t* counter, int32_t inc, void* stream) {
  RCV_REQUIRE(counter, RCV_ERR_BAD_ARG, "counter_add: bad arg");
  rcv_launch(counter_add_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, counter, inc);
  RCV_CHECK_LAUNCH("counter_add");
  return RCV_OK;
}

namespace {
int sgd_launch(bool det, int64_t n, float* p, const float* g, float* buf, const uint8_t* mask, float lr,
               float momentum, float weight_decay, float grad_scale, int first_step, float l1_decay, double* l1_sum,
               const float* lr_dev, void* scratch, void* stream) {
  RCV_REQUIRE(n > 0 && p && g && (momentum == 0.f || buf), RCV_ERR_BAD_ARG, "sgd_step: bad arg");
  rcv_launch(det ? sgd_kernel<true> : sgd_kernel<false>, dim3(blocks_for(n)), dim3(NT), 0, (cudaStream_t)stream, n,
             p, g, buf, mask, lr, momentum, weight_decay, grad_scale, first_step, l1_decay, l1_sum, lr_dev, scratch);
  RCV_CHECK_LAUNCH("sgd_step");
  return RCV_OK;
}
}  // namespace

extern "C" int rcv_sgd_step(int64_t n, float* p, const float* g, float* buf, const uint8_t* mask,
                            float lr, float momentum, float weight_decay, float grad_scale,
                            int first_step, float l1_decay, double* l1_sum, const float* lr_dev,
                            void* stream) {
  return sgd_launch(false, n, p, g, buf, mask, lr, momentum, weight_decay, grad_scale, first_step, l1_decay, l1_sum,
                    lr_dev, nullptr, stream);
}

extern "C" int rcv_sgd_step_det(int64_t n, float* p, const float* g, float* buf, const uint8_t* mask,
                                float lr, float momentum, float weight_decay, float grad_scale,
                                int first_step, float l1_decay, double* l1_sum, const float* lr_dev,
                                void* scratch, uint64_t scratch_bytes, void* stream) {
  RCV_L1_SCRATCH_CHECK("sgd_step_det");
  return sgd_launch(true, n, p, g, buf, mask, lr, momentum, weight_decay, grad_scale, first_step, l1_decay, l1_sum,
                    lr_dev, scratch, stream);
}

// Stream-ordered memset (a memset node when captured into a CUDA graph: no kernel): the zero fill of the
// accumulators a step sums into (gradient arena, BatchNorm statistics, loss sums).
extern "C" int rcv_zero(void* ptr, size_t bytes, void* stream) {
  RCV_REQUIRE(ptr || bytes == 0, RCV_ERR_BAD_ARG, "zero: NULL pointer");
  if (bytes == 0) return RCV_OK;
  cudaError_t e = cudaMemsetAsync(ptr, 0, bytes, (cudaStream_t)stream);
  if (e != cudaSuccess) {
    rcv_set_error("zero: %s", cudaGetErrorString(e));
    return RCV_ERR_CUDA;
  }
  return RCV_OK;
}
