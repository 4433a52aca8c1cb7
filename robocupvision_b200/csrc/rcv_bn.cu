// BatchNorm2d (training mode) pieces, ReLU backward and per-channel sums.
// All are HBM-bound streaming kernels over [N, C, HW] fp32 tensors: float4
// accesses along HW, one channel per blockIdx.x so per-channel constants live
// in registers and the reductions finish with one double atomic per block.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "rcv_common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int NT = 256;

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = l < (NT / 32) ? sh[l] : 0.0;
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  }
  return r;  // valid in thread 0
}

__global__ void bn_finalize_kernel(int C, double count, const double* __restrict__ stats,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* running_mean, float* running_var, float momentum, float eps,
                                   float* scale, float* shift, float* save_mean, float* save_invstd,
                                   long long* nbt) {
  rcv_pdl_enter();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (c == 0 && nbt) *nbt += 1;  // BatchNorm2d.num_batches_tracked
  const double mean = stats[c] / count;
  double var = stats[C + c] / count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
  const float sc = g * invstd;
  scale[c] = sc;
  shift[c] = b - (float)mean * sc;
  if (save_mean) save_mean[c] = (float)mean;
  if (save_invstd) save_invstd[c] = invstd;
  if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
  if (running_var) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

__global__ void bn_fold_kernel(int C, const float* __restrict__ gamma, const float* __restrict__ beta,
                               const float* __restrict__ mean, const float* __restrict__ var,
                               float eps, float* scale, float* shift) {
  rcv_pdl_enter();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  // same operation order as ATen's eval batch_norm: invstd = 1/sqrt(var+eps)
  const float invstd = 1.f / sqrtf(var[c] + eps);
  const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
  const float sc = g * invstd;
  scale[c] = sc;
  shift[c] = b - mean[c] * sc;
}

// index into a residual tensor that has only the first RC of the C channels ([N, RC, HW]; RC == C: the same index):
// i = element (or float4) index in [N, C, HW], plane = i / HW = n * C + c
__device__ __forceinline__ int64_t res_index(int64_t i, int64_t plane, int64_t hw, int C, int RC) {
  return RC == C ? i : i - (plane / C) * (int64_t)(C - RC) * hw;
}

// y = act(sc*z+sh) + residual ; flat float4 grid-stride
template <bool VEC>
__global__ void __launch_bounds__(NT) bn_apply_kernel(int64_t total, int C, int64_t HW,
                                                       const float* __restrict__ z,
                                                       const float* __restrict__ scale,
                                                       const float* __restrict__ shift, int relu,
                                                       const float* __restrict__ residual, int RC,
                                                       float* __restrict__ y) {
  rcv_pdl_enter();
  const int64_t stride = (int64_t)gridDim.x * NT;
  if (VEC) {
    const int64_t hw4 = HW >> 2, tot4 = total >> 2;
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < tot4; i += stride) {
      const int64_t plane = i / hw4;
      const int c = (int)(plane % C);
      const float sc = __ldg(scale + c), sh = __ldg(shift + c);
      float4 v = __ldg(reinterpret_cast<const float4*>(z) + i);
      v.x = fmaf(sc, v.x, sh); v.y = fmaf(sc, v.y, sh); v.z = fmaf(sc, v.z, sh); v.w = fmaf(sc, v.w, sh);
      if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
      if (residual && c < RC) {
        const float4 r = __ldg(reinterpret_cast<const float4*>(residual) + res_index(i, plane, hw4, C, RC));
        v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
      }
      reinterpret_cast<float4*>(y)[i] = v;
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < total; i += stride) {
      const int64_t plane = i / HW;
      const int c = (int)(plane % C);
      float v = fmaf(__ldg(scale + c), z[i], __ldg(shift + c));
      if (relu) v = fmaxf(v, 0.f);
      if (residual && c < RC) v += residual[res_index(i, plane, HW, C, RC)];
      y[i] = v;
    }
  }
}

// bn_finalize fused into bn_apply: each block re-derives the per-channel scale / shift from the fp64
// statistics (C <= 1024 values: negligible next to the streaming pass) into shared memory; block 0
// publishes them for the backward pass and updates the running statistics.
template <bool VEC>
__global__ void __launch_bounds__(NT) bn_finalize_apply_kernel(
    int64_t total, int C, int64_t HW, double count, const double* __restrict__ stats,
    const float* __restrict__ gamma, const float* __restrict__ beta, float* running_mean, float* running_var,
    float momentum, float eps, const float* __restrict__ z, int relu, const float* __restrict__ residual, int RC,
    float* __restrict__ y, float* scale_out, float* shift_out, float* save_mean, float* save_invstd,
    long long* nbt) {
  rcv_pdl_enter();
  extern __shared__ float s_ss[];  // [2][C]
  if (blockIdx.x == 0 && threadIdx.x == 0 && nbt) *nbt += 1;  // BatchNorm2d.num_batches_tracked
  for (int c = threadIdx.x; c < C; c += NT) {
    const double mean = stats[c] / count;
    double var = stats[C + c] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    const float sc = g * invstd;
    const float sh = b - (float)mean * sc;
    s_ss[c] = sc;
    s_ss[C + c] = sh;
    if (blockIdx.x == 0) {
      scale_out[c] = sc;
      shift_out[c] = sh;
      if (save_mean) save_mean[c] = (float)mean;
      if (save_invstd) save_invstd[c] = invstd;
      if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
      if (running_var) {
        const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
      }
    }
  }
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * NT;
  if (VEC) {
    const int64_t hw4 = HW >> 2, tot4 = total >> 2;
    // two quads per trip: both loads (and the two residual loads) are in flight before either is used
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < tot4; i += 2 * stride) {
      const int64_t i2 = i + stride;
      const bool two = i2 < tot4;
      float4 v = __ldg(reinterpret_cast<const float4*>(z) + i);
      float4 w = two ? __ldg(reinterpret_cast<const float4*>(z) + i2) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f), q = r;
      const int64_t pl = i / hw4, pl2 = two ? i2 / hw4 : pl;
      const int c = (int)(pl % C), c2 = (int)(pl2 % C);
      if (residual) {
        if (c < RC) r = __ldg(reinterpret_cast<const float4*>(residual) + res_index(i, pl, hw4, C, RC));
        if (two && c2 < RC) q = __ldg(reinterpret_cast<const float4*>(residual) + res_index(i2, pl2, hw4, C, RC));
      }
      const float sc = s_ss[c], sh = s_ss[C + c], sc2 = s_ss[c2], sh2 = s_ss[C + c2];
      v.x = fmaf(sc, v.x, sh); v.y = fmaf(sc, v.y, sh); v.z = fmaf(sc, v.z, sh); v.w = fmaf(sc, v.w, sh);
      w.x = fmaf(sc2, w.x, sh2); w.y = fmaf(sc2, w.y, sh2); w.z = fmaf(sc2, w.z, sh2); w.w = fmaf(sc2, w.w, sh2);
      if (relu) {
        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
        w.x = fmaxf(w.x, 0.f); w.y = fmaxf(w.y, 0.f); w.z = fmaxf(w.z, 0.f); w.w = fmaxf(w.w, 0.f);
      }
      v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
      reinterpret_cast<float4*>(y)[i] = v;
      if (two) {
        w.x += q.x; w.y += q.y; w.z += q.z; w.w += q.w;
        reinterpret_cast<float4*>(y)[i2] = w;
      }
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < total; i += stride) {
      const int c = (int)((i / HW) % C);
      float v = fmaf(s_ss[c], z[i], s_ss[C + c]);
      if (relu) v = fmaxf(v, 0.f);
      if (residual && c < RC) v += residual[res_index(i, i / HW, HW, C, RC)];
      y[i] = v;
    }
  }
}

// One channel per blockIdx.x, blockIdx.y splits the N*HW elements of the channel.
// PASS 0: reduce (sum g, sum g*xhat).  PASS 1: apply + dbias.
template <int PASS>
__global__ void __launch_bounds__(NT) bn_bwd_kernel(int N, int C, int64_t HW, int order,
                                                     const float* __restrict__ dy,
                                                     const float* __restrict__ z,
                                                     const float* __restrict__ scale,
                                                     const float* __restrict__ shift,
                                                     const float* __restrict__ save_mean,
                                                     const float* __restrict__ save_invstd,
                                                     double* sums, float* __restrict__ dconv,
                                                     float* dgamma, float* dbeta, float* dbias) {
  rcv_pdl_enter();
  __shared__ double sh[NT / 32];
  const int c = blockIdx.x;
  const float sc = scale[c], sft = shift[c], mean = save_mean[c], invstd = save_invstd[c];
  const int64_t E = (int64_t)N * HW;  // elements of this channel
  const double cnt = (double)E;
  // The two channel means the apply pass subtracts are kept as fp32 hi + lo pairs of their fp64 values.  Where the
  // incoming gradient is almost all common mode (|g - mean g| << |g|: measured ~1/4000 at the decoder's first
  // blocks), a mean rounded to fp32 leaves the SAME offset on every pixel of the channel, which the next input
  // and weight gradients sum coherently: 10x the error of the fp32 reference, whose CPU kernel does this
  // subtraction in double (tools/grad_accuracy.py).
  float m1 = 0.f, m2 = 0.f, m1l = 0.f, m2l = 0.f;
  if (PASS == 1) {
    const double m1d = sums[c] / cnt, m2d = sums[C + c] / cnt;
    m1 = (float)m1d;
    m1l = (float)(m1d - (double)m1);
    m2 = (float)m2d;
    m2l = (float)(m2d - (double)m2);
  }
  const bool vec = (HW & 3) == 0;
  const int64_t per = (E + gridDim.y - 1) / gridDim.y;
  int64_t beg = (int64_t)blockIdx.y * per;
  beg = vec ? (beg & ~(int64_t)3) : beg;
  int64_t end = (int64_t)(blockIdx.y + 1) * per;
  end = vec ? (end & ~(int64_t)3) : end;
  if (blockIdx.y == gridDim.y - 1) end = E;
  if (end > E) end = E;
  double s1 = 0.0, s2 = 0.0;
  float fs1 = 0.f, fs2 = 0.f;

  auto elem = [&](float g, float zz, float& out) {
    if (order == RCV_EPI_AFFINE_RELU) g = (fmaf(sc, zz, sft) > 0.f) ? g : 0.f;
    const float xh = (zz - mean) * invstd;
    if (PASS == 0) {
      fs1 += g;
      fs2 += g * xh;
    } else {
      float d = sc * fmaf(-xh, m2l, fmaf(-xh, m2, (g - m1) - m1l));
      if (order == RCV_EPI_RELU_AFFINE) d = zz > 0.f ? d : 0.f;
      out = d;
      fs1 += d;
    }
  };

  if (vec) {
    const int step = NT * 4;
    int iter = 0;
    // two quads per trip: all four loads are in flight before the first is used
    for (int64_t e = beg + (int64_t)threadIdx.x * 4; e < end; e += 2 * step) {
      const int64_t e2 = e + step;
      const bool two = e2 < end;
      const int64_t n = e / HW, r = e - n * HW;
      const size_t off = ((size_t)n * C + c) * HW + r;
      size_t off2 = off;
      if (two) {
        const int64_t n2 = e2 / HW, r2 = e2 - n2 * HW;
        off2 = ((size_t)n2 * C + c) * HW + r2;
      }
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(dy + off));
      const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + off));
      const float4 h4 = __ldg(reinterpret_cast<const float4*>(dy + off2));
      const float4 y4 = __ldg(reinterpret_cast<const float4*>(z + off2));
      float4 o;
      elem(g4.x, z4.x, o.x); elem(g4.y, z4.y, o.y); elem(g4.z, z4.z, o.z); elem(g4.w, z4.w, o.w);
      if (PASS == 1) *reinterpret_cast<float4*>(dconv + off) = o;
      if (two) {
        elem(h4.x, y4.x, o.x); elem(h4.y, y4.y, o.y); elem(h4.z, y4.z, o.z); elem(h4.w, y4.w, o.w);
        if (PASS == 1) *reinterpret_cast<float4*>(dconv + off2) = o;
      }
      if ((++iter & 7) == 0) { s1 += fs1; s2 += fs2; fs1 = fs2 = 0.f; }
    }
  } else {
    int iter = 0;
    for (int64_t e = beg + threadIdx.x; e < end; e += NT) {
      const int64_t n = e / HW, r = e - n * HW;
      const size_t off = ((size_t)n * C + c) * HW + r;
      float o = 0.f;
      elem(dy[off], z[off], o);
      if (PASS == 1) dconv[off] = o;
      if ((++iter & 63) == 0) { s1 += fs1; s2 += fs2; fs1 = fs2 = 0.f; }
    }
  }
  s1 += fs1;
  s2 += fs2;
  const double t1 = block_sum(s1, sh);
  if (PASS == 0) {
    const double t2 = block_sum(s2, sh);
    if (threadIdx.x == 0) {
      atomicAdd(sums + c, t1);
      atomicAdd(sums + C + c, t2);
    }
  } else if (threadIdx.x == 0) {
    if (dbias) atomicAdd(dbias + c, (float)t1);
    if (blockIdx.y == 0) {
      if (dgamma) atomicAdd(dgamma + c, (float)(sums[C + c]));
      if (dbeta) atomicAdd(dbeta + c, (float)(sums[c]));
    }
  }
}


// ---------------------------------------------------------------------------------------------------------------
// BatchNorm backward in ONE launch (reduce + apply) for the layers whose channels split into <= 8 CTA-sized slices.
// A channel's reduction (sum g, sum g*xhat) only spans that channel, so no grid-wide barrier is needed: a THREAD-
// BLOCK CLUSTER of CS CTAs owns one channel (grid = C * CS), every CTA reduces its slice, the cluster synchronises,
// every CTA sums the CS partial pairs through distributed shared memory IN RANK ORDER (bitwise reproducible, unlike
// the fp64 atomics of the two-pass form) and applies -- re-reading a slice that is now in L1 / L2.  Clusters are
// co-scheduled by the hardware, so unlike a cooperative grid this runs beside the weight-gradient kernels of the
// side stream.  One launch and one tail instead of two on the backward critical path.
constexpr int BNF_NT = 512;

__device__ __forceinline__ double block_sum_f(double v, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = l < (BNF_NT / 32) ? sh[l] : 0.0;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  }
  return r;  // valid in thread 0
}

__global__ void __launch_bounds__(BNF_NT) bn_bwd_cluster_kernel(int N, int C, int64_t HW, int order,
                                                                const float* __restrict__ dy,
                                                                const float* __restrict__ z,
                                                                const float* __restrict__ scale,
                                                                const float* __restrict__ shift,
                                                                const float* __restrict__ save_mean,
                                                                const float* __restrict__ save_invstd,
                                                                float* __restrict__ dconv, float* dgamma, float* dbeta,
                                                                float* dbias) {
  rcv_pdl_enter();
  cg::cluster_group cluster = cg::this_cluster();
  const int CS = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  __shared__ double sh[BNF_NT / 32];
  __shared__ double part[2];  // this CTA's partial sums; the cluster reads them through distributed shared memory
  __shared__ double tot[2];
  const int c = blockIdx.x / CS;
  const float sc = scale[c], sft = shift[c], mean = save_mean[c], invstd = save_invstd[c];
  const int64_t E = (int64_t)N * HW;  // elements of this channel (HW % 4 == 0: checked by the launcher)
  const int64_t per = (((E + CS - 1) / CS) + 3) & ~(int64_t)3;
  const int64_t beg = (int64_t)rank * per;
  int64_t end = beg + per;
  if (end > E) end = E;
  const int step = BNF_NT * 4;

  auto masked = [&](float g, float zz) {  // the gradient that reaches the BatchNorm output
    return (order == RCV_EPI_AFFINE_RELU && !(fmaf(sc, zz, sft) > 0.f)) ? 0.f : g;
  };
  // ---- phase 1: sum g, sum g * xhat over this CTA's slice (two quads in flight) ----
  double s1 = 0.0, s2 = 0.0;
  {
    float fs1 = 0.f, fs2 = 0.f;
    int iter = 0;
    for (int64_t e = beg + (int64_t)threadIdx.x * 4; e < end; e += 2 * step) {
      const int64_t e2 = e + step;
      const bool two = e2 < end;
      const int64_t n = e / HW, r = e - n * HW;
      const size_t off = ((size_t)n * C + c) * HW + r;
      size_t off2 = off;
      if (two) {
        const int64_t n2 = e2 / HW, r2 = e2 - n2 * HW;
        off2 = ((size_t)n2 * C + c) * HW + r2;
      }
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(dy + off));
      const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + off));
      const float4 h4 = __ldg(reinterpret_cast<const float4*>(dy + off2));
      const float4 y4 = __ldg(reinterpret_cast<const float4*>(z + off2));
      const float gg[8] = {g4.x, g4.y, g4.z, g4.w, h4.x, h4.y, h4.z, h4.w};
      const float zz[8] = {z4.x, z4.y, z4.z, z4.w, y4.x, y4.y, y4.z, y4.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (i >= 4 && !two) break;
        const float g = masked(gg[i], zz[i]);
        fs1 += g;
        fs2 += g * ((zz[i] - mean) * invstd);
      }
      if ((++iter & 7) == 0) { s1 += fs1; s2 += fs2; fs1 = fs2 = 0.f; }
    }
    s1 += fs1;
    s2 += fs2;
  }
  const double t1 = block_sum_f(s1, sh);
  const double t2 = block_sum_f(s2, sh);
  if (threadIdx.x == 0) { part[0] = t1; part[1] = t2; }
  cluster.sync();
  if (threadIdx.x == 0) {
    double S1 = 0.0, S2 = 0.0;
    for (int r = 0; r < CS; ++r) {  // rank order: the sums do not depend on scheduling
      const double* rp = cluster.map_shared_rank(part, r);
      S1 += rp[0];
      S2 += rp[1];
    }
    tot[0] = S1;
    tot[1] = S2;
  }
  cluster.sync();  // (also: no CTA leaves while a peer may still read its partials)
  const double S1 = tot[0], S2 = tot[1];
  const double cnt = (double)E;
  const double m1d = S1 / cnt, m2d = S2 / cnt;
  const float m1 = (float)m1d, m1l = (float)(m1d - (double)m1), m2 = (float)m2d, m2l = (float)(m2d - (double)m2);
  // ---- phase 2: apply (the slice is in L1 / L2 now) ----
  double sd = 0.0;
  {
    float fd = 0.f;
    int iter = 0;
    for (int64_t e = beg + (int64_t)threadIdx.x * 4; e < end; e += 2 * step) {
      const int64_t e2 = e + step;
      const bool two = e2 < end;
      const int64_t n = e / HW, r = e - n * HW;
      const size_t off = ((size_t)n * C + c) * HW + r;
      size_t off2 = off;
      if (two) {
        const int64_t n2 = e2 / HW, r2 = e2 - n2 * HW;
        off2 = ((size_t)n2 * C + c) * HW + r2;
      }
      const float4 g4 = __ldg(reinterpret_cast<const float4*>(dy + off));
      const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + off));
      const float4 h4 = __ldg(reinterpret_cast<const float4*>(dy + off2));
      const float4 y4 = __ldg(reinterpret_cast<const float4*>(z + off2));
      const float gg[8] = {g4.x, g4.y, g4.z, g4.w, h4.x, h4.y, h4.z, h4.w};
      const float zz[8] = {z4.x, z4.y, z4.z, z4.w, y4.x, y4.y, y4.z, y4.w};
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float g = masked(gg[i], zz[i]);
        const float xh = (zz[i] - mean) * invstd;
        float d = sc * fmaf(-xh, m2l, fmaf(-xh, m2, (g - m1) - m1l));
        if (order == RCV_EPI_RELU_AFFINE) d = zz[i] > 0.f ? d : 0.f;
        o[i] = d;
        if (i < 4 || two) fd += d;
      }
      *reinterpret_cast<float4*>(dconv + off) = make_float4(o[0], o[1], o[2], o[3]);
      if (two) *reinterpret_cast<float4*>(dconv + off2) = make_float4(o[4], o[5], o[6], o[7]);
      if ((++iter & 7) == 0) { sd += fd; fd = 0.f; }
    }
    sd += fd;
  }
  const double td = block_sum_f(sd, sh);
  if (threadIdx.x == 0) {
    if (dbias) atomicAdd(dbias + c, (float)td);
    if (rank == 0) {
      if (dgamma) atomicAdd(dgamma + c, (float)S2);
      if (dbeta) atomicAdd(dbeta + c, (float)S1);
    }
  }
}

// cluster size for the one-launch form (0: use the two-pass kernels): enough CTAs to cover the SMs, slices of at
// most 16 k elements (both tensors of a slice then stay in L1 for the second phase).  Measured alone (CUDA graph,
// batch 64): 128 ch @15x20 12.3 -> 11.6 us, 64 ch @30x40 19.1 -> 17.1 us; whole step +0.5 %.
int fused_cluster_size(int C, int64_t E, int64_t HW) {
  static const int on = getenv("RCV_BN_BWD_FUSED") ? atoi(getenv("RCV_BN_BWD_FUSED")) : 1;
  if (!on || (HW & 3) != 0 || C <= 0) return 0;
  int cs = 1;
  while (cs < 8 && ((int64_t)C * cs < 148 || E / cs > 12288)) cs *= 2;
  if (E / cs > 16384) return 0;  // measured: 38 k-element slices (16 channels @60x80 x64) 26.6 us vs 19.1 us in two passes
  return cs;
}

__global__ void __launch_bounds__(NT) relu_bwd_kernel(int64_t n, const float* __restrict__ dy,
                                                       const float* __restrict__ y,
                                                       float* __restrict__ dx) {
  rcv_pdl_enter();
  const int64_t stride = (int64_t)gridDim.x * NT;
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < n4; i += stride) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(dy) + i);
    const float4 v = __ldg(reinterpret_cast<const float4*>(y) + i);
    float4 o;
    o.x = v.x > 0.f ? g.x : 0.f; o.y = v.y > 0.f ? g.y : 0.f;
    o.z = v.z > 0.f ? g.z : 0.f; o.w = v.w > 0.f ? g.w : 0.f;
    reinterpret_cast<float4*>(dx)[i] = o;
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * NT + threadIdx.x; i < n; i += stride)
    dx[i] = y[i] > 0.f ? dy[i] : 0.f;
}

__global__ void __launch_bounds__(NT) channel_sum_kernel(int N, int C, int64_t HW,
                                                          const float* __restrict__ dy, float* dbias) {
  rcv_pdl_enter();
  __shared__ double sh[NT / 32];
  const int c = blockIdx.x;
  const int64_t E = (int64_t)N * HW;
  const int64_t per = (E + gridDim.y - 1) / gridDim.y;
  const int64_t beg = (int64_t)blockIdx.y * per;
  int64_t end = beg + per;
  if (end > E) end = E;
  double s = 0.0;
  float fs = 0.f;
  int iter = 0;
  for (int64_t e = beg + threadIdx.x; e < end; e += NT) {
    const int64_t n = e / HW, r = e - n * HW;
    fs += __ldg(dy + ((size_t)n * C + c) * HW + r);
    if ((++iter & 63) == 0) { s += fs; fs = 0.f; }
  }
  s += fs;
  const double t = block_sum(s, sh);
  if (threadIdx.x == 0) atomicAdd(dbias + c, (float)t);
}

int ew_blocks(int64_t work_items) {
  int64_t b = (work_items + NT - 1) / NT;
  const int64_t cap = 148 * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// bn_finalize_apply: every block re-derives scale / shift from the fp64 statistics, so fewer, fatter blocks:
// one resident wave (8 x 256 threads per SM) and at least two quads per thread
int fa_blocks(int64_t quads) {
  int64_t b = (quads + 2 * NT - 1) / (2 * NT);
  const int64_t cap = 148 * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

int chan_splits(int C, int64_t E) {
  // ONE wave: six CTAs of 256 threads are resident per SM (40 registers), so at most 148 * 6 CTAs.  A grid of 148 * 8
  // ran a second, third-full wave with too few warps per SM to hide the load latency: 42.1 -> 36.4 us for the pair of
  // passes on 8 channels @120x160, 19.0 -> 17.1 us on 16 channels @60x80 (batch 64; 4, 5, 7 and 12 per SM all slower).
  int s = (148 * 6) / C;
  const int64_t maxs = (E + NT * 16 - 1) / (NT * 16);
  if (s > maxs) s = (int)maxs;
  if (s < 1) s = 1;
  if (s > 65535) s = 65535;
  return s;
}

}  // namespace

extern "C" int rcv_bn_finalize(int32_t C, int64_t count, const double* stats, const float* gamma,
                               const float* beta, float* running_mean, float* running_var,
                               float momentum, float eps, float* scale, float* shift,
                               float* save_mean, float* save_invstd, int64_t* num_batches_tracked,
                               void* stream) {
  RCV_REQUIRE(C > 0 && count > 0 && stats && scale && shift, RCV_ERR_BAD_ARG, "bn_finalize: bad arg");
  rcv_launch(bn_finalize_kernel, dim3(rcv_cdiv(C, 128)), dim3(128), 0, (cudaStream_t)stream, C, (double)count, stats,
             gamma, beta, running_mean, running_var, momentum, eps, scale, shift, save_mean, save_invstd,
             reinterpret_cast<long long*>(num_batches_tracked));
  RCV_CHECK_LAUNCH("bn_finalize");
  return RCV_OK;
}

extern "C" int rcv_bn_fold(int32_t C, const float* gamma, const float* beta, const float* mean,
                           const float* var, float eps, float* scale, float* shift, void* stream) {
  RCV_REQUIRE(C > 0 && mean && var && scale && shift, RCV_ERR_BAD_ARG, "bn_fold: bad arg");
  rcv_launch(bn_fold_kernel, dim3(rcv_cdiv(C, 128)), dim3(128), 0, (cudaStream_t)stream, C, gamma, beta, mean, var,
             eps, scale, shift);
  RCV_CHECK_LAUNCH("bn_fold");
  return RCV_OK;
}

extern "C" int rcv_bn_apply(int32_t N, int32_t C, int64_t HW, const float* z, const float* scale,
                            const float* shift, int relu, const float* residual, int32_t res_channels, float* y,
                            void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && HW > 0 && z && scale && shift && y, RCV_ERR_BAD_ARG,
              "bn_apply: bad arg");
  const int64_t total = (int64_t)N * C * HW;
  RCV_REQUIRE(res_channels >= 0 && res_channels <= C, RCV_ERR_BAD_ARG, "bn_apply: res_channels %d outside [0, %d]", res_channels, C);
  const int rc_ = res_channels > 0 ? res_channels : C;
  if ((HW & 3) == 0)
    rcv_launch(bn_apply_kernel<true>, dim3(ew_blocks(total / 4)), dim3(NT), 0, (cudaStream_t)stream, total, C, HW, z,
               scale, shift, relu, residual, rc_, y);
  else
    rcv_launch(bn_apply_kernel<false>, dim3(ew_blocks(total)), dim3(NT), 0, (cudaStream_t)stream, total, C, HW, z,
               scale, shift, relu, residual, rc_, y);
  RCV_CHECK_LAUNCH("bn_apply");
  return RCV_OK;
}

// the statistics in `stats` were summed over `count_` elements per channel: N*HW on one rank, more when the sums were
// added up over the ranks of a global batch (TrainStep(global_batch=True))
extern "C" int rcv_bn_finalize_apply_count(int32_t N, int32_t C, int64_t HW, int64_t count_, const double* stats,
                                           const float* gamma, const float* beta, float* running_mean,
                                           float* running_var, float momentum, float eps, const float* z, int relu,
                                           const float* residual, int32_t res_channels, float* y, float* scale,
                                           float* shift, float* save_mean, float* save_invstd,
                                           int64_t* num_batches_tracked, void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && HW > 0 && count_ > 0 && stats && z && y && scale && shift, RCV_ERR_BAD_ARG,
              "bn_finalize_apply: bad arg");
  RCV_REQUIRE(C <= 4096, RCV_ERR_UNSUPPORTED, "bn_finalize_apply: C=%d > 4096", C);
  const int64_t total = (int64_t)N * C * HW;
  const double count = (double)count_;
  const size_t smem = (size_t)2 * C * sizeof(float);
  RCV_REQUIRE(res_channels >= 0 && res_channels <= C, RCV_ERR_BAD_ARG, "bn_finalize_apply: res_channels %d outside [0, %d]",
              res_channels, C);
  const int rc_ = res_channels > 0 ? res_channels : C;
  if ((HW & 3) == 0)
    rcv_launch(bn_finalize_apply_kernel<true>, dim3(fa_blocks(total / 4)), dim3(NT), smem, (cudaStream_t)stream,
               total, C, HW, count, stats, gamma, beta, running_mean, running_var, momentum, eps, z, relu, residual,
               rc_, y, scale, shift, save_mean, save_invstd, reinterpret_cast<long long*>(num_batches_tracked));
  else
    rcv_launch(bn_finalize_apply_kernel<false>, dim3(ew_blocks(total)), dim3(NT), smem, (cudaStream_t)stream, total,
               C, HW, count, stats, gamma, beta, running_mean, running_var, momentum, eps, z, relu, residual, rc_, y,
               scale, shift, save_mean, save_invstd, reinterpret_cast<long long*>(num_batches_tracked));
  RCV_CHECK_LAUNCH("bn_finalize_apply");
  return RCV_OK;
}

extern "C" int rcv_bn_finalize_apply(int32_t N, int32_t C, int64_t HW, const double* stats, const float* gamma,
                                     const float* beta, float* running_mean, float* running_var, float momentum,
                                     float eps, const float* z, int relu, const float* residual,
                                     int32_t res_channels, float* y,
                                     float* scale, float* shift, float* save_mean, float* save_invstd,
                                     int64_t* num_batches_tracked, void* stream) {
  return rcv_bn_finalize_apply_count(N, C, HW, (int64_t)N * HW, stats, gamma, beta, running_mean, running_var,
                                     momentum, eps, z, relu, residual, res_channels, y, scale, shift, save_mean,
                                     save_invstd, num_batches_tracked, stream);
}

extern "C" int rcv_bn_bwd_reduce(int32_t N, int32_t C, int64_t HW, int order, const float* dy,
                                 const float* z, const float* scale, const float* shift,
                                 const float* save_mean, const float* save_invstd, double* sums,
                                 void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && HW > 0 && dy && z && scale && shift && save_mean && save_invstd && sums,
              RCV_ERR_BAD_ARG, "bn_bwd_reduce: bad arg");
  RCV_REQUIRE(order == RCV_EPI_RELU_AFFINE || order == RCV_EPI_AFFINE_RELU || order == RCV_EPI_AFFINE,
              RCV_ERR_BAD_ARG, "bn_bwd_reduce: bad order %d", order);
  dim3 grid(C, chan_splits(C, (int64_t)N * HW));
  rcv_launch(bn_bwd_kernel<0>, dim3(grid), dim3(NT), 0, (cudaStream_t)stream, N, C, HW, order, dy, z, scale, shift,
             save_mean, save_invstd, sums, nullptr, nullptr, nullptr, nullptr);
  RCV_CHECK_LAUNCH("bn_bwd_reduce");
  return RCV_OK;
}

extern "C" int rcv_bn_bwd_apply(int32_t N, int32_t C, int64_t HW, int order, const float* dy,
                                const float* z, const float* scale, const float* shift,
                                const float* save_mean, const float* save_invstd, const double* sums,
                                float* dconv, float* dgamma, float* dbeta, float* dbias,
                                void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && HW > 0 && dy && z && scale && shift && save_mean && save_invstd &&
                  sums && dconv,
              RCV_ERR_BAD_ARG, "bn_bwd_apply: bad arg");
  RCV_REQUIRE(order == RCV_EPI_RELU_AFFINE || order == RCV_EPI_AFFINE_RELU || order == RCV_EPI_AFFINE,
              RCV_ERR_BAD_ARG, "bn_bwd_apply: bad order %d", order);
  dim3 grid(C, chan_splits(C, (int64_t)N * HW));
  rcv_launch(bn_bwd_kernel<1>, dim3(grid), dim3(NT), 0, (cudaStream_t)stream, N, C, HW, order, dy, z, scale, shift,
             save_mean, save_invstd, const_cast<double*>(sums), dconv, dgamma, dbeta, dbias);
  RCV_CHECK_LAUNCH("bn_bwd_apply");
  return RCV_OK;
}


// 1 if rcv_bn_bwd runs this tensor (16-byte aligned pointers assumed) as one cluster launch, else 0 (two passes)
extern "C" int rcv_bn_bwd_is_fused(int32_t N, int32_t C, int64_t HW) {
  if (N <= 0 || C <= 0 || HW <= 0) return 0;
  return fused_cluster_size(C, (int64_t)N * HW, HW) > 0 ? 1 : 0;
}

// reduce + apply: one cluster launch where the tensor suits it, else the two passes above
extern "C" int rcv_bn_bwd(int32_t N, int32_t C, int64_t HW, int order, const float* dy, const float* z,
                          const float* scale, const float* shift, const float* save_mean, const float* save_invstd,
                          double* sums, float* dconv, float* dgamma, float* dbeta, float* dbias, void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && HW > 0 && dy && z && scale && shift && save_mean && save_invstd && sums && dconv,
              RCV_ERR_BAD_ARG, "bn_bwd: bad arg");
  RCV_REQUIRE(order == RCV_EPI_RELU_AFFINE || order == RCV_EPI_AFFINE_RELU || order == RCV_EPI_AFFINE,
              RCV_ERR_BAD_ARG, "bn_bwd: bad order %d", order);
  const int cs = ((((uintptr_t)dy | (uintptr_t)z | (uintptr_t)dconv) & 15) == 0) ? fused_cluster_size(C, (int64_t)N * HW, HW) : 0;
  if (cs == 0) {
    int rc = rcv_bn_bwd_reduce(N, C, HW, order, dy, z, scale, shift, save_mean, save_invstd, sums, stream);
    if (rc) return rc;
    return rcv_bn_bwd_apply(N, C, HW, order, dy, z, scale, shift, save_mean, save_invstd, sums, dconv, dgamma, dbeta,
                            dbias, stream);
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(C * cs);
  cfg.blockDim = dim3(BNF_NT);
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attrs[2];
  memset(attrs, 0, sizeof(attrs));
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = cs;
  attrs[0].val.clusterDim.y = 1;
  attrs[0].val.clusterDim.z = 1;
  cfg.numAttrs = 1;
  if (rcv_pdl_enabled()) {
    attrs[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
  cfg.attrs = attrs;
  int n = N, cc = C;
  int64_t hw = HW;
  (void)cudaLaunchKernelEx(&cfg, bn_bwd_cluster_kernel, n, cc, hw, order, dy, z, scale, shift, save_mean, save_invstd,
                           dconv, dgamma, dbeta, dbias);
  RCV_CHECK_LAUNCH("bn_bwd_cluster");
  return RCV_OK;
}

extern "C" int rcv_relu_bwd(int64_t n, const float* dy, const float* y, float* dx, void* stream) {
  RCV_REQUIRE(n > 0 && dy && y && dx, RCV_ERR_BAD_ARG, "relu_bwd: bad arg");
  RCV_REQUIRE((((uintptr_t)dy | (uintptr_t)y | (uintptr_t)dx) & 15) == 0, RCV_ERR_BAD_ARG,
              "relu_bwd: pointers must be 16-byte aligned");
  rcv_launch(relu_bwd_kernel, dim3(ew_blocks(n / 4 + 1)), dim3(NT), 0, (cudaStream_t)stream, n, dy, y, dx);
  RCV_CHECK_LAUNCH("relu_bwd");
  return RCV_OK;
}

extern "C" int rcv_channel_sum(int32_t N, int32_t C, int64_t HW, const float* dy, float* dbias,
                               void* stream) {
  RCV_REQUIRE(N > 0 && C > 0 && HW > 0 && dy && dbias, RCV_ERR_BAD_ARG, "channel_sum: bad arg");
  dim3 grid(C, chan_splits(C, (int64_t)N * HW));
  rcv_launch(channel_sum_kernel, dim3(grid), dim3(NT), 0, (cudaStream_t)stream, N, C, HW, dy, dbias);
  RCV_CHECK_LAUNCH("channel_sum");
  return RCV_OK;
}
