// norm.cu -- BatchNorm2d (training mode) and InstanceNorm2d on NHWC fp32 tensors.
//
// Reference call sites: nn.BatchNorm2d(128) / (C, 0.8) dcgan.py:53,56,60,80 (second positional
// argument is eps = 0.8, momentum stays 0.1); nn.InstanceNorm2d(C) pix2pix/models.py:25,40,117,
// cyclegan/models.py:29,33,51,61,76,108 (affine=False, no running stats, eps 1e-5).
// Statistics are kept per "group": g = c (BatchNorm) or n*C + c (InstanceNorm).  Normalisation
// uses the biased variance; running_var is updated with the unbiased one (torch semantics).
// All kernels are HBM-bound streaming passes: float4 accesses along C, fp64 accumulation only
// at the final atomic so that E[x^2]-E[x]^2 does not cancel catastrophically.
#include "common.cuh"
#include <stdlib.h>

namespace b200gan {

// ---- statistics ---------------------------------------------------------------------------
// grid: (ceil(C/32), row_blocks, N or 1).  block (32, 8).
__global__ void __launch_bounds__(256)
norm_stats_kernel(const float *__restrict__ x, double *__restrict__ stats, int C, int64_t rows,
                  int64_t rows_per_block, int G, int per_sample) {
  __shared__ float s1[8][33], s2[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t base_row = per_sample ? (int64_t)blockIdx.z * rows : 0;
  int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  int64_t r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  float a = 0.f, b = 0.f;
  if (c < C) {
    const float *xp = x + (base_row + r0) * C + c;
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      float v = __ldg(xp + (r - r0) * C);
      a += v;
      b = fmaf(v, v, b);
    }
  }
  s1[threadIdx.y][threadIdx.x] = a;
  s2[threadIdx.y][threadIdx.x] = b;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    double ta = 0.0, tb = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      ta += (double)s1[i][threadIdx.x];
      tb += (double)s2[i][threadIdx.x];
    }
    int g = per_sample ? blockIdx.z * C + c : c;
    atomicAdd(stats + g, ta);
    atomicAdd(stats + G + g, tb);
  }
}

__global__ void norm_finalize_kernel(double *__restrict__ stats, const float *__restrict__ gamma,
                                     const float *__restrict__ beta, float *__restrict__ mean_rstd,
                                     float *__restrict__ scale_shift, float *running_mean,
                                     float *running_var, int64_t *nbt, int G, int C, double count,
                                     float eps, float momentum) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0 && nbt) *nbt += 1;
  if (g >= G) return;
  double mean = stats[g] / count;
  double var = stats[G + g] / count - mean * mean;
  stats[g] = 0.0;      // the accumulator is consumed: leave it zeroed for its next use (no memset launch needed)
  stats[G + g] = 0.0;
  if (var < 0.0) var = 0.0;
  float rstd = (float)(1.0 / sqrt(var + (double)eps));
  int c = g % C;
  float ga = gamma ? gamma[c] : 1.f;
  float be = beta ? beta[c] : 0.f;
  mean_rstd[g] = (float)mean;
  mean_rstd[G + g] = rstd;
  float sc = ga * rstd;
  scale_shift[g] = sc;
  scale_shift[G + g] = be - (float)mean * sc;
  if (running_mean) {
    double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[g] = (1.f - momentum) * running_mean[g] + momentum * (float)mean;
    running_var[g] = (1.f - momentum) * running_var[g] + momentum * (float)unbiased;
  }
}

// ---- apply: y = act(x*scale + shift) ----------------------------------------------------------
// One thread per float4 along C (C % 4 == 0) or per element.
template <int VEC>
__global__ void __launch_bounds__(256)
norm_apply_kernel(const float *__restrict__ x, const float *__restrict__ scale_shift,
                  float *__restrict__ y, int64_t total_vec, int C, int64_t HW, int G, int per_sample,
                  int act, float slope, int rtf) {
  const int CV = C / VEC;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (int64_t)gridDim.x * blockDim.x) {
    int cv = (int)(i % CV);
    int64_t row = i / CV;
    int gbase = per_sample ? (int)(row / HW) * C : 0;
    float v[VEC], sc[VEC], sh[VEC];
    if (VEC == 4) {
      float4 t = __ldg(reinterpret_cast<const float4 *>(x) + i);
      v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
      v[0] = __ldg(x + i);
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      int g = gbase + cv * VEC + j;
      sc[j] = __ldg(scale_shift + g);
      sh[j] = __ldg(scale_shift + G + g);
      float o = apply_act(fmaf(v[j], sc[j], sh[j]), act, slope);
      v[j] = rtf ? round_tf32(o) : o;
    }
    if (VEC == 4) {
      reinterpret_cast<float4 *>(y)[i] = make_float4(v[0], v[1], v[2], v[3]);
    } else {
      y[i] = v[0];
    }
  }
}

// ---- backward -----------------------------------------------------------------------------
// pass 1: sums[g] += sum dy', sums[G+g] += sum dy' * xhat   with dy' = dy * act'(y)
__global__ void __launch_bounds__(256)
norm_bwd_reduce_kernel(const float *__restrict__ dy, const float *__restrict__ x,
                       const float *__restrict__ y, const float *__restrict__ mean_rstd,
                       double *__restrict__ sums, int C, int64_t rows, int64_t rows_per_block, int G,
                       int per_sample, int act, float slope) {
  __shared__ float s1[8][33], s2[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t base_row = per_sample ? (int64_t)blockIdx.z * rows : 0;
  int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  int64_t r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  float a = 0.f, b = 0.f;
  if (c < C) {
    int g = per_sample ? blockIdx.z * C + c : c;
    float mean = __ldg(mean_rstd + g), rstd = __ldg(mean_rstd + G + g);
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      int64_t idx = (base_row + r) * C + c;
      float d = __ldg(dy + idx);
      if (act != B200GAN_ACT_NONE) d *= act_grad_from_out(__ldg(y + idx), act, slope);
      float xh = (__ldg(x + idx) - mean) * rstd;
      a += d;
      b = fmaf(d, xh, b);
    }
  }
  s1[threadIdx.y][threadIdx.x] = a;
  s2[threadIdx.y][threadIdx.x] = b;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    double ta = 0.0, tb = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      ta += (double)s1[i][threadIdx.x];
      tb += (double)s2[i][threadIdx.x];
    }
    int g = per_sample ? blockIdx.z * C + c : c;
    atomicAdd(sums + g, ta);
    atomicAdd(sums + G + g, tb);
  }
}

// pass 2: dx = gamma*rstd * (dy' - mean(dy') - xhat * mean(dy' xhat)); also dgamma/dbeta
template <int VEC>
__global__ void __launch_bounds__(256)
norm_bwd_apply_kernel(const float *__restrict__ dy, const float *__restrict__ x,
                      const float *__restrict__ y, const float *__restrict__ mean_rstd,
                      const float *__restrict__ gamma, const double *__restrict__ sums,
                      float *__restrict__ dx, int64_t total_vec, int C, int64_t HW, int G,
                      int per_sample, float inv_count, int act, float slope, int rtf) {
  const int CV = C / VEC;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (int64_t)gridDim.x * blockDim.x) {
    int cv = (int)(i % CV);
    int64_t row = i / CV;
    int gbase = per_sample ? (int)(row / HW) * C : 0;
    float d[VEC], xv[VEC], yv[VEC];
    if (VEC == 4) {
      float4 t = __ldg(reinterpret_cast<const float4 *>(dy) + i);
      d[0] = t.x; d[1] = t.y; d[2] = t.z; d[3] = t.w;
      t = __ldg(reinterpret_cast<const float4 *>(x) + i);
      xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w;
      if (act != B200GAN_ACT_NONE) {
        t = __ldg(reinterpret_cast<const float4 *>(y) + i);
        yv[0] = t.x; yv[1] = t.y; yv[2] = t.z; yv[3] = t.w;
      }
    } else {
      d[0] = __ldg(dy + i);
      xv[0] = __ldg(x + i);
      if (act != B200GAN_ACT_NONE) yv[0] = __ldg(y + i);
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      int c = cv * VEC + j;
      int g = gbase + c;
      float mean = __ldg(mean_rstd + g), rstd = __ldg(mean_rstd + G + g);
      float ga = gamma ? __ldg(gamma + c) : 1.f;
      float m1 = (float)(sums[g]) * inv_count;
      float m2 = (float)(sums[G + g]) * inv_count;
      float dd = d[j];
      if (act != B200GAN_ACT_NONE) dd *= act_grad_from_out(yv[j], act, slope);
      float xh = (xv[j] - mean) * rstd;
      float o = ga * rstd * (dd - m1 - xh * m2);
      d[j] = rtf ? round_tf32(o) : o;
    }
    if (VEC == 4) {
      reinterpret_cast<float4 *>(dx)[i] = make_float4(d[0], d[1], d[2], d[3]);
    } else {
      dx[i] = d[0];
    }
  }
}

__global__ void norm_bwd_params_kernel(double *__restrict__ sums, float *__restrict__ dgb, int G) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  if (dgb) {
    dgb[g] = (float)sums[G + g];  // dgamma = sum dy' * xhat
    dgb[G + g] = (float)sums[g];  // dbeta  = sum dy'
  }
  sums[g] = 0.0;  // workspace handed back zeroed
  sums[G + g] = 0.0;
}


// ---- fast paths (C % 4 == 0, 256 % (C/4) == 0): a thread keeps ONE float4 channel group for its whole loop, so there is
// no index arithmetic beyond an add per element (the generic kernels above spend most of their time in 64-bit div/mod).
// grid = (row blocks, samples): blockIdx.y selects the sample for per-sample (InstanceNorm) groups, else gridDim.y == 1.
__global__ void __launch_bounds__(256)
norm_apply_v4_kernel(const float *__restrict__ x, const float *__restrict__ scale_shift, float *__restrict__ y,
                     int64_t rows, int C, int G, int act, float slope, int rtf) {
  const int CV = C >> 2, cv = threadIdx.x % CV, rpb = 256 / CV;
  const int gbase = (gridDim.y > 1 ? blockIdx.y * C : 0) + cv * 4;
  const float4 sc = __ldg(reinterpret_cast<const float4 *>(scale_shift + gbase));
  const float4 sh = __ldg(reinterpret_cast<const float4 *>(scale_shift + G + gbase));
  const int64_t base = (gridDim.y > 1 ? (int64_t)blockIdx.y * rows : 0);
  const float4 *x4 = reinterpret_cast<const float4 *>(x) + base * CV + cv;
  float4 *y4 = reinterpret_cast<float4 *>(y) + base * CV + cv;
  const int64_t step = (int64_t)gridDim.x * rpb;
#pragma unroll 4
  for (int64_t r = (int64_t)blockIdx.x * rpb + threadIdx.x / CV; r < rows; r += step) {
    const float4 v = __ldg(x4 + r * CV);
    float4 o;
    o.x = apply_act(fmaf(v.x, sc.x, sh.x), act, slope);
    o.y = apply_act(fmaf(v.y, sc.y, sh.y), act, slope);
    o.z = apply_act(fmaf(v.z, sc.z, sh.z), act, slope);
    o.w = apply_act(fmaf(v.w, sc.w, sh.w), act, slope);
    if (rtf) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
    y4[r * CV] = o;
  }
}

// derivative of the fused activation: from the pre-activation value recomputed from x (scale_shift given: LeakyReLU /
// ReLU masks need no saved output) or from the saved output y
__device__ __forceinline__ float norm_act_grad(float xv, float sc, float sh, float yv, bool from_x, int act, float slope) {
  if (act == B200GAN_ACT_NONE) return 1.f;
  if (from_x) {
    const float pre = fmaf(xv, sc, sh);
    return act == B200GAN_ACT_LRELU ? (pre > 0.f ? 1.f : slope) : (pre > 0.f ? 1.f : 0.f);
  }
  return act_grad_from_out(yv, act, slope);
}

__global__ void __launch_bounds__(256)
norm_bwd_reduce_v4_kernel(const float *__restrict__ dy, const float *__restrict__ x, const float *__restrict__ y,
                          const float *__restrict__ mean_rstd, const float *__restrict__ scale_shift,
                          double *__restrict__ sums, int64_t rows, int C, int G, int act, float slope) {
  __shared__ float red[256][8];
  const int CV = C >> 2, cv = threadIdx.x % CV, rpb = 256 / CV;
  const int gbase = (gridDim.y > 1 ? blockIdx.y * C : 0) + cv * 4;
  const bool from_x = scale_shift != nullptr && (act == B200GAN_ACT_LRELU || act == B200GAN_ACT_RELU);
  float mean[4], rstd[4], sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mean[j] = __ldg(mean_rstd + gbase + j);
    rstd[j] = __ldg(mean_rstd + G + gbase + j);
    if (from_x) {
      sc[j] = __ldg(scale_shift + gbase + j);
      sh[j] = __ldg(scale_shift + G + gbase + j);
    }
  }
  const int64_t base = (gridDim.y > 1 ? (int64_t)blockIdx.y * rows : 0);
  const float4 *dy4 = reinterpret_cast<const float4 *>(dy) + base * CV + cv;
  const float4 *x4 = reinterpret_cast<const float4 *>(x) + base * CV + cv;
  const float4 *y4 = reinterpret_cast<const float4 *>(y) + base * CV + cv;
  const bool need_y = act != B200GAN_ACT_NONE && !from_x;
  float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
  const int64_t step = (int64_t)gridDim.x * rpb;
#pragma unroll 4
  for (int64_t r = (int64_t)blockIdx.x * rpb + threadIdx.x / CV; r < rows; r += step) {
    const float4 d = __ldg(dy4 + r * CV), xv = __ldg(x4 + r * CV);
    float4 yv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (need_y) yv = __ldg(y4 + r * CV);
    const float dd[4] = {d.x, d.y, d.z, d.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w}, yy[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float dz = dd[j] * norm_act_grad(xx[j], sc[j], sh[j], yy[j], from_x, act, slope);
      a[j] += dz;
      b[j] = fmaf(dz, (xx[j] - mean[j]) * rstd[j], b[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[threadIdx.x][j] = a[j];
    red[threadIdx.x][4 + j] = b[j];
  }
  __syncthreads();
  if (threadIdx.x < CV) {
    double t[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < rpb; ++r)
#pragma unroll
      for (int j = 0; j < 8; ++j) t[j] += (double)red[r * CV + threadIdx.x][j];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      atomicAdd(sums + gbase + j, t[j]);
      atomicAdd(sums + G + gbase + j, t[4 + j]);
    }
  }
}

__global__ void __launch_bounds__(256)
norm_bwd_apply_v4_kernel(const float *__restrict__ dy, const float *__restrict__ x, const float *__restrict__ y,
                         const float *__restrict__ mean_rstd, const float *__restrict__ scale_shift,
                         const float *__restrict__ gamma, const double *__restrict__ sums, float *__restrict__ dx,
                         int64_t rows, int C, int G, float inv_count, int act, float slope, int rtf) {
  const int CV = C >> 2, cv = threadIdx.x % CV, rpb = 256 / CV;
  const int gbase = (gridDim.y > 1 ? blockIdx.y * C : 0) + cv * 4;
  const bool from_x = scale_shift != nullptr && (act == B200GAN_ACT_LRELU || act == B200GAN_ACT_RELU);
  float mean[4], rstd[4], gr[4], m1[4], m2[4], sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mean[j] = __ldg(mean_rstd + gbase + j);
    rstd[j] = __ldg(mean_rstd + G + gbase + j);
    gr[j] = (gamma ? __ldg(gamma + cv * 4 + j) : 1.f) * rstd[j];
    m1[j] = (float)sums[gbase + j] * inv_count;
    m2[j] = (float)sums[G + gbase + j] * inv_count;
    if (from_x) {
      sc[j] = __ldg(scale_shift + gbase + j);
      sh[j] = __ldg(scale_shift + G + gbase + j);
    }
  }
  const int64_t base = (gridDim.y > 1 ? (int64_t)blockIdx.y * rows : 0);
  const float4 *dy4 = reinterpret_cast<const float4 *>(dy) + base * CV + cv;
  const float4 *x4 = reinterpret_cast<const float4 *>(x) + base * CV + cv;
  const float4 *y4 = reinterpret_cast<const float4 *>(y) + base * CV + cv;
  float4 *dx4 = reinterpret_cast<float4 *>(dx) + base * CV + cv;
  const bool need_y = act != B200GAN_ACT_NONE && !from_x;
  const int64_t step = (int64_t)gridDim.x * rpb;
#pragma unroll 4
  for (int64_t r = (int64_t)blockIdx.x * rpb + threadIdx.x / CV; r < rows; r += step) {
    const float4 d = __ldg(dy4 + r * CV), xv = __ldg(x4 + r * CV);
    float4 yv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (need_y) yv = __ldg(y4 + r * CV);
    const float dd[4] = {d.x, d.y, d.z, d.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w}, yy[4] = {yv.x, yv.y, yv.z, yv.w};
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float dz = dd[j] * norm_act_grad(xx[j], sc[j], sh[j], yy[j], from_x, act, slope);
      const float v = gr[j] * (dz - m1[j] - ((xx[j] - mean[j]) * rstd[j]) * m2[j]);
      o[j] = rtf ? round_tf32(v) : v;
    }
    dx4[r * CV] = make_float4(o[0], o[1], o[2], o[3]);
  }
}

static bool fast_path(const b200gan_norm_desc *d, const void *a, const void *b, const void *c, const void *e) {
  static const bool enabled = !(getenv("B200GAN_NORM_FAST") && atoi(getenv("B200GAN_NORM_FAST")) == 0);
  if (!enabled || d->C % 4 != 0) return false;
  const int CV = d->C / 4;
  if (CV > 256 || 256 % CV != 0) return false;
  return (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c | (uintptr_t)e) & 15) == 0;
}
// (row blocks, samples) with ~8 blocks per SM in total
static dim3 fast_grid(const b200gan_norm_desc *d, int64_t &rows) {
  rows = d->per_sample ? (int64_t)d->HW : (int64_t)d->N * d->HW;
  const int ny = d->per_sample ? d->N : 1;
  const int rpb = 256 / (d->C / 4);
  int64_t want = (148 * 8 + ny - 1) / ny;
  int64_t maxb = ceil_div64(rows, (int64_t)rpb * 4);
  if (want > maxb) want = maxb;
  if (want < 1) want = 1;
  return dim3((unsigned)want, (unsigned)ny, 1);
}

static void reduce_grid(const b200gan_norm_desc *d, dim3 &grid, int64_t &rows, int64_t &rpb) {
  rows = d->per_sample ? (int64_t)d->HW : (int64_t)d->N * d->HW;
  int xb = ceil_div(d->C, 32);
  int zb = d->per_sample ? d->N : 1;
  int64_t want = (148 * 8) / ((int64_t)xb * zb);
  if (want < 1) want = 1;
  rpb = ceil_div64(rows, want);
  if (rpb < 32) rpb = 32;
  int64_t yb = ceil_div64(rows, rpb);
  grid = dim3((unsigned)xb, (unsigned)yb, (unsigned)zb);
}

// ---- double backward of training-mode BatchNorm2d [+ LeakyReLU / ReLU] (gradient penalties of BatchNorm critics) ----
// Per channel over its M elements, with xhat = (x - mean) * r, g = dy * m (m: the activation mask, recomputed from the
// sign of x * scale + shift) and u = dL/d(dx), ggg = dL/d(dgamma), ggb = dL/d(dbeta):
//   A = mean g, B = mean g xhat, U = mean u, Cu = mean u xhat, D = mean u g, E = D - U A - Cu B
//   dL/dx     = r (ggg - gamma r Cu) (g - A - xhat B) - gamma r^2 B (u - U - xhat Cu) - gamma r^2 E xhat
//   dL/ddy    = m (gamma r (u - U - xhat Cu) + ggg xhat + ggb)
//   dL/dgamma = r M E
// One reduction pass gives the five sums [5][C] (sum g, g xhat, u, u xhat, u g); one element-wise pass writes both
// outputs; the parameter kernel writes dL/dgamma and hands the workspace back zeroed.
struct BbCoef {
  float mean, rstd, sc, sh;   // xhat = (x - mean) * rstd; mask from x * sc + sh
  float A, B, U, Cu;          // channel means
  float k1, k2, k3;           // dL/dx = k1 (g - A - xhat B) - k2 (u - U - xhat Cu) - k3 xhat
  float gr, ggg, ggb;         // dL/ddy = m (gr (u - U - xhat Cu) + ggg xhat + ggb)
};

__device__ __forceinline__ BbCoef bb_coef(int c, int C, const float *__restrict__ mean_rstd,
                                          const float *__restrict__ scale_shift, const float *__restrict__ gamma,
                                          const float *__restrict__ gg_gamma, const float *__restrict__ gg_beta,
                                          const double *__restrict__ sums, double inv_count) {
  BbCoef k;
  k.mean = __ldg(mean_rstd + c);
  k.rstd = __ldg(mean_rstd + C + c);
  k.sc = scale_shift ? __ldg(scale_shift + c) : 1.f;
  k.sh = scale_shift ? __ldg(scale_shift + C + c) : 0.f;
  const double A = sums[c] * inv_count, B = sums[C + c] * inv_count, U = sums[2 * C + c] * inv_count;
  const double Cu = sums[3 * C + c] * inv_count, D = sums[4 * C + c] * inv_count;
  const double r = (double)k.rstd, gr = (gamma ? (double)__ldg(gamma + c) : 1.0) * r;
  const double ggg = gg_gamma ? (double)__ldg(gg_gamma + c) : 0.0;
  k.A = (float)A; k.B = (float)B; k.U = (float)U; k.Cu = (float)Cu;
  k.k1 = (float)(r * (ggg - gr * Cu));
  k.k2 = (float)(r * gr * B);
  k.k3 = (float)(r * gr * (D - U * A - Cu * B));
  k.gr = (float)gr;
  k.ggg = (float)ggg;
  k.ggb = gg_beta ? __ldg(gg_beta + c) : 0.f;
  return k;
}

__device__ __forceinline__ float bb_mask(float xv, const BbCoef &k, int act, float slope) {
  if (act == B200GAN_ACT_NONE) return 1.f;
  const float pre = fmaf(xv, k.sc, k.sh);
  return pre > 0.f ? 1.f : (act == B200GAN_ACT_LRELU ? slope : 0.f);
}

// element-wise: both outputs of one element from its three inputs
__device__ __forceinline__ void bb_apply(float dyv, float xv, float uv, const BbCoef &k, int act, float slope,
                                         float &gx, float &gdy) {
  const float m = bb_mask(xv, k, act, slope);
  const float g = dyv * m;
  const float xh = (xv - k.mean) * k.rstd;
  const float t = g - k.A - xh * k.B;
  const float v = uv - k.U - xh * k.Cu;
  gx = fmaf(k.k1, t, -fmaf(k.k2, v, k.k3 * xh));
  gdy = m * fmaf(k.gr, v, fmaf(k.ggg, xh, k.ggb));
}

// generic reduction: block (32 channels, 8 row lanes), grid (ceil(C/32), row blocks)
__global__ void __launch_bounds__(256)
norm_bwd_bwd_reduce_kernel(const float *__restrict__ dy, const float *__restrict__ x, const float *__restrict__ u,
                           const float *__restrict__ mean_rstd, const float *__restrict__ scale_shift,
                           double *__restrict__ sums, int C, int64_t rows, int64_t rows_per_block, int act,
                           float slope) {
  __shared__ float s[5][8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  int64_t r1 = r0 + rows_per_block;
  if (r1 > rows) r1 = rows;
  float p[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  if (c < C) {
    const float mean = __ldg(mean_rstd + c), rstd = __ldg(mean_rstd + C + c);
    const float sc = scale_shift ? __ldg(scale_shift + c) : 1.f, sh = scale_shift ? __ldg(scale_shift + C + c) : 0.f;
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) {
      const int64_t idx = r * C + c;
      const float xv = __ldg(x + idx), uv = __ldg(u + idx);
      float g = __ldg(dy + idx);
      if (act != B200GAN_ACT_NONE) {
        const float pre = fmaf(xv, sc, sh);
        g *= pre > 0.f ? 1.f : (act == B200GAN_ACT_LRELU ? slope : 0.f);
      }
      const float xh = (xv - mean) * rstd;
      p[0] += g;
      p[1] = fmaf(g, xh, p[1]);
      p[2] += uv;
      p[3] = fmaf(uv, xh, p[3]);
      p[4] = fmaf(uv, g, p[4]);
    }
  }
#pragma unroll
  for (int j = 0; j < 5; ++j) s[j][threadIdx.y][threadIdx.x] = p[j];
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += (double)s[j][i][threadIdx.x];
      atomicAdd(sums + j * C + c, t);
    }
  }
}

// generic element-wise pass: one thread per float4 along C (C % 4 == 0) or per element
template <int VEC>
__global__ void __launch_bounds__(256)
norm_bwd_bwd_apply_kernel(const float *__restrict__ dy, const float *__restrict__ x, const float *__restrict__ u,
                          const float *__restrict__ mean_rstd, const float *__restrict__ scale_shift,
                          const float *__restrict__ gamma, const float *__restrict__ gg_gamma,
                          const float *__restrict__ gg_beta, const double *__restrict__ sums, float *__restrict__ gx,
                          float *__restrict__ gdy, int64_t total_vec, int C, double inv_count, int act, float slope) {
  const int CV = C / VEC;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    float d[VEC], xv[VEC], uv[VEC], ox[VEC], od[VEC];
    if (VEC == 4) {
      float4 t = __ldg(reinterpret_cast<const float4 *>(dy) + i);
      d[0] = t.x; d[1] = t.y; d[2] = t.z; d[3] = t.w;
      t = __ldg(reinterpret_cast<const float4 *>(x) + i);
      xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w;
      t = __ldg(reinterpret_cast<const float4 *>(u) + i);
      uv[0] = t.x; uv[1] = t.y; uv[2] = t.z; uv[3] = t.w;
    } else {
      d[0] = __ldg(dy + i);
      xv[0] = __ldg(x + i);
      uv[0] = __ldg(u + i);
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const BbCoef k = bb_coef(cv * VEC + j, C, mean_rstd, scale_shift, gamma, gg_gamma, gg_beta, sums, inv_count);
      bb_apply(d[j], xv[j], uv[j], k, act, slope, ox[j], od[j]);
    }
    if (VEC == 4) {
      reinterpret_cast<float4 *>(gx)[i] = make_float4(ox[0], ox[1], ox[2], ox[3]);
      reinterpret_cast<float4 *>(gdy)[i] = make_float4(od[0], od[1], od[2], od[3]);
    } else {
      gx[i] = ox[0];
      gdy[i] = od[0];
    }
  }
}

// fast reduction (C % 4 == 0, 256 % (C/4) == 0): a thread keeps one float4 channel group; lanes of a warp that share
// it are combined with shuffles, the warps (or row slots) through shared memory, then one fp64 atomic per sum
__global__ void __launch_bounds__(256)
norm_bwd_bwd_reduce_v4_kernel(const float *__restrict__ dy, const float *__restrict__ x, const float *__restrict__ u,
                              const float *__restrict__ mean_rstd, const float *__restrict__ scale_shift,
                              double *__restrict__ sums, int64_t rows, int C, int act, float slope) {
  __shared__ float red[20][256];
  const int CV = C >> 2, cv = threadIdx.x % CV, rpb = 256 / CV;
  float mean[4], rstd[4], sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mean[j] = __ldg(mean_rstd + cv * 4 + j);
    rstd[j] = __ldg(mean_rstd + C + cv * 4 + j);
    if (act != B200GAN_ACT_NONE) {
      sc[j] = __ldg(scale_shift + cv * 4 + j);
      sh[j] = __ldg(scale_shift + C + cv * 4 + j);
    }
  }
  const float4 *dy4 = reinterpret_cast<const float4 *>(dy) + cv;
  const float4 *x4 = reinterpret_cast<const float4 *>(x) + cv;
  const float4 *u4 = reinterpret_cast<const float4 *>(u) + cv;
  float p[20];
#pragma unroll
  for (int j = 0; j < 20; ++j) p[j] = 0.f;
  const int64_t step = (int64_t)gridDim.x * rpb;
#pragma unroll 2
  for (int64_t r = (int64_t)blockIdx.x * rpb + threadIdx.x / CV; r < rows; r += step) {
    const float4 d = __ldg(dy4 + r * CV), xv = __ldg(x4 + r * CV), uv = __ldg(u4 + r * CV);
    const float dd[4] = {d.x, d.y, d.z, d.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w}, uu[4] = {uv.x, uv.y, uv.z, uv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float g = dd[j];
      if (act != B200GAN_ACT_NONE) {
        const float pre = fmaf(xx[j], sc[j], sh[j]);
        g *= pre > 0.f ? 1.f : (act == B200GAN_ACT_LRELU ? slope : 0.f);
      }
      const float xh = (xx[j] - mean[j]) * rstd[j];
      p[j] += g;
      p[4 + j] = fmaf(g, xh, p[4 + j]);
      p[8 + j] += uu[j];
      p[12 + j] = fmaf(uu[j], xh, p[12 + j]);
      p[16 + j] = fmaf(uu[j], g, p[16 + j]);
    }
  }
  const int lane = threadIdx.x & 31;
  int slot, nslots;
  bool writer;
  if (CV < 32) {
    for (int off = 16; off >= CV; off >>= 1)
#pragma unroll
      for (int j = 0; j < 20; ++j) p[j] += __shfl_xor_sync(0xffffffffu, p[j], off);
    slot = threadIdx.x >> 5;
    nslots = 8;
    writer = lane < CV;
  } else {
    slot = threadIdx.x / CV;
    nslots = rpb;
    writer = true;
  }
  if (writer)
#pragma unroll
    for (int j = 0; j < 20; ++j) red[j][slot * CV + cv] = p[j];
  __syncthreads();
  if (threadIdx.x < CV) {
#pragma unroll
    for (int j = 0; j < 20; ++j) {
      double t = 0.0;
      for (int s = 0; s < nslots; ++s) t += (double)red[j][s * CV + threadIdx.x];
      // p[4q + jj]: sum q of channel 4 cv + jj
      atomicAdd(sums + (j >> 2) * C + threadIdx.x * 4 + (j & 3), t);
    }
  }
}

__global__ void __launch_bounds__(256)
norm_bwd_bwd_apply_v4_kernel(const float *__restrict__ dy, const float *__restrict__ x, const float *__restrict__ u,
                             const float *__restrict__ mean_rstd, const float *__restrict__ scale_shift,
                             const float *__restrict__ gamma, const float *__restrict__ gg_gamma,
                             const float *__restrict__ gg_beta, const double *__restrict__ sums,
                             float *__restrict__ gx, float *__restrict__ gdy, int64_t rows, int C, double inv_count,
                             int act, float slope) {
  const int CV = C >> 2, cv = threadIdx.x % CV, rpb = 256 / CV;
  BbCoef k[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)
    k[j] = bb_coef(cv * 4 + j, C, mean_rstd, scale_shift, gamma, gg_gamma, gg_beta, sums, inv_count);
  const float4 *dy4 = reinterpret_cast<const float4 *>(dy) + cv;
  const float4 *x4 = reinterpret_cast<const float4 *>(x) + cv;
  const float4 *u4 = reinterpret_cast<const float4 *>(u) + cv;
  float4 *gx4 = reinterpret_cast<float4 *>(gx) + cv;
  float4 *gdy4 = reinterpret_cast<float4 *>(gdy) + cv;
  const int64_t step = (int64_t)gridDim.x * rpb;
#pragma unroll 2
  for (int64_t r = (int64_t)blockIdx.x * rpb + threadIdx.x / CV; r < rows; r += step) {
    const float4 d = __ldg(dy4 + r * CV), xv = __ldg(x4 + r * CV), uv = __ldg(u4 + r * CV);
    float4 ox, od;
    bb_apply(d.x, xv.x, uv.x, k[0], act, slope, ox.x, od.x);
    bb_apply(d.y, xv.y, uv.y, k[1], act, slope, ox.y, od.y);
    bb_apply(d.z, xv.z, uv.z, k[2], act, slope, ox.z, od.z);
    bb_apply(d.w, xv.w, uv.w, k[3], act, slope, ox.w, od.w);
    gx4[r * CV] = ox;
    gdy4[r * CV] = od;
  }
}

// dL/dgamma = r M E = r (S_ug - S_u S_g / M - S_uxh S_gxh / M); the workspace is handed back zeroed
__global__ void norm_bwd_bwd_params_kernel(double *__restrict__ sums, const float *__restrict__ mean_rstd,
                                           float *__restrict__ dgamma, int C, double count) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (dgamma) {
    const double sg = sums[c], sgx = sums[C + c], su = sums[2 * C + c], sux = sums[3 * C + c], sug = sums[4 * C + c];
    dgamma[c] = (float)((double)mean_rstd[C + c] * (sug - (su * sg + sux * sgx) / count));
  }
#pragma unroll
  for (int j = 0; j < 5; ++j) sums[j * C + c] = 0.0;
}

static int check_desc(const b200gan_norm_desc *d) {
  B2_CHECK_ARG(d != nullptr, "norm: null descriptor");
  B2_CHECK_ARG(d->N > 0 && d->HW > 0 && d->C > 0, "norm: bad dims N=%d HW=%d C=%d", d->N, d->HW, d->C);
  B2_CHECK_ARG(!d->per_sample || d->N <= 65535, "norm: N too large for per-sample grid");
  return B200GAN_OK;
}

}  // namespace b200gan

using namespace b200gan;

extern "C" int b200gan_norm_stats(const b200gan_norm_desc *d, const float *x, double *stats,
                                  void *stream) {
  if (int e = check_desc(d)) return e;
  B2_CHECK_ARG(x && stats, "norm_stats: null pointer");
  dim3 grid;
  int64_t rows, rpb;
  reduce_grid(d, grid, rows, rpb);
  int G = d->per_sample ? d->N * d->C : d->C;
  norm_stats_kernel<<<grid, dim3(32, 8), 0, as_stream(stream)>>>(x, stats, d->C, rows, rpb, G,
                                                                 d->per_sample);
  B2_LAUNCH_CHECK();
  return B200GAN_OK;
}

extern "C" int b200gan_norm_finalize(const b200gan_norm_desc *d, double *stats,
                                     const float *gamma, const float *beta, float *mean_rstd,
                                     float *scale_shift, float *running_mean, float *running_var,
                                     int64_t *num_batches_tracked, void *stream) {
  if (int e = check_desc(d)) return e;
  B2_CHECK_ARG(stats && mean_rstd && scale_shift, "norm_finalize: null pointer");
  B2_CHECK_ARG(!(running_mean && d->per_sample), "norm_finalize: running stats with per-sample norm");
  B2_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr),
               "norm_finalize: running_mean/var must both be given");
  int G = d->per_sample ? d->N * d->C : d->C;
  double count = d->per_sample ? (double)d->HW : (double)d->N * (double)d->HW;
  norm_finalize_kernel<<<ceil_div(G, 128), 128, 0, as_stream(stream)>>>(
      stats, gamma, beta, mean_rstd, scale_shift, running_mean, running_var, num_batches_tracked, G,
      d->C, count, d->eps, d->momentum);
  B2_LAUNCH_CHECK();
  return B200GAN_OK;
}

extern "C" int b200gan_norm_apply(const b200gan_norm_desc *d, const float *x,
                                  const float *scale_shift, float *y, void *stream) {
  if (int e = check_desc(d)) return e;
  B2_CHECK_ARG(x && scale_shift && y, "norm_apply: null pointer");
  int G = d->per_sample ? d->N * d->C : d->C;
  int64_t total = (int64_t)d->N * d->HW * d->C;
  if (fast_path(d, x, y, scale_shift, x) && G % 4 == 0) {
    int64_t rows;
    dim3 grid = fast_grid(d, rows);
    norm_apply_v4_kernel<<<grid, 256, 0, as_stream(stream)>>>(x, scale_shift, y, rows, d->C, G, d->act, d->slope,
                                                              d->round_tf32);
    B2_LAUNCH_CHECK();
    return B200GAN_OK;
  }
  bool vec = (d->C % 4 == 0) && (((uintptr_t)x | (uintptr_t)y) % 16 == 0);
  int64_t tv = vec ? total / 4 : total;
  int64_t blocks = ceil_div64(tv, 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (vec)
    norm_apply_kernel<4><<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
        x, scale_shift, y, tv, d->C, d->HW, G, d->per_sample, d->act, d->slope, d->round_tf32);
  else
    norm_apply_kernel<1><<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(
        x, scale_shift, y, tv, d->C, d->HW, G, d->per_sample, d->act, d->slope, d->round_tf32);
  B2_LAUNCH_CHECK();
  return B200GAN_OK;
}

extern "C" int b200gan_norm_bwd(const b200gan_norm_desc *d, const float *dy, const float *x,
                                const float *y, const float *mean_rstd, const float *scale_shift,
                                const float *gamma, double *sums, float *dx, float *dgamma_dbeta, void *stream) {
  if (int e = check_desc(d)) return e;
  B2_CHECK_ARG(dy && x && mean_rstd && sums && dx, "norm_bwd: null pointer");
  const bool from_x = scale_shift && (d->act == B200GAN_ACT_LRELU || d->act == B200GAN_ACT_RELU);
  B2_CHECK_ARG(d->act == B200GAN_ACT_NONE || from_x || y != nullptr,
               "norm_bwd: fused activation needs the saved output y (or scale_shift for LeakyReLU / ReLU)");
  cudaStream_t st = as_stream(stream);
  int G = d->per_sample ? d->N * d->C : d->C;
  if (fast_path(d, dy, x, dx, y ? (const void *)y : (const void *)x) && G % 4 == 0 &&
      (((uintptr_t)mean_rstd | (uintptr_t)(scale_shift ? scale_shift : mean_rstd)) & 3) == 0) {
    int64_t rows2;
    dim3 g2 = fast_grid(d, rows2);
    const float *yy = y ? y : x;  // never dereferenced when the mask comes from x
    norm_bwd_reduce_v4_kernel<<<g2, 256, 0, st>>>(dy, x, yy, mean_rstd, scale_shift, sums, rows2, d->C, G, d->act, d->slope);
    B2_LAUNCH_CHECK();
    float inv = (float)(1.0 / (d->per_sample ? (double)d->HW : (double)d->N * (double)d->HW));
    norm_bwd_apply_v4_kernel<<<g2, 256, 0, st>>>(dy, x, yy, mean_rstd, scale_shift, gamma, sums, dx, rows2, d->C, G, inv,
                                                 d->act, d->slope, d->round_tf32);
    B2_LAUNCH_CHECK();
    norm_bwd_params_kernel<<<ceil_div(G, 128), 128, 0, st>>>(sums, dgamma_dbeta, G);
    B2_LAUNCH_CHECK();
    return B200GAN_OK;
  }
  B2_CHECK_ARG(d->act == B200GAN_ACT_NONE || y != nullptr, "norm_bwd: this geometry needs the saved output y");
  dim3 grid;
  int64_t rows, rpb;
  reduce_grid(d, grid, rows, rpb);
  norm_bwd_reduce_kernel<<<grid, dim3(32, 8), 0, st>>>(dy, x, y, mean_rstd, sums, d->C, rows, rpb, G,
                                                       d->per_sample, d->act, d->slope);
  B2_LAUNCH_CHECK();
  int64_t total = (int64_t)d->N * d->HW * d->C;
  bool vec = (d->C % 4 == 0) &&
             (((uintptr_t)x | (uintptr_t)dy | (uintptr_t)dx | (uintptr_t)(y ? y : x)) % 16 == 0);
  int64_t tv = vec ? total / 4 : total;
  int64_t blocks = ceil_div64(tv, 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  float inv_count = (float)(1.0 / (d->per_sample ? (double)d->HW : (double)d->N * (double)d->HW));
  if (vec)
    norm_bwd_apply_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(
        dy, x, y, mean_rstd, gamma, sums, dx, tv, d->C, d->HW, G, d->per_sample, inv_count, d->act,
        d->slope, d->round_tf32);
  else
    norm_bwd_apply_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(
        dy, x, y, mean_rstd, gamma, sums, dx, tv, d->C, d->HW, G, d->per_sample, inv_count, d->act,
        d->slope, d->round_tf32);
  B2_LAUNCH_CHECK();
  norm_bwd_params_kernel<<<ceil_div(G, 128), 128, 0, st>>>(sums, dgamma_dbeta, G);
  B2_LAUNCH_CHECK();
  return B200GAN_OK;
}

extern "C" int b200gan_norm_bwd_bwd(const b200gan_norm_desc *d, const float *dy, const float *x, const float *u,
                                    const float *mean_rstd, const float *scale_shift, const float *gamma,
                                    const float *gg_gamma, const float *gg_beta, double *sums, float *gx, float *gdy,
                                    float *dgamma, void *stream) {
  if (int e = check_desc(d)) return e;
  B2_CHECK_ARG(!d->per_sample, "norm_bwd_bwd: per-sample (InstanceNorm) statistics are not supported");
  B2_CHECK_ARG(dy && x && u && mean_rstd && sums && gx && gdy, "norm_bwd_bwd: null pointer");
  B2_CHECK_ARG(d->act == B200GAN_ACT_NONE || d->act == B200GAN_ACT_LRELU || d->act == B200GAN_ACT_RELU,
               "norm_bwd_bwd: fused activation %d (only LeakyReLU / ReLU / none)", d->act);
  B2_CHECK_ARG(d->act == B200GAN_ACT_NONE || scale_shift, "norm_bwd_bwd: the activation mask needs scale_shift");
  cudaStream_t st = as_stream(stream);
  const int C = d->C;
  const int64_t rows = (int64_t)d->N * d->HW;
  const double count = (double)rows, inv = 1.0 / count;
  if (fast_path(d, dy, x, u, gx) && ((uintptr_t)gdy & 15) == 0) {
    int64_t rows2;
    dim3 g2 = fast_grid(d, rows2);
    norm_bwd_bwd_reduce_v4_kernel<<<g2, 256, 0, st>>>(dy, x, u, mean_rstd, scale_shift, sums, rows2, C, d->act,
                                                      d->slope);
    B2_LAUNCH_CHECK();
    norm_bwd_bwd_apply_v4_kernel<<<g2, 256, 0, st>>>(dy, x, u, mean_rstd, scale_shift, gamma, gg_gamma, gg_beta, sums,
                                                     gx, gdy, rows2, C, inv, d->act, d->slope);
    B2_LAUNCH_CHECK();
  } else {
    dim3 grid;
    int64_t rows1, rpb;
    reduce_grid(d, grid, rows1, rpb);
    norm_bwd_bwd_reduce_kernel<<<grid, dim3(32, 8), 0, st>>>(dy, x, u, mean_rstd, scale_shift, sums, C, rows1, rpb,
                                                             d->act, d->slope);
    B2_LAUNCH_CHECK();
    const bool vec = (C % 4 == 0) && (((uintptr_t)dy | (uintptr_t)x | (uintptr_t)u | (uintptr_t)gx |
                                       (uintptr_t)gdy) % 16 == 0);
    const int64_t tv = vec ? rows * C / 4 : rows * C;
    int64_t blocks = ceil_div64(tv, 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (vec)
      norm_bwd_bwd_apply_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(dy, x, u, mean_rstd, scale_shift, gamma, gg_gamma,
                                                                     gg_beta, sums, gx, gdy, tv, C, inv, d->act,
                                                                     d->slope);
    else
      norm_bwd_bwd_apply_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(dy, x, u, mean_rstd, scale_shift, gamma, gg_gamma,
                                                                     gg_beta, sums, gx, gdy, tv, C, inv, d->act,
                                                                     d->slope);
    B2_LAUNCH_CHECK();
  }
  norm_bwd_bwd_params_kernel<<<ceil_div(C, 128), 128, 0, st>>>(sums, mean_rstd, dgamma, C, count);
  B2_LAUNCH_CHECK();
  return B200GAN_OK;
}
