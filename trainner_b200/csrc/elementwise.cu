// HBM-bound kernels of the ESRGAN step: BatchNorm(+LeakyReLU) fwd/bwd, MaxPool fwd/bwd,
// nearest-upsample backward, L1 losses, layout conversion.  All NHWC bf16 with 128-bit accesses
// and warp-shuffle / shared-memory reductions.
#include "common.cuh"

namespace b200 {
namespace {

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return u;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

inline int grid_for(long long work_items, int threads, int max_blocks = 148 * 16) {
  long long b = (work_items + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return (int)b;
}

// ------------------------------------------------------------------ BatchNorm
// Each thread owns one 8-channel vector lane (c/8 lanes per pixel) and strides over pixels.
// per-channel statistics -> mean / invstd (+ running statistics, unbiased variance, like nn.BatchNorm2d)
__device__ __forceinline__ void bn_finalize_channel(const float* stats, float* mean_invstd, float* running_mean,
                                                    float* running_var, long long npix, int c, float momentum,
                                                    float eps, int ch) {
  const double n = (double)npix;
  const double mean = stats[ch] / n;
  double var = stats[c + ch] / n - mean * mean;
  if (var < 0) var = 0;
  mean_invstd[ch] = (float)mean;
  mean_invstd[c + ch] = (float)(1.0 / sqrt(var + (double)eps));
  if (running_mean) {
    const double unbiased = npix > 1 ? var * n / (n - 1.0) : var;
    running_mean[ch] = (float)((1.0 - momentum) * running_mean[ch] + momentum * mean);
    running_var[ch] = (float)((1.0 - momentum) * running_var[ch] + momentum * unbiased);
  }
}

// blockDim = 256; lanes_per_pix = c/8 must divide 256 or be a multiple handled by the loop.
template <int MODE>  // 0: stats of z ; 1: bwd reduce (sum dbn, sum dbn*zhat)
__global__ void bn_reduce_kernel(const __nv_bfloat16* __restrict__ z,
                                 const __nv_bfloat16* __restrict__ da,
                                 const float* __restrict__ mean_invstd,
                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                 float* __restrict__ sums, long long npix, int c, float slope,
                                 float* __restrict__ part, unsigned* __restrict__ counter,
                                 float* __restrict__ dgamma, float* __restrict__ dbeta,
                                 float* __restrict__ fin_mean_invstd, float* __restrict__ running_mean,
                                 float* __restrict__ running_var, float momentum, float eps) {
  pdl_trigger();
  pdl_wait();
  const int vec_per_pix = c / 8;
  const long long total_vec = npix * vec_per_pix;
  const long long stride = (long long)gridDim.x * blockDim.x;
  // make every thread keep a fixed channel lane: stride must be a multiple of vec_per_pix
  // (host guarantees blockDim.x * gridDim.x % vec_per_pix == 0)
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int cv = (int)(i % vec_per_pix) * 8;
  float s0[8], s1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s0[j] = s1[j] = 0.f;
  float mu[8], is[8], ga[8], be[8];
  if (MODE == 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      mu[j] = mean_invstd[cv + j];
      is[j] = mean_invstd[c + cv + j];
      ga[j] = gamma[cv + j];
      be[j] = beta[cv + j];
    }
  }
  constexpr int U = 4;
  for (; i < total_vec; i += U * stride) {
    uint4 zv[U], gv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long iu = i + u * stride;
      zv[u] = iu < total_vec ? reinterpret_cast<const uint4*>(z)[iu] : make_uint4(0, 0, 0, 0);
      if (MODE == 1) gv[u] = iu < total_vec ? reinterpret_cast<const uint4*>(da)[iu] : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i + u * stride >= total_vec) break;
      float f[8];
      unpack8(zv[u], f);
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s0[j] += f[j];
          s1[j] = fmaf(f[j], f[j], s1[j]);
        }
      } else {
        float g[8];
        unpack8(gv[u], g);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float zh = (f[j] - mu[j]) * is[j];
          const float bn = fmaf(ga[j], zh, be[j]);
          const float d = bn > 0.f ? g[j] : g[j] * slope;
          s0[j] += d;
          s1[j] = fmaf(d, zh, s1[j]);
        }
      }
    }
  }
  // block reduction without shared-memory float atomics (a CAS loop under 32-way same-address
  // contention was most of this kernel's time): every thread parks its 16 partial sums, then one
  // thread per output adds the 256 / vec_per_pix threads that share its channel lane.
  extern __shared__ float sh[];  // [16][256]
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sh[j * 256 + threadIdx.x] = s0[j];
    sh[(8 + j) * 256 + threadIdx.x] = s1[j];
  }
  __syncthreads();
  for (int k = threadIdx.x; k < 2 * c; k += blockDim.x) {
    const int which = k / c, ch = k - which * c;
    const int ln = ch >> 3, j = (ch & 7) + 8 * which;
    float t = 0.f;
    for (int q = ln; q < 256; q += vec_per_pix) t += sh[j * 256 + q];
    part[(size_t)k * gridDim.x + blockIdx.x] = t;
  }
  // deterministic two-level grid reduction (common.cuh)
  const bool fin = det_reduce(part, part + (size_t)2 * c * gridDim.x, counter, gridDim.x, 2 * c, [&](int k, float t) {
    sums[k] = t;
    // MODE 1: sums[0..c) = sum dbn = d(beta), sums[c..2c) = sum dbn * zhat = d(gamma): accumulated here instead of
    // two extra launches per layer
    if (MODE == 1) {
      if (k < c) {
        if (dbeta) dbeta[k] += t;
      } else if (dgamma) {
        dgamma[k - c] += t;
      }
    }
  });
  if (MODE == 0 && fin && fin_mean_invstd) {
    // the block that produced the totals also turns them into mean / invstd and the running statistics
    // (bn_finalize_channel, as in the other finalize kernels): one launch less per BatchNorm layer
    __syncthreads();
    for (int ch = threadIdx.x; ch < c; ch += blockDim.x)
      bn_finalize_channel(sums, fin_mean_invstd, running_mean, running_var, npix, c, momentum, eps, ch);
  }
}

__global__ void bn_finalize_multi_kernel(const b200_bn_finalize_entry* __restrict__ table) {
  pdl_trigger();
  pdl_wait();
  const b200_bn_finalize_entry e = table[blockIdx.y];
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= e.c) return;
  bn_finalize_channel(e.stats, e.mean_invstd, e.running_mean, e.running_var, e.npix, e.c, e.momentum, e.eps, ch);
}

// BatchNorm statistics from the per-tile partial sums the conv epilogue wrote (conv_igemm EPI = 3; output-major
// part[(which * c + ch) * rows + r]): one warp per channel adds the rows in a fixed order (lane-strided, then a
// butterfly), so the result is deterministic, then finishes the channel with bn_finalize_channel.
__global__ void __launch_bounds__(256) bn_partials_finalize_kernel(const float* __restrict__ part, int rows,
                                                                   float* __restrict__ stats,
                                                                   float* __restrict__ mean_invstd,
                                                                   float* __restrict__ running_mean,
                                                                   float* __restrict__ running_var, long long npix, int c,
                                                                   float momentum, float eps) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31, ch = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (ch >= c) return;
  float s0 = 0.f, s1 = 0.f;
  const float* p0 = part + (size_t)ch * rows;
  const float* p1 = part + (size_t)(c + ch) * rows;
  for (int i = lane; i < rows; i += 32) {
    s0 += p0[i];
    s1 += p1[i];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
  }
  if (lane == 0) {
    stats[ch] = s0;
    stats[c + ch] = s1;
    bn_finalize_channel(stats, mean_invstd, running_mean, running_var, npix, c, momentum, eps, ch);
  }
}

template <int MODE>  // 0: fwd apply+lrelu ; 1: bwd apply (dz)
__global__ void bn_apply_kernel(const __nv_bfloat16* __restrict__ z,
                                const __nv_bfloat16* __restrict__ da,
                                const float* __restrict__ mean_invstd,
                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                const float* __restrict__ sums, __nv_bfloat16* __restrict__ out,
                                long long npix, int c, float slope, int use_batch_stats) {
  pdl_trigger();
  pdl_wait();
  const int vec_per_pix = c / 8;
  const long long total_vec = npix * vec_per_pix;
  const long long stride = (long long)gridDim.x * blockDim.x;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int cv = (int)(i % vec_per_pix) * 8;
  float mu[8], is[8], ga[8], be[8], m0[8], m1[8];
  // eval mode (running statistics): the normalisation is a fixed per-channel affine map, so the batch-mean terms
  // of the train-mode gradient vanish
  const float inv_n = use_batch_stats ? 1.f / (float)npix : 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    mu[j] = mean_invstd[cv + j];
    is[j] = mean_invstd[c + cv + j];
    ga[j] = gamma[cv + j];
    be[j] = beta[cv + j];
    if (MODE == 1) {
      m0[j] = sums[cv + j] * inv_n;
      m1[j] = sums[c + cv + j] * inv_n;
    }
  }
  constexpr int U = 2;
  for (; i < total_vec; i += U * stride) {
    uint4 zv[U], gv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long iu = i + u * stride;
      zv[u] = iu < total_vec ? reinterpret_cast<const uint4*>(z)[iu] : make_uint4(0, 0, 0, 0);
      if (MODE == 1) gv[u] = iu < total_vec ? reinterpret_cast<const uint4*>(da)[iu] : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long iu = i + u * stride;
      if (iu >= total_vec) break;
      float f[8], o[8];
      unpack8(zv[u], f);
      if (MODE == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float bn = fmaf(ga[j], (f[j] - mu[j]) * is[j], be[j]);
          o[j] = bn > 0.f ? bn : bn * slope;
        }
      } else {
        float g[8];
        unpack8(gv[u], g);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float zh = (f[j] - mu[j]) * is[j];
          const float bn = fmaf(ga[j], zh, be[j]);
          const float d = bn > 0.f ? g[j] : g[j] * slope;
          o[j] = ga[j] * is[j] * (d - m0[j] - zh * m1[j]);
        }
      }
      reinterpret_cast<uint4*>(out)[iu] = pack8(o);
    }
  }
}

__global__ void add_small_kernel(float* __restrict__ dst, const float* __restrict__ src, int n) {
  pdl_trigger();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// ------------------------------------------------------------------ PixelShuffle(2) (block.py:383)
// out[n, 2y+i, 2x+j, c] = act(z[n, y, x, 4c + 2i + j]).  One thread moves 32 input channels (8 output
// channels for each of the 4 sub-pixels): four 16-byte loads, four 16-byte stores.
template <int BWD>
__global__ void pixel_shuffle2_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                      int n, int h, int w, int c, int act, float slope) {
  pdl_trigger();
  pdl_wait();
  const int qn = c / 8;
  const long long total = (long long)n * h * w * qn;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(idx % qn);
    long long r = idx / qn;
    const int x = (int)(r % w);
    r /= w;
    const int y = (int)(r % h);
    const int b = (int)(r / h);
    const long long zoff = ((((long long)b * h + y) * w + x) * 4 * c) + 32 * q;          // [.., 4c] pixel
    float v[32];
    if (BWD == 0) {
#pragma unroll
      for (int u = 0; u < 4; ++u) unpack8(*reinterpret_cast<const uint4*>(src + zoff + 8 * u), v + 8 * u);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long ooff = ((((long long)b * 2 * h + 2 * y + (k >> 1)) * 2 * w + 2 * x + (k & 1)) * c) + 8 * q;
      float o[8];
      if (BWD == 0) {
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {
          const float t = v[cc * 4 + k];
          o[cc] = (act && t < 0.f) ? t * slope : t;
        }
        *reinterpret_cast<uint4*>(dst + ooff) = pack8(o);
      } else {
        unpack8(*reinterpret_cast<const uint4*>(src + ooff), o);
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) v[cc * 4 + k] = o[cc];
      }
    }
    if (BWD == 1) {
#pragma unroll
      for (int u = 0; u < 4; ++u) *reinterpret_cast<uint4*>(dst + zoff + 8 * u) = pack8(v + 8 * u);
    }
  }
}

// ------------------------------------------------------------------ MaxPool 2x2
__global__ void maxpool_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y,
                               int n, int h, int w, int c) {
  pdl_trigger();
  pdl_wait();
  const int ho = h / 2, wo = w / 2, cv = c / 8;
  const long long total = (long long)n * ho * wo * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % cv);
    long long r = i / cv;
    const int xo = (int)(r % wo);
    r /= wo;
    const int yo = (int)(r % ho);
    const int b = (int)(r / ho);
    const uint4* base = reinterpret_cast<const uint4*>(x) +
                        (((long long)b * h + 2 * yo) * w + 2 * xo) * cv + v;
    float a[8], t[8];
    unpack8(base[0], a);
    unpack8(base[cv], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > a[j] ? t[j] : a[j];
    unpack8(base[(long long)w * cv], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > a[j] ? t[j] : a[j];
    unpack8(base[(long long)w * cv + cv], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > a[j] ? t[j] : a[j];
    reinterpret_cast<uint4*>(y)[i] = pack8(a);
  }
}

// dx = dy routed to the first maximum of each window, times ReLU'(x) (x is a post-ReLU tensor)
__global__ void maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ x,
                                   const __nv_bfloat16* __restrict__ dy,
                                   __nv_bfloat16* __restrict__ dx, int n, int h, int w, int c) {
  pdl_trigger();
  pdl_wait();
  const int ho = h / 2, wo = w / 2, cv = c / 8;
  const long long total = (long long)n * ho * wo * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % cv);
    long long r = i / cv;
    const int xo = (int)(r % wo);
    r /= wo;
    const int yo = (int)(r % ho);
    const int b = (int)(r / ho);
    const long long o00 = (((long long)b * h + 2 * yo) * w + 2 * xo) * cv + v;
    const long long offs[4] = {o00, o00 + cv, o00 + (long long)w * cv, o00 + (long long)w * cv + cv};
    float q[4][8], g[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) unpack8(reinterpret_cast<const uint4*>(x)[offs[k]], q[k]);
    unpack8(reinterpret_cast<const uint4*>(dy)[i], g);
    float o[4][8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int arg = 0;
      float best = q[0][j];
#pragma unroll
      for (int k = 1; k < 4; ++k)
        if (q[k][j] > best) {
          best = q[k][j];
          arg = k;
        }
#pragma unroll
      for (int k = 0; k < 4; ++k) o[k][j] = (k == arg && best > 0.f) ? g[j] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) reinterpret_cast<uint4*>(dx)[offs[k]] = pack8(o[k]);
  }
}

__global__ void sumpool_mask_kernel(const __nv_bfloat16* __restrict__ dy,
                                    const __nv_bfloat16* __restrict__ mask,
                                    __nv_bfloat16* __restrict__ dx, int n, int h, int w, int c,
                                    float slope) {
  pdl_trigger();
  pdl_wait();
  // dx: [n,h,w,c]; dy: [n,2h,2w,c]
  const int cv = c / 8;
  const long long total = (long long)n * h * w * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % cv);
    long long r = i / cv;
    const int xo = (int)(r % w);
    r /= w;
    const int yo = (int)(r % h);
    const int b = (int)(r / h);
    const long long o00 = (((long long)b * 2 * h + 2 * yo) * 2 * w + 2 * xo) * cv + v;
    float a[8], t[8];
    unpack8(reinterpret_cast<const uint4*>(dy)[o00], a);
    unpack8(reinterpret_cast<const uint4*>(dy)[o00 + cv], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += t[j];
    unpack8(reinterpret_cast<const uint4*>(dy)[o00 + (long long)2 * w * cv], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += t[j];
    unpack8(reinterpret_cast<const uint4*>(dy)[o00 + (long long)2 * w * cv + cv], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += t[j];
    if (mask) {  // mask_up: the upsampled activation, sampled at (2y, 2x)
      unpack8(reinterpret_cast<const uint4*>(mask)[o00], t);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = t[j] > 0.f ? a[j] : a[j] * slope;
    }
    reinterpret_cast<uint4*>(dx)[i] = pack8(a);
  }
}

__global__ void lrelu_mask_mul_kernel(const __nv_bfloat16* __restrict__ g,
                                      const __nv_bfloat16* __restrict__ y,
                                      __nv_bfloat16* __restrict__ out, long long nvec, float slope) {
  pdl_trigger();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec;
       i += (long long)gridDim.x * blockDim.x) {
    float a[8], t[8];
    unpack8(reinterpret_cast<const uint4*>(g)[i], a);
    unpack8(reinterpret_cast<const uint4*>(y)[i], t);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = t[j] > 0.f ? a[j] : a[j] * slope;
    reinterpret_cast<uint4*>(out)[i] = pack8(a);
  }
}

// ------------------------------------------------------------------ L1 loss (+ gradient)
template <typename T>
__device__ __forceinline__ float ld_as_float(const T* p, long long i);
template <>
__device__ __forceinline__ float ld_as_float<float>(const float* p, long long i) { return p[i]; }
template <>
__device__ __forceinline__ float ld_as_float<__nv_bfloat16>(const __nv_bfloat16* p, long long i) {
  return __bfloat162float(p[i]);
}
__device__ __forceinline__ void st_from_float(float* p, long long i, float v) { p[i] = v; }
__device__ __forceinline__ void st_from_float(__nv_bfloat16* p, long long i, float v) {
  p[i] = __float2bfloat16(v);
}

template <typename T>
__global__ void l1_loss_kernel(const T* __restrict__ a, const T* __restrict__ b,
                               float* __restrict__ loss_out, T* __restrict__ grad_a, long long numel,
                               float scale, float* __restrict__ part, unsigned* __restrict__ counter) {
  pdl_trigger();
  pdl_wait();
  // scale = weight / numel
  float s = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < numel;
       i += (long long)gridDim.x * blockDim.x) {
    const float d = ld_as_float(a, i) - ld_as_float(b, i);
    s += fabsf(d);
    if (grad_a) st_from_float(grad_a, i, d > 0.f ? scale : (d < 0.f ? -scale : 0.f));
  }
  s = warp_sum(s);
  __shared__ float red[32];
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) red[w] = s;
  __syncthreads();
  if (w == 0) {
    s = l < (blockDim.x >> 5) ? red[l] : 0.f;
    s = warp_sum(s);
    if (l == 0) part[blockIdx.x] = s;
  }
  // deterministic two-level grid reduction (common.cuh)
  det_reduce(part, part + gridDim.x, counter, gridDim.x, 1, [&](int, float t) { *loss_out = t * scale; });
}

// ------------------------------------------------------------------ layout conversion
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int n,
                                    int c, int h, int w, int cy, int coff) {
  pdl_trigger();
  pdl_wait();
  const long long hw = (long long)h * w;
  const long long total = (long long)n * hw * c;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(i % c);
    const long long pix = i / c;
    const long long b = pix / hw, p = pix % hw;
    y[pix * cy + coff + ch] = __float2bfloat16(x[(b * c + ch) * hw + p]);
  }
}
__global__ void nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, int n,
                                    int c, int h, int w, int cx, int coff) {
  pdl_trigger();
  pdl_wait();
  const long long total = (long long)n * c * h * w;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long hw = i % ((long long)h * w);
    const long long r = i / ((long long)h * w);
    const int ch = (int)(r % c);
    const long long b = r / c;
    y[i] = __bfloat162float(x[(b * h * w + hw) * cx + coff + ch]);
  }
}
// grid such that (grid*256) % vec_per_pix == 0 so each thread keeps one channel lane
inline int bn_grid(long long npix, int c, int per_thread, int max_blocks = 148 * 8) {
  const int vpp = c / 8;
  long long total = (npix * vpp + per_thread - 1) / per_thread;
  int g = grid_for(total, 256, max_blocks);
  // 256 * g divisible by vpp: vpp is a power of two <= 64 for c in {64,128,256,512}; otherwise fix up
  while ((256LL * g) % vpp != 0) ++g;
  return g;
}

}  // namespace
}  // namespace b200

using namespace b200;
typedef __nv_bfloat16 bf16;

extern "C" {

int b200_bn_stats_finalize(const void* z, float* stats, float* mean_invstd, float* running_mean,
                           float* running_var, int64_t npix, int32_t c, float momentum, float eps,
                           b200_stream_t stream) {
  B200_REQUIRE(mean_invstd != nullptr, "b200_bn_stats_finalize: mean_invstd is required");
  B200_REQUIRE(c % 8 == 0 && c <= 2048 && 256 % (c / 8) == 0,
               "b200_bn_stats_finalize: c/8 must be a power of two <= 256 (c=%d)", c);
  const int grid = bn_grid(npix, c, 4, 148 * 2);   // the last block adds the per-block partials: keep them few
  DetScratch ds;
  if (det_scratch(&ds, (size_t)(grid + det_groups(grid)) * 2 * c, 1 + det_groups(grid))) return 1;
  ::b200::launch_kernel(bn_reduce_kernel<0>, grid, 256, 16 * 256 * sizeof(float), as_stream(stream),
      (const bf16*)z, nullptr, nullptr, nullptr, nullptr, stats, (long long)npix, c, 0.f, ds.part, ds.counters, nullptr, nullptr,
      mean_invstd, running_mean, running_var, momentum, eps);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_bn_finalize_multi(const b200_bn_finalize_entry* table_dev, int32_t count, int32_t c_max,
                           b200_stream_t stream) {
  if (count <= 0) return 0;
  B200_REQUIRE(table_dev && c_max > 0, "b200_bn_finalize_multi: bad arguments");
  ::b200::launch_kernel(bn_finalize_multi_kernel, dim3((c_max + 127) / 128, count), 128, 0, as_stream(stream), table_dev);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_bn_partials_finalize(const float* part, int32_t rows, float* stats, float* mean_invstd,
                              float* running_mean, float* running_var, int64_t npix, int32_t c, float momentum,
                              float eps, b200_stream_t stream) {
  B200_REQUIRE(part && stats && mean_invstd && rows > 0, "b200_bn_partials_finalize: bad arguments");
  ::b200::launch_kernel(bn_partials_finalize_kernel, (c + 7) / 8, 256, 0, as_stream(stream),
      part, (int)rows, stats, mean_invstd, running_mean, running_var, (long long)npix, (int)c, momentum, eps);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_bn_apply_lrelu(const void* z, const float* mean_invstd, const float* gamma,
                        const float* beta, void* a, int64_t npix, int32_t c, float slope,
                        b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0, "b200_bn_apply_lrelu: c must be a multiple of 8");
  ::b200::launch_kernel(bn_apply_kernel<0>, bn_grid(npix, c, 2), 256, 0, as_stream(stream), 
      (const bf16*)z, nullptr, mean_invstd, gamma, beta, nullptr, (bf16*)a, npix, c, slope, 1);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_bn_bwd_reduce(const void* z, const void* da, const float* mean_invstd, const float* gamma,
                       const float* beta, float* sums, float* dgamma, float* dbeta, int64_t npix, int32_t c,
                       float slope, b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0 && c <= 2048 && 256 % (c / 8) == 0, "b200_bn_bwd_reduce: c/8 must be a power of two <= 256 (c=%d)", c);
  const int grid = bn_grid(npix, c, 4, 148 * 2);   // the last block adds the per-block partials: keep them few
  DetScratch ds;
  if (det_scratch(&ds, (size_t)(grid + det_groups(grid)) * 2 * c, 1 + det_groups(grid))) return 1;
  ::b200::launch_kernel(bn_reduce_kernel<1>, grid, 256, 16 * 256 * sizeof(float), as_stream(stream), 
      (const bf16*)z, (const bf16*)da, mean_invstd, gamma, beta, sums, npix, c, slope, ds.part, ds.counters, dgamma, dbeta,
      nullptr, nullptr, nullptr, 0.f, 0.f);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_bn_bwd_apply(const void* z, const void* da, const float* mean_invstd, const float* gamma,
                      const float* beta, const float* sums, void* dz, int64_t npix, int32_t c, float slope,
                      int32_t use_batch_stats, b200_stream_t stream) {
  ::b200::launch_kernel(bn_apply_kernel<1>, bn_grid(npix, c, 2), 256, 0, as_stream(stream), 
      (const bf16*)z, (const bf16*)da, mean_invstd, gamma, beta, sums, (bf16*)dz, npix, c, slope, (int)use_batch_stats);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_maxpool2x2(const void* x, void* y, int32_t n, int32_t h, int32_t w, int32_t c,
                    b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "b200_maxpool2x2: bad shape");
  const long long total = (long long)n * (h / 2) * (w / 2) * (c / 8);
  ::b200::launch_kernel(maxpool_kernel, grid_for(total, 256), 256, 0, as_stream(stream), (const bf16*)x, (bf16*)y, n, h,
                                                                     w, c);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_maxpool2x2_bwd(const void* x, const void* dy, void* dx, int32_t n, int32_t h, int32_t w,
                        int32_t c, b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "b200_maxpool2x2_bwd: bad shape");
  const long long total = (long long)n * (h / 2) * (w / 2) * (c / 8);
  ::b200::launch_kernel(maxpool_bwd_kernel, grid_for(total, 256), 256, 0, as_stream(stream), 
      (const bf16*)x, (const bf16*)dy, (bf16*)dx, n, h, w, c);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_sumpool2x2_mask(const void* dy, const void* mask, void* dx, int32_t n, int32_t h,
                         int32_t w, int32_t c, float slope, b200_stream_t stream) {
  B200_REQUIRE(c % 8 == 0, "b200_sumpool2x2_mask: bad shape");
  const long long total = (long long)n * h * w * (c / 8);
  ::b200::launch_kernel(sumpool_mask_kernel, grid_for(total, 256), 256, 0, as_stream(stream), 
      (const bf16*)dy, (const bf16*)mask, (bf16*)dx, n, h, w, c, slope);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_pixel_shuffle2(const void* z, void* out, int32_t n, int32_t h, int32_t w, int32_t c, int32_t act,
                        float slope, b200_stream_t stream) {
  B200_REQUIRE(z && out && c % 8 == 0, "b200_pixel_shuffle2: c (output channels) must be a multiple of 8");
  const long long total = (long long)n * h * w * (c / 8);
  ::b200::launch_kernel(pixel_shuffle2_kernel<0>, grid_for(total, 256), 256, 0, as_stream(stream),
                        (const bf16*)z, (bf16*)out, n, h, w, c, act, slope);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_pixel_unshuffle2(const void* dout, void* dz, int32_t n, int32_t h, int32_t w, int32_t c,
                          b200_stream_t stream) {
  B200_REQUIRE(dout && dz && c % 8 == 0, "b200_pixel_unshuffle2: c (output channels) must be a multiple of 8");
  const long long total = (long long)n * h * w * (c / 8);
  ::b200::launch_kernel(pixel_shuffle2_kernel<1>, grid_for(total, 256), 256, 0, as_stream(stream),
                        (const bf16*)dout, (bf16*)dz, n, h, w, c, 0, 0.f);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_l1_loss_f32(const float* a, const float* b, float* loss_out, float* grad_a, int64_t numel,
                     float weight, b200_stream_t stream) {
  const int grid = grid_for(numel, 256, 148 * 4);
  DetScratch ds;
  if (det_scratch(&ds, (size_t)grid + det_groups(grid), 1 + det_groups(grid))) return 1;
  ::b200::launch_kernel(l1_loss_kernel<float>, grid, 256, 0, as_stream(stream), 
      a, b, loss_out, grad_a, numel, weight / (float)numel, ds.part, ds.counters);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_l1_loss_bf16(const void* a, const void* b, float* loss_out, void* grad_a, int64_t numel,
                      float weight, b200_stream_t stream) {
  const int grid = grid_for(numel, 256, 148 * 4);
  DetScratch ds;
  if (det_scratch(&ds, (size_t)grid + det_groups(grid), 1 + det_groups(grid))) return 1;
  ::b200::launch_kernel(l1_loss_kernel<bf16>, grid, 256, 0, as_stream(stream), 
      (const bf16*)a, (const bf16*)b, loss_out, (bf16*)grad_a, numel, weight / (float)numel, ds.part, ds.counters);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_lrelu_mask_mul(const void* g, const void* y, void* out, int64_t numel, float slope,
                        b200_stream_t stream) {
  B200_REQUIRE(numel % 8 == 0, "b200_lrelu_mask_mul: numel must be a multiple of 8");
  ::b200::launch_kernel(lrelu_mask_mul_kernel, grid_for(numel / 8, 256), 256, 0, as_stream(stream), 
      (const bf16*)g, (const bf16*)y, (bf16*)out, numel / 8, slope);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_nchw_f32_to_nhwc_bf16(const float* x, void* y, int32_t n, int32_t c, int32_t h, int32_t w,
                               int32_t cy, int32_t y_coff, b200_stream_t stream) {
  ::b200::launch_kernel(nchw_to_nhwc_kernel, grid_for((long long)n * h * w * c, 256), 256, 0, as_stream(stream), 
      x, (bf16*)y, n, c, h, w, cy, y_coff);
  B200_LAUNCH_CHECK();
  return 0;
}

int b200_nhwc_bf16_to_nchw_f32(const void* x, float* y, int32_t n, int32_t c, int32_t h, int32_t w,
                               int32_t cx, int32_t x_coff, b200_stream_t stream) {
  ::b200::launch_kernel(nhwc_to_nchw_kernel, grid_for((long long)n * c * h * w, 256), 256, 0, as_stream(stream), 
      (const bf16*)x, y, n, c, h, w, cx, x_coff);
  B200_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
