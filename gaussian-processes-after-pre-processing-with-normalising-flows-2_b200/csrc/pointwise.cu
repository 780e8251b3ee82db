// Fused pointwise layers of the Flow++ conditioner for the TRAINING path (forward + backward each in one pass):
//   concat_elu(x) = elu(cat(x, -x))                 flow_modules/mixlogcdf_nn.py:8-10
//   glu(x)        = x[:, :C] * sigmoid(x[:, C:])    flow_modules/mixlogcdf_nn.py:149-151,257-258
// Tensors are viewed as [outer, channels, inner]: inner = H*W for the NCHW convolutional branch (split along dim 1),
// inner = 1 for the NHWC attention branch (split along the last dim).  HBM-bound: 12 B / 12 B per input element.
#include <cuda_fp16.h>
#include "common.cuh"

namespace flowk {

__device__ __forceinline__ float elu_f(float x) { return x > 0.f ? x : expm1f(x); }
__device__ __forceinline__ float elu_grad(float x) { return x > 0.f ? 1.f : expf(x); }

// Index type I: unsigned when the tensor has < 2^31 elements (one 32-bit division per VEC elements instead of a 64-bit
// one per element - the division, not the memory system, bounded the first version); VEC = 4 when C*inner % 4 == 0.
// `mask` (nullable, [outer, 2C]): feature dropout applied to the OUTPUT channels (nn.Dropout2d right after concat_elu in
// GatedConv, mixlogcdf_nn.py:251-256): y[o, c', :] *= mask[o, c'].  With VEC = 4 the host guarantees inner % 4 == 0.
template <typename I, int VEC>
__global__ void concat_elu_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, const float* __restrict__ mask,
                                      unsigned long long inner, I total_v, I per_v) {
  const I inner_i = (I)inner, C = (I)(per_v * VEC / inner_i);
  for (I i = blockIdx.x * (I)blockDim.x + threadIdx.x; i < total_v; i += (I)gridDim.x * blockDim.x) {
    const I o = i / per_v, r = i - o * per_v;
    const size_t src = (size_t)i * VEC, dst = ((size_t)o * 2 * per_v + r) * VEC, half = (size_t)per_v * VEC;
    float m1 = 1.f, m2 = 1.f;
    if (mask) {
      const I c = (r * VEC) / inner_i;
      m1 = mask[(size_t)o * 2 * C + c];
      m2 = mask[(size_t)o * 2 * C + C + c];
    }
    if (VEC == 4) {
      const float4 v = *reinterpret_cast<const float4*>(x + src);
      *reinterpret_cast<float4*>(y + dst) = make_float4(m1 * elu_f(v.x), m1 * elu_f(v.y), m1 * elu_f(v.z), m1 * elu_f(v.w));
      *reinterpret_cast<float4*>(y + dst + half) =
          make_float4(m2 * elu_f(-v.x), m2 * elu_f(-v.y), m2 * elu_f(-v.z), m2 * elu_f(-v.w));
    } else {
      const float v = x[src];
      y[dst] = m1 * elu_f(v);
      y[dst + half] = m2 * elu_f(-v);
    }
  }
}
template <typename I, int VEC>
__global__ void concat_elu_bwd_kernel(const float* __restrict__ x, const float* __restrict__ gy, float* __restrict__ gx,
                                      const float* __restrict__ mask, unsigned long long inner, I total_v, I per_v) {
  const I inner_i = (I)inner, C = (I)(per_v * VEC / inner_i);
  for (I i = blockIdx.x * (I)blockDim.x + threadIdx.x; i < total_v; i += (I)gridDim.x * blockDim.x) {
    const I o = i / per_v, r = i - o * per_v;
    const size_t src = (size_t)i * VEC, dst = ((size_t)o * 2 * per_v + r) * VEC, half = (size_t)per_v * VEC;
    float m1 = 1.f, m2 = 1.f;
    if (mask) {
      const I c = (r * VEC) / inner_i;
      m1 = mask[(size_t)o * 2 * C + c];
      m2 = mask[(size_t)o * 2 * C + C + c];
    }
    if (VEC == 4) {
      const float4 v = *reinterpret_cast<const float4*>(x + src);
      const float4 g1 = *reinterpret_cast<const float4*>(gy + dst), g2 = *reinterpret_cast<const float4*>(gy + dst + half);
      *reinterpret_cast<float4*>(gx + src) =
          make_float4(m1 * g1.x * elu_grad(v.x) - m2 * g2.x * elu_grad(-v.x), m1 * g1.y * elu_grad(v.y) - m2 * g2.y * elu_grad(-v.y),
                      m1 * g1.z * elu_grad(v.z) - m2 * g2.z * elu_grad(-v.z), m1 * g1.w * elu_grad(v.w) - m2 * g2.w * elu_grad(-v.w));
    } else {
      const float v = x[src];
      gx[src] = m1 * gy[dst] * elu_grad(v) - m2 * gy[dst + half] * elu_grad(-v);
    }
  }
}
__device__ __forceinline__ float sigmoid_f(float b) { return 1.f / (1.f + expf(-b)); }
template <typename I, int VEC>
__global__ void glu_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, I total_v, I per_v) {
  for (I i = blockIdx.x * (I)blockDim.x + threadIdx.x; i < total_v; i += (I)gridDim.x * blockDim.x) {
    const I o = i / per_v, r = i - o * per_v;
    const size_t dst = (size_t)i * VEC, src = ((size_t)o * 2 * per_v + r) * VEC, half = (size_t)per_v * VEC;
    if (VEC == 4) {
      const float4 a = *reinterpret_cast<const float4*>(x + src), b = *reinterpret_cast<const float4*>(x + src + half);
      *reinterpret_cast<float4*>(y + dst) =
          make_float4(a.x * sigmoid_f(b.x), a.y * sigmoid_f(b.y), a.z * sigmoid_f(b.z), a.w * sigmoid_f(b.w));
    } else {
      y[dst] = x[src] * sigmoid_f(x[src + half]);
    }
  }
}
template <typename I, int VEC>
__global__ void glu_bwd_kernel(const float* __restrict__ x, const float* __restrict__ gy, float* __restrict__ gx, I total_v,
                               I per_v) {
  for (I i = blockIdx.x * (I)blockDim.x + threadIdx.x; i < total_v; i += (I)gridDim.x * blockDim.x) {
    const I o = i / per_v, r = i - o * per_v;
    const size_t dst = (size_t)i * VEC, src = ((size_t)o * 2 * per_v + r) * VEC, half = (size_t)per_v * VEC;
    if (VEC == 4) {
      const float4 a = *reinterpret_cast<const float4*>(x + src), b = *reinterpret_cast<const float4*>(x + src + half);
      const float4 g = *reinterpret_cast<const float4*>(gy + dst);
      const float s0 = sigmoid_f(b.x), s1 = sigmoid_f(b.y), s2 = sigmoid_f(b.z), s3 = sigmoid_f(b.w);
      *reinterpret_cast<float4*>(gx + src) = make_float4(g.x * s0, g.y * s1, g.z * s2, g.w * s3);
      *reinterpret_cast<float4*>(gx + src + half) =
          make_float4(g.x * a.x * s0 * (1.f - s0), g.y * a.y * s1 * (1.f - s1), g.z * a.z * s2 * (1.f - s2),
                      g.w * a.w * s3 * (1.f - s3));
    } else {
      const float a = x[src], g = gy[dst], sg = sigmoid_f(x[src + half]);
      gx[src] = g * sg;
      gx[src + half] = g * a * sg * (1.f - sg);
    }
  }
}

static int grid_for(long long total) {
  long long b = (total + 255) / 256;
  return (int)(b < 148 * 16 ? b : 148 * 16);
}

}  // namespace flowk

using namespace flowk;

// picks (index type, vector width) and launches KERNEL<I, VEC>(args..., total / VEC, C * inner / VEC)
#define FLOWK_POINTWISE_ENTRY(KERNEL, ALIGNED, ...)                                                                     \
  if (outer < 0 || C < 1 || inner < 1) return FLOWK_ERR_SHAPE;                                                          \
  if (outer == 0) return FLOWK_OK;                                                                                      \
  {                                                                                                                     \
    const long long per = (long long)C * inner, total = outer * per;                                                    \
    const bool v4 = (per % 4 == 0) && (ALIGNED);                                                                        \
    const long long tv = v4 ? total / 4 : total, pv = v4 ? per / 4 : per;                                               \
    const int grid = grid_for(tv);                                                                                      \
    if (2 * total < 0x7fffffffLL) {                                                                                     \
      if (v4) KERNEL<unsigned, 4><<<grid, 256, 0, stream>>>(__VA_ARGS__, (unsigned)tv, (unsigned)pv);                   \
      else KERNEL<unsigned, 1><<<grid, 256, 0, stream>>>(__VA_ARGS__, (unsigned)tv, (unsigned)pv);                      \
    } else {                                                                                                            \
      if (v4) KERNEL<unsigned long long, 4><<<grid, 256, 0, stream>>>(__VA_ARGS__, (unsigned long long)tv,              \
                                                                      (unsigned long long)pv);                         \
      else KERNEL<unsigned long long, 1><<<grid, 256, 0, stream>>>(__VA_ARGS__, (unsigned long long)tv,                 \
                                                                   (unsigned long long)pv);                            \
    }                                                                                                                   \
  }                                                                                                                     \
  return launch_status();

extern "C" int flowk_concat_elu_fwd(const float* x, float* y, const float* mask, long long outer, int C, long long inner,
                                    flowk_stream_t stream) {
  if (outer > 0 && (!x || !y)) return FLOWK_ERR_ARG;
  FLOWK_POINTWISE_ENTRY(concat_elu_fwd_kernel, aligned16(x) && aligned16(y) && (!mask || inner % 4 == 0), x, y, mask,
                        (unsigned long long)inner)
}
extern "C" int flowk_concat_elu_bwd(const float* x, const float* gy, float* gx, const float* mask, long long outer, int C,
                                    long long inner, flowk_stream_t stream) {
  if (outer > 0 && (!x || !gy || !gx)) return FLOWK_ERR_ARG;
  FLOWK_POINTWISE_ENTRY(concat_elu_bwd_kernel, aligned16(x) && aligned16(gy) && aligned16(gx) && (!mask || inner % 4 == 0), x,
                        gy, gx, mask, (unsigned long long)inner)
}
extern "C" int flowk_glu_fwd(const float* x, float* y, long long outer, int C, long long inner, flowk_stream_t stream) {
  if (outer > 0 && (!x || !y)) return FLOWK_ERR_ARG;
  FLOWK_POINTWISE_ENTRY(glu_fwd_kernel, aligned16(x) && aligned16(y), x, y)
}
extern "C" int flowk_glu_bwd(const float* x, const float* gy, float* gx, long long outer, int C, long long inner,
                             flowk_stream_t stream) {
  if (outer > 0 && (!x || !gy || !gx)) return FLOWK_ERR_ARG;
  FLOWK_POINTWISE_ENTRY(glu_bwd_kernel, aligned16(x) && aligned16(gy) && aligned16(gx), x, gy, gx)
}

// ---------------------------------------------------------------------------------------------------------------
// Weight normalisation (old-style weight_g / weight_v, mixlogcdf_nn.py:19-21 `weight_norm(nn.Conv2d)`) fused with the
// construction of the tcgen05 GEMM weight operands.  v: [N, cin, taps] (torch conv / linear weight layout).
//   norm[n] = ||v[n]||,  s[n] = g[n] / norm[n],  w = v * s
//   forward operand  [N, taps, cin_pad]  (K-major rows of W),            hi/lo TF32 split
//   dgrad operand    [cin, taps, n_pad]  = w[n, ci, taps-1-t] (taps flipped, transposed), hi/lo TF32 split
// Two launches per layer instead of ~10 torch kernels; the backward is one kernel:
//   dot = sum(gw * v);  gg = dot / norm;  gv = gw * s - v * (dot * g / norm^3)
namespace flowk {

__device__ __forceinline__ void split_tf32_rna(float x, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
  lo = __uint_as_float((__float_as_uint(x - hi) + 0x1000u) & 0xffffe000u);
}

__global__ void wn_norm_kernel(const float* __restrict__ v, float* __restrict__ norm, int rows, int cols) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* p = v + (size_t)row * cols;
  float s = 0.f;
  for (int i = threadIdx.x & 31; i < cols; i += 32) s = fmaf(p[i], p[i], s);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) norm[row] = sqrtf(s);
}

__global__ void wn_operands_kernel(const float* __restrict__ v, const float* __restrict__ g, const float* __restrict__ norm,
                                   int N, int cin, int taps, int cin_pad, int n_pad, float* __restrict__ w,
                                   float* __restrict__ fwd_hi, float* __restrict__ fwd_lo, float* __restrict__ dg_hi,
                                   float* __restrict__ dg_lo) {
  const long long stride = (long long)gridDim.x * blockDim.x, t0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (w) {
    const long long total = (long long)N * cin * taps, per = (long long)cin * taps;
    for (long long i = t0; i < total; i += stride) {
      const int n = (int)(i / per);
      w[i] = v[i] * (g[n] / norm[n]);
    }
  }
  if (fwd_hi) {
    const long long total = (long long)N * taps * cin_pad;
    for (long long i = t0; i < total; i += stride) {
      const int c = (int)(i % cin_pad);
      const int t = (int)((i / cin_pad) % taps);
      const int n = (int)(i / ((long long)cin_pad * taps));
      float val = 0.f;
      if (c < cin) val = v[((size_t)n * cin + c) * taps + t] * (g[n] / norm[n]);
      float hi, lo;
      split_tf32_rna(val, hi, lo);
      fwd_hi[i] = hi;
      fwd_lo[i] = lo;
    }
  }
  if (dg_hi) {
    const long long total = (long long)cin * taps * n_pad;
    for (long long i = t0; i < total; i += stride) {
      const int n = (int)(i % n_pad);
      const int t = (int)((i / n_pad) % taps);
      const int c = (int)(i / ((long long)n_pad * taps));
      float val = 0.f;
      if (n < N) val = v[((size_t)n * cin + c) * taps + (taps - 1 - t)] * (g[n] / norm[n]);
      float hi, lo;
      split_tf32_rna(val, hi, lo);
      dg_hi[i] = hi;
      dg_lo[i] = lo;
    }
  }
}

__global__ void wn_bwd_kernel(const float* __restrict__ v, const float* __restrict__ g, const float* __restrict__ norm,
                              const float* __restrict__ gw, float* __restrict__ gv, float* __restrict__ gg, int cols) {
  __shared__ float part[4];
  const int row = blockIdx.x;
  const float* pv = v + (size_t)row * cols;
  const float* pg = gw + (size_t)row * cols;
  float d = 0.f;
  for (int i = threadIdx.x; i < cols; i += 128) d = fmaf(pg[i], pv[i], d);
  d = warp_sum(d);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = d;
  __syncthreads();
  const float dot = (part[0] + part[1]) + (part[2] + part[3]);
  const float nr = norm[row], gr = g[row];
  const float s = gr / nr, k = dot * gr / (nr * nr * nr);
  if (threadIdx.x == 0) gg[row] = dot / nr;
  for (int i = threadIdx.x; i < cols; i += 128) gv[(size_t)row * cols + i] = pg[i] * s - pv[i] * k;
}

// Same, with gw given as the split-K partial sums of flowk_conv_wgrad: partial[s][t][n][c] (or [s][t][c][n] when
// transposed); the slices are added in index order.  The reduced row is staged in shared memory (cols floats).
__global__ void __launch_bounds__(256) wn_bwd_partials_kernel(
    const float* __restrict__ v, const float* __restrict__ g, const float* __restrict__ norm,
    const float* __restrict__ partial, float* __restrict__ gv, float* __restrict__ gg, int N, int cin, int taps, int splits,
    int transposed) {
  extern __shared__ float gw_row[];           // [cols] in (t, c) order
  __shared__ float part[8];
  const int row = blockIdx.x, cols = cin * taps;
  const size_t split_stride = (size_t)taps * N * cin;
  float d = 0.f;
  for (int j = threadIdx.x; j < cols; j += 256) {
    const int t = j / cin, c = j - t * cin;
    const float* q = transposed ? partial + ((size_t)t * cin + c) * N + row : partial + ((size_t)t * N + row) * cin + c;
    float acc = 0.f;
    int s = 0;
    for (; s + 4 <= splits; s += 4) {          // four independent loads in flight, summed in index order
      const float a0 = q[(size_t)s * split_stride], a1 = q[(size_t)(s + 1) * split_stride];
      const float a2 = q[(size_t)(s + 2) * split_stride], a3 = q[(size_t)(s + 3) * split_stride];
      acc = (((acc + a0) + a1) + a2) + a3;
    }
    for (; s < splits; ++s) acc += q[(size_t)s * split_stride];
    gw_row[j] = acc;
    d = fmaf(acc, v[(size_t)row * cols + (size_t)c * taps + t], d);
  }
  d = warp_sum(d);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = d;
  __syncthreads();
  float dot = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) dot += part[k];
  const float nr = norm[row], gr = g[row];
  const float sc = gr / nr, k3 = dot * gr / (nr * nr * nr);
  if (threadIdx.x == 0) gg[row] = dot / nr;
  // second pass in v's own (c, t) order so the gv stores coalesce
  for (int i = threadIdx.x; i < cols; i += 256) {
    const int c = i / taps, t = i - c * taps;
    const size_t at = (size_t)row * cols + i;
    gv[at] = gw_row[t * cin + c] * sc - v[at] * k3;
  }
}

// Transposed partials ([s][t][c][n]: the output channel is the fastest index): one CTA takes R consecutive output channels,
// so every load is a whole 16- / 32-byte run of one sector instead of one float per sector.  Narrow layers (cols <= 128:
// the Linear layers, up to 64 split-K slices) leave most of the 256 threads without a column, so the slices are dealt out
// to SG = 256 / cols thread groups (contiguous ranges, each summed in index order) and the group sums are added in group
// order: a fixed summation tree, bit-reproducible.
template <int R>
__global__ void __launch_bounds__(256) wn_bwd_partials_t_kernel(
    const float* __restrict__ v, const float* __restrict__ g, const float* __restrict__ norm,
    const float* __restrict__ partial, float* __restrict__ gv, float* __restrict__ gg, int N, int cin, int taps, int splits) {
  extern __shared__ float wn_sm[];            // gw_rows [R][cols] in (t, c) order, then psum [SG][R][cols] when SG > 1
  __shared__ float part[8][R];
  const int row0 = blockIdx.x * R, cols = cin * taps;
  const int jt = cols >= 256 ? 256 : (cols + 31) / 32 * 32;      // column lanes
  const int sgs = 256 / jt;                                      // split groups
  const int jl = threadIdx.x % jt, sg = threadIdx.x / jt;
  const int chunk = (splits + sgs - 1) / sgs;
  float* gw_rows = wn_sm;
  float* psum = wn_sm + R * cols;
  const size_t split_stride = (size_t)taps * N * cin;
  float d[R];
#pragma unroll
  for (int r = 0; r < R; ++r) d[r] = 0.f;
  for (int j0 = 0; j0 < cols; j0 += jt) {
    const int j = j0 + jl;
    const bool live = j < cols && sg < sgs;
    const int t = live ? j / cin : 0, c = live ? j - t * cin : 0;
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.f;
    if (live) {
      const float4* q = reinterpret_cast<const float4*>(partial + ((size_t)t * cin + c) * N + row0);
      int s = sg * chunk;
      const int s_end = s + chunk < splits ? s + chunk : splits;
      for (; s + 8 <= s_end; s += 8) {         // eight slices' loads in flight (L2-latency-bound), added in index order
        float4 a[8][R / 4];
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
          for (int h = 0; h < R / 4; ++h) a[u][h] = __ldg(q + ((size_t)(s + u) * split_stride) / 4 + h);
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
          for (int h = 0; h < R / 4; ++h) {
            acc[4 * h] += a[u][h].x;
            acc[4 * h + 1] += a[u][h].y;
            acc[4 * h + 2] += a[u][h].z;
            acc[4 * h + 3] += a[u][h].w;
          }
      }
      for (; s + 4 <= s_end; s += 4) {         // four slices' loads in flight
        float4 a[4][R / 4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int h = 0; h < R / 4; ++h) a[u][h] = __ldg(q + ((size_t)(s + u) * split_stride) / 4 + h);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int h = 0; h < R / 4; ++h) {
            acc[4 * h] += a[u][h].x;
            acc[4 * h + 1] += a[u][h].y;
            acc[4 * h + 2] += a[u][h].z;
            acc[4 * h + 3] += a[u][h].w;
          }
      }
      for (; s < s_end; ++s)
#pragma unroll
        for (int h = 0; h < R / 4; ++h) {
          const float4 a = __ldg(q + ((size_t)s * split_stride) / 4 + h);
          acc[4 * h] += a.x;
          acc[4 * h + 1] += a.y;
          acc[4 * h + 2] += a.z;
          acc[4 * h + 3] += a.w;
        }
    }
    if (sgs > 1) {                             // (then cols <= jt: a single pass of this loop)
      if (live) {
#pragma unroll
        for (int r = 0; r < R; ++r) psum[(sg * R + r) * cols + j] = acc[r];
      }
      __syncthreads();
      if (live && sg == 0) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          float tot = acc[r];
          for (int k = 1; k < sgs; ++k) tot += psum[(k * R + r) * cols + j];
          acc[r] = tot;
        }
      }
    }
    if (live && sg == 0) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        gw_rows[r * cols + j] = acc[r];
        d[r] = fmaf(acc[r], v[(size_t)(row0 + r) * cols + (size_t)c * taps + t], d[r]);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) d[r] = warp_sum(d[r]);
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int r = 0; r < R; ++r) part[threadIdx.x >> 5][r] = d[r];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < R * cols; i += 256) {
    const int r = i / cols, ii = i - r * cols;
    const int c = ii / taps, t = ii - c * taps;
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) dot += part[k][r];
    const float nr = norm[row0 + r], gr = g[row0 + r];
    const float sc = gr / nr, k3 = dot * gr / (nr * nr * nr);
    if (ii == 0) gg[row0 + r] = dot / nr;
    const size_t at = (size_t)(row0 + r) * cols + ii;
    gv[at] = gw_rows[r * cols + t * cin + c] * sc - v[at] * k3;
  }
}

}  // namespace flowk

extern "C" int flowk_weight_norm_bwd_partials(const float* v, const float* g, const float* norm, const float* partial,
                                              float* gv, float* gg, int N, int cin, int taps, int splits,
                                              int transposed, flowk_stream_t stream) {
  if (N < 1 || cin < 1 || taps < 1 || splits < 1) return FLOWK_ERR_SHAPE;
  if (!v || !g || !norm || !partial || !gv || !gg) return FLOWK_ERR_ARG;
  if ((size_t)cin * taps * sizeof(float) > 48 * 1024) return FLOWK_ERR_SHAPE;
  const size_t row_bytes = (size_t)cin * taps * sizeof(float);
  const bool al16 = aligned16(partial) && ((size_t)taps * N * cin) % 4 == 0;
  // shared memory: the R reduced rows, plus one copy per split group when the layer is narrow (cols <= 128)
  const int cols = cin * taps, jt = cols >= 256 ? 256 : (cols + 31) / 32 * 32, sgs = 256 / jt;
  const size_t per_row = row_bytes * (sgs > 1 ? 1 + sgs : 1);
  if (transposed && al16 && N % 8 == 0 && 8 * per_row <= 48 * 1024)
    wn_bwd_partials_t_kernel<8><<<N / 8, 256, 8 * per_row, stream>>>(v, g, norm, partial, gv, gg, N, cin, taps, splits);
  else if (transposed && al16 && N % 4 == 0 && 4 * per_row <= 48 * 1024)
    wn_bwd_partials_t_kernel<4><<<N / 4, 256, 4 * per_row, stream>>>(v, g, norm, partial, gv, gg, N, cin, taps, splits);
  else
    wn_bwd_partials_kernel<<<N, 256, row_bytes, stream>>>(v, g, norm, partial, gv, gg, N, cin, taps, splits, transposed);
  return launch_status();
}

// ---- all layers of a model in two launches: the per-layer kernels above are launch-bound (N*cols is tiny), and a
// training step re-normalises ~500 weight tensors.  jobs: device array, one entry per layer (pointers are stable: the
// optimizer updates parameters in place and the outputs are preallocated by the caller).
namespace flowk {

__global__ void wn_norm_batched_kernel(const flowk_wn_job* __restrict__ jobs) {
  const flowk_wn_job j = jobs[blockIdx.y];
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= j.N) return;
  const int cols = j.cin * j.taps;
  const float* p = j.v + (size_t)row * cols;
  float s = 0.f, mx = 0.f;
  for (int i = threadIdx.x & 31; i < cols; i += 32) {
    s = fmaf(p[i], p[i], s);
    mx = fmaxf(mx, fabsf(p[i]));
  }
  s = warp_sum(s);
  if (j.fwd_f16) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    const float nr = sqrtf(s);
    j.norm[row] = nr;
    if (j.fwd_f16) {                                       // max |w| of the layer -> norm[N] (zeroed by the caller)
      const float top = fabsf(j.g[row] / nr) * mx;
      if (top > 0.f && top <= 3.0e38f) atomicMax(reinterpret_cast<unsigned*>(j.norm + j.N), __float_as_uint(top));
    }
  }
}

__global__ void wn_operands_batched_kernel(const flowk_wn_job* __restrict__ jobs) {
  // 32-bit index math throughout (a weight tensor has far fewer than 2^31 elements)
  const flowk_wn_job j = jobs[blockIdx.y];
  const unsigned stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned N = j.N, cin = j.cin, taps = j.taps, cin_pad = j.cin_pad, n_pad = j.n_pad;
  if (j.w) {
    const unsigned total = N * cin * taps, per = cin * taps;
    for (unsigned i = t0; i < total; i += stride) {
      const unsigned n = i / per;
      j.w[i] = j.v[i] * (j.g[n] / j.norm[n]);
    }
  }
  if (j.fwd_hi && j.fwd_f16) {
    // fp16 (hi, lo) forward operand, pre-scaled by the power of two that puts the layer's max |w| into [2^14, 2^15)
    // (FLOWK_OPERAND_F16, see flowk_pack_weight_f16); 1 / scale goes to norm[N + 1] for flowk_conv_gemm's acc_scale_ptr
    const unsigned bits = reinterpret_cast<const unsigned*>(j.norm)[N];
    int e = 0;
    if (bits != 0u) {
      const int field = (int)((bits >> 23) & 0xffu);
      e = field == 0 ? 24 : 14 - (field - 127);
      e = e < -14 ? -14 : (e > 24 ? 24 : e);
    }
    const float scale = __int_as_float((127 + e) << 23);
    if (t0 == 0) j.norm[N + 1] = __int_as_float((127 - e) << 23);
    unsigned short* hi16 = reinterpret_cast<unsigned short*>(j.fwd_hi);
    unsigned short* lo16 = reinterpret_cast<unsigned short*>(j.fwd_lo);
    const unsigned total = N * taps * cin_pad, row = taps * cin_pad;
    for (unsigned i = t0; i < total; i += stride) {
      const unsigned n = i / row, r = i - n * row;
      const unsigned t = r / cin_pad, c = r - t * cin_pad;
      float val = 0.f;
      if (c < cin) val = (j.v[(n * cin + c) * taps + t] * (j.g[n] / j.norm[n])) * scale;
      unsigned short h, l;
      split_f16(val, h, l);
      hi16[i] = h;
      lo16[i] = l;
    }
  } else if (j.fwd_hi) {
    const unsigned total = N * taps * cin_pad, row = taps * cin_pad;
    for (unsigned i = t0; i < total; i += stride) {
      const unsigned n = i / row, r = i - n * row;
      const unsigned t = r / cin_pad, c = r - t * cin_pad;
      float val = 0.f;
      if (c < cin) val = j.v[(n * cin + c) * taps + t] * (j.g[n] / j.norm[n]);
      float hi, lo;
      split_tf32_rna(val, hi, lo);
      j.fwd_hi[i] = hi;
      j.fwd_lo[i] = lo;
    }
  }
  if (j.dg_hi) {
    const unsigned total = cin * taps * n_pad, row = taps * n_pad;
    for (unsigned i = t0; i < total; i += stride) {
      const unsigned c = i / row, r = i - c * row;
      const unsigned t = r / n_pad, n = r - t * n_pad;
      float val = 0.f;
      if (n < N) val = j.v[(n * cin + c) * taps + (taps - 1 - t)] * (j.g[n] / j.norm[n]);
      float hi, lo;
      split_tf32_rna(val, hi, lo);
      j.dg_hi[i] = hi;
      j.dg_lo[i] = lo;
    }
  }
}

}  // namespace flowk

extern "C" int flowk_weight_norm_operands_batched(const flowk_wn_job* jobs_device, int njobs, int max_rows,
                                                  flowk_stream_t stream) {
  if (njobs < 0 || max_rows < 1) return FLOWK_ERR_SHAPE;
  if (njobs == 0) return FLOWK_OK;
  if (!jobs_device) return FLOWK_ERR_ARG;
  wn_norm_batched_kernel<<<dim3((max_rows + 3) / 4, njobs), 128, 0, stream>>>(jobs_device);
  wn_operands_batched_kernel<<<dim3(96, njobs), 256, 0, stream>>>(jobs_device);
  return launch_status();
}

extern "C" int flowk_weight_norm_operands(const float* v, const float* g, int N, int cin, int taps, int cin_pad, int n_pad,
                                          float* norm, float* w, float* fwd_hi, float* fwd_lo, float* dg_hi, float* dg_lo,
                                          flowk_stream_t stream) {
  if (N < 1 || cin < 1 || taps < 1) return FLOWK_ERR_SHAPE;
  if (!v || !g || !norm || (fwd_hi && !fwd_lo) || (dg_hi && !dg_lo)) return FLOWK_ERR_ARG;
  if ((fwd_hi && cin_pad < cin) || (dg_hi && n_pad < N)) return FLOWK_ERR_SHAPE;
  const int cols = cin * taps;
  wn_norm_kernel<<<(N + 3) / 4, 128, 0, stream>>>(v, norm, N, cols);
  long long most = w ? (long long)N * cols : 0;
  if (fwd_hi && (long long)N * taps * cin_pad > most) most = (long long)N * taps * cin_pad;
  if (dg_hi && (long long)cin * taps * n_pad > most) most = (long long)cin * taps * n_pad;
  if (most > 0)
    wn_operands_kernel<<<grid_for(most), 256, 0, stream>>>(v, g, norm, N, cin, taps, cin_pad, n_pad, w, fwd_hi, fwd_lo,
                                                            dg_hi, dg_lo);
  return launch_status();
}

extern "C" int flowk_weight_norm_bwd(const float* v, const float* g, const float* norm, const float* gw, float* gv, float* gg,
                                     int N, int cols, flowk_stream_t stream) {
  if (N < 1 || cols < 1) return FLOWK_ERR_SHAPE;
  if (!v || !g || !norm || !gw || !gv || !gg) return FLOWK_ERR_ARG;
  wn_bwd_kernel<<<N, 128, 0, stream>>>(v, g, norm, gw, gv, gg, cols);
  return launch_status();
}

// ---------------------------------------------------------------------------------------------------------------
// Residual add + LayerNorm over channels (ConvAttnBlock, mixlogcdf_nn.py:226-234): y = LN_C(a + b) * gamma + beta.
// Rows are pixels m = (b, h, w); either side may be NCHW ([B, C, HW]) or NHWC rows ([M, C]) so the block's two
// permutes cost nothing: the tile of 32 pixels x C channels is transposed through shared memory.
// Forward also stores s = a + b (rows) and mean / rstd for the backward pass.
namespace flowk {

constexpr int kLnPix = 32;
constexpr int kLnThreads = 256;

__device__ __forceinline__ size_t ln_addr(bool nchw, long long m, int c, int C, int HW) {
  if (!nchw) return (size_t)m * C + c;
  const long long b = m / HW;
  return ((size_t)b * C + c) * HW + (size_t)(m - b * HW);
}

// tile[c * 33 + p].  NCHW: a thread keeps its pixel (p = tid & 31) and walks the channels, so the (image, offset)
// split of the pixel index - an integer division - is done once per thread, not once per element.
template <typename F>
__device__ __forceinline__ void ln_tile_io(bool nchw, long long m0, long long M, int C, int HW, F f) {
  if (nchw) {
    const int p = threadIdx.x & 31;
    const long long m = m0 + p;
    if (m < M) {
      const long long b = m / HW;
      const size_t base = (size_t)b * C * HW + (size_t)(m - b * HW);
#pragma unroll 4
      for (int c = threadIdx.x >> 5; c < C; c += kLnThreads / 32) f(c, p, base + (size_t)c * HW);
    }
  } else {
    const unsigned total = (unsigned)C * kLnPix, uc = (unsigned)C;
    const size_t base = (size_t)m0 * C;
    const unsigned limit = (M - m0 >= kLnPix) ? total : (unsigned)(M - m0) * uc;      // rows past M are skipped
#pragma unroll 4
    for (unsigned i = threadIdx.x; i < limit; i += kLnThreads) {
      const unsigned p = i / uc, c = i - p * uc;
      f((int)c, (int)p, base + i);                       // row-major: element i of the tile is at base + i
    }
  }
}

__global__ void __launch_bounds__(kLnThreads) add_layernorm_fwd_kernel(
    const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ gamma, const float* __restrict__ beta,
    float* __restrict__ y, float* __restrict__ s_out, float* __restrict__ mean_out, float* __restrict__ rstd_out,
    long long M, int C, int HW, int in_nchw, int out_nchw, float eps) {
  extern __shared__ float tile[];
  __shared__ float s_mean[kLnPix], s_rstd[kLnPix];
  const long long m0 = (long long)blockIdx.x * kLnPix;
  ln_tile_io(in_nchw, m0, M, C, HW, [&](int c, int p, size_t at) { tile[c * 33 + p] = a[at] + (b ? b[at] : 0.f); });
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int p = warp; p < kLnPix; p += kLnThreads / 32) {
    float sum = 0.f;
    for (int c = lane; c < C; c += 32) sum += tile[c * 33 + p];
    const float mean = warp_sum(sum) / C;
    float var = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float d = tile[c * 33 + p] - mean;
      var = fmaf(d, d, var);
    }
    const float rstd = rsqrtf(warp_sum(var) / C + eps);
    if (lane == 0) {
      s_mean[p] = mean;
      s_rstd[p] = rstd;
      if (m0 + p < M) {
        mean_out[m0 + p] = mean;
        rstd_out[m0 + p] = rstd;
      }
    }
  }
  __syncthreads();
  ln_tile_io(false, m0, M, C, HW, [&](int c, int p, size_t at) { s_out[at] = tile[c * 33 + p]; });
  ln_tile_io(out_nchw, m0, M, C, HW, [&](int c, int p, size_t at) {
    y[at] = (tile[c * 33 + p] - s_mean[p]) * s_rstd[p] * gamma[c] + beta[c];
  });
}

// gs = rstd * (gamma*gy - mean_c(gamma*gy) - xhat * mean_c(gamma*gy*xhat));  partial dgamma/dbeta per CTA
__global__ void __launch_bounds__(kLnThreads) add_layernorm_bwd_kernel(
    const float* __restrict__ gy, const float* __restrict__ s, const float* __restrict__ mean, const float* __restrict__ rstd,
    const float* __restrict__ gamma, float* __restrict__ gs, float* __restrict__ part, long long M, int C, int HW,
    int in_nchw, int out_nchw) {
  extern __shared__ float tile[];
  float* tg = tile;                 // gy
  float* tx = tile + C * 33;        // xhat
  __shared__ float s_m1[kLnPix], s_m2[kLnPix], s_rstd[kLnPix];
  const long long m0 = (long long)blockIdx.x * kLnPix;
  for (int i = threadIdx.x; i < C * 33; i += kLnThreads) tg[i] = tx[i] = 0.f;      // pixels past M contribute zero
  __syncthreads();
  ln_tile_io(out_nchw, m0, M, C, HW, [&](int c, int p, size_t at) { tg[c * 33 + p] = gy[at]; });
  ln_tile_io(false, m0, M, C, HW, [&](int c, int p, size_t at) {
    tx[c * 33 + p] = (s[at] - mean[m0 + p]) * rstd[m0 + p];
  });
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int p = warp; p < kLnPix; p += kLnThreads / 32) {
    float m1 = 0.f, m2 = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float gg = gamma[c] * tg[c * 33 + p];
      m1 += gg;
      m2 = fmaf(gg, tx[c * 33 + p], m2);
    }
    m1 = warp_sum(m1) / C;
    m2 = warp_sum(m2) / C;
    if (lane == 0) {
      s_m1[p] = m1;
      s_m2[p] = m2;
      s_rstd[p] = (m0 + p < M) ? rstd[m0 + p] : 0.f;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += kLnThreads) {
    float dg = 0.f, db = 0.f;
#pragma unroll 8
    for (int p = 0; p < kLnPix; ++p) {
      const float g = tg[c * 33 + p];
      dg = fmaf(g, tx[c * 33 + p], dg);
      db += g;
    }
    part[((size_t)blockIdx.x * 2) * C + c] = dg;
    part[((size_t)blockIdx.x * 2 + 1) * C + c] = db;
  }
  ln_tile_io(in_nchw, m0, M, C, HW, [&](int c, int p, size_t at) {
    gs[at] = s_rstd[p] * (gamma[c] * tg[c * 33 + p] - s_m1[p] - tx[c * 33 + p] * s_m2[p]);
  });
}

// dgamma[c] = sum over CTAs of part[cta][0][c], dbeta likewise; fixed order -> deterministic
__global__ void layernorm_param_grad_kernel(const float* __restrict__ part, float* __restrict__ dgamma,
                                            float* __restrict__ dbeta, int ctas, int C) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), which = blockIdx.y, slice = threadIdx.x >> 5;
  float acc = 0.f;
  if (c < C)
    for (int i = slice; i < ctas; i += 8) acc += part[((size_t)i * 2 + which) * C + c];
  red[slice][threadIdx.x & 31] = acc;
  __syncthreads();
  if (slice == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    (which ? dbeta : dgamma)[c] = t;
  }
}

}  // namespace flowk

extern "C" long long flowk_add_layernorm_workspace_bytes(long long M, int C) {
  return ((M + kLnPix - 1) / kLnPix) * 2 * (long long)C * (long long)sizeof(float);
}

extern "C" int flowk_add_layernorm_fwd(const float* a, const float* b, const float* gamma, const float* beta, float* y,
                                       float* s, float* mean, float* rstd, long long M, int C, int HW, int in_nchw,
                                       int out_nchw, float eps, flowk_stream_t stream) {
  if (M < 0 || C < 1 || C > 512 || HW < 1 || M % HW) return FLOWK_ERR_SHAPE;
  if (M == 0) return FLOWK_OK;
  if (!a || !gamma || !beta || !y || !s || !mean || !rstd) return FLOWK_ERR_ARG;
  const size_t smem = (size_t)C * 33 * sizeof(float);
  static bool attr = false;
  if (!attr) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(add_layernorm_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 512 * 33 * 4));
    FLOWK_CUDA_OK(cudaFuncSetAttribute(add_layernorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 512 * 33 * 4));
    attr = true;
  }
  add_layernorm_fwd_kernel<<<(unsigned)((M + kLnPix - 1) / kLnPix), kLnThreads, smem, stream>>>(
      a, b, gamma, beta, y, s, mean, rstd, M, C, HW, in_nchw, out_nchw, eps);
  return launch_status();
}

extern "C" int flowk_add_layernorm_bwd(const float* gy, const float* s, const float* mean, const float* rstd,
                                       const float* gamma, float* gs, float* dgamma, float* dbeta, void* workspace,
                                       long long M, int C, int HW, int in_nchw, int out_nchw, flowk_stream_t stream) {
  if (M < 1 || C < 1 || C > 512 || HW < 1 || M % HW) return FLOWK_ERR_SHAPE;
  if (!gy || !s || !mean || !rstd || !gamma || !gs || !dgamma || !dbeta || !workspace) return FLOWK_ERR_ARG;
  const size_t smem = (size_t)2 * C * 33 * sizeof(float);
  static bool attr = false;
  if (!attr) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(add_layernorm_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 512 * 33 * 4));
    FLOWK_CUDA_OK(cudaFuncSetAttribute(add_layernorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 512 * 33 * 4));
    attr = true;
  }
  const unsigned ctas = (unsigned)((M + kLnPix - 1) / kLnPix);
  add_layernorm_bwd_kernel<<<ctas, kLnThreads, smem, stream>>>(gy, s, mean, rstd, gamma, gs, (float*)workspace, M, C, HW,
                                                                in_nchw, out_nchw);
  layernorm_param_grad_kernel<<<dim3((C + 31) / 32, 2), 256, 0, stream>>>((const float*)workspace, dgamma, dbeta,
                                                                           (int)ctas, C);
  return launch_status();
}

// ---------------------------------------------------------------------------------------------------------------
// Bias gradient: out[c] = sum over (b, p) of x[b, c, p]  (NCHW, inner = H*W)  or  sum over rows of x[m, c] (inner = 1).
// Stage 1: grid (chunks, C-tiles) of fixed-order partial sums; stage 2 adds the chunks in index order (deterministic).
namespace flowk {

constexpr int kSumChunks = 64;

__global__ void __launch_bounds__(256) channel_sum_nchw_kernel(const float* __restrict__ x, float* __restrict__ part, int B,
                                                              int C, int HW) {
  // one CTA per (channel, chunk of samples); the chunk's B' x HW values are B' contiguous runs of HW floats
  __shared__ float red[8];
  const int c = blockIdx.x, chunk = blockIdx.y, chunks = gridDim.y;
  const int b0 = (int)((long long)B * chunk / chunks), b1 = (int)((long long)B * (chunk + 1) / chunks);
  float acc = 0.f;
  if ((HW & 3) == 0) {
    const int hw4 = HW >> 2, total = (b1 - b0) * hw4;
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int i = threadIdx.x; i < total; i += 256) {
      const int b = b0 + i / hw4, j = i - (i / hw4) * hw4;
      const float4 v = __ldg(reinterpret_cast<const float4*>(x + ((size_t)b * C + c) * HW) + j);
      a4.x += v.x; a4.y += v.y; a4.z += v.z; a4.w += v.w;
    }
    acc = (a4.x + a4.y) + (a4.z + a4.w);
  } else {
    for (int b = b0; b < b1; ++b) {
      const float* p = x + ((size_t)b * C + c) * HW;
      for (int i = threadIdx.x; i < HW; i += 256) acc += p[i];
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k];
    part[(size_t)chunk * C + c] = t;
  }
}

__global__ void channel_sum_rows_kernel(const float* __restrict__ x, float* __restrict__ part, long long M, int C) {
  // CTA = 32 columns x 8 row-slices; chunk of rows per blockIdx.y
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), slice = threadIdx.x >> 5, chunk = blockIdx.y, chunks = gridDim.y;
  const long long m0 = M * chunk / chunks, m1 = M * (chunk + 1) / chunks;
  float acc = 0.f;
  if (c < C)
    for (long long m = m0 + slice; m < m1; m += 8) acc += x[(size_t)m * C + c];
  red[slice][threadIdx.x & 31] = acc;
  __syncthreads();
  if (slice == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    part[(size_t)chunk * C + c] = t;
  }
}

__global__ void channel_sum_final_kernel(const float* __restrict__ part, float* __restrict__ out, int chunks, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float t = 0.f;
  for (int k = 0; k < chunks; ++k) t += part[(size_t)k * C + c];
  out[c] = t;
}

}  // namespace flowk

extern "C" long long flowk_channel_sum_workspace_bytes(int C) { return (long long)kSumChunks * C * (long long)sizeof(float); }

extern "C" int flowk_channel_sum(const float* x, float* out, void* workspace, long long outer, int C, long long inner,
                                 flowk_stream_t stream) {
  if (outer < 1 || C < 1 || inner < 1 || inner > 0x7fffffff || outer > 0x7fffffff) return FLOWK_ERR_SHAPE;
  if (!x || !out || !workspace) return FLOWK_ERR_ARG;
  float* part = (float*)workspace;
  int chunks;
  if (inner > 1) {
    chunks = (int)(outer < kSumChunks ? outer : kSumChunks);
    while (chunks > 1 && (long long)chunks * C > 148 * 6) chunks >>= 1;
    channel_sum_nchw_kernel<<<dim3(C, chunks), 256, 0, stream>>>(x, part, (int)outer, C, (int)inner);
  } else {
    chunks = (int)(outer / 64 < 1 ? 1 : (outer / 64 > kSumChunks ? kSumChunks : outer / 64));
    channel_sum_rows_kernel<<<dim3((C + 31) / 32, chunks), 256, 0, stream>>>(x, part, outer, C);
  }
  channel_sum_final_kernel<<<(C + 127) / 128, 128, 0, stream>>>(part, out, chunks, C);
  return launch_status();
}

// ---------------------------------------------------------------------------------------------------------------
// log N(z; 0, I) per sample, added to the running objective: out[b] = (in ? in[b] : 0) - (sum_i z[b, i]^2 + n log 2 pi) / 2
// (the default prior of FlowNet.encode: GaussianDiag.logp with zero mean / log-std, common_modules.py:223-240, summed into
// the log-det, marscf_main.py:159-164).  One CTA per sample, fixed-order block reduction; z may be a channel slice
// (`sample_stride` floats between samples).
namespace flowk {

__global__ void __launch_bounds__(256) std_normal_logp_kernel(const float* __restrict__ z, long long sample_stride,
                                                              const float* __restrict__ in, float* __restrict__ out,
                                                              long long n) {
  __shared__ float part[8];
  const float* p = z + (size_t)blockIdx.x * sample_stride;
  float s = 0.f;
  if ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
    for (long long i = threadIdx.x; i < (n >> 2); i += 256) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(p) + i);
      s += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    }
  } else {
    for (long long i = threadIdx.x; i < n; i += 256) s = fmaf(p[i], p[i], s);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += part[k];
    out[blockIdx.x] = (in ? in[blockIdx.x] : 0.f) - 0.5f * (tot + (float)n * 1.8378770664093453f);
  }
}

}  // namespace flowk

extern "C" int flowk_std_normal_logp(const float* z, long long sample_stride, const float* in, float* out, int B, long long n,
                                     flowk_stream_t stream) {
  if (B < 0 || n < 1 || sample_stride < n) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!z || !out) return FLOWK_ERR_ARG;
  flowk::std_normal_logp_kernel<<<B, 256, 0, stream>>>(z, sample_stride, in, out, n);
  return flowk::launch_status();
}

// ---------------------------------------------------------------------------------------------------------------
// ConvLSTM cell backward of one time step (the cell of mar_prior/convolutional_rnn/functional.py:30-52, forward in the
// PRE_LSTM epilogue of csrc/tc_gemm.cu).  Rows [M, 4 hid] of gate pre-activations a = gi + hh ([i | f | g | o], hh the
// recomputed hidden-to-hidden term with b_hh), cell states c_{t-1}, c_t [M, hid]; dh = dh_a (+ dh_b), the gradient of h_t
// from the layer above and from step t+1; dc_next = dL/dc_t arriving from step t+1 (already multiplied by f_{t+1}):
//   dc = dh o tanh'(c_t) + dc_next      do = dh tanh(c_t) o'      di = dc g i'      df = dc c_{t-1} f'      dg = dc i tanh'(g)
// -> dgates [M, 4 hid] fp32 and as the TF32 (hi, lo) pair the input-gradient GEMM reads, and dc_prev = dc f (dL/dc_{t-1}).
// Sigmoid' = s(a) s(-a) and tanh' = 4e / (1 + e)^2 with e = exp(-2|x|) keep their relative accuracy in saturated gates.
// One thread per (row, unit): the four gates of a unit are independent of every other unit.  dc_prev may alias dc_next.
namespace flowk {

__device__ __forceinline__ float sigm(float a) { return 1.f / (1.f + expf(-a)); }
__device__ __forceinline__ float dtanh_of(float x) {
  const float e = expf(-2.f * fabsf(x));
  return 4.f * e / ((1.f + e) * (1.f + e));
}
__device__ __forceinline__ void tf32_pair(float v, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
  lo = __uint_as_float((__float_as_uint(v - hi) + 0x1000u) & 0xffffe000u);
}

__global__ void __launch_bounds__(256) lstm_cell_bwd_kernel(const float* __restrict__ gi, const float* __restrict__ hh,
                                                            const float* __restrict__ c_prev, const float* __restrict__ c,
                                                            const float* __restrict__ dh_a, const float* __restrict__ dh_b,
                                                            const float* dc_next, float* __restrict__ dgates,
                                                            float* __restrict__ dg_hi, float* __restrict__ dg_lo,
                                                            float* dc_prev, long long total, int hid) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long m = e / hid;
    const int j = (int)(e - m * hid);
    const size_t g0 = (size_t)m * 4 * hid + j;
    float a[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) a[q] = __ldg(hh + g0 + (size_t)q * hid) + __ldg(gi + g0 + (size_t)q * hid);
    const float ig = sigm(a[0]), fg = sigm(a[1]), gg = tanhf(a[2]), og = sigm(a[3]);
    const float ct = __ldg(c + e), cp = __ldg(c_prev + e);
    const float dh = __ldg(dh_a + e) + (dh_b ? __ldg(dh_b + e) : 0.f);
    const float dc = dh * og * dtanh_of(ct) + (dc_next ? dc_next[e] : 0.f);
    float d[4];
    d[0] = dc * gg * (ig * sigm(-a[0]));
    d[1] = dc * cp * (fg * sigm(-a[1]));
    d[2] = dc * ig * dtanh_of(a[2]);
    d[3] = dh * tanhf(ct) * (og * sigm(-a[3]));
    dc_prev[e] = dc * fg;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const size_t o = g0 + (size_t)q * hid;
      float h, l;
      tf32_pair(d[q], h, l);
      dgates[o] = d[q];
      dg_hi[o] = h;
      dg_lo[o] = l;
    }
  }
}

// fp16 (hi, lo) operand rows [M, C] -> fp32 rows [M, C_out] = hi + lo, columns C..C_out-1 zero (the weight-gradient
// kernels read fp32 containers with whole 32-channel blocks)
__global__ void __launch_bounds__(256) f16_pair_to_f32_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo,
                                                              float* __restrict__ out, long long total, int C, int C_out) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long m = e / C_out;
    const int c = (int)(e - m * C_out);
    out[e] = c < C ? __half2float(hi[(size_t)m * C + c]) + __half2float(lo[(size_t)m * C + c]) : 0.f;
  }
}

}  // namespace flowk

extern "C" int flowk_lstm_cell_bwd(const float* gi, const float* hh, const float* c_prev, const float* c, const float* dh,
                                   const float* dh_rec, const float* dc_next, float* dgates, float* dg_hi, float* dg_lo,
                                   float* dc_prev, long long M, int hid, flowk_stream_t stream) {
  if (M < 0 || hid < 1) return FLOWK_ERR_SHAPE;
  if (M == 0) return FLOWK_OK;
  if (!gi || !hh || !c_prev || !c || !dh || !dgates || !dg_hi || !dg_lo || !dc_prev) return FLOWK_ERR_ARG;
  flowk::lstm_cell_bwd_kernel<<<grid_for(M * hid), 256, 0, stream>>>(gi, hh, c_prev, c, dh, dh_rec, dc_next, dgates, dg_hi,
                                                                      dg_lo, dc_prev, M * hid, hid);
  return flowk::launch_status();
}

extern "C" int flowk_f16_pair_to_f32(const void* hi, const void* lo, float* out, long long M, int C, int C_out,
                                     flowk_stream_t stream) {
  if (M < 0 || C < 1 || C_out < C) return FLOWK_ERR_SHAPE;
  if (M == 0) return FLOWK_OK;
  if (!hi || !lo || !out) return FLOWK_ERR_ARG;
  flowk::f16_pair_to_f32_kernel<<<grid_for(M * C_out), 256, 0, stream>>>(
      reinterpret_cast<const __half*>(hi), reinterpret_cast<const __half*>(lo), out, M * C_out, C, C_out);
  return flowk::launch_status();
}
