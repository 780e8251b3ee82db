// Training-time self-attention core of GatedAttn (flow_modules/mixlogcdf_nn.py:134-147,154-173) with attention-weight
// dropout (:143, `F.dropout(weight, p, training)`), forward and backward, flash-attention style on mma.sync m16n8k8
// TF32 with the 3xTF32 split (fp32 accuracy) - the counterpart of attention.cu's inference kernel:
//     P = softmax_j(q_i k_j / sqrt(d)),   Pd = P * M  (M = 0 or 1/(1-p)),   O = Pd V
//     dV = Pd^T dO;  dPd = dO V^T;  delta_i = dO_i . O_i;  dS = P * (dPd * M - delta_i);  dQ = dS K / sqrt(d);  dK = dS^T q'
// Nothing of size seq x seq touches HBM: the forward stores the row log-sum-exp, the backward recomputes S = q' K^T
// and regenerates the dropout mask from a counter-based hash of (seed, image*head, query, key).  Two backward kernels,
// no atomics: one owns 16 queries per warp (dQ), one owns 16 keys per warp (dK, dV) -> deterministic; they share no
// intermediate (each computes delta itself), so they may run concurrently on two streams.
// Rows of qkv [M, 3C] are (k | v | q) (:136-139); dqkv has the same layout.
#include "common.cuh"
#include "attention_dropout.cuh"

namespace flowk {
namespace attn_train {

__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void split_bits(float x, uint32_t& hi, uint32_t& lo) {   // round-to-nearest TF32 split
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = (__float_as_uint(x - __uint_as_float(hi)) + 0x1000u) & 0xffffe000u;
}
// D += A B with A = (ah, al), B = (bh, bl) split operands: three TF32 passes
__device__ __forceinline__ void mma3(float (&c)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4], uint32_t bh0,
                                     uint32_t bh1, uint32_t bl0, uint32_t bl1) {
  mma_tf32(c, ah, bh0, bh1);
  mma_tf32(c, al, bh0, bh1);
  mma_tf32(c, ah, bl0, bl1);
}

// stage `tile_rows` rows of D floats (row j at src + j*row_stride, rows >= `rows` are zero) as (hi, lo), pitch D + 4
template <int D>
__device__ __forceinline__ void stage_rows(uint32_t* hi, uint32_t* lo, const float* __restrict__ src, size_t row_stride,
                                           int rows, int tile_rows, float scale) {
  constexpr int V4 = D / 4, P = D + 4;
  for (int i = threadIdx.x; i < tile_rows * V4; i += blockDim.x) {
    const int j = i / V4, v4 = i - j * V4;
    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < rows) val = __ldg(reinterpret_cast<const float4*>(src + (size_t)j * row_stride) + v4);
    uint4 h, l;
    split_bits(val.x * scale, h.x, l.x); split_bits(val.y * scale, h.y, l.y);
    split_bits(val.z * scale, h.z, l.z); split_bits(val.w * scale, h.w, l.w);
    *reinterpret_cast<uint4*>(hi + (size_t)j * P + v4 * 4) = h;
    *reinterpret_cast<uint4*>(lo + (size_t)j * P + v4 * 4) = l;
  }
}

// A-operand fragments (rows g / g+8 of a 16-row block, all D columns) of a row-major matrix, split once
template <int D>
__device__ __forceinline__ void load_a_frags(uint32_t (&fh)[D / 8][4], uint32_t (&fl)[D / 8][4], const float* __restrict__ row_lo,
                                             const float* __restrict__ row_hi, bool ok_lo, bool ok_hi, int t, float scale) {
#pragma unroll
  for (int ks = 0; ks < D / 8; ++ks) {
    const float v0 = ok_lo ? __ldg(row_lo + ks * 8 + t) * scale : 0.f, v1 = ok_hi ? __ldg(row_hi + ks * 8 + t) * scale : 0.f;
    const float v2 = ok_lo ? __ldg(row_lo + ks * 8 + t + 4) * scale : 0.f, v3 = ok_hi ? __ldg(row_hi + ks * 8 + t + 4) * scale : 0.f;
    split_bits(v0, fh[ks][0], fl[ks][0]); split_bits(v1, fh[ks][1], fl[ks][1]);
    split_bits(v2, fh[ks][2], fl[ks][2]); split_bits(v3, fh[ks][3], fl[ks][3]);
  }
}

constexpr int kTile = 128;      // rows of the streamed operand staged per iteration

// ---------------------------------------------------------------------------------------------------------------
// forward: O = dropout(softmax(q' K^T)) V, lse = row log-sum-exp.  grid (pairs, ceil(S / (16*warps))), a warp = 16 queries
// ---------------------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) fwd_kernel(const float* __restrict__ qkv, float* __restrict__ out, float* __restrict__ lse,
                                                  const unsigned* __restrict__ seed_dev, unsigned salt, uint32_t thresh,
                                                  float inv_keep, int S, int C, int heads, float scale) {
  extern __shared__ __align__(16) uint32_t smem_u[];
  constexpr int P = D + 4, KS = D / 8;
  uint32_t* Kh = smem_u;
  uint32_t* Kl = Kh + kTile * P;
  uint32_t* Vh = Kl + kTile * P;
  uint32_t* Vl = Vh + kTile * P;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int pair = blockIdx.x, b = pair / heads, h = pair - b * heads;
  const int q0 = (blockIdx.y * (blockDim.x >> 5) + warp) * 16;
  const int row_stride = 3 * C;
  const uint32_t seed = layer_seed(seed_dev, salt);
  const bool ok_lo = q0 + g < S, ok_hi = q0 + g + 8 < S;
  const float* base = qkv + (size_t)b * S * row_stride + h * D;
  uint32_t qh[KS][4], ql[KS][4];
  load_a_frags<D>(qh, ql, base + (size_t)(ok_lo ? q0 + g : 0) * row_stride + 2 * C,
                  base + (size_t)(ok_hi ? q0 + g + 8 : 0) * row_stride + 2 * C, ok_lo, ok_hi, t, scale);
  float o[KS][4];
#pragma unroll
  for (int nb = 0; nb < KS; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
  float mx_lo = -INFINITY, mx_hi = -INFINITY, l_lo = 0.f, l_hi = 0.f;
  for (int kt0 = 0; kt0 < S; kt0 += kTile) {
    const int keys_here = S - kt0 < kTile ? S - kt0 : kTile;
    __syncthreads();
    stage_rows<D>(Kh, Kl, base + (size_t)kt0 * row_stride, row_stride, keys_here, keys_here, 1.f);
    stage_rows<D>(Vh, Vl, base + (size_t)kt0 * row_stride + C, row_stride, keys_here, keys_here, 1.f);
    __syncthreads();
    for (int k0 = 0; k0 < keys_here; k0 += 8) {
      float sc[4] = {0.f, 0.f, 0.f, 0.f};
      const size_t ko = (size_t)(k0 + g) * P + t;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks)
        mma3(sc, qh[ks], ql[ks], Kh[ko + ks * 8], Kh[ko + ks * 8 + 4], Kl[ko + ks * 8], Kl[ko + ks * 8 + 4]);
      float m_lo = fmaxf(sc[0], sc[1]), m_hi = fmaxf(sc[2], sc[3]);
      m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 1)); m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 2));
      m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 1)); m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 2));
      const float nm_lo = fmaxf(mx_lo, m_lo), nm_hi = fmaxf(mx_hi, m_hi);
      const float c_lo = __expf(mx_lo - nm_lo), c_hi = __expf(mx_hi - nm_hi);
      mx_lo = nm_lo; mx_hi = nm_hi;
      l_lo *= c_lo; l_hi *= c_hi;
#pragma unroll
      for (int nb = 0; nb < KS; ++nb) { o[nb][0] *= c_lo; o[nb][1] *= c_lo; o[nb][2] *= c_hi; o[nb][3] *= c_hi; }
      float p0 = __expf(sc[0] - mx_lo), p1 = __expf(sc[1] - mx_lo), p2 = __expf(sc[2] - mx_hi), p3 = __expf(sc[3] - mx_hi);
      l_lo += p0 + p1;
      l_hi += p2 + p3;
      const uint32_t key = (uint32_t)(kt0 + k0 + 2 * t);
      p0 *= drop_scale(seed, pair, q0 + g, key, S, thresh, inv_keep);
      p1 *= drop_scale(seed, pair, q0 + g, key + 1, S, thresh, inv_keep);
      p2 *= drop_scale(seed, pair, q0 + g + 8, key, S, thresh, inv_keep);
      p3 *= drop_scale(seed, pair, q0 + g + 8, key + 1, S, thresh, inv_keep);
      uint32_t ph[4], pl[4];
      split_bits(p0, ph[0], pl[0]); split_bits(p2, ph[1], pl[1]); split_bits(p1, ph[2], pl[2]); split_bits(p3, ph[3], pl[3]);
      const size_t vo = (size_t)(k0 + 2 * t) * P + g;
#pragma unroll
      for (int nb = 0; nb < KS; ++nb)
        mma3(o[nb], ph, pl, Vh[vo + nb * 8], Vh[vo + P + nb * 8], Vl[vo + nb * 8], Vl[vo + P + nb * 8]);
    }
  }
  l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1); l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
  l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1); l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
  const float i_lo = 1.0f / l_lo, i_hi = 1.0f / l_hi;
  if (t == 0) {
    if (ok_lo) lse[(size_t)pair * S + q0 + g] = mx_lo + logf(l_lo);
    if (ok_hi) lse[(size_t)pair * S + q0 + g + 8] = mx_hi + logf(l_hi);
  }
#pragma unroll
  for (int nb = 0; nb < KS; ++nb) {
    const int col = h * D + nb * 8 + 2 * t;
    if (ok_lo) *reinterpret_cast<float2*>(out + (size_t)(b * S + q0 + g) * C + col) = make_float2(o[nb][0] * i_lo, o[nb][1] * i_lo);
    if (ok_hi) *reinterpret_cast<float2*>(out + (size_t)(b * S + q0 + g + 8) * C + col) = make_float2(o[nb][2] * i_hi, o[nb][3] * i_hi);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// backward, query side: delta_i = dO_i . O_i, dQ = scale * dS K.  a warp = 16 queries
// ---------------------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) bwd_dq_kernel(const float* __restrict__ qkv, const float* __restrict__ out,
                                                     const float* __restrict__ dout, const float* __restrict__ lse,
                                                     float* __restrict__ dqkv,
                                                     const unsigned* __restrict__ seed_dev, unsigned salt, uint32_t thresh,
                                                     float inv_keep, int S, int C, int heads, float scale) {
  extern __shared__ __align__(16) uint32_t smem_u[];
  constexpr int P = D + 4, KS = D / 8;
  uint32_t* Kh = smem_u;
  uint32_t* Kl = Kh + kTile * P;
  uint32_t* Vh = Kl + kTile * P;
  uint32_t* Vl = Vh + kTile * P;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int pair = blockIdx.x, b = pair / heads, h = pair - b * heads;
  const int q0 = (blockIdx.y * (blockDim.x >> 5) + warp) * 16;
  const int row_stride = 3 * C;
  const uint32_t seed = layer_seed(seed_dev, salt);
  const bool ok_lo = q0 + g < S, ok_hi = q0 + g + 8 < S;
  const int r_lo = ok_lo ? q0 + g : 0, r_hi = ok_hi ? q0 + g + 8 : 0;
  const float* base = qkv + (size_t)b * S * row_stride + h * D;
  uint32_t qh[KS][4], ql[KS][4], gh[KS][4], gl[KS][4];
  load_a_frags<D>(qh, ql, base + (size_t)r_lo * row_stride + 2 * C, base + (size_t)r_hi * row_stride + 2 * C, ok_lo, ok_hi, t, scale);
  const float* do_lo = dout + (size_t)(b * S + r_lo) * C + h * D;
  const float* do_hi = dout + (size_t)(b * S + r_hi) * C + h * D;
  load_a_frags<D>(gh, gl, do_lo, do_hi, ok_lo, ok_hi, t, 1.f);
  // delta = dO . O per row (each lane holds columns t, t+4 of every 8-column block; a row lives in one quad)
  float d_lo = 0.f, d_hi = 0.f;
  {
    const float* o_lo = out + (size_t)(b * S + r_lo) * C + h * D;
    const float* o_hi = out + (size_t)(b * S + r_hi) * C + h * D;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      if (ok_lo) d_lo += __ldg(do_lo + ks * 8 + t) * __ldg(o_lo + ks * 8 + t) + __ldg(do_lo + ks * 8 + t + 4) * __ldg(o_lo + ks * 8 + t + 4);
      if (ok_hi) d_hi += __ldg(do_hi + ks * 8 + t) * __ldg(o_hi + ks * 8 + t) + __ldg(do_hi + ks * 8 + t + 4) * __ldg(o_hi + ks * 8 + t + 4);
    }
    d_lo += __shfl_xor_sync(0xffffffffu, d_lo, 1); d_lo += __shfl_xor_sync(0xffffffffu, d_lo, 2);
    d_hi += __shfl_xor_sync(0xffffffffu, d_hi, 1); d_hi += __shfl_xor_sync(0xffffffffu, d_hi, 2);
  }
  const float L_lo = ok_lo ? __ldg(lse + (size_t)pair * S + r_lo) : 0.f, L_hi = ok_hi ? __ldg(lse + (size_t)pair * S + r_hi) : 0.f;
  float dq[KS][4];
#pragma unroll
  for (int nb = 0; nb < KS; ++nb) dq[nb][0] = dq[nb][1] = dq[nb][2] = dq[nb][3] = 0.f;
  for (int kt0 = 0; kt0 < S; kt0 += kTile) {
    const int keys_here = S - kt0 < kTile ? S - kt0 : kTile;
    __syncthreads();
    stage_rows<D>(Kh, Kl, base + (size_t)kt0 * row_stride, row_stride, keys_here, keys_here, 1.f);
    stage_rows<D>(Vh, Vl, base + (size_t)kt0 * row_stride + C, row_stride, keys_here, keys_here, 1.f);
    __syncthreads();
    for (int k0 = 0; k0 < keys_here; k0 += 8) {
      float sc[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
      const size_t ko = (size_t)(k0 + g) * P + t;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        mma3(sc, qh[ks], ql[ks], Kh[ko + ks * 8], Kh[ko + ks * 8 + 4], Kl[ko + ks * 8], Kl[ko + ks * 8 + 4]);
        mma3(dp, gh[ks], gl[ks], Vh[ko + ks * 8], Vh[ko + ks * 8 + 4], Vl[ko + ks * 8], Vl[ko + ks * 8 + 4]);
      }
      const uint32_t key = (uint32_t)(kt0 + k0 + 2 * t);
      const float ds0 = __expf(sc[0] - L_lo) * (dp[0] * drop_scale(seed, pair, q0 + g, key, S, thresh, inv_keep) - d_lo);
      const float ds1 = __expf(sc[1] - L_lo) * (dp[1] * drop_scale(seed, pair, q0 + g, key + 1, S, thresh, inv_keep) - d_lo);
      const float ds2 = __expf(sc[2] - L_hi) * (dp[2] * drop_scale(seed, pair, q0 + g + 8, key, S, thresh, inv_keep) - d_hi);
      const float ds3 = __expf(sc[3] - L_hi) * (dp[3] * drop_scale(seed, pair, q0 + g + 8, key + 1, S, thresh, inv_keep) - d_hi);
      uint32_t ah[4], al[4];
      split_bits(ds0, ah[0], al[0]); split_bits(ds2, ah[1], al[1]); split_bits(ds1, ah[2], al[2]); split_bits(ds3, ah[3], al[3]);
      const size_t vo = (size_t)(k0 + 2 * t) * P + g;
#pragma unroll
      for (int nb = 0; nb < KS; ++nb)
        mma3(dq[nb], ah, al, Kh[vo + nb * 8], Kh[vo + P + nb * 8], Kl[vo + nb * 8], Kl[vo + P + nb * 8]);
    }
  }
#pragma unroll
  for (int nb = 0; nb < KS; ++nb) {
    const int col = 2 * C + h * D + nb * 8 + 2 * t;
    if (ok_lo) *reinterpret_cast<float2*>(dqkv + (size_t)(b * S + q0 + g) * row_stride + col) = make_float2(dq[nb][0] * scale, dq[nb][1] * scale);
    if (ok_hi) *reinterpret_cast<float2*>(dqkv + (size_t)(b * S + q0 + g + 8) * row_stride + col) = make_float2(dq[nb][2] * scale, dq[nb][3] * scale);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// backward, key side: dV = Pd^T dO, dK = dS^T q'.  a warp = 16 keys; queries (q', dO, lse, delta) stream through smem.
// Independent of the query-side kernel (delta is recomputed here), so the two can run on different streams.
// ---------------------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) bwd_dkv_kernel(const float* __restrict__ qkv, const float* __restrict__ out,
                                                      const float* __restrict__ dout, const float* __restrict__ lse,
                                                      float* __restrict__ dqkv, const unsigned* __restrict__ seed_dev,
                                                      unsigned salt, uint32_t thresh, float inv_keep, int S, int C, int heads,
                                                      float scale) {
  extern __shared__ __align__(16) uint32_t smem_u[];
  constexpr int P = D + 4, KS = D / 8;
  uint32_t* Qh = smem_u;
  uint32_t* Ql = Qh + kTile * P;
  uint32_t* Gh = Ql + kTile * P;
  uint32_t* Gl = Gh + kTile * P;
  float* Ls = reinterpret_cast<float*>(Gl + kTile * P);
  float* Ds = Ls + kTile;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int pair = blockIdx.x, b = pair / heads, h = pair - b * heads;
  const int k0w = (blockIdx.y * (blockDim.x >> 5) + warp) * 16;          // first key of this warp
  const int row_stride = 3 * C;
  const uint32_t seed = layer_seed(seed_dev, salt);
  const bool ok_lo = k0w + g < S, ok_hi = k0w + g + 8 < S;
  const int r_lo = ok_lo ? k0w + g : 0, r_hi = ok_hi ? k0w + g + 8 : 0;
  const float* base = qkv + (size_t)b * S * row_stride + h * D;
  uint32_t kh[KS][4], kl[KS][4], vh[KS][4], vl[KS][4];
  load_a_frags<D>(kh, kl, base + (size_t)r_lo * row_stride, base + (size_t)r_hi * row_stride, ok_lo, ok_hi, t, 1.f);
  load_a_frags<D>(vh, vl, base + (size_t)r_lo * row_stride + C, base + (size_t)r_hi * row_stride + C, ok_lo, ok_hi, t, 1.f);
  float dk[KS][4], dv[KS][4];
#pragma unroll
  for (int nb = 0; nb < KS; ++nb) { dk[nb][0] = dk[nb][1] = dk[nb][2] = dk[nb][3] = 0.f; dv[nb][0] = dv[nb][1] = dv[nb][2] = dv[nb][3] = 0.f; }
  for (int qt0 = 0; qt0 < S; qt0 += kTile) {
    const int q_here = S - qt0 < kTile ? S - qt0 : kTile;
    __syncthreads();
    stage_rows<D>(Qh, Ql, base + (size_t)qt0 * row_stride + 2 * C, row_stride, q_here, q_here, scale);
    stage_rows<D>(Gh, Gl, dout + (size_t)(b * S + qt0) * C + h * D, (size_t)C, q_here, q_here, 1.f);
    for (int i = threadIdx.x; i < q_here; i += blockDim.x) Ls[i] = __ldg(lse + (size_t)pair * S + qt0 + i);
    // delta_i = dO_i . O_i: eight lanes per row (D / 4 <= 10 float4 per row, so lanes 0..7 take one or two each), reduced
    // with shuffles in a fixed order - coalesced row reads, deterministic
    for (int i0 = 0; i0 < q_here * 8; i0 += blockDim.x) {
      const int i = i0 + threadIdx.x, row = i >> 3, part = i & 7;
      float acc = 0.f;
      if (row < q_here) {
        const float4* po = reinterpret_cast<const float4*>(out + (size_t)(b * S + qt0 + row) * C + h * D);
        const float4* pg = reinterpret_cast<const float4*>(dout + (size_t)(b * S + qt0 + row) * C + h * D);
        for (int v4 = part; v4 < D / 4; v4 += 8) {
          const float4 o4 = __ldg(po + v4), g4 = __ldg(pg + v4);
          acc += o4.x * g4.x + o4.y * g4.y + o4.z * g4.z + o4.w * g4.w;
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if (part == 0 && row < q_here) Ds[row] = acc;
    }
    __syncthreads();
    for (int q0 = 0; q0 < q_here; q0 += 8) {
      float st[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
      const size_t qo = (size_t)(q0 + g) * P + t;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        mma3(st, kh[ks], kl[ks], Qh[qo + ks * 8], Qh[qo + ks * 8 + 4], Ql[qo + ks * 8], Ql[qo + ks * 8 + 4]);
        mma3(dp, vh[ks], vl[ks], Gh[qo + ks * 8], Gh[qo + ks * 8 + 4], Gl[qo + ks * 8], Gl[qo + ks * 8 + 4]);
      }
      // c0: (key g, query 2t), c1: (key g, query 2t+1), c2 / c3: key g+8
      const int qa = q0 + 2 * t;
      const uint32_t query = (uint32_t)(qt0 + qa);
      const float La = Ls[qa], Lb = Ls[qa + 1], Da = Ds[qa], Db = Ds[qa + 1];
      const float m0 = drop_scale(seed, pair, query, k0w + g, S, thresh, inv_keep);
      const float m1 = drop_scale(seed, pair, query + 1, k0w + g, S, thresh, inv_keep);
      const float m2 = drop_scale(seed, pair, query, k0w + g + 8, S, thresh, inv_keep);
      const float m3 = drop_scale(seed, pair, query + 1, k0w + g + 8, S, thresh, inv_keep);
      const float p0 = __expf(st[0] - La), p1 = __expf(st[1] - Lb), p2 = __expf(st[2] - La), p3 = __expf(st[3] - Lb);
      uint32_t ah[4], al[4];
      split_bits(p0 * m0, ah[0], al[0]); split_bits(p2 * m2, ah[1], al[1]); split_bits(p1 * m1, ah[2], al[2]); split_bits(p3 * m3, ah[3], al[3]);
      const size_t go = (size_t)(q0 + 2 * t) * P + g;
#pragma unroll
      for (int nb = 0; nb < KS; ++nb)
        mma3(dv[nb], ah, al, Gh[go + nb * 8], Gh[go + P + nb * 8], Gl[go + nb * 8], Gl[go + P + nb * 8]);
      split_bits(p0 * (dp[0] * m0 - Da), ah[0], al[0]); split_bits(p2 * (dp[2] * m2 - Da), ah[1], al[1]);
      split_bits(p1 * (dp[1] * m1 - Db), ah[2], al[2]); split_bits(p3 * (dp[3] * m3 - Db), ah[3], al[3]);
#pragma unroll
      for (int nb = 0; nb < KS; ++nb)
        mma3(dk[nb], ah, al, Qh[go + nb * 8], Qh[go + P + nb * 8], Ql[go + nb * 8], Ql[go + P + nb * 8]);
    }
  }
#pragma unroll
  for (int nb = 0; nb < KS; ++nb) {
    const int col = h * D + nb * 8 + 2 * t;
    if (ok_lo) {
      float* row = dqkv + (size_t)(b * S + k0w + g) * row_stride;
      *reinterpret_cast<float2*>(row + col) = make_float2(dk[nb][0], dk[nb][1]);
      *reinterpret_cast<float2*>(row + C + col) = make_float2(dv[nb][0], dv[nb][1]);
    }
    if (ok_hi) {
      float* row = dqkv + (size_t)(b * S + k0w + g + 8) * row_stride;
      *reinterpret_cast<float2*>(row + col) = make_float2(dk[nb][2], dk[nb][3]);
      *reinterpret_cast<float2*>(row + C + col) = make_float2(dv[nb][2], dv[nb][3]);
    }
  }
}

__global__ void mask_kernel(const unsigned* __restrict__ seed_dev, unsigned salt, uint32_t thresh, float inv_keep, int pairs,
                            int S, float* __restrict__ mask) {
  const uint32_t seed = layer_seed(seed_dev, salt);
  const long long total = (long long)pairs * S * S;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t k = (uint32_t)(i % S), q = (uint32_t)((i / S) % S), pair = (uint32_t)(i / ((long long)S * S));
    mask[i] = drop_scale(seed, pair, q, k, S, thresh, inv_keep);
  }
}

struct Launch {
  dim3 grid, block;
  size_t smem;
  uint32_t thresh;
  float inv_keep, scale;
};
static bool plan(int B, int S, int C, int heads, float p_drop, int D, Launch* l) {
  if (B < 1 || S < 8 || S % 8 || C < 1 || heads < 1 || C % heads || C / heads != D) return false;
  if (!(p_drop >= 0.f) || p_drop >= 1.f) return false;
  if ((long long)B * heads * S * S >= 0xffffffffLL) return false;         // the mask counter is 32 bits
  int warps = (S + 15) / 16;
  if (warps > 8) warps = 8;
  l->grid = dim3(B * heads, (S + warps * 16 - 1) / (warps * 16));
  l->block = dim3(32 * warps);
  l->smem = (size_t)4 * kTile * (D + 4) * 4 + 2 * kTile * 4;
  l->thresh = (uint32_t)((double)p_drop * 4294967296.0);
  l->inv_keep = 1.f / (1.f - p_drop);
  l->scale = 1.f / sqrtf((float)D);
  return true;
}

template <int D>
static int run_fwd(const float* qkv, float* out, float* lse, const unsigned* seed, unsigned salt, float p, int B, int S, int C,
                   int heads, cudaStream_t st) {
  Launch l;
  if (!plan(B, S, C, heads, p, D, &l)) return FLOWK_ERR_SHAPE;
  FLOWK_CUDA_OK(cudaFuncSetAttribute(fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem));
  fwd_kernel<D><<<l.grid, l.block, l.smem, st>>>(qkv, out, lse, seed, salt, l.thresh, l.inv_keep, S, C, heads, l.scale);
  return launch_status();
}
template <int D>
static int run_bwd(int which, const float* qkv, const float* out, const float* dout, const float* lse, float* dqkv,
                   const unsigned* seed, unsigned salt, float p, int B, int S, int C, int heads, cudaStream_t st) {
  Launch l;
  if (!plan(B, S, C, heads, p, D, &l)) return FLOWK_ERR_SHAPE;
  if (which & 1) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(bwd_dq_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem));
    bwd_dq_kernel<D><<<l.grid, l.block, l.smem, st>>>(qkv, out, dout, lse, dqkv, seed, salt, l.thresh, l.inv_keep, S, C, heads,
                                                      l.scale);
  }
  if (which & 2) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(bwd_dkv_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem));
    bwd_dkv_kernel<D><<<l.grid, l.block, l.smem, st>>>(qkv, out, dout, lse, dqkv, seed, salt, l.thresh, l.inv_keep, S, C, heads,
                                                       l.scale);
  }
  return launch_status();
}

}  // namespace attn_train
}  // namespace flowk

using namespace flowk;
using namespace flowk::attn_train;

extern "C" int flowk_attention_train_fwd(const float* qkv, float* out, float* lse, const unsigned* seed_device, unsigned salt,
                                         float p_drop, int B, int HW, int C, int heads, flowk_stream_t stream) {
  if (B == 0) return FLOWK_OK;
  if (!qkv || !out || !lse) return FLOWK_ERR_ARG;
  if (heads < 1 || C % heads) return FLOWK_ERR_SHAPE;
  switch (C / heads) {
    case 8: return run_fwd<8>(qkv, out, lse, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 16: return run_fwd<16>(qkv, out, lse, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 24: return run_fwd<24>(qkv, out, lse, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 32: return run_fwd<32>(qkv, out, lse, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 40: return run_fwd<40>(qkv, out, lse, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 64: return run_fwd<64>(qkv, out, lse, seed_device, salt, p_drop, B, HW, C, heads, stream);
    default: return FLOWK_ERR_SHAPE;
  }
}

// which: 1 = query side (dq columns of dqkv), 2 = key side (dk, dv columns), 3 = both on `stream`
extern "C" int flowk_attention_train_bwd(int which, const float* qkv, const float* out, const float* dout, const float* lse,
                                         float* dqkv, const unsigned* seed_device, unsigned salt, float p_drop, int B, int HW,
                                         int C, int heads, flowk_stream_t stream) {
  if (B == 0) return FLOWK_OK;
  if (which < 1 || which > 3) return FLOWK_ERR_ARG;
  if (!qkv || !out || !dout || !lse || !dqkv) return FLOWK_ERR_ARG;
  if (heads < 1 || C % heads) return FLOWK_ERR_SHAPE;
  switch (C / heads) {
    case 8: return run_bwd<8>(which, qkv, out, dout, lse, dqkv, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 16: return run_bwd<16>(which, qkv, out, dout, lse, dqkv, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 24: return run_bwd<24>(which, qkv, out, dout, lse, dqkv, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 32: return run_bwd<32>(which, qkv, out, dout, lse, dqkv, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 40: return run_bwd<40>(which, qkv, out, dout, lse, dqkv, seed_device, salt, p_drop, B, HW, C, heads, stream);
    case 64: return run_bwd<64>(which, qkv, out, dout, lse, dqkv, seed_device, salt, p_drop, B, HW, C, heads, stream);
    default: return FLOWK_ERR_SHAPE;
  }
}

extern "C" int flowk_attention_dropout_mask(const unsigned* seed_device, unsigned salt, float p_drop, int pairs, int HW,
                                            float* mask, flowk_stream_t stream) {
  if (pairs < 1 || HW < 1 || !(p_drop >= 0.f) || p_drop >= 1.f || (long long)pairs * HW * HW >= 0xffffffffLL) return FLOWK_ERR_SHAPE;
  if (!mask) return FLOWK_ERR_ARG;
  mask_kernel<<<148 * 8, 256, 0, stream>>>(seed_device, salt, (uint32_t)((double)p_drop * 4294967296.0), 1.f / (1.f - p_drop),
                                          pairs, HW, mask);
  return launch_status();
}
