// `Transformer_attn` (the fork's invertible patch attention, reference flow_modules/transformer.py:123-326, used twice per
// FlowStep at marscf_main.py:50-51,69-70) as ONE pass over the activations, inference / sampling.
//
// The image is a 2x2 grid of patches of side p = W/2; patch n, flattened index l = (c, i, j).  Entries with (n + l) even
// (odd when `permute`) condition the attention and pass through; the others are mixed between the patches of equal
// parity by two 2x2 matrices.  With G = sum_i Wq_i^T Wk_i (the six 1x1 convs and three Q K^T products collapsed, built on
// the host side once per weight version):
//
//   score[n, m] = sum_{(i,j)} u_n(i,j)^T G u_m(i,j),   u_n(i,j) = masked channel vector of patch n at in-patch pixel (i,j)
//   attn        = sigmoid(score / scale + offset2) + offset3,   M1 = attn[{0,2},{0,2}] + offset I,  M2 = attn[{1,3},{1,3}] + offset I
//   forward     free entries of patches (0, 2) <- M1 (x0, x2),  of patches (1, 3) <- M2 (x1, x3);  ldj += (log|det M1| + log|det M2|) p (p/2) C
//   reverse     the same with the closed-form inverses; ldj -= ...
//
// One CTA per sample: the sample ([C, H, W] fp32, <= 48 KB) and G sit in shared memory, the eight scores are a fixed-order
// block reduction (bit-reproducible), the mixing pass re-reads shared memory: HBM traffic is one read + one write of the
// activations (8 B per element), the same as the fused ActNorm / 1x1-conv kernel.
//
// Training (forward direction only) runs the same kernel with the raw scores as an extra [B, 8] output, and
// patch_attention_bwd_kernel below differentiates it per sample in closed form (the 2x2 matrices make every step local).
#include "common.cuh"

namespace flowk {

constexpr int PA_THREADS = 256;

__global__ void __launch_bounds__(PA_THREADS) patch_attention_kernel(const float* __restrict__ x, const float* __restrict__ G,
                                                                      const float* __restrict__ prm, float* __restrict__ y,
                                                                      const float* __restrict__ ldj_in, float* __restrict__ ldj_out,
                                                                      float* __restrict__ scores, int C, int H, int W, int permute,
                                                                      int reverse) {
  extern __shared__ __align__(16) float sm[];
  const int HW = H * W, n_el = C * HW, p = W >> 1, pp = p * p;
  float* xs = sm;                         // [C][H][W]
  float* xm = sm + ((n_el + 3) & ~3);     // the same with the free entries zeroed (the conditioning part the scores see)
  float* gs = xm + ((n_el + 3) & ~3);     // [C][C]
  __shared__ float red[PA_THREADS / 32][8];
  __shared__ float mat[8];                // a1 b1 c1 d1 a2 b2 c2 d2 (already inverted when reverse)
  const int b = blockIdx.x;
  const float* xb = x + (size_t)b * n_el;
  float* yb = y + (size_t)b * n_el;
  // conditioning mask of entry l = c p^2 + i p + j of patch n: (n + l) even, inverted by `permute`
  const int perm = permute ? 1 : 0;
  auto is_cond = [&](int n, int c, int i, int j) -> bool { return (((n + c * pp + i * p + j) & 1) ^ perm) == 0; };
  for (int e = threadIdx.x; e < n_el; e += PA_THREADS) {
    const float v = __ldcs(xb + e);
    const int xx = e % W, t = e / W, yy = t % H, c = t / H;
    const int lower = yy >= p, right = xx >= p;
    xs[e] = v;
    xm[e] = is_cond((lower << 1) | right, c, yy - (lower ? p : 0), xx - (right ? p : 0)) ? v : 0.f;
  }
  for (int i = threadIdx.x; i < C * C; i += PA_THREADS) gs[i] = __ldg(G + i);
  __syncthreads();

  // ---- scores: item = (patch m, in-patch pixel, output channel c): v = sum_c' G[c, c'] u_m[c'], then u_n[c] v for both n
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};      // (0,0) (0,2) (2,0) (2,2) (1,1) (1,3) (3,1) (3,3)
  for (int it = threadIdx.x; it < n_el; it += PA_THREADS) {
    const int c = it % C, r = it / C, m = r & 3, pix = r >> 2;
    const int i = pix / p, j = pix - i * p;
    const int ym = i + ((m >> 1) ? p : 0), xm_col = j + ((m & 1) ? p : 0);
    float v = 0.f;
    const float* grow = gs + c * C;
    const float* xcol = xm + ym * W + xm_col;
#pragma unroll 4
    for (int cc = 0; cc < C; ++cc) v = fmaf(grow[cc], xcol[cc * HW], v);
    // rows n of equal parity: n = m & 1 (upper patch) and n = (m & 1) + 2 (lower patch)
    const int n0 = m & 1, n1 = n0 + 2;
    const int y0 = i, x0 = j + (n0 ? p : 0), y1 = i + p, x1 = x0;
    const float u0 = xm[(c * H + y0) * W + x0];
    const float u1 = xm[(c * H + y1) * W + x1];
    const int base = (m & 1) ? 4 : 0, col = m >> 1;               // score[n, m]: column index of m within its parity class
    acc[base + col] += u0 * v;                                     // n = n0 (row 0 of the 2x2 block)
    acc[base + 2 + col] += u1 * v;                                 // n = n1 (row 1)
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = warp_sum(acc[k]);
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) red[threadIdx.x >> 5][k] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float s[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float t = 0.f;
      for (int w = 0; w < PA_THREADS / 32; ++w) t += red[w][k];
      s[k] = t;
    }
    if (scores) {
#pragma unroll
      for (int k = 0; k < 8; ++k) scores[(size_t)b * 8 + k] = s[k];
    }
    const float off = prm[0], off2 = prm[1], off3 = prm[2], scale = prm[3];
    float mm[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) mm[k] = 1.0f / (1.0f + expf(-(s[k] / scale + off2))) + off3;
    mm[0] += off; mm[3] += off; mm[4] += off; mm[7] += off;        // diagonals
    const float det1 = mm[0] * mm[3] - mm[1] * mm[2], det2 = mm[4] * mm[7] - mm[5] * mm[6];
    const float ld = (logf(fabsf(det1)) + logf(fabsf(det2))) * (float)(p * (p / 2) * C);
    if (reverse) {
      const float a1 = mm[3] / det1, b1 = -mm[1] / det1, c1 = -mm[2] / det1, d1 = mm[0] / det1;
      const float a2 = mm[7] / det2, b2 = -mm[5] / det2, c2 = -mm[6] / det2, d2 = mm[4] / det2;
      mm[0] = a1; mm[1] = b1; mm[2] = c1; mm[3] = d1; mm[4] = a2; mm[5] = b2; mm[6] = c2; mm[7] = d2;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) mat[k] = mm[k];
    if (ldj_out) ldj_out[b] = (ldj_in ? ldj_in[b] : 0.f) + (reverse ? -ld : ld);
  }
  __syncthreads();

  // ---- mixing: conditioning entries pass through, free entries are mixed with the same entry of the partner patch
  for (int e = threadIdx.x; e < n_el; e += PA_THREADS) {
    const int xx = e % W, t = e / W, yy = t % H, c = t / H;
    float v = xs[e];
    const int lower = yy >= p, right = xx >= p;
    if (!is_cond((lower << 1) | right, c, yy - (lower ? p : 0), xx - (right ? p : 0))) {
      const float partner = xs[(c * H + (lower ? yy - p : yy + p)) * W + xx];
      const float* mtx = mat + (right ? 4 : 0);
      // upper patch (row 0): a x_n + b x_partner;  lower patch (row 1): c x_partner + d x_n
      v = lower ? fmaf(mtx[2], partner, mtx[3] * v) : fmaf(mtx[0], v, mtx[1] * partner);
    }
    __stcs(yb + e, v);
  }
}

// Backward of the forward direction, one CTA per sample (notation as above; class e = 0 for patches (0, 2), 1 for (1, 3); row
// r of patch n is n >> 1; K = p (p/2) C; gl = d loss / d ldj_out):
//
//   gM_e[r,s] = sum_free gy_{n_r} x_{n_s} + gl K M_e^-T[r,s]     gZ = gM (.) sig (1 - sig)     gS = gZ / scale
//   g_offset = sum diag gM,  g_offset3 = sum gM,  g_offset2 = sum gZ,  g_scale = -sum gZ (.) S / scale^2
//   free entries:          gx_{n_s} = sum_r M_e[r,s] gy_{n_r}
//   conditioning entries:  gx_n = gy_n + G W_n + G^T V_n,   W_n = sum_s gS[r(n), s] u_{n_s},   V_n = sum_r gS[r, r(n)] u_{n_r}
//   gG = sum_pixels sum_n u_n W_n^T  (C x C per sample, reduced over the batch by the caller)
//
// Shared memory: x, its masked copy u, gy and G (3 C H W + C^2 floats); x is dead after the gM sums and its slot holds W.
// Every sum has a fixed order (fixed item -> thread maps, warp shuffles, warps added in index order): bit-reproducible.
__global__ void __launch_bounds__(PA_THREADS) patch_attention_bwd_kernel(
    const float* __restrict__ x, const float* __restrict__ G, const float* __restrict__ prm,
    const float* __restrict__ scores, const float* __restrict__ gy, const float* __restrict__ gldj, float* __restrict__ gx,
    float* __restrict__ partials, int C, int H, int W, int permute) {
  extern __shared__ __align__(16) float sm[];
  const int HW = H * W, n_el = C * HW, p = W >> 1, pp = p * p, n4 = (n_el + 3) & ~3;
  float* xs = sm;                         // [C][H][W]; later W_n at the same index
  float* xm = sm + n4;                    // u: x with the free entries zeroed
  float* gys = xm + n4;                   // [C][H][W]
  float* gs = gys + n4;                   // [C][C]
  __shared__ float red[PA_THREADS / 32][8];
  __shared__ float mat[8];                // M_0, M_1 row-major (a b c d)
  __shared__ float gsc[8];                // gS_0, gS_1 row-major
  __shared__ float gpart[PA_THREADS];     // sliced partial sums of gG
  const int b = blockIdx.x;
  const float* xb = x + (size_t)b * n_el;
  const float* gyb = gy + (size_t)b * n_el;
  const int perm = permute ? 1 : 0;
  auto is_cond = [&](int n, int c, int i, int j) -> bool { return (((n + c * pp + i * p + j) & 1) ^ perm) == 0; };
  for (int e = threadIdx.x; e < n_el; e += PA_THREADS) {
    const float v = __ldg(xb + e);
    const int xx = e % W, t = e / W, yy = t % H, c = t / H;
    const int lower = yy >= p, right = xx >= p;
    xs[e] = v;
    xm[e] = is_cond((lower << 1) | right, c, yy - (lower ? p : 0), xx - (right ? p : 0)) ? v : 0.f;
    gys[e] = __ldcs(gyb + e);
  }
  for (int i = threadIdx.x; i < C * C; i += PA_THREADS) gs[i] = __ldg(G + i);
  __syncthreads();

  // ---- gM data term: item = entry (c, i, jj) of the upper patch row; its lower partner is the row-1 entry of the class
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};      // gM_0 (a b c d), gM_1 (a b c d)
  for (int it = threadIdx.x; it < n_el / 2; it += PA_THREADS) {
    const int xx = it % W, t = it / W, yy = t % p, c = t / p;
    const int right = xx >= p;
    if (is_cond(right, c, yy, xx - (right ? p : 0))) continue;    // the partner (n + 2) has the same mask
    const int eu = (c * H + yy) * W + xx, el = eu + p * W;
    const float xu = xs[eu], xl = xs[el], gu = gys[eu], gl = gys[el];
    if (right) {
      acc[4] = fmaf(gu, xu, acc[4]); acc[5] = fmaf(gu, xl, acc[5]); acc[6] = fmaf(gl, xu, acc[6]); acc[7] = fmaf(gl, xl, acc[7]);
    } else {
      acc[0] = fmaf(gu, xu, acc[0]); acc[1] = fmaf(gu, xl, acc[1]); acc[2] = fmaf(gl, xu, acc[2]); acc[3] = fmaf(gl, xl, acc[3]);
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) acc[k] = warp_sum(acc[k]);
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 8; ++k) red[threadIdx.x >> 5][k] = acc[k];
  }
  __syncthreads();
  float* part = partials + (size_t)b * (C * C + 4);
  if (threadIdx.x == 0) {
    const float off = prm[0], off2 = prm[1], off3 = prm[2], scale = prm[3];
    const float glk = gldj[b] * (float)(p * (p / 2) * C);
    float g_off = 0.f, g_off2 = 0.f, g_off3 = 0.f, g_scale = 0.f;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float s[4], sig[4], m[4], gm[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        s[k] = scores[(size_t)b * 8 + 4 * e + k];
        sig[k] = 1.0f / (1.0f + expf(-(s[k] / scale + off2)));   // the forward's expression
        m[k] = sig[k] + off3;
        float t = 0.f;
        for (int w = 0; w < PA_THREADS / 32; ++w) t += red[w][4 * e + k];
        gm[k] = t;
      }
      m[0] += off; m[3] += off;
      const float det = m[0] * m[3] - m[1] * m[2];
      // d log|det M| / dM = M^-T = [d, -c; -b, a] / det
      gm[0] = fmaf(glk, m[3] / det, gm[0]); gm[1] = fmaf(glk, -m[2] / det, gm[1]);
      gm[2] = fmaf(glk, -m[1] / det, gm[2]); gm[3] = fmaf(glk, m[0] / det, gm[3]);
      g_off += gm[0] + gm[3];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float gz = gm[k] * sig[k] * (1.0f - sig[k]);
        g_off3 += gm[k];
        g_off2 += gz;
        g_scale -= gz * s[k] / (scale * scale);
        gsc[4 * e + k] = gz / scale;
        mat[4 * e + k] = m[k];
      }
    }
    part[C * C + 0] = g_off;
    part[C * C + 1] = g_off2;
    part[C * C + 2] = g_off3;
    part[C * C + 3] = g_scale;
  }
  __syncthreads();

  // ---- W_n = gS[r, r] u_n + gS[r, 1 - r] u_partner into the x slot
  for (int e = threadIdx.x; e < n_el; e += PA_THREADS) {
    const int xx = e % W, t = e / W, yy = t % H;
    const int lower = yy >= p, right = xx >= p;
    const float* g2 = gsc + 4 * right + 2 * lower;                // row r = lower of the class matrix
    const float up = xm[lower ? e - p * W : e + p * W];
    xs[e] = lower ? fmaf(g2[0], up, g2[1] * xm[e]) : fmaf(g2[0], xm[e], g2[1] * up);
  }
  __syncthreads();

  // ---- gx: item = entry pair (2q, 2q + 1) of one image row; exactly one of the two conditions (the parity of n + j flips
  // from one to the next, also across the patch boundary where p is odd), so every thread does one C-long dot product
  float* gxb = gx + (size_t)b * n_el;
  for (int q = threadIdx.x; q < n_el / 2; q += PA_THREADS) {
    const int e0 = 2 * q;
    const int xx0 = e0 % W, t = e0 / W, yy = t % H, c = t / H;
    const int lower = yy >= p, i = yy - (lower ? p : 0);
    const int right0 = xx0 >= p;
    const int ec = is_cond((lower << 1) | right0, c, i, xx0 - (right0 ? p : 0)) ? e0 : e0 + 1;
    const int ef = e0 + e0 + 1 - ec;
    const int pw = lower ? -p * W : p * W;                       // offset to the partner patch of the class
    {                                                            // free entry: gx_{n_s} = sum_r M[r, s] gy_{n_r}, s = lower
      const int right = (ef % W) >= p;
      const float* mt = mat + 4 * right;
      const float g_self = gys[ef], g_part = gys[ef + pw];
      __stcs(gxb + ef, lower ? fmaf(mt[1], g_part, mt[3] * g_self) : fmaf(mt[0], g_self, mt[2] * g_part));
    }
    {                                                            // conditioning entry: gy + G W + G^T V
      const int right = (ec % W) >= p, sp = ec - c * HW;
      const float* g2 = gsc + 4 * right;
      const float v_self = g2[3 * lower], v_part = g2[lower ? 1 : 2];   // gS[r, r], gS[1 - r, r]
      const float* grow = gs + c * C;
      const float* gcol = gs + c;
      const float* wc = xs + sp;
      const float* uc = xm + sp;
      float t_w = 0.f, t_s = 0.f, t_p = 0.f;
#pragma unroll 4
      for (int cc = 0; cc < C; ++cc) {
        const float gc = gcol[cc * C];
        t_w = fmaf(grow[cc], wc[cc * HW], t_w);
        t_s = fmaf(gc, uc[cc * HW], t_s);
        t_p = fmaf(gc, uc[cc * HW + pw], t_p);
      }
      __stcs(gxb + ec, gys[ec] + t_w + fmaf(v_self, t_s, v_part * t_p));
    }
  }

  // ---- gG[c, c'] = sum_pixels u[c] W[c']: C^2 dot products over HW, split into `slices` fixed ranges when C^2 < threads
  const int n_out = C * C, slices = n_out >= PA_THREADS ? 1 : PA_THREADS / n_out;
  for (int o0 = 0; o0 < n_out; o0 += PA_THREADS) {
    const int tid = threadIdx.x, o = o0 + tid % n_out, sl = tid / n_out;
    if (o < n_out && sl < slices && (slices == 1 || o0 + tid < n_out * slices)) {
      const int c = o / C, c2 = o - c * C;
      const int s0 = (int)((long long)HW * sl / slices), s1 = (int)((long long)HW * (sl + 1) / slices), len = s1 - s0;
      const int rot = len ? c2 % len : 0;                         // staggered start: neighbouring c' hit different banks
      const float* u = xm + c * HW;
      const float* wv = xs + c2 * HW;
      float a = 0.f;
      for (int s = s0 + rot; s < s1; ++s) a = fmaf(u[s], wv[s], a);
      for (int s = s0; s < s0 + rot; ++s) a = fmaf(u[s], wv[s], a);
      if (slices == 1) part[o] = a;
      else gpart[tid] = a;
    }
  }
  if (slices > 1) {
    __syncthreads();
    if (threadIdx.x < n_out) {
      float a = 0.f;
      for (int sl = 0; sl < slices; ++sl) a += gpart[sl * n_out + threadIdx.x];
      part[threadIdx.x] = a;
    }
  }
}

}  // namespace flowk

using namespace flowk;

namespace {

bool pa_shape_ok(int B, int C, int H, int W) { return B >= 0 && C >= 1 && H >= 2 && H == W && !(W & 1); }

// dynamic shared memory: a [C, H, W] sample held `copies` times, plus G
size_t pa_smem(int C, int H, int W, int copies) {
  return ((size_t)copies * (((size_t)C * H * W + 3) & ~(size_t)3) + (size_t)C * C) * sizeof(float);
}

int pa_forward(const float* x, const float* G, const float* prm, float* y, const float* ldj_in, float* ldj_out,
               float* scores, bool need_scores, int B, int C, int H, int W, int permute, int reverse, cudaStream_t stream) {
  if (!pa_shape_ok(B, C, H, W)) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!x || !G || !prm || !y || (need_scores && !scores)) return FLOWK_ERR_ARG;
  const size_t smem = pa_smem(C, H, W, 2);
  if (smem > 200 * 1024) return FLOWK_ERR_SHAPE;
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(patch_attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  patch_attention_kernel<<<B, PA_THREADS, smem, stream>>>(x, G, prm, y, ldj_in, ldj_out, scores, C, H, W, permute, reverse);
  return launch_status();
}

}  // namespace

// x, y [B, C, H, W] fp32 (H == W, even); G [C, C] = sum_i Wq_i^T Wk_i; prm = device {offset, offset2, offset3, scale};
// ldj_in / ldj_out [B] (either may be NULL).  reference: flow_modules/transformer.py:123-326.
extern "C" int flowk_patch_attention(const float* x, const float* G, const float* prm, float* y, const float* ldj_in,
                                     float* ldj_out, int B, int C, int H, int W, int permute, int reverse,
                                     flowk_stream_t stream) {
  return pa_forward(x, G, prm, y, ldj_in, ldj_out, nullptr, false, B, C, H, W, permute, reverse, stream);
}

// Forward direction for training: flowk_patch_attention plus the raw scores [B, 8] that flowk_patch_attention_bwd takes.
extern "C" int flowk_patch_attention_train_fwd(const float* x, const float* G, const float* prm, float* y,
                                               const float* ldj_in, float* ldj_out, float* scores, int B, int C, int H,
                                               int W, int permute, flowk_stream_t stream) {
  return pa_forward(x, G, prm, y, ldj_in, ldj_out, scores, true, B, C, H, W, permute, 0, stream);
}

// gx [B, C, H, W]; partials [B, C*C + 4] = per-sample gG (row-major), g_offset, g_offset2, g_offset3, g_scale.
extern "C" int flowk_patch_attention_bwd(const float* x, const float* G, const float* prm, const float* scores,
                                         const float* gy, const float* gldj, float* gx, float* partials, int B, int C,
                                         int H, int W, int permute, flowk_stream_t stream) {
  if (!pa_shape_ok(B, C, H, W)) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!x || !G || !prm || !scores || !gy || !gldj || !gx || !partials) return FLOWK_ERR_ARG;
  const size_t smem = pa_smem(C, H, W, 3);
  if (smem > 200 * 1024) return FLOWK_ERR_SHAPE;
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(patch_attention_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  patch_attention_bwd_kernel<<<B, PA_THREADS, smem, stream>>>(x, G, prm, scores, gy, gldj, gx, partials, C, H, W, permute);
  return launch_status();
}
