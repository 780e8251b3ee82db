// Training-time self-attention core of GatedAttn (flow_modules/mixlogcdf_nn.py:134-147) with attention-weight dropout on
// the 5th-gen tensor cores, for head dim D = 64 and seq S in {128, 256} (the width-256 model at 16x16 / 8x16).  Same
// function, layouts and dropout mask as attention_train.cu (which keeps head dims 8-40 and the shorter sequences):
//     P = softmax_j(q_i k_j / sqrt(d)),   Pd = P * M,   O = Pd V,   lse_i = log sum_j exp(s_ij)
//     dV = Pd^T dO;  dP = dO V^T;  delta_i = dO_i . O_i;  dS = P * (dP * M - delta_i);  dQ = dS K / sqrt(d);  dK = dS^T q'
//
// One kernel template, three modes; a CTA of 128 threads owns 128 rows of one (image, head) pair - thread t = TMEM lane t =
// own row t - and streams the pair's other rows through shared memory in blocks of NB:
//   FWD  own = 128 queries (Q' = Q / sqrt d),  blocks of 64 keys:     S = Q' K^T;  online softmax in registers;  O_b = Pd V
//   DQ   own = 128 queries (Q', dO),           blocks of 32 keys:     S = Q' K^T, dP = dO V^T;  dQ += dS K   (TMEM accumulator)
//   DKV  own = 128 keys (K, V),                blocks of 32 queries:  S^T = K Q'^T, dP^T = V dO^T;  dV += Pd^T dO, dK += dS^T Q'
// Every product is tcgen05.mma kind::tf32, M = 128, with fp32 accuracy from (hi, lo) TF32 operand pairs and three MMAs
// (hi hi + lo hi + hi lo), the scheme of the training GEMMs.  Operands are K-major SWIZZLE_128B tiles (32 fp32 per 128-byte
// row) written by the threads from the fp32 rows: the streamed matrix as it lies (score B operand) and transposed (B
// operand of the accumulating product), the softmax weights Pd / dS row by row (its A operand).  Nothing of size S x S
// touches HBM; the backward recomputes S from lse and regenerates the dropout mask (attention_dropout.cuh).  The two
// backward modes share no intermediate (each computes delta itself) and use no atomics: results are deterministic.
// The phases of a block run in order (stage -> score MMAs -> softmax -> accumulating MMAs); the shared-memory carve (up to
// 225 KB) leaves one CTA per SM.  A timed-out mbarrier wait writes NaN into the CTA's outputs instead of hanging.
#include <cuda.h>
#include "common.cuh"
#include "umma.cuh"
#include "attention_tile.cuh"
#include "attention_dropout.cuh"

namespace flowk {
namespace attn_train_tc {

using namespace flowk::tc;
using flowk::attn_train::drop_scale;
using flowk::attn_train::layer_seed;

constexpr int D = 64;                 // head dim: two 32-float K blocks per row
constexpr int OWN = 128;              // own rows per CTA = MMA M = threads
enum Mode { FWD = 0, DQ = 1, DKV = 2 };

template <int MODE> struct Cfg {
  static constexpr int NB = MODE == FWD ? 64 : 32;                // streamed rows per block
  static constexpr int OWN_T = MODE == FWD ? 1 : 2;               // own operand tiles [128 x 64]
  static constexpr int DIR_T = MODE == FWD ? 1 : 2;               // streamed tiles as they lie [NB x 64]
  static constexpr int TR_T = MODE == DQ ? 1 : (MODE == FWD ? 1 : 2);   // streamed tiles transposed [64 x NB]
  static constexpr int OWN_B = OWN * D * 4 * 2;                   // (hi, lo)
  static constexpr int DIR_B = NB * D * 4 * 2;
  static constexpr int TR_B = D * NB * 4 * 2;
  static constexpr int W_B = OWN * NB * 4 * 2;
  static constexpr int SMEM = OWN_T * OWN_B + DIR_T * DIR_B + TR_T * TR_B + W_B + 1024;
  // TMEM: scores [0, NB) (+ dP [NB, 2 NB)), then one or two 64-column accumulators
  static constexpr int ACC0 = MODE == FWD ? NB : 2 * NB;
  static constexpr int TMEM_COLS = MODE == DKV ? 256 : 128;
};

// 8 consecutive fp32 (K index k, k % 8 == 0) of row r of a K-major SWIZZLE_128B tile of R rows, as TF32 (hi, lo)
__device__ __forceinline__ void put8(uint8_t* hi, uint8_t* lo, int R, int r, int k, const float* v) {
  const uint32_t o0 = (uint32_t)((k >> 5) * R * ROW_B) + sw_off(r, (k & 31) >> 2);
  const uint32_t o1 = (uint32_t)((k >> 5) * R * ROW_B) + sw_off(r, ((k & 31) >> 2) + 1);
  float h[8], l[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) split_tf32(v[i], h[i], l[i]);
  *reinterpret_cast<float4*>(hi + o0) = make_float4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<float4*>(lo + o0) = make_float4(l[0], l[1], l[2], l[3]);
  *reinterpret_cast<float4*>(hi + o1) = make_float4(h[4], h[5], h[6], h[7]);
  *reinterpret_cast<float4*>(lo + o1) = make_float4(l[4], l[5], l[6], l[7]);
}
// one fp32 at (row r, K index k) of a K-major SWIZZLE_128B tile of R rows
__device__ __forceinline__ void put1(uint8_t* hi, uint8_t* lo, int R, int r, int k, float v) {
  const uint32_t o = (uint32_t)((k >> 5) * R * ROW_B) + sw_off(r, (k & 31) >> 2) + ((k & 3) << 2);
  float h, l;
  split_tf32(v, h, l);
  *reinterpret_cast<float*>(hi + o) = h;
  *reinterpret_cast<float*>(lo + o) = l;
}

// `rows` rows of D floats (row j at src + j * stride) scaled by `sc`: as they lie into (dhi, dlo) [rows x D] and, if thi,
// transposed into (thi, tlo) [D x rows]
__device__ __forceinline__ void stage(const float* __restrict__ src, size_t stride, int rows, float sc, uint8_t* dhi,
                                      uint8_t* dlo, uint8_t* thi, uint8_t* tlo) {
  for (int i = threadIdx.x; i < rows * (D / 8); i += OWN) {
    const int r = i >> 3, k = (i & 7) * 8;
    const float4* g = reinterpret_cast<const float4*>(src + (size_t)r * stride + k);
    const float4 a = __ldg(g), c = __ldg(g + 1);
    const float v[8] = {a.x * sc, a.y * sc, a.z * sc, a.w * sc, c.x * sc, c.y * sc, c.z * sc, c.w * sc};
    if (dhi) put8(dhi, dlo, rows, r, k, v);
    if (thi) {
#pragma unroll
      for (int u = 0; u < 8; ++u) put1(thi, tlo, D, k + u, r, v[u]);
    }
  }
}

// D[128 x N] (+)= A[128 x K] B[N x K]^T, both (hi, lo) K-major tiles, three TF32 MMAs per 8-wide K step (issued by the
// whole warp, the instruction predicated on the elected lane)
__device__ __forceinline__ void mma3(uint32_t tmem_d, const uint8_t* a_hi, const uint8_t* a_lo, const uint8_t* b_hi,
                                     const uint8_t* b_lo, int N, int K, bool accumulate, uint32_t leader) {
  const uint32_t idesc = make_idesc(N);
#pragma unroll 1
  for (int kb = 0; kb < K / 32; ++kb) {
    const uint64_t ah = make_smem_desc(smem_u32(a_hi + kb * OWN * ROW_B)), al = make_smem_desc(smem_u32(a_lo + kb * OWN * ROW_B));
    const uint64_t bh = make_smem_desc(smem_u32(b_hi + kb * N * ROW_B)), bl = make_smem_desc(smem_u32(b_lo + kb * N * ROW_B));
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint64_t ko = (uint64_t)(ks * 2);          // 32 bytes per K = 8 step, in 16-byte units
      umma_elect<false>(tmem_d, ah + ko, bh + ko, idesc, (accumulate || kb || ks) ? 1u : 0u, leader);
      umma_elect<false>(tmem_d, al + ko, bh + ko, idesc, 1u, leader);
      umma_elect<false>(tmem_d, ah + ko, bl + ko, idesc, 1u, leader);
    }
  }
}

struct Params {
  const float* qkv;          // [B, S, 3C] rows (k | v | q)
  const float* out;          // FWD: written; backward: the forward's output
  const float* dout;         // [B, S, C]
  float* out_w;              // FWD: out
  float* lse;                // [B * heads, S]
  float* dqkv;               // [B, S, 3C]
  const unsigned* seed_dev;
  unsigned salt;
  uint32_t thresh;
  float inv_keep, scale;
  int S, C, heads;
};

template <int MODE>
__global__ void __launch_bounds__(OWN, 1) attn_train_tc_kernel(const Params p) {
  using CF = Cfg<MODE>;
  constexpr int NB = CF::NB;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar_s, bar_o, bar_k;
  __shared__ uint32_t tmem_slot;
  __shared__ int failed_flag;
  __shared__ float blk_lse[NB], blk_delta[NB];
  volatile int* failed = &failed_flag;

  const int tid = threadIdx.x, warp = tid >> 5;
  const int pair = blockIdx.x, b = pair / p.heads, h = pair - b * p.heads;
  const int S = p.S, C = p.C, rs = 3 * C;
  const int row0 = blockIdx.y * OWN, row = row0 + tid;
  const float* base = p.qkv + (size_t)b * S * rs + h * D;               // k at +0, v at +C, q at +2C
  const float* gbase = p.dout + (size_t)b * S * C + h * D;
  const uint32_t seed = layer_seed(p.seed_dev, p.salt);

  uint8_t* own_hi[2];
  uint8_t* own_lo[2];
  uint8_t* dir_hi[2];
  uint8_t* dir_lo[2];
  uint8_t* tr_hi[2];
  uint8_t* tr_lo[2];
  uint8_t* cur = smem;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    own_hi[i] = i < CF::OWN_T ? cur : nullptr; own_lo[i] = i < CF::OWN_T ? cur + CF::OWN_B / 2 : nullptr;
    if (i < CF::OWN_T) cur += CF::OWN_B;
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    dir_hi[i] = i < CF::DIR_T ? cur : nullptr; dir_lo[i] = i < CF::DIR_T ? cur + CF::DIR_B / 2 : nullptr;
    if (i < CF::DIR_T) cur += CF::DIR_B;
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    tr_hi[i] = i < CF::TR_T ? cur : nullptr; tr_lo[i] = i < CF::TR_T ? cur + CF::TR_B / 2 : nullptr;
    if (i < CF::TR_T) cur += CF::TR_B;
  }
  uint8_t* w_hi = cur;
  uint8_t* w_lo = cur + CF::W_B / 2;

  if (tid == 0) {
    failed_flag = 0;
    mbar_init(&bar_s, 1);
    mbar_init(&bar_o, 1);
    mbar_init(&bar_k, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_slot, (uint32_t)CF::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);
  const uint32_t leader = warp == 0 ? elect_one() : 0u;

  // ---- own rows: FWD / DQ: Q' (and dO); DKV: K, V ----
  if constexpr (MODE == DKV) {
    stage(base + (size_t)row0 * rs, rs, OWN, 1.f, own_hi[0], own_lo[0], nullptr, nullptr);
    stage(base + (size_t)row0 * rs + C, rs, OWN, 1.f, own_hi[1], own_lo[1], nullptr, nullptr);
  } else {
    stage(base + (size_t)row0 * rs + 2 * C, rs, OWN, p.scale, own_hi[0], own_lo[0], nullptr, nullptr);
    if (MODE == DQ) stage(gbase + (size_t)row0 * C, C, OWN, 1.f, own_hi[1], own_lo[1], nullptr, nullptr);
  }
  // per-row state of the query modes: lse and delta (DQ), running max / sum / output (FWD)
  float L = 0.f, delta = 0.f, mx = -INFINITY, lsum = 0.f;
  float o[MODE == FWD ? D : 1];
  if constexpr (MODE == FWD) {
#pragma unroll
    for (int i = 0; i < D; ++i) o[i] = 0.f;
  }
  if constexpr (MODE == DQ) {
    L = __ldg(p.lse + (size_t)pair * S + row);
    const float4* po = reinterpret_cast<const float4*>(p.out + (size_t)(b * S + row) * C + h * D);
    const float4* pg = reinterpret_cast<const float4*>(gbase + (size_t)row * C);
#pragma unroll 4
    for (int v4 = 0; v4 < D / 4; ++v4) {
      const float4 a = __ldg(po + v4), g = __ldg(pg + v4);
      delta += a.x * g.x + a.y * g.y + a.z * g.z + a.w * g.w;
    }
  }

  const int nblk = S / NB;
  for (int blk = 0; blk < nblk; ++blk) {
    const int j0 = blk * NB;
    const uint32_t ph = (uint32_t)(blk & 1);
    // ---- stage the block (the previous block's MMAs have retired: every thread waited for them) ----
    if constexpr (MODE == FWD) {
      stage(base + (size_t)j0 * rs, rs, NB, 1.f, dir_hi[0], dir_lo[0], nullptr, nullptr);              // K
      stage(base + (size_t)j0 * rs + C, rs, NB, 1.f, nullptr, nullptr, tr_hi[0], tr_lo[0]);            // V^T
    } else if constexpr (MODE == DQ) {
      stage(base + (size_t)j0 * rs, rs, NB, 1.f, dir_hi[0], dir_lo[0], tr_hi[0], tr_lo[0]);            // K, K^T
      stage(base + (size_t)j0 * rs + C, rs, NB, 1.f, dir_hi[1], dir_lo[1], nullptr, nullptr);          // V
    } else {
      stage(base + (size_t)j0 * rs + 2 * C, rs, NB, p.scale, dir_hi[0], dir_lo[0], tr_hi[0], tr_lo[0]); // Q', Q'^T
      stage(gbase + (size_t)j0 * C, C, NB, 1.f, dir_hi[1], dir_lo[1], tr_hi[1], tr_lo[1]);             // dO, dO^T
      if (tid < NB) blk_lse[tid] = __ldg(p.lse + (size_t)pair * S + j0 + tid);
      // delta of the block's queries: four threads per row, a fixed reduction order
      {
        const int r = tid >> 2, part = tid & 3;
        const float4* po = reinterpret_cast<const float4*>(p.out + (size_t)(b * S + j0 + r) * C + h * D);
        const float4* pg = reinterpret_cast<const float4*>(gbase + (size_t)(j0 + r) * C);
        float acc = 0.f;
#pragma unroll
        for (int v4 = part; v4 < D / 4; v4 += 4) {
          const float4 a = __ldg(po + v4), g = __ldg(pg + v4);
          acc += a.x * g.x + a.y * g.y + a.z * g.z + a.w * g.w;
        }
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        if (part == 0) blk_delta[r] = acc;
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();

    // ---- score MMAs: S [0, NB) (+ dP [NB, 2 NB)) ----
    if (warp == 0) {
      tc_fence_after();
      mma3(tmem, own_hi[0], own_lo[0], dir_hi[0], dir_lo[0], NB, D, false, leader);
      if constexpr (MODE != FWD) mma3(tmem + NB, own_hi[1], own_lo[1], dir_hi[1], dir_lo[1], NB, D, false, leader);
      umma_commit_elect(&bar_s, leader);
    }
    mbar_wait(&bar_s, ph, failed);
    tc_fence_after();

    float s[NB];
    if constexpr (MODE == FWD) {
      tmem_ld32(tlane, s);
      tmem_ld32(tlane + 32, s + 32);
      float m = mx;
#pragma unroll
      for (int j = 0; j < NB; ++j) m = fmaxf(m, s[j]);
      const float corr = __expf(mx - m);
      mx = m;
      lsum *= corr;
#pragma unroll
      for (int i = 0; i < D; ++i) o[i] *= corr;
#pragma unroll
      for (int j = 0; j < NB; ++j) {
        s[j] = __expf(s[j] - m);
        lsum += s[j];
        s[j] *= drop_scale(seed, pair, row, j0 + j, S, p.thresh, p.inv_keep);
      }
#pragma unroll
      for (int j = 0; j < NB; j += 8) put8(w_hi, w_lo, OWN, tid, j, s + j);
      fence_proxy_async();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        mma3(tmem + CF::ACC0, w_hi, w_lo, tr_hi[0], tr_lo[0], D, NB, false, leader);     // O_b = Pd V
        umma_commit_elect(&bar_o, leader);
      }
      mbar_wait(&bar_o, ph, failed);
      tc_fence_after();
      float ob[32];
      tmem_ld32(tlane + CF::ACC0, ob);
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] += ob[i];
      tmem_ld32(tlane + CF::ACC0 + 32, ob);
#pragma unroll
      for (int i = 0; i < 32; ++i) o[32 + i] += ob[i];
    } else {
      float dp[NB];
      tmem_ld32(tlane, s);
      tmem_ld32(tlane + NB, dp);
      if constexpr (MODE == DQ) {
#pragma unroll
        for (int j = 0; j < NB; ++j)
          s[j] = __expf(s[j] - L) * (dp[j] * drop_scale(seed, pair, row, j0 + j, S, p.thresh, p.inv_keep) - delta);
#pragma unroll
        for (int j = 0; j < NB; j += 8) put8(w_hi, w_lo, OWN, tid, j, s + j);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
          tc_fence_after();
          mma3(tmem + CF::ACC0, w_hi, w_lo, tr_hi[0], tr_lo[0], D, NB, blk > 0, leader);   // dQ += dS K
          umma_commit_elect(&bar_o, leader);
        }
        mbar_wait(&bar_o, ph, failed);
        tc_fence_after();
      } else {
        // thread = key `row`; column j = query j0 + j
#pragma unroll
        for (int j = 0; j < NB; ++j) {
          const float m = drop_scale(seed, pair, j0 + j, row, S, p.thresh, p.inv_keep);
          const float pj = __expf(s[j] - blk_lse[j]);
          s[j] = pj * m;                                          // Pd^T
          dp[j] = pj * (dp[j] * m - blk_delta[j]);               // dS^T
        }
#pragma unroll
        for (int j = 0; j < NB; j += 8) put8(w_hi, w_lo, OWN, tid, j, s + j);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
          tc_fence_after();
          mma3(tmem + CF::ACC0, w_hi, w_lo, tr_hi[1], tr_lo[1], D, NB, blk > 0, leader);   // dV += Pd^T dO
          umma_commit_elect(&bar_o, leader);
        }
        mbar_wait(&bar_o, ph, failed);
        tc_fence_after();
#pragma unroll
        for (int j = 0; j < NB; j += 8) put8(w_hi, w_lo, OWN, tid, j, dp + j);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
          tc_fence_after();
          mma3(tmem + CF::ACC0 + D, w_hi, w_lo, tr_hi[0], tr_lo[0], D, NB, blk > 0, leader);   // dK += dS^T Q'
          umma_commit_elect(&bar_k, leader);
        }
        mbar_wait(&bar_k, ph, failed);
        tc_fence_after();
      }
    }
    tc_fence_before();
    __syncthreads();                                   // every thread is past this block's MMAs: its buffers may be restaged
  }

  // ---- epilogue ----
  const bool bad = *failed != 0;
  const float nan = __int_as_float(0x7fc00000);
  if constexpr (MODE == FWD) {
    const float inv = 1.f / lsum;
    p.lse[(size_t)pair * S + row] = bad ? nan : mx + logf(lsum);
    float4* dst = reinterpret_cast<float4*>(p.out_w + (size_t)(b * S + row) * C + h * D);
#pragma unroll
    for (int i = 0; i < D / 4; ++i)
      dst[i] = bad ? make_float4(nan, nan, nan, nan)
                   : make_float4(o[4 * i] * inv, o[4 * i + 1] * inv, o[4 * i + 2] * inv, o[4 * i + 3] * inv);
  } else {
    float* drow = p.dqkv + (size_t)(b * S + row) * rs + h * D;
#pragma unroll
    for (int part = 0; part < (MODE == DQ ? 1 : 2); ++part) {
      // DQ: dQ -> columns 2C + h D (times 1/sqrt d); DKV: dV -> C + h D, dK -> h D
      float4* dst = reinterpret_cast<float4*>(drow + (MODE == DQ ? 2 * C : (part == 0 ? C : 0)));
      const float sc = MODE == DQ ? p.scale : 1.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float v[32];
        tmem_ld32(tlane + CF::ACC0 + part * D + half * 32, v);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          dst[half * 8 + i] = bad ? make_float4(nan, nan, nan, nan)
                                  : make_float4(v[4 * i] * sc, v[4 * i + 1] * sc, v[4 * i + 2] * sc, v[4 * i + 3] * sc);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, (uint32_t)CF::TMEM_COLS);
}

// argument checks of both entry points; fills the launch constants
static int plan(const float* const* ptrs, int nptrs, float p_drop, int B, int S, int C, int heads, Params* p) {
  for (int i = 0; i < nptrs; ++i)
    if (!ptrs[i]) return FLOWK_ERR_ARG;
  if (B < 1 || heads < 1 || C % heads || C / heads != D || (S != 128 && S != 256)) return FLOWK_ERR_SHAPE;
  if (!(p_drop >= 0.f) || p_drop >= 1.f) return FLOWK_ERR_SHAPE;
  if ((long long)B * heads * S * S >= 0xffffffffLL) return FLOWK_ERR_SHAPE;     // the mask counter is 32 bits
  p->thresh = (uint32_t)((double)p_drop * 4294967296.0);
  p->inv_keep = 1.f / (1.f - p_drop);
  p->scale = 1.f / sqrtf((float)D);
  p->S = S;
  p->C = C;
  p->heads = heads;
  return FLOWK_OK;
}

template <int MODE>
static int launch(const Params& p, int B, cudaStream_t st) {
  const int smem = Cfg<MODE>::SMEM;
  FLOWK_CUDA_OK(cudaFuncSetAttribute(attn_train_tc_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  attn_train_tc_kernel<MODE><<<dim3(B * p.heads, p.S / OWN), OWN, smem, st>>>(p);
  return launch_status();
}

}  // namespace attn_train_tc
}  // namespace flowk

using namespace flowk;
using namespace flowk::attn_train_tc;

extern "C" int flowk_attention_train_tc_fwd(const float* qkv, float* out, float* lse, const unsigned* seed_device, unsigned salt,
                                            float p_drop, int B, int HW, int C, int heads, flowk_stream_t stream) {
  if (B == 0) return FLOWK_OK;
  const float* ptrs[3] = {qkv, out, lse};
  Params p{};
  const int rc = plan(ptrs, 3, p_drop, B, HW, C, heads, &p);
  if (rc != FLOWK_OK) return rc;
  p.qkv = qkv;
  p.out_w = out;
  p.lse = lse;
  p.seed_dev = seed_device;
  p.salt = salt;
  return launch<FWD>(p, B, stream);
}

// which: 1 = query side (dq columns of dqkv), 2 = key side (dk, dv columns), 3 = both on `stream`
extern "C" int flowk_attention_train_tc_bwd(int which, const float* qkv, const float* out, const float* dout, const float* lse,
                                            float* dqkv, const unsigned* seed_device, unsigned salt, float p_drop, int B, int HW,
                                            int C, int heads, flowk_stream_t stream) {
  if (B == 0) return FLOWK_OK;
  if (which < 1 || which > 3) return FLOWK_ERR_ARG;
  const float* ptrs[5] = {qkv, out, dout, lse, dqkv};
  Params p{};
  const int rc = plan(ptrs, 5, p_drop, B, HW, C, heads, &p);
  if (rc != FLOWK_OK) return rc;
  p.qkv = qkv;
  p.out = out;
  p.dout = dout;
  p.lse = const_cast<float*>(lse);
  p.dqkv = dqkv;
  p.seed_dev = seed_device;
  p.salt = salt;
  if (which & 1) {
    const int r = launch<DQ>(p, B, stream);
    if (r != FLOWK_OK) return r;
  }
  if (which & 2) return launch<DKV>(p, B, stream);
  return FLOWK_OK;
}
