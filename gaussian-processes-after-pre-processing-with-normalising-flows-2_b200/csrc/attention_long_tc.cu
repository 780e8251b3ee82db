// Self-attention core of GatedAttn (flow_modules/mixlogcdf_nn.py:134-147) on the 5th-gen tensor cores, inference, for long
// sequences: the level-1 maps of 64x64 images (seq = 32 * 32 = 1024 tokens) and longer.
//
//   att[q, :] = softmax_k(q . k / sqrt(d)) v        per (image, head); seq = H*W a multiple of 128, >= 512; d in {24, 32, 40, 64}
//
// attention_tc.cu stages the whole K and V^T of an (image, head) in shared memory, which stops at 256 keys.  Here one CTA owns
// one 128-query tile of one (image, head) and streams the keys in 128-key blocks:
//   1. stage Q_t (pre-scaled by log2(e) / sqrt(d)), K_0 and V_0^T as fp16 (hi, lo) operand tiles, K-major SWIZZLE_128B (the
//      layouts of attention_tc_kernel); the head dim is zero-padded to dk = ceil16(d);
//   2. per key block b:
//      a. S_b = Q_t K_b^T (tcgen05.mma kind::f16, M = 128, N = 128, three products Qh Kh + Ql Kh + Qh Kl) into TMEM [0, 128);
//      b. softmax of the block with its own row maximum m_b: p = 2^(s - m_b) goes back into the same TMEM columns as packed
//         fp16, the TS-mode A operand of O_b (as in attention_tc_v2_kernel); row sum l_b.  Keys [16 j, 16 j + 16) of the
//         block: hi in columns [16 j, 16 j + 8), lo in [16 j + 8, 16 j + 16), i.e. over the S columns of those same keys, so
//         a thread only overwrites scores it has read itself (the thread sharing its row still reads the other 64 columns);
//      c. O_b = P_b V_b (N = dk, the three products again) into TMEM [128, 128 + dk) while the threads stage K_{b+1} over the
//         K tile S_b no longer needs;
//      d. the threads fold O_b into the running output in registers, o = o 2^(m - m') + O_b 2^(m_b - m'), l alike, with
//         m' = max(m, m_b) (the fold of attention_train_tc.cu's FWD mode), then S_{b+1} is issued and V_{b+1} staged over
//         V_b under it;
//   3. epilogue: o / l -> the (hi, lo) operand pair of the attention-gate GEMM (fp16, or TF32 values in fp32 containers).
// The query tile is the fastest grid index, so the tiles of one (image, head) run side by side and read its K and V from
// L2.  256 threads (2 per score row, 64 keys of a block each), 256 TMEM columns and <= 97 KB of shared memory: two CTAs
// share an SM, and each one's softmax runs under the other's MMAs.  Nothing of size seq x seq touches HBM; no atomics, and
// the blocks are folded in key order, so two calls give the same bits.
#include <cuda.h>
#include "common.cuh"
#include "umma.cuh"
#include "attention_tile.cuh"

namespace flowk {
namespace tc {

constexpr int LONG_THREADS = 256;               // 8 warps: warps w and w + 4 share TMEM lanes 32 (w % 4) .. +31, 64 keys each
constexpr int LONG_TMEM_COLS = 256;             // S / P [0, 128), O_b [128, 128 + dk)
constexpr int LONG_TILE_B = 128 * ROW_B;        // one 128-row K-major operand tile (hi or lo)

struct LongAttParams {
  const float* qkv;         // [B*HW, 3C], columns (k | v | q)
  float* out_hi;            // [B*HW, C] operand pair (fp16 when out_f16, else TF32 values in fp32 containers)
  float* out_lo;
  int out_f16;
  int HW, C, heads, D;      // D = C / heads
  float qscale;             // log2(e) / sqrt(D)
  int* status;
  long long* trace;         // optional device [3]: clock64 stamps of CTA 0 (start, after the key loop, end), NULL in production
};

template <int KCH>           // KCH = dk / 8: 16-byte chunks per staged Q / K row (4, 6 or 8)
__global__ void __launch_bounds__(LONG_THREADS, 2) attention_long_tc_kernel(const LongAttParams p) {
  constexpr int DK = KCH * 8;
  constexpr int VT_TILE = 2 * DK * ROW_B;       // one 64-key block of V^T: [DK rows of hi | DK rows of lo][128 B]
  constexpr int OCH = (KCH + 1) / 2;            // output chunks per thread: chunks half, half + 2, ...
  constexpr int BATCH = KCH == 8 ? 1 : 2;        // staging items (2 x 16 B loads) in flight per thread: what the registers beside o allow
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar_s, bar_o;
  __shared__ uint32_t tmem_slot;
  __shared__ int failed_flag;
  __shared__ float red_max[2][128], red_sum[2][128];
  volatile int* failed = &failed_flag;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int HW = p.HW, D = p.D, C = p.C, row_stride = 3 * C;
  const int tiles = HW >> 7, nblocks = tiles;
  const int pair = blockIdx.x / tiles, t = blockIdx.x - pair * tiles;
  const int b = pair / p.heads, h = pair - b * p.heads;
  const int chunks = D >> 3;                    // 16-byte chunks of real data per row (the rest up to KCH are zero)

  if (threadIdx.x == 0) {
    failed_flag = 0;
    mbar_init(&bar_s, 1);
    mbar_init(&bar_o, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_slot, (uint32_t)LONG_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const bool tracing = p.trace && blockIdx.x == 0 && threadIdx.x == 0;
  griddep_launch();
  griddep_wait();                               // the in_proj GEMM's rows are complete from here on
  if (tracing) p.trace[0] = clock64();

  uint8_t* q_hi = smem;                         // [128 rows][128 B] each, SWIZZLE_128B
  uint8_t* q_lo = q_hi + LONG_TILE_B;
  uint8_t* k_hi = q_lo + LONG_TILE_B;
  uint8_t* k_lo = k_hi + LONG_TILE_B;
  uint8_t* v_t = k_lo + LONG_TILE_B;            // [2 blocks of 64 keys][VT_TILE]
  const float* base = p.qkv + (size_t)b * HW * row_stride + h * D;

  // 128 rows of Q (col = 2C, scaled) or K (col = 0) of rows [r0, r0 + 128): K-major rows, chunks >= `chunks` zero
  auto stage_rows = [&](int r0, int col, float sc, uint8_t* dst_hi, uint8_t* dst_lo) {
    constexpr int ITEMS = 128 * KCH / LONG_THREADS;   // KCH / 2 per thread, in batches of BATCH: loads, then convert and store
#pragma unroll
    for (int u0 = 0; u0 < ITEMS; u0 += BATCH) {
    float4 a[BATCH], c[BATCH];
#pragma unroll
    for (int u = 0; u < BATCH && u0 + u < ITEMS; ++u) {
      const int i = threadIdx.x + (u0 + u) * LONG_THREADS, r = i / KCH, ch = i % KCH;
      a[u] = c[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ch < chunks) {
        const float4* g = reinterpret_cast<const float4*>(base + (size_t)(r0 + r) * row_stride + col + ch * 8);
        a[u] = __ldg(g);
        c[u] = __ldg(g + 1);
      }
    }
#pragma unroll
    for (int u = 0; u < BATCH && u0 + u < ITEMS; ++u) {
      const int i = threadIdx.x + (u0 + u) * LONG_THREADS, r = i / KCH, ch = i % KCH;
      const float v[8] = {a[u].x * sc, a[u].y * sc, a[u].z * sc, a[u].w * sc, c[u].x * sc, c[u].y * sc, c[u].z * sc, c[u].w * sc};
      uint4 hi, lo;
      cvt8(v, hi, lo);
      *reinterpret_cast<uint4*>(dst_hi + sw_off(r, ch)) = hi;
      *reinterpret_cast<uint4*>(dst_lo + sw_off(r, ch)) = lo;
    }
    }
  };
  // V^T of keys [k0, k0 + 128): rows = head dims (zero past D), the keys along the 128-byte rows; consecutive threads take
  // consecutive keys
  auto stage_vt = [&](int k0) {
    constexpr int ITEMS = 128 * KCH / LONG_THREADS;
#pragma unroll
    for (int u0 = 0; u0 < ITEMS; u0 += BATCH) {
    float4 a[BATCH], c[BATCH];
#pragma unroll
    for (int u = 0; u < BATCH && u0 + u < ITEMS; ++u) {
      const int i = threadIdx.x + (u0 + u) * LONG_THREADS, key = i & 127, ch = i >> 7;
      a[u] = c[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ch < chunks) {
        const float4* g = reinterpret_cast<const float4*>(base + (size_t)(k0 + key) * row_stride + C + ch * 8);
        a[u] = __ldg(g);
        c[u] = __ldg(g + 1);
      }
    }
#pragma unroll
    for (int u = 0; u < BATCH && u0 + u < ITEMS; ++u) {
      const int i = threadIdx.x + (u0 + u) * LONG_THREADS, key = i & 127, ch = i >> 7;
      const float v[8] = {a[u].x, a[u].y, a[u].z, a[u].w, c[u].x, c[u].y, c[u].z, c[u].w};
      uint8_t* tile = v_t + (key >> 6) * VT_TILE;
      const int kk = key & 63;
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const int dim = ch * 8 + jj;
        unsigned short hh, ll;
        split_f16(v[jj], hh, ll);
        *reinterpret_cast<unsigned short*>(tile + sw_off(dim, kk >> 3) + ((kk & 7) << 1)) = hh;
        *reinterpret_cast<unsigned short*>(tile + sw_off(DK + dim, kk >> 3) + ((kk & 7) << 1)) = ll;
      }
    }
    }
  };

  // ---- 1. Q_t, K_0, V_0^T ----------------------------------------------------------------------------------------------
  stage_rows(t * 128, 2 * C, p.qscale, q_hi, q_lo);
  stage_rows(0, 0, 1.f, k_hi, k_lo);
  stage_vt(0);
  fence_proxy_async();                          // generic-proxy smem writes -> visible to the tensor core
  __syncthreads();

  const uint32_t leader = warp == 0 ? elect_one() : 0u;
  auto issue_s = [&]() {                        // warp 0: S = Q_t K^T into columns [0, 128)
    tc_fence_after();
    const uint32_t idesc = make_idesc_f16(128);
    const uint64_t dq_hi = make_smem_desc(smem_u32(q_hi)), dq_lo = make_smem_desc(smem_u32(q_lo));
    const uint64_t dk_hi = make_smem_desc(smem_u32(k_hi)), dk_lo = make_smem_desc(smem_u32(k_lo));
#pragma unroll
    for (int ks = 0; ks < DK / 16; ++ks) {
      const uint64_t ko = (uint64_t)(ks * 2);   // 32 bytes per K = 16 step, in 16-byte units
      umma_elect<true>(tmem_base, dq_hi + ko, dk_hi + ko, idesc, ks == 0 ? 0u : 1u, leader);
      umma_elect<true>(tmem_base, dq_lo + ko, dk_hi + ko, idesc, 1u, leader);
      umma_elect<true>(tmem_base, dq_hi + ko, dk_lo + ko, idesc, 1u, leader);
    }
    umma_commit_elect(&bar_s, leader);
  };
  if (warp == 0) issue_s();

  const int lane_grp = warp & 3, half = warp >> 2;
  const int row = lane_grp * 32 + lane;
  const uint32_t lane_addr = tmem_base + ((uint32_t)(lane_grp * 32) << 16);
  float o[OCH][8];
  float m = 0.f, l = 0.f;
#pragma unroll
  for (int j = 0; j < OCH; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i) o[j][i] = 0.f;

#pragma unroll 1
  for (int kb = 0; kb < nblocks; ++kb) {
    // ---- 2b. block maximum of this thread's 64 scores, then p = 2^(s - m_b) as packed fp16 (hi, lo) into S_b's columns
    mbar_wait(&bar_s, (uint32_t)(kb & 1), failed);
    tc_fence_after();
    float mx = -INFINITY;
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {
      float s[16];
      tmem_ld16(lane_addr + (uint32_t)(half * 64 + g * 16), s);
#pragma unroll
      for (int i = 0; i < 16; ++i) mx = fmaxf(mx, s[i]);
    }
    red_max[half][row] = mx;
    tc_fence_before();                          // every load of S_b is complete before anyone writes P over it
    __syncthreads();
    tc_fence_after();
    const float mb = fmaxf(red_max[0][row], red_max[1][row]);
    float sum = 0.f;
#pragma unroll 1
    for (int g = 0; g < 4; ++g) {               // keys 64 half + 16 g + [0, 16): hi over the first 8 of their 16 S columns, lo over the rest
      float s[16];
      tmem_ld16(lane_addr + (uint32_t)(half * 64 + g * 16), s);
      uint32_t ph[8], pl[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float e0 = ex2_fast(s[2 * i] - mb), e1 = ex2_fast(s[2 * i + 1] - mb);
        sum += e0 + e1;
        ph[i] = pack_h2(e0, e1);
        float a0, a1;
        unpack_h2(ph[i], a0, a1);
        pl[i] = pack_h2(e0 - a0, e1 - a1);
      }
      const uint32_t col = (uint32_t)(half * 64 + g * 16);   // only columns this thread has read: the other half still reads
      tmem_st8u(lane_addr + col, ph);
      tmem_st8u(lane_addr + col + 8, pl);
    }
    red_sum[half][row] = sum;
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    const float lb = red_sum[0][row] + red_sum[1][row];

    // ---- 2c. O_b = P_hi V_hi + P_lo V_hi + P_hi V_lo (N = dk, K = 128 keys); K_{b+1} is staged under it
    if (warp == 0) {
      tc_fence_after();
      const uint32_t idesc = make_idesc_f16(DK);
      const uint32_t d = tmem_base + 128u;
#pragma unroll
      for (int j = 0; j < 8; ++j) {             // K = 16 keys per step: 8 packed columns of P, 32 bytes of a V^T row
        const uint8_t* vb = v_t + (j >> 2) * VT_TILE;
        const uint64_t ko = (uint64_t)((j & 3) * 2);
        const uint64_t dv_hi = make_smem_desc(smem_u32(vb)) + ko, dv_lo = make_smem_desc(smem_u32(vb + DK * ROW_B)) + ko;
        const uint32_t a_hi = tmem_base + (uint32_t)(j * 16), a_lo = a_hi + 8u;
        umma_f16_ts_elect(d, a_hi, dv_hi, idesc, j == 0 ? 0u : 1u, leader);
        umma_f16_ts_elect(d, a_lo, dv_hi, idesc, 1u, leader);
        umma_f16_ts_elect(d, a_hi, dv_lo, idesc, 1u, leader);
      }
      umma_commit_elect(&bar_o, leader);
    }
    const bool more = kb + 1 < nblocks;
    if (more) stage_rows((kb + 1) * 128, 0, 1.f, k_hi, k_lo);   // S_b has retired: K_b is dead

    // ---- 2d. fold O_b into the running output (thread: row `row`, chunks half, half + 2, ...)
    mbar_wait(&bar_o, (uint32_t)(kb & 1), failed);
    tc_fence_after();
    const float mn = kb == 0 ? mb : fmaxf(m, mb);
    const float wa = kb == 0 ? 0.f : ex2_fast(m - mn), wb = ex2_fast(mb - mn);
    m = mn;
    l = l * wa + lb * wb;
#pragma unroll
    for (int j = 0; j < OCH; ++j) {
      const int ch = half + 2 * j;
      if (ch < chunks) {
        float ob[8];
        tmem_ld8(lane_addr + 128u + (uint32_t)(ch * 8), ob);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[j][i] = o[j][i] * wa + ob[i] * wb;
      }
    }
    if (more) fence_proxy_async();              // K_{b+1}
    tc_fence_before();                          // O_b's loads are complete before O_{b+1} overwrites it
    __syncthreads();
    if (more) {
      if (warp == 0) issue_s();                 // P_b has been read (O_b retired): S_{b+1} may overwrite it
      stage_vt((kb + 1) * 128);                 // O_b has retired: V_b is dead
      fence_proxy_async();                      // V_{b+1}: visible to the tensor core after the next block's barriers
    }
  }
  if (tracing) p.trace[1] = clock64();

  // ---- 3. epilogue: o / l -> operand pair
  const float inv = 1.0f / l;
  const size_t o0 = ((size_t)b * HW + t * 128 + row) * C + (size_t)h * D;
#pragma unroll
  for (int j = 0; j < OCH; ++j) {
    const int ch = half + 2 * j;
    if (ch < chunks) {
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = o[j][i] * inv;
      if (p.out_f16) {
        uint4 hi, lo;
        cvt8(v, hi, lo);
        *reinterpret_cast<uint4*>(reinterpret_cast<unsigned short*>(p.out_hi) + o0 + ch * 8) = hi;
        *reinterpret_cast<uint4*>(reinterpret_cast<unsigned short*>(p.out_lo) + o0 + ch * 8) = lo;
      } else {
#pragma unroll
        for (int i = 0; i < 8; i += 2) store_pair(p.out_hi, p.out_lo, o0 + ch * 8 + i, v[i], v[i + 1], 0);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tracing) p.trace[2] = clock64();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)LONG_TMEM_COLS);
  if (threadIdx.x == 0 && failed_flag && p.status) *p.status = 1;
}

}  // namespace tc
}  // namespace flowk

using namespace flowk;
using namespace flowk::tc;

namespace {
template <int KCH>
int attention_long_tc_launch(const LongAttParams& p, int B, cudaStream_t stream) {
  // Q_t (hi, lo), K_b (hi, lo), V_b^T (two 64-key blocks of hi and lo rows) + alignment of the 1024-byte swizzle atoms
  const size_t smem = (size_t)4 * LONG_TILE_B + (size_t)2 * (2 * KCH * 8 * ROW_B) + 1024;
  static size_t smem_set = 0;
  if (smem > smem_set) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(attention_long_tc_kernel<KCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    FLOWK_CUDA_OK(cudaFuncSetAttribute(attention_long_tc_kernel<KCH>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
    smem_set = smem;
  }
  const long long ctas = (long long)B * p.heads * (p.HW / 128);
  FLOWK_CUDA_OK(launch_pdl(attention_long_tc_kernel<KCH>, dim3((unsigned)ctas), dim3(LONG_THREADS), smem, stream, p));
  return launch_status();
}
}  // namespace

// Same arguments and outputs as flowk_attention_tc (include/flowk.h): seq a multiple of 128 and >= 512, C / heads in
// {24, 32, 40, 64}.
extern "C" int flowk_attention_long_tc(const float* qkv, void* out_hi, void* out_lo, int out_f16, int B, int HW, int C,
                                       int heads, int* status, long long* trace, flowk_stream_t stream) {
  if (B < 0 || HW < 512 || HW % 128 || C < 1 || heads < 1 || C % heads) return FLOWK_ERR_SHAPE;
  const int D = C / heads;
  if (D != 24 && D != 32 && D != 40 && D != 64) return FLOWK_ERR_SHAPE;
  if ((long long)B * heads * (HW / 128) > 0x7fffffffLL) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!qkv || !out_hi || !out_lo) return FLOWK_ERR_ARG;
  LongAttParams p{};
  p.qkv = qkv;
  p.out_hi = reinterpret_cast<float*>(out_hi);
  p.out_lo = reinterpret_cast<float*>(out_lo);
  p.out_f16 = out_f16;
  p.HW = HW;
  p.C = C;
  p.heads = heads;
  p.D = D;
  p.qscale = 1.4426950408889634f / sqrtf((float)D);
  p.status = status;
  p.trace = trace;
  switch ((D + 15) / 16) {
    case 2: return attention_long_tc_launch<4>(p, B, stream);
    case 3: return attention_long_tc_launch<6>(p, B, stream);
    default: return attention_long_tc_launch<8>(p, B, stream);
  }
}
