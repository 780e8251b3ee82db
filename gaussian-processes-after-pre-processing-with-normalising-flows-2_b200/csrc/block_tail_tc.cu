// The attention half of a ConvAttnBlock (flow_modules/mixlogcdf_nn.py:81-102, GatedAttn :124-152) in ONE launch for feature
// maps whose images fit whole into a 128-row M tile (H*W <= 128, 128 % (H*W) == 0: cfg2's 8x8 and 4x4 levels), inference:
//
//   x1 = LayerNorm1(GLU(gate(c1)) + x)                               gate: 1x1, K = 2C, N = 2C
//   (k | v | q) = (x1 + pos) W_in^T                                  in_proj: K = C, N = 3C
//   a = softmax(q k^T / sqrt(d)) v        per image and head          block-diagonal over the tile's images
//   x2 = LayerNorm2(GLU(attn_gate(a)) + x1)                           attention gate: K = C, N = 2C
//   out = concat_elu(x2) (or x2 for the last block) as the next layer's fp16 (hi, lo) operand pair, and x2 in fp32
//
// One CTA per 128-row tile; every row attention and the two LayerNorms need is already in the CTA, so x1, q, k, v and the
// attention output never leave the SM.  Phases (serial inside the CTA; the launch has only M / 128 CTAs):
//   1. gate GEMM: the c1 pair (TMA, SWIZZLE_64B, 32-channel slices) x the gate weights streamed through a two-stage ring by a
//      producer warp that runs ahead through all three GEMMs' weights; accumulator in TMEM [0, 2C);
//   2. GLU + bias + x (staged into an fp32 slab in shared memory during step 1), LayerNorm -> x1 (over x in the slab: the
//      residual of step 6) and x1 + pos as the fp16 (hi, lo) A operand of in_proj, in the SWIZZLE_64B layout the MMA reads;
//   3. in_proj GEMM (three-product split, 1 or 2 MMAs of N <= 256) into TMEM [2C, 5C);
//   4. per head (d = 24 or 32, padded to 32): drain q (scaled by log2(e) / sqrt(d)), k, v from TMEM into fp16 pair tiles;
//      S = Q K^T (M = N = 128); a thread owns 32 keys of a row and masks the keys of other images (a 32-key quarter that
//      holds none of its row's image writes zero weights without loading S); P = 2^(s - max) packed into TMEM over S;
//      O = P V (TS-mode MMA); O / rowsum -> the head's columns of the attention gate's A operand pair in shared memory;
//   5. attention-gate GEMM into TMEM [0, 2C);
//   6. GLU + bias + x1, LayerNorm -> x2 (over x1 in the slab), then x2 (fp32 rows) and the next layer's operand pair
//      written out row-contiguously.
// Same numerics as the three launches it replaces: the two-term fp16 split with three products per GEMM, the chained gate's
// GLU / LayerNorm epilogue and the one-wave attention kernel's softmax (csrc/tc_gemm.cu, csrc/attention_tc.cu).
//
// PAIR = true (flowk_block_tail_pair_tc): 16x16 maps, where an image's 256 rows span two tiles.  A cluster of two CTAs per
// image, rank r owning image rows [128 r, 128 r + 128); phases 1-3, 5 and 6 are the per-CTA ones above (the positional
// encoding rows offset by 128 r, no mask: all 256 keys of the image are valid).  Phase 4, per head:
//   * after its drain a CTA also sends the head's K pair and V^T (32 KB, one cp.async.bulk shared::cta -> shared::cluster)
//     into the peer's "remote" buffer, completing on the peer's rfull barrier;
//   * S and P V run over four 64-key blocks, the CTA's own keys 0-63 and 64-127 first (the first S never waits for the
//     peer), then the peer's from the remote buffer.  A dedicated MMA warp keeps two S / P buffers in flight: S_{b+2} is
//     issued into block b's buffer as soon as P_b V has retired, so the softmax of block b runs under P_{b-1} V and
//     S_{b+1}.  Each block has its own row maximum m_b; the compute threads fold O_b into registers as it retires with a
//     running maximum, o = o 2^(m_old - m) + O_b 2^(m_b - m) (the split-key combination of the one-wave attention kernel,
//     applied block by block), which frees O_b's TMEM for P_{b+2} V;
//   * once the P V that read the remote buffer has retired, the CTA arrives on the peer's pempty barrier; a CTA waits
//     there before its next drain (so its bulk copy of the previous head has been read) and before sending a head.
//   TMEM: two S / P buffers [s, s + 64), [s + 64, s + 128) and two O buffers of 32 columns after them, over the drained
//   gate accumulator at C = 96.  Shared memory: the remote buffer lies over the ring stage the attention gate's second
//   weight slice goes to; the producer loads that slice only after the last P V has retired (rfree barrier), the first
//   slice goes to the other stage.  All tcgen05 instructions stay cta_group::1.
#include <cuda.h>
#include "common.cuh"
#include "umma.cuh"
#include "attention_tile.cuh"

namespace flowk {
namespace tc {

constexpr int BT_WARPS = 16;                    // compute warps: 4 per TMEM lane group, a quarter of each row's columns each
// + one TMA producer warp, and (PAIR) one warp that issues the attention's MMAs
constexpr int bt_threads(bool pair) { return 32 * BT_WARPS + (pair ? 64 : 32); }
constexpr int BT_SLICE = 128 * V2_ROW_B;        // one 32-channel slice of a 128-row operand (hi or lo), SWIZZLE_64B: 8 KB
constexpr int BT_DK = 32;                       // head dim padded to the MMA's K = 16 granule (one 64-byte row)
constexpr int BT_VT_B = 2 * BT_DK * ROW_B;      // one 64-key block of V^T: [32 rows of hi | 32 rows of lo][128 B]
constexpr int BT_QKV_B = 4 * BT_SLICE + 2 * BT_VT_B;   // one head's Q pair, K pair and V^T: 48 KB
constexpr int BT_REM_B = 2 * BT_SLICE + 2 * BT_VT_B;   // PAIR: the peer's K pair and V^T of one head: 32 KB

// elu(x) = x > 0 ? x : e^x - 1 and the logistic sigmoid, as the GEMM epilogues of csrc/tc_gemm.cu compute them
__device__ __forceinline__ float bt_elu(float x) { return x > 0.f ? x : ex2_fast(x * kLog2e) - 1.f; }
__device__ __forceinline__ float bt_sigmoid(float x) { return __fdividef(1.f, 1.f + ex2_fast(-x * kLog2e)); }

struct BlockTailParams {
  const float* bias_g;      // gate bias [2C]
  const float* x;           // block input [M, C] fp32 (the residual of the first LayerNorm)
  const float* gamma1;      // LayerNorm 1 [C]
  const float* beta1;
  const float* pos;         // positional encoding [HW, C]
  const float* bias_a;      // attention-gate bias [2C]
  const float* gamma2;      // LayerNorm 2 [C]
  const float* beta2;
  float* x2;                // [M, C] fp32
  uint16_t* out_hi;         // [M, 2C] concat-ELU pair (celu) or [M, C] plain pair, fp16
  uint16_t* out_lo;
  int celu;
  float sc_g, sc_i, sc_a;   // undo the power-of-two pre-scaling of the three weight operands
  float qscale;             // log2(e) / sqrt(d)
  int HW, heads, D;
  int n_ip;                 // in_proj MMA N: 3C in one MMA, or two of 3C / 2 when 3C > 256
  int s_col;                // TMEM column of S / P; O follows at s_col + 128
  int qkv_off, r2_off, ring_off, stage_b, slab_off;   // shared-memory carve (bytes)
  int rem_off, rem_alias;   // PAIR: the remote K / V^T buffer, and whether it lies over a ring stage
  int* status;
  long long* trace;         // optional device [8]: clock64 stamps of CTA 0 (profiling), NULL in production
};

__device__ __forceinline__ void bt_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * BT_WARPS) : "memory"); }
// PAIR: the compute warps and the attention MMA warp, once per head (its q, k and v are drained)
__device__ __forceinline__ void bt_sync_mma() { asm volatile("bar.sync 2, %0;" ::"n"(32 * BT_WARPS + 32) : "memory"); }

template <int NKB, bool PAIR>   // C = 32 NKB channels; PAIR: two-CTA clusters over 256-row images
__global__ void __launch_bounds__(bt_threads(PAIR), 1)
block_tail_tc_kernel(const BlockTailParams p, const __grid_constant__ CUtensorMap map_c1_hi,
                     const __grid_constant__ CUtensorMap map_c1_lo, const __grid_constant__ CUtensorMap map_wg_hi,
                     const __grid_constant__ CUtensorMap map_wg_lo, const __grid_constant__ CUtensorMap map_wi_hi,
                     const __grid_constant__ CUtensorMap map_wi_lo, const __grid_constant__ CUtensorMap map_wa_hi,
                     const __grid_constant__ CUtensorMap map_wa_lo) {
  constexpr int C = 32 * NKB;
  constexpr int NG = 2 * NKB;                   // 32-channel K slices of the gate GEMM (K = 2C)
  constexpr int NSL = NG + 2 * NKB;             // weight slices through the ring: gate, in_proj, attention gate
  constexpr int PITCH = C + 4;                  // x1 slab row pitch (floats): 16-byte shift per row, conflict-free chunks
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar_a, bar_full[2], bar_empty[2], bar_g, bar_i, bar_s[PAIR ? 2 : 1], bar_o[PAIR ? 2 : 1], bar_ag;
  __shared__ uint64_t bar_p[2];                 // PAIR: P of the S / P buffer written (one arrival per compute warp)
  __shared__ uint64_t bar_rfull, bar_pempty, bar_rfree;   // PAIR: remote buffer filled / peer's buffer free / ring stage free
  __shared__ uint32_t tmem_slot;
  __shared__ int failed_flag;
  __shared__ float red[PAIR ? 3 : 2][4][128];   // per-row partials of the four threads that share a row
  volatile int* failed = &failed_flag;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  if (threadIdx.x == 0) {
    failed_flag = 0;
    mbar_init(&bar_a, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_empty[s], 1);
    }
    mbar_init(&bar_g, 1);
    mbar_init(&bar_i, 1);
    for (int s = 0; s < (PAIR ? 2 : 1); ++s) {
      mbar_init(&bar_s[s], 1);
      mbar_init(&bar_o[s], 1);
      if (PAIR) mbar_init(&bar_p[s], BT_WARPS);
    }
    mbar_init(&bar_ag, 1);
    mbar_init(&bar_rfull, 1);
    mbar_init(&bar_pempty, 1);
    mbar_init(&bar_rfree, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_slot, 512u);
  if (warp == BT_WARPS && lane == 0) {
    prefetch_tmap(&map_c1_hi);
    prefetch_tmap(&map_c1_lo);
    prefetch_tmap(&map_wg_hi);
    prefetch_tmap(&map_wg_lo);
    prefetch_tmap(&map_wi_hi);
    prefetch_tmap(&map_wi_lo);
    prefetch_tmap(&map_wa_hi);
    prefetch_tmap(&map_wa_lo);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (PAIR) cluster_sync_all();                 // the peer's barriers are initialised before anything signals them
  const uint32_t tmem = tmem_slot;
  const bool tracing = p.trace && blockIdx.x == 0 && threadIdx.x == 0;
  griddep_launch();
  griddep_wait();                               // the producing launches' outputs are complete from here on
  if (tracing) p.trace[0] = clock64();

  if (warp == BT_WARPS) {
    // ===================== TMA producer: the c1 tile, then every weight slice of the three GEMMs ======================
    if (lane == 0) {
      mbar_expect_tx(&bar_a, (uint32_t)(NG * 2 * BT_SLICE));
      for (int s = 0; s < NG; ++s) {
        tma_load_2d(smem + s * 2 * BT_SLICE, &map_c1_hi, &bar_a, s * 32, tile * 128);
        tma_load_2d(smem + s * 2 * BT_SLICE + BT_SLICE, &map_c1_lo, &bar_a, s * 32, tile * 128);
      }
      for (int g = 0; g < NSL; ++g) {
        const int st = g & 1;
        mbar_wait(&bar_empty[st], (uint32_t)(((g >> 1) & 1) ^ 1), failed);
        if (PAIR && g == NG + NKB + 1 && p.rem_alias) mbar_wait(&bar_rfree, 0, failed);  // the remote buffer's stage
        uint8_t* w = smem + p.ring_off + st * p.stage_b;
        if (g < NG || g >= NG + NKB) {          // gate / attention gate: 2C rows, one box each
          const bool gate = g < NG;
          const int k = gate ? g : g - NG - NKB;
          mbar_expect_tx(&bar_full[st], (uint32_t)(2 * 2 * C * V2_ROW_B));
          tma_load_2d(w, gate ? &map_wg_hi : &map_wa_hi, &bar_full[st], k * 32, 0);
          tma_load_2d(w + 2 * C * V2_ROW_B, gate ? &map_wg_lo : &map_wa_lo, &bar_full[st], k * 32, 0);
        } else {                                // in_proj: 3C rows in boxes of n_ip rows
          const int k = g - NG;
          mbar_expect_tx(&bar_full[st], (uint32_t)(2 * 3 * C * V2_ROW_B));
          for (int r = 0; r < 3 * C; r += p.n_ip) {
            tma_load_2d(w + r * V2_ROW_B, &map_wi_hi, &bar_full[st], k * 32, r);
            tma_load_2d(w + (3 * C + r) * V2_ROW_B, &map_wi_lo, &bar_full[st], k * 32, r);
          }
        }
      }
    }
  } else if (PAIR && warp == BT_WARPS + 1) {
    // ===================== PAIR: phase 4's MMAs, per head over four 64-key blocks b (own 0-63, 64-127, peer's 0-63, 64-127)
    // S_b = Q K_b^T -> S / P buffer b & 1 at [s_col + 64 (b & 1), + 64); O_b = P_b V_b -> [s_col + 128 + 32 (b & 1), + 32)
    const uint32_t leader = elect_one();
    const uint8_t* q_t = smem + p.qkv_off;
    const uint8_t* k_t = q_t + 2 * BT_SLICE;
    const uint8_t* v_t = q_t + 4 * BT_SLICE;
    const uint8_t* rem = smem + p.rem_off;
    const uint32_t sc_col = (uint32_t)p.s_col, o_col = sc_col + 128u;
    const uint64_t dq_hi = make_smem_desc_sw64(smem_u32(q_t)), dq_lo = make_smem_desc_sw64(smem_u32(q_t + BT_SLICE));
    auto issue_s = [&](int b) {
      tc_fence_after();
      const uint32_t idesc = make_idesc_f16(64), d = tmem + sc_col + (uint32_t)(64 * (b & 1));
      const uint8_t* kt = (b < 2 ? k_t : rem) + (b & 1) * 64 * V2_ROW_B;   // 64 rows of the SWIZZLE_64B K pair: 4 KB
      const uint64_t dk_hi = make_smem_desc_sw64(smem_u32(kt)), dk_lo = make_smem_desc_sw64(smem_u32(kt + BT_SLICE));
#pragma unroll
      for (int ks = 0; ks < BT_DK / 16; ++ks) {
        const uint64_t ko = (uint64_t)(ks * 2);
        umma_elect<true>(d, dq_hi + ko, dk_hi + ko, idesc, ks == 0 ? 0u : 1u, leader);
        umma_elect<true>(d, dq_lo + ko, dk_hi + ko, idesc, 1u, leader);
        umma_elect<true>(d, dq_hi + ko, dk_lo + ko, idesc, 1u, leader);
      }
      umma_commit_elect(&bar_s[b & 1], leader);
    };
#pragma unroll 1
    for (int h = 0; h < p.heads; ++h) {
      bt_sync_mma();                            // Q, K, V^T of head h are in shared memory
      issue_s(0);
      issue_s(1);
#pragma unroll 1
      for (int b = 0; b < 4; ++b) {
        const int it = h * 4 + b;               // blocks done: buffer it & 1, phase (it >> 1) & 1 of bar_p / bar_o / bar_s
        mbar_wait(&bar_p[b & 1], (uint32_t)((it >> 1) & 1), failed);   // P_b written, O buffer b & 1 drained
        tc_fence_after();
        // O_b = P_hi V_hi + P_lo V_hi + P_hi V_lo (N = 32, K = 64 keys)
        const uint32_t idesc = make_idesc_f16(BT_DK), od = tmem + o_col + (uint32_t)(BT_DK * (b & 1));
        const uint32_t pc = tmem + sc_col + (uint32_t)(64 * (b & 1));
        const uint8_t* vb = b < 2 ? v_t + b * BT_VT_B : rem + 2 * BT_SLICE + (b - 2) * BT_VT_B;
        const uint64_t dv_hi = make_smem_desc(smem_u32(vb)), dv_lo = make_smem_desc(smem_u32(vb + BT_DK * ROW_B));
#pragma unroll
        for (int j = 0; j < 4; ++j) {           // 16 keys per step: 8 packed columns of P, 32 bytes of a V^T row
          const uint64_t ko = (uint64_t)(j * 2);
          umma_f16_ts_elect(od, pc + (uint32_t)(j * 8), dv_hi + ko, idesc, j == 0 ? 0u : 1u, leader);
          umma_f16_ts_elect(od, pc + (uint32_t)(32 + j * 8), dv_hi + ko, idesc, 1u, leader);
          umma_f16_ts_elect(od, pc + (uint32_t)(j * 8), dv_lo + ko, idesc, 1u, leader);
        }
        umma_commit_elect(&bar_o[b & 1], leader);
        if (b < 2) {                            // S_{b+2} overwrites the P_b that this P V reads: wait for it to retire
          mbar_wait(&bar_o[b & 1], (uint32_t)((it >> 1) & 1), failed);
          if (b == 0) mbar_wait(&bar_rfull, (uint32_t)(h & 1), failed);   // the peer's K / V^T of head h have landed
          issue_s(b + 2);
        }
      }
      if (h == p.heads - 1) umma_commit_elect(&bar_rfree, leader);   // the remote buffer is read
    }
  } else {
    // ===================== compute warps: MMA issue (warp 0, elected lane; PAIR: phase 4's from the MMA warp above),
    // epilogues and softmax (all)
    const uint32_t leader = warp == 0 ? elect_one() : 0u;
    const int lane_grp = warp & 3, quarter = warp >> 2;
    const int row = lane_grp * 32 + lane;       // TMEM lane = tile row
    const uint32_t lane_addr = tmem + ((uint32_t)(lane_grp * 32) << 16);
    float* slab = reinterpret_cast<float*>(smem + p.slab_off);
    uint8_t* r1 = smem;                         // in_proj A operand (x1 + pos pair), then one head's Q / K / V^T
    uint8_t* r2 = smem + p.r2_off;              // attention gate A operand (attention output pair)

    // warp 0: D[d0 + c n, ...] (+)= A W^T over `n` weight slices of the ring starting at global slice g0; A slice k = pair
    // at a + 2 k BT_SLICE; W stage = [hi: rows][lo: rows] x 64 B, one MMA of N = rows / n_mma per column group
    auto gemm = [&](int g0, int n, const uint8_t* a, int rows, int n_mma, uint32_t d0, uint64_t* done) {
      tc_fence_after();
      const int nn = rows / n_mma;
      const uint32_t idesc = make_idesc_f16(nn);
      for (int k = 0; k < n; ++k) {
        const int g = g0 + k, st = g & 1;
        mbar_wait(&bar_full[st], (uint32_t)((g >> 1) & 1), failed);
        tc_fence_after();
        const uint8_t* w = smem + p.ring_off + st * p.stage_b;
        const uint64_t da_hi = make_smem_desc_sw64(smem_u32(a + k * 2 * BT_SLICE));
        const uint64_t da_lo = make_smem_desc_sw64(smem_u32(a + k * 2 * BT_SLICE + BT_SLICE));
        for (int c = 0; c < n_mma; ++c) {
          const uint64_t dw_hi = make_smem_desc_sw64(smem_u32(w + c * nn * V2_ROW_B));
          const uint64_t dw_lo = make_smem_desc_sw64(smem_u32(w + (rows + c * nn) * V2_ROW_B));
          const uint32_t d = tmem + d0 + (uint32_t)(c * nn);
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {      // K = 16 per MMA: two per 64-byte row
            const uint64_t ko = (uint64_t)(kk * 2);
            umma_elect<true>(d, da_hi + ko, dw_hi + ko, idesc, (k | kk) == 0 ? 0u : 1u, leader);
            umma_elect<true>(d, da_lo + ko, dw_hi + ko, idesc, 1u, leader);
            umma_elect<true>(d, da_hi + ko, dw_lo + ko, idesc, 1u, leader);
          }
        }
        umma_commit_elect(&bar_empty[st], leader);
      }
      umma_commit_elect(done, leader);
    };

    // row-wise LayerNorm of the thread's NKB chunks of 8 columns (column j = 32 i + 8 quarter + e), statistics combined
    // across the four threads of the row through shared memory
    auto layer_norm = [&](float (&v)[NKB][8], float psum, const float* gamma, const float* beta) {
      red[0][quarter][row] = psum;
      bt_sync();
      const float mu = ((red[0][0][row] + red[0][1][row]) + (red[0][2][row] + red[0][3][row])) / (float)C;
      float pvar = 0.f;
#pragma unroll
      for (int i = 0; i < NKB; ++i)
#pragma unroll
        for (int e = 0; e < 8; ++e) pvar = fmaf(v[i][e] - mu, v[i][e] - mu, pvar);
      red[1][quarter][row] = pvar;
      bt_sync();
      const float rs = rsqrtf(((red[1][0][row] + red[1][1][row]) + (red[1][2][row] + red[1][3][row])) / (float)C + 1e-5f);
#pragma unroll
      for (int i = 0; i < NKB; ++i) {
        const int j = i * 32 + quarter * 8;
        const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + j)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + j + 4));
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + j)), b1 = __ldg(reinterpret_cast<const float4*>(beta + j + 4));
        const float gs[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bs[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) v[i][e] = fmaf((v[i][e] - mu) * rs, gs[e], bs[e]);
      }
    };

    // GLU over the accumulator's [a | b] halves at TMEM columns [0, 2C) + bias + residual; returns the row partial sum
    auto glu = [&](float (&v)[NKB][8], const float* bias, float sc, const float* res, int res_pitch) {
      float psum = 0.f;
#pragma unroll
      for (int i = 0; i < NKB; ++i) {
        const int j = i * 32 + quarter * 8;
        float a[8], b[8];
        tmem_ld8(lane_addr + (uint32_t)j, a);
        tmem_ld8(lane_addr + (uint32_t)(C + j), b);
        const float4 ba0 = __ldg(reinterpret_cast<const float4*>(bias + j)), ba1 = __ldg(reinterpret_cast<const float4*>(bias + j + 4));
        const float4 bb0 = __ldg(reinterpret_cast<const float4*>(bias + C + j));
        const float4 bb1 = __ldg(reinterpret_cast<const float4*>(bias + C + j + 4));
        const float4 r0 = *reinterpret_cast<const float4*>(res + (size_t)row * res_pitch + j);
        const float4 r1_ = *reinterpret_cast<const float4*>(res + (size_t)row * res_pitch + j + 4);
        const float bas[8] = {ba0.x, ba0.y, ba0.z, ba0.w, ba1.x, ba1.y, ba1.z, ba1.w};
        const float bbs[8] = {bb0.x, bb0.y, bb0.z, bb0.w, bb1.x, bb1.y, bb1.z, bb1.w};
        const float rs[8] = {r0.x, r0.y, r0.z, r0.w, r1_.x, r1_.y, r1_.z, r1_.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) v[i][e] = fmaf(a[e], sc, bas[e]) * bt_sigmoid(fmaf(b[e], sc, bbs[e])) + rs[e];
#pragma unroll
        for (int e = 0; e < 8; e += 4) psum += (v[i][e] + v[i][e + 1]) + (v[i][e + 2] + v[i][e + 3]);
      }
      return psum;
    };

    // ---- 1. gate GEMM ----------------------------------------------------------------------------------------------------
    if (warp == 0) {
      mbar_wait(&bar_a, 0, failed);
      gemm(0, NG, smem, 2 * C, 1, 0u, &bar_g);
    }
    {   // the tile's residual rows x -> slab, coalesced, while the gate GEMM runs
      const float4* xs = reinterpret_cast<const float4*>(p.x + (size_t)tile * 128 * C);
      for (int i = threadIdx.x; i < 128 * C / 4; i += 32 * BT_WARPS) {
        const int r = i / (C / 4), c4 = i - r * (C / 4);
        *reinterpret_cast<float4*>(slab + r * PITCH + 4 * c4) = __ldg(xs + i);
      }
    }
    bt_sync();
    mbar_wait(&bar_g, 0, failed);
    tc_fence_after();
    if (tracing) p.trace[1] = clock64();

    // ---- 2. GLU + x, LayerNorm 1 -> x1 (slab) and x1 + pos (in_proj operand) ---------------------------------------------
    {
      float v[NKB][8];
      const float psum = glu(v, p.bias_g, p.sc_g, slab, PITCH);   // x1 then replaces x in the slab, row by row
      layer_norm(v, psum, p.gamma1, p.beta1);
      const float* pr = p.pos + (size_t)((tile * 128 + row) % p.HW) * C;   // the row's position in its image
#pragma unroll
      for (int i = 0; i < NKB; ++i) {
        const int j = i * 32 + quarter * 8;
        float* sl = slab + row * PITCH + j;
        *reinterpret_cast<float4*>(sl) = make_float4(v[i][0], v[i][1], v[i][2], v[i][3]);
        *reinterpret_cast<float4*>(sl + 4) = make_float4(v[i][4], v[i][5], v[i][6], v[i][7]);
        const float4 p0 = __ldg(reinterpret_cast<const float4*>(pr + j)), p1 = __ldg(reinterpret_cast<const float4*>(pr + j + 4));
        const float t[8] = {v[i][0] + p0.x, v[i][1] + p0.y, v[i][2] + p0.z, v[i][3] + p0.w,
                            v[i][4] + p1.x, v[i][5] + p1.y, v[i][6] + p1.z, v[i][7] + p1.w};
        uint4 hi, lo;
        cvt8(t, hi, lo);
        *reinterpret_cast<uint4*>(r1 + i * 2 * BT_SLICE + sw64_off(row, quarter)) = hi;
        *reinterpret_cast<uint4*>(r1 + i * 2 * BT_SLICE + BT_SLICE + sw64_off(row, quarter)) = lo;
      }
    }
    fence_proxy_async();                        // generic-proxy smem writes -> visible to the tensor core
    tc_fence_before();
    bt_sync();
    if (tracing) p.trace[2] = clock64();

    // ---- 3. in_proj GEMM -> (k | v | q) in TMEM [2C, 5C) -------------------------------------------------------------------
    if (warp == 0) gemm(NG, NKB, r1, 3 * C, 3 * C / p.n_ip, (uint32_t)(2 * C), &bar_i);
    mbar_wait(&bar_i, 0, failed);
    tc_fence_after();
    if (PAIR && threadIdx.x == 0) mbar_arrive_cluster(mapa_rank(&bar_pempty, cluster_ctarank() ^ 1u));   // in_proj has read the ring stage
    if (tracing) p.trace[3] = clock64();

    // ---- 4. attention, one head at a time ----------------------------------------------------------------------------------
    if constexpr (!PAIR) {   // deep levels: one 128-key block per head, MMAs from warp 0
      uint8_t* q_t = smem + p.qkv_off;          // [hi | lo][128 rows][64 B], SWIZZLE_64B (over the dead in_proj operand)
      uint8_t* k_t = q_t + 2 * BT_SLICE;
      uint8_t* v_t = q_t + 4 * BT_SLICE;        // 2 blocks of 64 keys, SWIZZLE_128B
      const int D = p.D, chunks = D >> 3;
      const uint32_t ip = (uint32_t)(2 * C), sc_col = (uint32_t)p.s_col, o_col = sc_col + 128u;
      const int klo = row / p.HW * p.HW, khi = klo + p.HW;  // the keys of this row's image
      const int k0 = quarter * 32;
      const bool live = k0 < khi && k0 + 32 > klo;          // warp-uniform: a warp's 32 rows meet the same quarters
      constexpr int NB = 1;                     // key blocks per head
#pragma unroll 1
      for (int h = 0; h < p.heads; ++h) {
        // 4a. drain: thread (row, quarter) takes dims [8 quarter, 8 quarter + 8) of the head's k, v and q; dims >= D are zero
        {
          const uint32_t col = lane_addr + ip + (uint32_t)(h * D + quarter * 8);
          float v[8];
          uint4 hi, lo;
          const bool has = quarter < chunks;
          if (has) {
            tmem_ld8(col, v);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] *= p.sc_i;
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = 0.f;
          }
          cvt8(v, hi, lo);
          *reinterpret_cast<uint4*>(k_t + sw64_off(row, quarter)) = hi;
          *reinterpret_cast<uint4*>(k_t + BT_SLICE + sw64_off(row, quarter)) = lo;
          if (has) {
            tmem_ld8(col + 2 * C, v);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = v[e] * p.sc_i * p.qscale;
          }
          cvt8(v, hi, lo);
          *reinterpret_cast<uint4*>(q_t + sw64_off(row, quarter)) = hi;
          *reinterpret_cast<uint4*>(q_t + BT_SLICE + sw64_off(row, quarter)) = lo;
          if (has) {
            tmem_ld8(col + C, v);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] *= p.sc_i;
          }
          // V^T: rows = head dims, contraction (keys) along the 128-byte rows; hi rows then lo rows per 64-key block
          uint8_t* blk = v_t + (row >> 6) * BT_VT_B;
          const int kk = row & 63;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int dim = quarter * 8 + e;
            unsigned short hh, ll;
            split_f16(v[e], hh, ll);
            *reinterpret_cast<unsigned short*>(blk + sw_off(dim, kk >> 3) + ((kk & 7) << 1)) = hh;
            *reinterpret_cast<unsigned short*>(blk + sw_off(BT_DK + dim, kk >> 3) + ((kk & 7) << 1)) = ll;
          }
        }
        fence_proxy_async();
        tc_fence_before();
        bt_sync();

        // 4b. S = Q K^T into TMEM [s_col, s_col + 128) (warp 0; `kt` = the key block's K pair)
        auto issue_s = [&](const uint8_t* kt) {
          tc_fence_after();
          const uint32_t idesc = make_idesc_f16(128);
          const uint64_t dq_hi = make_smem_desc_sw64(smem_u32(q_t)), dq_lo = make_smem_desc_sw64(smem_u32(q_t + BT_SLICE));
          const uint64_t dk_hi = make_smem_desc_sw64(smem_u32(kt)), dk_lo = make_smem_desc_sw64(smem_u32(kt + BT_SLICE));
#pragma unroll
          for (int ks = 0; ks < BT_DK / 16; ++ks) {
            const uint64_t ko = (uint64_t)(ks * 2);
            umma_elect<true>(tmem + sc_col, dq_hi + ko, dk_hi + ko, idesc, ks == 0 ? 0u : 1u, leader);
            umma_elect<true>(tmem + sc_col, dq_lo + ko, dk_hi + ko, idesc, 1u, leader);
            umma_elect<true>(tmem + sc_col, dq_hi + ko, dk_lo + ko, idesc, 1u, leader);
          }
          umma_commit_elect(&bar_s[0], leader);
        };
        if (warp == 0) issue_s(k_t);
        float mx = 0.f, l = 0.f;                // the last key block's row maximum and sum
#pragma unroll 1
        for (int kb = 0; kb < NB; ++kb) {
          const int it = h * NB + kb;             // key blocks done: phase of bar_s / bar_o
          mbar_wait(&bar_s[0], (uint32_t)(it & 1), failed);
          tc_fence_after();
          if (tracing && it == 0) p.trace[4] = clock64();

          // 4c. masked row maximum over this thread's 32 keys
          float s[32];
          mx = -INFINITY;
          if (live) {
            tmem_ld32(lane_addr + sc_col + (uint32_t)k0, s);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int key = k0 + i;
              s[i] = (key >= klo && key < khi) ? s[i] : -INFINITY;
              mx = fmaxf(mx, s[i]);
            }
          }
          red[0][quarter][row] = mx;
          tc_fence_before();                      // every load of S is complete before anyone writes P over it
          bt_sync();
          tc_fence_after();
          mx = fmaxf(fmaxf(red[0][0][row], red[0][1][row]), fmaxf(red[0][2][row], red[0][3][row]));

          // 4d. p = 2^(s - max) (0 for other images' keys) as packed fp16 (hi, lo): keys (2i, 2i + 1) in column i of each half
          float sum = 0.f;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t ph[8], pl[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float e0 = 0.f, e1 = 0.f;
              if (live) {
                e0 = ex2_fast(s[16 * half + 2 * i] - mx);       // masked keys: 2^-inf = 0
                e1 = ex2_fast(s[16 * half + 2 * i + 1] - mx);
              }
              sum += e0 + e1;
              ph[i] = pack_h2(e0, e1);
              float a0, a1;
              unpack_h2(ph[i], a0, a1);
              pl[i] = pack_h2(e0 - a0, e1 - a1);
            }
            tmem_st8u(lane_addr + sc_col + (uint32_t)(quarter * 16 + half * 8), ph);
            tmem_st8u(lane_addr + sc_col + (uint32_t)(64 + quarter * 16 + half * 8), pl);
          }
          red[1][quarter][row] = sum;
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          tc_fence_before();
          bt_sync();
          l = (red[1][0][row] + red[1][1][row]) + (red[1][2][row] + red[1][3][row]);

          // 4e. O_kb = P_hi V_hi + P_lo V_hi + P_hi V_lo (N = 32, K = 128 keys) into TMEM [o_col + 32 kb, o_col + 32 kb + 32)
          if (warp == 0) {
            tc_fence_after();
            const uint32_t idesc = make_idesc_f16(BT_DK), od = tmem + o_col + (uint32_t)(kb * BT_DK);
            const uint8_t* vt = v_t;
#pragma unroll
            for (int j = 0; j < 8; ++j) {         // 16 keys per step: 8 packed columns of P, 32 bytes of a V^T row
              const int key = j * 16;
              const uint8_t* vb = vt + (key >> 6) * BT_VT_B;
              const uint64_t ko = (uint64_t)(((key & 63) >> 4) * 2);
              const uint64_t dv_hi = make_smem_desc(smem_u32(vb)) + ko, dv_lo = make_smem_desc(smem_u32(vb + BT_DK * ROW_B)) + ko;
              const uint32_t a_hi = tmem + sc_col + (uint32_t)(j * 8), a_lo = tmem + sc_col + (uint32_t)(64 + j * 8);
              umma_f16_ts_elect(od, a_hi, dv_hi, idesc, j == 0 ? 0u : 1u, leader);
              umma_f16_ts_elect(od, a_lo, dv_hi, idesc, 1u, leader);
              umma_f16_ts_elect(od, a_hi, dv_lo, idesc, 1u, leader);
            }
            umma_commit_elect(&bar_o[0], leader);
          }
        }
        mbar_wait(&bar_o[0], (uint32_t)((h * NB + NB - 1) & 1), failed);
        tc_fence_after();

        // 4f. O / rowsum -> columns [h D, h D + D) of the attention gate's operand pair
        const float w0 = 1.0f / l;
        if (quarter < chunks) {
          float o[8];
          tmem_ld8(lane_addr + o_col + (uint32_t)(quarter * 8), o);
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] *= w0;
          uint4 hi, lo;
          cvt8(o, hi, lo);
          const int c = h * D + quarter * 8, kb = c >> 5, ch = (c & 31) >> 3;
          *reinterpret_cast<uint4*>(r2 + kb * 2 * BT_SLICE + sw64_off(row, ch)) = hi;
          *reinterpret_cast<uint4*>(r2 + kb * 2 * BT_SLICE + BT_SLICE + sw64_off(row, ch)) = lo;
        }
        // (the next head's drain barrier orders these TMEM loads before its MMAs overwrite S and O)
      }
    } else {                 // PAIR: four 64-key blocks per head, MMAs from the MMA warp
      uint8_t* q_t = smem + p.qkv_off;          // [hi | lo][128 rows][64 B], SWIZZLE_64B (over the dead in_proj operand)
      uint8_t* k_t = q_t + 2 * BT_SLICE;
      uint8_t* v_t = q_t + 4 * BT_SLICE;        // 2 blocks of 64 keys, SWIZZLE_128B
      const int D = p.D, chunks = D >> 3;
      const uint32_t ip = (uint32_t)(2 * C), sc_col = (uint32_t)p.s_col, o_col = sc_col + 128u;

      // 4a. drain: thread (row, quarter) takes dims [8 quarter, 8 quarter + 8) of the head's k, v and q; dims >= D are zero
      auto drain = [&](int h) {
        const uint32_t col = lane_addr + ip + (uint32_t)(h * D + quarter * 8);
        float v[8];
        uint4 hi, lo;
        const bool has = quarter < chunks;
        if (has) {
          tmem_ld8(col, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] *= p.sc_i;
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = 0.f;
        }
        cvt8(v, hi, lo);
        *reinterpret_cast<uint4*>(k_t + sw64_off(row, quarter)) = hi;
        *reinterpret_cast<uint4*>(k_t + BT_SLICE + sw64_off(row, quarter)) = lo;
        if (has) {
          tmem_ld8(col + 2 * C, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = v[e] * p.sc_i * p.qscale;
        }
        cvt8(v, hi, lo);
        *reinterpret_cast<uint4*>(q_t + sw64_off(row, quarter)) = hi;
        *reinterpret_cast<uint4*>(q_t + BT_SLICE + sw64_off(row, quarter)) = lo;
        if (has) {
          tmem_ld8(col + C, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] *= p.sc_i;
        }
        // V^T: rows = head dims, contraction (keys) along the 128-byte rows; hi rows then lo rows per 64-key block
        uint8_t* blk = v_t + (row >> 6) * BT_VT_B;
        const int kk = row & 63;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int dim = quarter * 8 + e;
          unsigned short hh, ll;
          split_f16(v[e], hh, ll);
          *reinterpret_cast<unsigned short*>(blk + sw_off(dim, kk >> 3) + ((kk & 7) << 1)) = hh;
          *reinterpret_cast<unsigned short*>(blk + sw_off(BT_DK + dim, kk >> 3) + ((kk & 7) << 1)) = ll;
        }
        fence_proxy_async();
        tc_fence_before();
      };
      // 4f. O / rowsum -> columns [h D, h D + D) of the attention gate's operand pair
      auto store_o = [&](int h, const float (&o)[8], float w) {
        float t[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) t[e] = o[e] * w;
        uint4 hi, lo;
        cvt8(t, hi, lo);
        const int c = h * D + quarter * 8, kb = c >> 5, ch = (c & 31) >> 3;
        *reinterpret_cast<uint4*>(r2 + kb * 2 * BT_SLICE + sw64_off(row, ch)) = hi;
        *reinterpret_cast<uint4*>(r2 + kb * 2 * BT_SLICE + BT_SLICE + sw64_off(row, ch)) = lo;
      };

      // Per head, four 64-key blocks b: own keys 0-63, 64-127, then the peer's 0-63, 64-127 from the remote buffer.  The
      // MMA warp keeps two S / P buffers in flight, so the softmax of block b runs while the tensor pipe does P_{b-1} V
      // and S_{b+1}.  A thread owns 16 keys of a row per block.  Each block has its own row maximum m_b; the thread
      // folds O_b into registers as it retires, m = max(m, m_b), o = o 2^(m_old - m) + O_b 2^(m_b - m), and likewise
      // its share of the row sum (the exact split-key combination, applied block by block).
      uint8_t* rem = smem + p.rem_off;        // the peer's K pair and V^T of the head, laid out as k_t, v_t
#pragma unroll 1
      for (int h = 0; h < p.heads; ++h) {
        mbar_wait(&bar_pempty, (uint32_t)(h & 1), failed);   // the peer is done with our previous head's copy
        drain(h);
        bt_sync_mma();
        if (warp == 1 && lane == 0) {         // K pair and V^T (contiguous from k_t) -> the peer's remote buffer
          mbar_expect_tx(&bar_rfull, (uint32_t)BT_REM_B);   // ... and the peer's into ours
          const uint32_t peer = cluster_ctarank() ^ 1u;
          bulk_copy_to_peer(mapa_rank(rem, peer), k_t, (uint32_t)BT_REM_B, mapa_rank(&bar_rfull, peer));
        }
        float m = -INFINITY, l = 0.f, o[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        // fold O_b (its P V committed on bar_o[b & 1]) with block maximum mb and this thread's block sum lb
        auto fold = [&](int b, float mb, float lb) {
          const int it = h * 4 + b;
          mbar_wait(&bar_o[b & 1], (uint32_t)((it >> 1) & 1), failed);
          tc_fence_after();
          const float mn = fmaxf(m, mb), a = ex2_fast(m - mn), c = ex2_fast(mb - mn);
          l = l * a + lb * c;
          m = mn;
          if (quarter < chunks) {
            float ob[8];
            tmem_ld8(lane_addr + o_col + (uint32_t)(BT_DK * (b & 1) + quarter * 8), ob);
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = o[e] * a + ob[e] * c;
          }
        };
        float mp = 0.f, lp = 0.f;             // the previous block's maximum and sum, folded one block later
#pragma unroll 1
        for (int b = 0; b < 4; ++b) {
          const int it = h * 4 + b;
          const uint32_t sb = lane_addr + sc_col + (uint32_t)(64 * (b & 1));
          mbar_wait(&bar_s[b & 1], (uint32_t)((it >> 1) & 1), failed);
          tc_fence_after();
          if (tracing && it == 0) p.trace[4] = clock64();
          float s[16];
          tmem_ld16(sb + (uint32_t)(quarter * 16), s);
          float mb = s[0];
#pragma unroll
          for (int i = 1; i < 16; ++i) mb = fmaxf(mb, s[i]);
          red[b & 1][quarter][row] = mb;
          tc_fence_before();                  // every load of S_b is complete before anyone writes P_b over it
          bt_sync();
          tc_fence_after();
          mb = fmaxf(fmaxf(red[b & 1][0][row], red[b & 1][1][row]), fmaxf(red[b & 1][2][row], red[b & 1][3][row]));
          // p = 2^(s - m_b) as packed fp16 (hi, lo): keys (2i, 2i + 1) of the block in column i of each 32-column half
          uint32_t ph[8], pl[8];
          float lb = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float e0 = ex2_fast(s[2 * i] - mb), e1 = ex2_fast(s[2 * i + 1] - mb);
            lb += e0 + e1;
            ph[i] = pack_h2(e0, e1);
            float a0, a1;
            unpack_h2(ph[i], a0, a1);
            pl[i] = pack_h2(e0 - a0, e1 - a1);
          }
          tmem_st8u(sb + (uint32_t)(quarter * 8), ph);
          tmem_st8u(sb + (uint32_t)(32 + quarter * 8), pl);
          asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
          tc_fence_before();
          __syncwarp();
          if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bar_p[b & 1])) : "memory");
          // O_{b-1} is drained before this warp's next arrival lets P_{b+1} V overwrite its buffer
          if (b > 0) fold(b - 1, mp, lp);
          mp = mb;
          lp = lb;
        }
        fold(3, mp, lp);
        // P_3 V has retired, and with it every MMA of the head that read the remote buffer
        if (h + 1 < p.heads && threadIdx.x == 0) mbar_arrive_cluster(mapa_rank(&bar_pempty, cluster_ctarank() ^ 1u));
        red[2][quarter][row] = l;
        bt_sync();
        l = (red[2][0][row] + red[2][1][row]) + (red[2][2][row] + red[2][3][row]);
        if (quarter < chunks) store_o(h, o, 1.0f / l);
        // (the next head's drain barrier orders these TMEM loads before its MMAs overwrite S and O)
      }
    }
    fence_proxy_async();
    tc_fence_before();
    bt_sync();
    if (tracing) p.trace[5] = clock64();

    // ---- 5. attention-gate GEMM into TMEM [0, 2C) --------------------------------------------------------------------------
    if (warp == 0) gemm(NG + NKB, NKB, r2, 2 * C, 1, 0u, &bar_ag);
    mbar_wait(&bar_ag, 0, failed);
    tc_fence_after();
    if (tracing) p.trace[6] = clock64();

    // ---- 6. GLU + x1, LayerNorm 2 -> x2 and the next layer's operand pair --------------------------------------------------
    {
      float v[NKB][8];
      const float psum = glu(v, p.bias_a, p.sc_a, slab, PITCH);
      layer_norm(v, psum, p.gamma2, p.beta2);
#pragma unroll
      for (int i = 0; i < NKB; ++i) {           // x2 over x1 in the slab (each thread rewrites the columns it read)
        float* sl = slab + row * PITCH + i * 32 + quarter * 8;
        *reinterpret_cast<float4*>(sl) = make_float4(v[i][0], v[i][1], v[i][2], v[i][3]);
        *reinterpret_cast<float4*>(sl + 4) = make_float4(v[i][4], v[i][5], v[i][6], v[i][7]);
      }
    }
    bt_sync();
    // write-out with consecutive threads on consecutive 8-column chunks of a row: every warp store is contiguous
    for (int i = threadIdx.x; i < 128 * C / 8; i += 32 * BT_WARPS) {
      const int r = i / (C / 8), j = (i - r * (C / 8)) * 8;
      const size_t mr = (size_t)tile * 128 + r;
      const float4 a = *reinterpret_cast<const float4*>(slab + r * PITCH + j);
      const float4 b = *reinterpret_cast<const float4*>(slab + r * PITCH + j + 4);
      const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
      float* xo = p.x2 + mr * C + j;
      *reinterpret_cast<float4*>(xo) = a;
      *reinterpret_cast<float4*>(xo + 4) = b;
      uint4 hi, lo;
      if (p.celu) {                             // concat_elu: [elu(x2) | elu(-x2)], width 2C
        float t[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) t[e] = bt_elu(v[e]);
        cvt8(t, hi, lo);
        *reinterpret_cast<uint4*>(p.out_hi + mr * 2 * C + j) = hi;
        *reinterpret_cast<uint4*>(p.out_lo + mr * 2 * C + j) = lo;
#pragma unroll
        for (int e = 0; e < 8; ++e) t[e] = bt_elu(-v[e]);
        cvt8(t, hi, lo);
        *reinterpret_cast<uint4*>(p.out_hi + mr * 2 * C + C + j) = hi;
        *reinterpret_cast<uint4*>(p.out_lo + mr * 2 * C + C + j) = lo;
      } else {
        cvt8(v, hi, lo);
        *reinterpret_cast<uint4*>(p.out_hi + mr * C + j) = hi;
        *reinterpret_cast<uint4*>(p.out_lo + mr * C + j) = lo;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();                 // neither CTA retires while the peer may still signal or copy into it
  if (tracing) p.trace[7] = clock64();
  if (warp == 0) tmem_dealloc(tmem, 512u);
  if (threadIdx.x == 0 && failed_flag && p.status) *p.status = 1;
}

}  // namespace tc
}  // namespace flowk

using namespace flowk;
using namespace flowk::tc;

namespace {
// Shapes the kernel takes and its shared-memory carve: [in_proj operand pair | one head's Q, K, V^T] [attention output pair]
// [weight ring: 2 stages] [x1 slab]; the c1 tile of the gate GEMM lies over the first two regions.  PAIR (HW = 256, two
// tiles per image): the remote K / V^T buffer lies over the ring stage of the attention gate's second weight slice when a
// stage holds it (C = 96), else after the slab.
bool block_tail_plan(long long M, int HW, int C, int heads, bool pair, BlockTailParams& p, size_t& smem) {
  if (pair ? HW != 256 || M % 256 : HW < 1 || HW > 128 || 128 % HW || M % 128) return false;
  if (C < 32 || C % 32 || 5 * C > 512 || heads < 1 || C % heads) return false;  // TMEM: gate [0, 2C) + in_proj [2C, 5C)
  const int D = C / heads;
  if (D != 24 && D != 32) return false;
  const int nkb = C / 32;
  p.HW = HW;
  p.heads = heads;
  p.D = D;
  p.qscale = 1.4426950408889634f / sqrtf((float)D);
  p.n_ip = 3 * C <= 256 ? 3 * C : 3 * C / 2;
  // S / P and O (PAIR: O_0, O_1) after in_proj, or over the drained gate accumulator
  p.s_col = 5 * C + 128 + (pair ? 2 : 1) * BT_DK <= 512 ? 5 * C : 0;
  const int r1 = 2 * nkb * BT_SLICE > BT_QKV_B ? 2 * nkb * BT_SLICE : BT_QKV_B;
  p.qkv_off = 0;
  p.r2_off = r1;
  p.ring_off = r1 + 2 * nkb * BT_SLICE;
  if (p.ring_off < 2 * nkb * 2 * BT_SLICE) return false;   // the c1 tile must fit below the ring
  p.stage_b = 2 * 3 * C * V2_ROW_B;
  p.slab_off = p.ring_off + 2 * p.stage_b;
  const int slab_end = p.slab_off + 128 * (C + 4) * 4;
  p.rem_alias = pair && p.stage_b >= BT_REM_B;
  p.rem_off = 0;
  if (p.rem_alias) p.rem_off = p.ring_off + ((3 * nkb + 1) & 1) * p.stage_b;   // the stage of weight slice 3 nkb + 1
  else if (pair) p.rem_off = (slab_end + 1023) / 1024 * 1024;
  smem = (size_t)(pair && !p.rem_alias ? p.rem_off + BT_REM_B : slab_end) + 1024;
  return smem + 8 * 1024 <= 227 * 1024;          // (+ the kernel's static shared memory)
}

template <int NKB, bool PAIR>
int block_tail_launch(const BlockTailParams& p, int tiles, size_t smem, const CUtensorMap* maps, cudaStream_t stream) {
  static size_t smem_set = 0;
  if (smem > smem_set) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(block_tail_tc_kernel<NKB, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    smem_set = smem;
  }
  FLOWK_CUDA_OK(launch_pdl_cluster(block_tail_tc_kernel<NKB, PAIR>, dim3(tiles), dim3(bt_threads(PAIR)), smem, stream,
                                   PAIR ? 2 : 1, p, maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], maps[6], maps[7]));
  return launch_status();
}

int block_tail_entry(bool pair, const void* c1_hi, const void* c1_lo, const void* wg_hi, const void* wg_lo, float sc_g,
                     const float* bias_g, const float* x, const float* gamma1, const float* beta1, const float* pos,
                     const void* wi_hi, const void* wi_lo, float sc_i, const void* wa_hi, const void* wa_lo, float sc_a,
                     const float* bias_a, const float* gamma2, const float* beta2, float* x2, void* out_hi, void* out_lo,
                     int celu, int B, int HW, int C, int heads, int* status, long long* trace, flowk_stream_t stream) {
  BlockTailParams p{};
  size_t smem = 0;
  const long long M = (long long)B * HW;
  if (B < 0 || !block_tail_plan(M, HW, C, heads, pair, p, smem)) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (M > 0x7fffffffLL) return FLOWK_ERR_SHAPE;
  const void* ptrs[] = {c1_hi, c1_lo, wg_hi, wg_lo, bias_g, x, gamma1, beta1, pos, wi_hi, wi_lo, wa_hi, wa_lo, bias_a,
                        gamma2, beta2, x2, out_hi, out_lo};
  for (const void* q : ptrs)
    if (!q) return FLOWK_ERR_ARG;
  for (const void* q : ptrs)
    if (!aligned16(q)) return FLOWK_ERR_ALIGN;
  if (!(sc_g > 0.f) || !(sc_i > 0.f) || !(sc_a > 0.f)) return FLOWK_ERR_ARG;
  p.bias_g = bias_g;
  p.x = x;
  p.gamma1 = gamma1;
  p.beta1 = beta1;
  p.pos = pos;
  p.bias_a = bias_a;
  p.gamma2 = gamma2;
  p.beta2 = beta2;
  p.x2 = x2;
  p.out_hi = reinterpret_cast<uint16_t*>(out_hi);
  p.out_lo = reinterpret_cast<uint16_t*>(out_lo);
  p.celu = celu ? 1 : 0;
  p.sc_g = sc_g;
  p.sc_i = sc_i;
  p.sc_a = sc_a;
  p.status = status;
  p.trace = trace;
  const long long k2 = (2LL * C + 63) / 64 * 64, k1 = (C + 63) / 64 * 64;
  CUtensorMap maps[8];
  if (!make_map_sw64(&maps[0], c1_hi, M, 2LL * C, 128) || !make_map_sw64(&maps[1], c1_lo, M, 2LL * C, 128) ||
      !make_map_sw64(&maps[2], wg_hi, 2LL * C, k2, 2 * C) || !make_map_sw64(&maps[3], wg_lo, 2LL * C, k2, 2 * C) ||
      !make_map_sw64(&maps[4], wi_hi, 3LL * C, k1, p.n_ip) || !make_map_sw64(&maps[5], wi_lo, 3LL * C, k1, p.n_ip) ||
      !make_map_sw64(&maps[6], wa_hi, 2LL * C, k1, 2 * C) || !make_map_sw64(&maps[7], wa_lo, 2LL * C, k1, 2 * C))
    return FLOWK_ERR_ARG;
  const int tiles = (int)(M / 128);
  switch (C / 32 + (pair ? 3 : 0)) {
    case 1: return block_tail_launch<1, false>(p, tiles, smem, maps, stream);
    case 2: return block_tail_launch<2, false>(p, tiles, smem, maps, stream);
    case 3: return block_tail_launch<3, false>(p, tiles, smem, maps, stream);
    case 4: return block_tail_launch<1, true>(p, tiles, smem, maps, stream);
    case 5: return block_tail_launch<2, true>(p, tiles, smem, maps, stream);
    default: return block_tail_launch<3, true>(p, tiles, smem, maps, stream);
  }
}
}  // namespace

extern "C" int flowk_block_tail_tc(const void* c1_hi, const void* c1_lo, const void* wg_hi, const void* wg_lo, float sc_g,
                                   const float* bias_g, const float* x, const float* gamma1, const float* beta1,
                                   const float* pos, const void* wi_hi, const void* wi_lo, float sc_i, const void* wa_hi,
                                   const void* wa_lo, float sc_a, const float* bias_a, const float* gamma2,
                                   const float* beta2, float* x2, void* out_hi, void* out_lo, int celu, int B, int HW, int C,
                                   int heads, int* status, long long* trace, flowk_stream_t stream) {
  return block_tail_entry(false, c1_hi, c1_lo, wg_hi, wg_lo, sc_g, bias_g, x, gamma1, beta1, pos, wi_hi, wi_lo, sc_i, wa_hi,
                          wa_lo, sc_a, bias_a, gamma2, beta2, x2, out_hi, out_lo, celu, B, HW, C, heads, status, trace,
                          stream);
}

extern "C" int flowk_block_tail_pair_tc(const void* c1_hi, const void* c1_lo, const void* wg_hi, const void* wg_lo,
                                        float sc_g, const float* bias_g, const float* x, const float* gamma1,
                                        const float* beta1, const float* pos, const void* wi_hi, const void* wi_lo,
                                        float sc_i, const void* wa_hi, const void* wa_lo, float sc_a, const float* bias_a,
                                        const float* gamma2, const float* beta2, float* x2, void* out_hi, void* out_lo,
                                        int celu, int B, int HW, int C, int heads, int* status, long long* trace,
                                        flowk_stream_t stream) {
  return block_tail_entry(true, c1_hi, c1_lo, wg_hi, wg_lo, sc_g, bias_g, x, gamma1, beta1, pos, wi_hi, wi_lo, sc_i, wa_hi,
                          wa_lo, sc_a, bias_a, gamma2, beta2, x2, out_hi, out_lo, celu, B, HW, C, heads, status, trace,
                          stream);
}
