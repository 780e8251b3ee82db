// Implicit-GEMM convolution / linear layer of the coupling conditioners on the 5th-gen tensor cores.
//
//   D[m, n] = sum_{tap, c} A[pos(m) + shift(tap), c] * Wt[n, tap*Cin + c]        (taps = 1 or 3x3, zero "same" padding)
//
// * activations NHWC fp32 [B,H,W,Cin]; an M tile = 128 consecutive positions = a (Bt x Ht x W) box, fetched per tap
//   by ONE 4-D TMA box load whose coordinates carry the tap shift - out-of-bounds rows/columns are zero-filled by
//   the TMA unit, which is the convolution's padding;
// * weights [N, taps*Cin] K-major, 2-D TMA;
// * tcgen05.mma, M=128, accumulators in TMEM.  fp32 accuracy (the 1e-4 parity budget rules out plain TF32 / bf16)
//   comes from a two-term operand split x = hi + lo and D += A_hi W_hi + A_lo W_hi + A_hi W_lo (dropped term ~2^-22):
//     - F16 = false (training path: gradients need fp32's exponent range): kind::tf32, hi / lo are TF32 values in
//       fp32 containers, 32 channels per 128-byte k-block, K = 8 per MMA;
//     - F16 = true (inference): kind::f16, hi / lo are fp16 (11 significant bits each - exactly TF32's - so the
//       split is as accurate, provided |x| < 65504; weights are pre-scaled by a power of two, undone by `acc_scale`):
//       HALF the operand bytes through TMA / shared memory (the bound of these layers, 4 B per element for the pair
//       = what ONE fp32 copy costs) and K = 16 per MMA, i.e. half the MMA instructions;
// * warp roles: warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer (one elected lane), warps 2..5 = epilogue,
//   each thread owning one accumulator row (TMEM lane) - so row-wise epilogues (GLU, residual, LayerNorm over the
//   channel dim) are thread-local;
// * fused epilogues produce exactly what the next layer consumes: fp32 rows, hi/lo operand pairs (optionally after
//   concat-ELU or after adding the positional encoding), or the NCHW parameter tensor the MixLogCDF kernel reads.
//
// Reference semantics: flow_modules/mixlogcdf_nn.py:12-29 (WNConv2d), :81-102 (ConvAttnBlock), :227-260 (GatedConv),
// :124-152 (GatedAttn projections), flow_modules/affine_coupling.py:27-80 (NN_net).
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "umma.cuh"

namespace flowk {
namespace tc {

constexpr int ROW_BYTES = 128;                          // one swizzle row = one k-block of a tile row (32 tf32 / 64 fp16)
constexpr int A_TILE_BYTES = BLOCK_M * ROW_BYTES;       // 16 KB
constexpr int EPI_WARPS = 16;                // 4 per TMEM lane group: they split the column chunks
constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
constexpr int MAX_CHUNKS = 2;

// elu(x) = x > 0 ? x : e^x - 1.  The result feeds a GEMM operand, so what matters is ABSOLUTE error (~1e-7 here).
__device__ __forceinline__ float elu1(float x) { return x > 0.f ? x : ex2_fast(x * kLog2e) - 1.f; }
__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.f, 1.f + ex2_fast(-x * kLog2e)); }

// --------------------------------------------------------------------------------------------------
// kernel parameters (device view)
// --------------------------------------------------------------------------------------------------
enum { PRE_BIAS = 0, PRE_GLU_RES_LN = 1, PRE_LSTM = 2 };
// one step of mAR ancestral sampling (flowk_mar_step): internal epilogues only, reached through that entry point
enum { PRE_MAR_EMBED = 3, PRE_MAR_LSTM = 4, PRE_MAR_SAMPLE = 5 };
enum { OUT_F32 = 1, OUT_HILO = 2, OUT_HILO_POS = 4, OUT_HILO_CELU = 8, OUT_NCHW = 16, OUT_HILO_RELU = 32 };

struct Params {
  int M, N, HW, W, H;              // M = B*H*W rows, N = total output columns of the GEMM
  int taps, kblocks_per_tap;       // K loop = taps * kblocks_per_tap blocks of 32 channels
  int ksz, dil;                    // taps = ksz * ksz (1, 3 or 5), tap (ky, kx) reads position + ((ky, kx) - ksz / 2) * dil
  int wt, ht, bt;                  // M tile = bt images x ht rows x wt (= W) columns
  int n_chunk, n_chunks;           // columns per MMA (<=256, %16) and MMAs per k-step; CTA covers n_chunk*n_chunks columns
  int tmem_cols, stages;
  int bar_offset;                  // byte offset of the mbarriers: past the pipeline stages AND the epilogue staging area
  int dxsplit, a_slots, w_slots;   // 3x3 "dx-split" mode: one accumulator per column shift, activation tile reused by 3 taps
  int pair, w_unit, pair_nmma;     // dx-split on CTA pairs (cta_group::2, M = 256 per MMA): each CTA of the pair stages half of
                                   // the weight rows, in TMA boxes of w_unit rows (umma.cuh)
  int pre, out_mask;
  const float* bias;               // [N] or null
  const float* res;                // [M, C] residual (PRE_GLU_RES_LN), C = N/2
  const float* gamma;              // LayerNorm weight/bias [C]
  const float* beta;
  const float* pos;                // positional encoding [HW, C] (OUT_HILO_POS)
  float* out_f32;                  // [M, Nout]
  float* out_hi;                   // [M, Nout] or [M, 2*Nout] (CELU)
  float* out_lo;
  float* out_nchw;                 // [B, N, HW]
  // chained second GEMM (GLU kernels only): rows (y [+ pos]) go from the epilogue straight into swizzled shared-memory
  // operand tiles and are multiplied by a second weight matrix [n2, C] in the same CTA (gate -> in_proj fusion)
  int chain, n2, n2_chunk, n2_chunks, a3_offset, w2_offset;
  float* out2_f32;                 // [M, n2]
  float acc_scale;                 // F16: the weights were scaled by 1 / acc_scale (a power of two)
  float acc_scale2;                // the same for the chained second GEMM's weights
  const float* acc_scale_ptr;      // non-null: device copy of acc_scale (read in the epilogue)
  int ksplit;                      // > 1: blockIdx.z takes a slice of every tap's channel blocks; fp32 partial rows go to
                                   // out_f32 + z*M*N (no bias) and flowk's split-K reduce kernel finishes the layer
  int* status;                     // set to 1 if a barrier wait timed out
  long long* trace;                // optional [16] clock64 stamps of CTA (0,0): setup, first full, last mma, epi start, epi end
  // PRE_MAR_*: up to two fp16-pair destinations, each with its own row pitch and first column (fp16 elements)
  void* dst_hi[2];
  void* dst_lo[2];
  int dst_pitch[2], dst_col[2];
  float* cell;                     // PRE_MAR_LSTM: c [M, hid], updated in place
  const float* noise;              // PRE_MAR_SAMPLE: [M] standard-normal draws
  float* z;                        // PRE_MAR_SAMPLE: z[b * z_stride + hw]
  long long z_stride;
};

// NV: 128-column groups per lane in the LayerNorm epilogue (1: C <= 128, 2: C <= 256); PAIR: the CTA-pair (cta_group::2)
// build of the dx-split main loop - a separate instantiation, because a kernel that contains cta_group::2 instructions can
// only be launched as a cluster
template <int PRE, int NV, bool F16, bool PAIR = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                 const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                 const __grid_constant__ CUtensorMap map_w2_hi, const __grid_constant__ CUtensorMap map_w2_lo,
                 const Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [stages][A_hi | A_lo | W_hi | W_lo], then barriers
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int BK = F16 ? 64 : BLOCK_K;                 // channels per k-block (128 bytes either way)
  const int w_tile_bytes = p.n_chunk * p.n_chunks * ROW_BYTES;
  const int stage_bytes = 2 * A_TILE_BYTES + 2 * w_tile_bytes;
  // normal mode:   full[stages], empty[stages], tmem_full
  // dx-split mode:  a_full[a_slots], a_empty[a_slots], w_full[w_slots], w_empty[w_slots], tmem_full
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + p.bar_offset);
  uint64_t* empty_bar = full_bar + (p.dxsplit ? p.a_slots : p.stages);
  uint64_t* wfull_bar = empty_bar + p.a_slots;
  uint64_t* wempty_bar = wfull_bar + p.w_slots;
  uint64_t* tmem_full_bar = p.dxsplit ? wempty_bar + p.w_slots : empty_bar + p.stages;
  uint64_t* a3_full_bar = tmem_full_bar + 1;      // chain: operand tiles written by the epilogue warps
  uint64_t* w2_full_bar = tmem_full_bar + 2;
  uint64_t* w2_empty_bar = tmem_full_bar + 3;
  uint64_t* acc2_full_bar = tmem_full_bar + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 5);
  volatile int* failed = reinterpret_cast<volatile int*>(tmem_slot + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x, n_tile = blockIdx.y;
  const int n_base = n_tile * p.n_chunk * p.n_chunks;
  // split-K (normal pipeline only): this CTA's slice [cb0, cb0 + kpt) of every tap's channel blocks
  const int ksp = p.ksplit > 1 ? p.ksplit : 1;
  const int cb0 = (int)((long long)p.kblocks_per_tap * blockIdx.z / ksp);
  const int kpt = (int)((long long)p.kblocks_per_tap * (blockIdx.z + 1) / ksp) - cb0;
  const int num_kb = p.taps * kpt;
  float* const out_f32 = p.out_f32 ? p.out_f32 + (size_t)blockIdx.z * p.M * p.N : nullptr;

  if (threadIdx.x == 0) {
    *failed = 0;
    if (p.dxsplit) {
      for (int s = 0; s < p.a_slots; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
      for (int s = 0; s < p.w_slots; ++s) { mbar_init(&wfull_bar[s], 1); mbar_init(&wempty_bar[s], 1); }
    } else {
      for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(a3_full_bar, EPI_WARPS);
    mbar_init(w2_full_bar, 1);
    mbar_init(w2_empty_bar, 1);
    mbar_init(acc2_full_bar, 1);
    fence_barrier_init();
    prefetch_tmap(&map_a_hi);
    prefetch_tmap(&map_a_lo);
    prefetch_tmap(&map_w_hi);
    prefetch_tmap(&map_w_lo);
  }
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;       // pair mode: rank 0 issues the MMAs of both CTAs
  if (warp == 1) {
    if (PAIR) tmem_alloc_pair(tmem_slot, (uint32_t)p.tmem_cols);
    else tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();         // the peer's barriers must be initialised before anything signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool tracing = p.trace && blockIdx.x == 0 && blockIdx.y == 0;
  if (tracing && threadIdx.x == 0) p.trace[0] = clock64();
  griddep_launch();                 // PDL: the next kernel may start its prologue; it waits on our completion itself

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      // position of this M tile in (b, h, w)
      const int tiles_per_img = (p.H * p.W) / (p.ht * p.wt);        // >= 1 when bt == 1
      int b0, h0;
      if (p.bt > 1) { b0 = m_tile * p.bt; h0 = 0; }
      else { b0 = m_tile / tiles_per_img; h0 = (m_tile % tiles_per_img) * p.ht; }
      griddep_wait();               // PDL: everything before this overlapped the previous kernel's tail; its output is
                                    // complete and visible from here on (all our global writes come after these loads)
      if (PAIR && p.dxsplit) {
        // CTA pair: the same groups; this CTA stages its own activation rows and its HALF of every MMA's weight rows
        // (MMA q of a k-step covers the stacked [dx][n] rows [q n_per, (q + 1) n_per): rank r holds the r-th half), in
        // boxes of w_unit rows that never straddle a dx block.  All transactions count on the LEADER's full barriers.
        uint8_t* w_ring = smem + (size_t)p.a_slots * 2 * A_TILE_BYTES;
        const int groups = 3 * p.kblocks_per_tap;
        const int n_total = 3 * p.n_chunk;
        int n_mma = (n_total + 255) / 256;
        if ((n_total / n_mma) % 16 || n_total % n_mma) n_mma = 3;
        if (p.pair_nmma) n_mma = p.pair_nmma;
        const int half = n_total / n_mma / 2;                        // rows of one MMA's weight tile held by this CTA
        const int lo_off = (n_total / 2) * ROW_BYTES;                // the lo tiles follow the hi tiles inside a slot
        for (int g = 0; g < groups; ++g) {
          const int dyi = g / p.kblocks_per_tap, cb = g % p.kblocks_per_tap;
          const int sa = g % p.a_slots;
          mbar_wait(&empty_bar[sa], (((uint32_t)(g / p.a_slots)) & 1u) ^ 1u, failed);
          uint8_t* at = smem + (size_t)sa * 2 * A_TILE_BYTES;
          const uint32_t afull = mapa_rank(&full_bar[sa], 0);
          if (cta_rank == 0) mbar_expect_tx(&full_bar[sa], 4u * A_TILE_BYTES);
          tma_load_4d_pair(at, &map_a_hi, afull, cb * BK, 0, h0 + dyi - 1, b0);
          tma_load_4d_pair(at + A_TILE_BYTES, &map_a_lo, afull, cb * BK, 0, h0 + dyi - 1, b0);
          const int sw = g % p.w_slots;
          mbar_wait(&wempty_bar[sw], (((uint32_t)(g / p.w_slots)) & 1u) ^ 1u, failed);
          uint8_t* wt = w_ring + (size_t)sw * 3 * w_tile_bytes;
          const uint32_t wfull = mapa_rank(&wfull_bar[sw], 0);
          if (cta_rank == 0) mbar_expect_tx(&wfull_bar[sw], 6u * (uint32_t)w_tile_bytes);
          for (int q = 0; q < n_mma; ++q)
            for (int j = 0; j < half; j += p.w_unit) {
              const int r = q * 2 * half + (int)cta_rank * half + j;  // stacked row = dx * n_chunk + n
              const int dxi = r / p.n_chunk, n = r - dxi * p.n_chunk;
              const int kcol = ((dyi * 3 + dxi) * p.kblocks_per_tap + cb) * BK;
              uint8_t* dst = wt + (size_t)(q * half + j) * ROW_BYTES;
              tma_load_2d_pair(dst, &map_w_hi, wfull, kcol, n_base + n);
              tma_load_2d_pair(dst + lo_off, &map_w_lo, wfull, kcol, n_base + n);
            }
        }
      } else if (p.dxsplit) {
        // group g = (dy, channel block): ONE activation tile (rows shifted by dy, columns unshifted) feeds the three
        // taps (dy, dx = -1, 0, +1); each tap streams its own weight tile.  Activation traffic / 3.
        uint8_t* w_ring = smem + (size_t)p.a_slots * 2 * A_TILE_BYTES;
        const int groups = 3 * p.kblocks_per_tap;
        for (int g = 0; g < groups; ++g) {
          const int dyi = g / p.kblocks_per_tap, cb = g % p.kblocks_per_tap;
          const int sa = g % p.a_slots;
          mbar_wait(&empty_bar[sa], (((uint32_t)(g / p.a_slots)) & 1u) ^ 1u, failed);
          uint8_t* at = smem + (size_t)sa * 2 * A_TILE_BYTES;
          mbar_expect_tx(&full_bar[sa], 2u * A_TILE_BYTES);
          tma_load_4d(at, &map_a_hi, &full_bar[sa], cb * BK, 0, h0 + dyi - 1, b0);
          tma_load_4d(at + A_TILE_BYTES, &map_a_lo, &full_bar[sa], cb * BK, 0, h0 + dyi - 1, b0);
          // the three taps (dy, dx=-1,0,+1) of this group: weight tiles back to back in ONE slot, so that the three
          // per-shift accumulators (adjacent TMEM column ranges) can be fed by wide MMAs
          const int sw = g % p.w_slots;
          mbar_wait(&wempty_bar[sw], (((uint32_t)(g / p.w_slots)) & 1u) ^ 1u, failed);
          uint8_t* wt = w_ring + (size_t)sw * 6 * w_tile_bytes;
          mbar_expect_tx(&wfull_bar[sw], 6u * (uint32_t)w_tile_bytes);
          for (int dxi = 0; dxi < 3; ++dxi) {
            const int kcol = ((dyi * 3 + dxi) * p.kblocks_per_tap + cb) * BK;
            tma_load_2d(wt + dxi * w_tile_bytes, &map_w_hi, &wfull_bar[sw], kcol, n_base);
            tma_load_2d(wt + (3 + dxi) * w_tile_bytes, &map_w_lo, &wfull_bar[sw], kcol, n_base);
          }
        }
      } else
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % p.stages;
        const uint32_t ph = (uint32_t)(kb / p.stages) & 1u;
        mbar_wait(&empty_bar[s], ph ^ 1u, failed);
        uint8_t* st = smem + (size_t)s * stage_bytes;
        const int tap = kb / kpt, cb = cb0 + kb % kpt;
        const int dy = (tap / p.ksz - (p.ksz >> 1)) * p.dil, dx = (tap % p.ksz - (p.ksz >> 1)) * p.dil;
        mbar_expect_tx(&full_bar[s], (uint32_t)stage_bytes);
        tma_load_4d(st, &map_a_hi, &full_bar[s], cb * BK, dx, h0 + dy, b0);
        tma_load_4d(st + A_TILE_BYTES, &map_a_lo, &full_bar[s], cb * BK, dx, h0 + dy, b0);
        const int kcol = (tap * p.kblocks_per_tap + cb) * BK;        // weights are [N, taps*Cin_pad], (tap, c) order
        for (int c = 0; c < p.n_chunks; ++c) {
          const int chunk_bytes = p.n_chunk * ROW_BYTES;
          tma_load_2d(st + 2 * A_TILE_BYTES + c * chunk_bytes, &map_w_hi, &full_bar[s], kcol, n_base + c * p.n_chunk);
          tma_load_2d(st + 2 * A_TILE_BYTES + w_tile_bytes + c * chunk_bytes, &map_w_lo, &full_bar[s], kcol,
                      n_base + c * p.n_chunk);
        }
      }
      if (p.chain) {
        // second GEMM's weights [n2, C]: their slot lies over the (now idle) pipeline stages, so wait for the first
        // GEMM to retire; the load then hides behind the GLU/LayerNorm epilogue
        mbar_wait(tmem_full_bar, 0, failed);
        const int w2_chunk_bytes = p.n2_chunk * ROW_BYTES, w2_half = w2_chunk_bytes * p.n2_chunks;
        const int kb2 = ((p.N >> 1) + BK - 1) / BK;
        for (int kb = 0; kb < kb2; ++kb) {
          mbar_wait(w2_empty_bar, ((uint32_t)kb & 1u) ^ 1u, failed);
          mbar_expect_tx(w2_full_bar, 2u * (uint32_t)w2_half);
          for (int c = 0; c < p.n2_chunks; ++c) {
            tma_load_2d(smem + p.w2_offset + c * w2_chunk_bytes, &map_w2_hi, w2_full_bar, kb * BK, c * p.n2_chunk);
            tma_load_2d(smem + p.w2_offset + w2_half + c * w2_chunk_bytes, &map_w2_lo, w2_full_bar, kb * BK,
                        c * p.n2_chunk);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // the whole warp runs the loop (uniform operands); only the elected lane's tcgen05 instructions execute (umma.cuh)
    const uint32_t leader = elect_one();
    {
      const uint32_t idesc = make_idesc_t<F16>(p.n_chunk);
      if (PAIR && p.dxsplit) {
        if (cta_rank == 0) {
          // M = 256 MMAs over both CTAs' activation tiles; each CTA's slot holds its half of every weight tile
          const uint32_t w_ring = smem_u32(smem + (size_t)p.a_slots * 2 * A_TILE_BYTES);
          const int groups = 3 * p.kblocks_per_tap;
          const int n_total = 3 * p.n_chunk;
          int n_mma = (n_total + 255) / 256;
          if ((n_total / n_mma) % 16 || n_total % n_mma) n_mma = 3;
          if (p.pair_nmma) n_mma = p.pair_nmma;
          const int n_per = n_total / n_mma;
          const uint32_t idesc_w = make_idesc_f16_pair(n_per);
          const uint64_t per_units = (uint64_t)((uint32_t)((n_per / 2) * ROW_BYTES) >> 4);
          const uint64_t lo_units = (uint64_t)((uint32_t)((n_total / 2) * ROW_BYTES) >> 4);
          for (int g = 0; g < groups; ++g) {
            const int sa = g % p.a_slots, sw = g % p.w_slots;
            mbar_wait(&full_bar[sa], ((uint32_t)(g / p.a_slots)) & 1u, failed);
            mbar_wait(&wfull_bar[sw], ((uint32_t)(g / p.w_slots)) & 1u, failed);
            tc_fence_after();
            if (tracing && lane == 0 && g == 0) p.trace[1] = clock64();
            if (tracing && lane == 0 && g == groups - 1) p.trace[2] = clock64();
            const uint32_t a_hi = smem_u32(smem + (size_t)sa * 2 * A_TILE_BYTES);
            const uint32_t w_hi = w_ring + (uint32_t)sw * 3u * (uint32_t)w_tile_bytes;
            const uint64_t da_hi = make_smem_desc(a_hi), da_lo = da_hi + (A_TILE_BYTES >> 4);
            const uint64_t db_hi = make_smem_desc(w_hi), db_lo = db_hi + lo_units;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ko = (uint64_t)(k * 2);
              for (int q = 0; q < n_mma; ++q) {
                const uint64_t bo = ko + q * per_units;
                const uint32_t d = tmem_base + q * n_per;
                umma_f16_pair_elect(d, da_hi + ko, db_hi + bo, idesc_w, (g | k) == 0 ? 0u : 1u, leader);
                umma_f16_pair_elect(d, da_lo + ko, db_hi + bo, idesc_w, 1u, leader);
                umma_f16_pair_elect(d, da_hi + ko, db_lo + bo, idesc_w, 1u, leader);
              }
            }
            umma_commit_pair_elect(&wempty_bar[sw], leader);
            umma_commit_pair_elect(&empty_bar[sa], leader);
          }
          umma_commit_pair_elect(tmem_full_bar, leader);
        }
      } else if (p.dxsplit) {
        const uint32_t w_ring = smem_u32(smem + (size_t)p.a_slots * 2 * A_TILE_BYTES);
        const int groups = 3 * p.kblocks_per_tap;
        // the three accumulators are the TMEM columns [0, 3*n_chunk): cover them with as few MMAs as possible
        // (a K=8 TF32 MMA costs ~100 cycles whatever its N, measured)
        const int n_total = 3 * p.n_chunk;
        int n_mma = (n_total + 255) / 256;
        if ((n_total / n_mma) % 16 || n_total % n_mma) n_mma = 3;
        const int n_per = n_total / n_mma;
        const uint32_t idesc_w = make_idesc_t<F16>(n_per);
        const uint64_t per_units = (uint64_t)((uint32_t)(n_per * ROW_BYTES) >> 4);
        for (int g = 0; g < groups; ++g) {
          const int sa = g % p.a_slots, sw = g % p.w_slots;
          mbar_wait(&full_bar[sa], ((uint32_t)(g / p.a_slots)) & 1u, failed);
          mbar_wait(&wfull_bar[sw], ((uint32_t)(g / p.w_slots)) & 1u, failed);
          tc_fence_after();
          if (tracing && lane == 0 && g == 0) p.trace[1] = clock64();
          if (tracing && lane == 0 && g == groups - 1) p.trace[2] = clock64();
          const uint32_t a_hi = smem_u32(smem + (size_t)sa * 2 * A_TILE_BYTES);
          const uint32_t w_hi = w_ring + (uint32_t)sw * 6u * (uint32_t)w_tile_bytes;
          const uint64_t da_hi = make_smem_desc(a_hi), da_lo = da_hi + (A_TILE_BYTES >> 4);
          const uint64_t db_hi = make_smem_desc(w_hi), db_lo = db_hi + ((3u * (uint32_t)w_tile_bytes) >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) {                               // 4 MMA k-steps of 32 bytes per 128-byte row
            const uint64_t ko = (uint64_t)(k * 2);
            for (int q = 0; q < n_mma; ++q) {
              const uint64_t bo = ko + q * per_units;
              const uint32_t d = tmem_base + q * n_per;
              umma_elect<F16>(d, da_hi + ko, db_hi + bo, idesc_w, (g | k) == 0 ? 0u : 1u, leader);
              umma_elect<F16>(d, da_lo + ko, db_hi + bo, idesc_w, 1u, leader);
              umma_elect<F16>(d, da_hi + ko, db_lo + bo, idesc_w, 1u, leader);
            }
          }
          umma_commit_elect(&wempty_bar[sw], leader);
          umma_commit_elect(&empty_bar[sa], leader);
        }
        umma_commit_elect(tmem_full_bar, leader);
      } else {
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % p.stages;
        const uint32_t ph = (uint32_t)(kb / p.stages) & 1u;
        mbar_wait(&full_bar[s], ph, failed);
        tc_fence_after();
        if (tracing && lane == 0 && kb == 0) p.trace[1] = clock64();
        if (tracing && lane == 0 && kb == num_kb - 1) p.trace[2] = clock64();
        const uint32_t a_hi = smem_u32(smem + (size_t)s * stage_bytes);
        const uint64_t da_hi0 = make_smem_desc(a_hi), da_lo0 = da_hi0 + (A_TILE_BYTES >> 4);
        const uint64_t db_hi0 = da_hi0 + (2 * A_TILE_BYTES >> 4), db_lo0 = db_hi0 + ((uint32_t)w_tile_bytes >> 4);
        const uint64_t chunk_units = (uint64_t)((uint32_t)(p.n_chunk * ROW_BYTES) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t ko = (uint64_t)(k * 2);                     // 16-byte units inside the 128-byte swizzle row
          for (int c = 0; c < p.n_chunks; ++c) {
            const uint64_t co = ko + c * chunk_units;
            const uint32_t d = tmem_base + c * p.n_chunk;
            umma_elect<F16>(d, da_hi0 + ko, db_hi0 + co, idesc, (kb | k) == 0 ? 0u : 1u, leader);
            umma_elect<F16>(d, da_lo0 + ko, db_hi0 + co, idesc, 1u, leader);
            umma_elect<F16>(d, da_hi0 + ko, db_lo0 + co, idesc, 1u, leader);
          }
        }
        umma_commit_elect(&empty_bar[s], leader);                                  // smem slot free once these MMAs retire
      }
      umma_commit_elect(tmem_full_bar, leader);                                    // accumulator complete
      }
      if (p.chain) {
        mbar_wait(a3_full_bar, 0, failed);                           // epilogue warps have written the operand tiles
        tc_fence_after();
        const uint32_t idesc2 = make_idesc_t<F16>(p.n2_chunk);
        const int kb2 = ((p.N >> 1) + BK - 1) / BK;
        const uint32_t w2_half = (uint32_t)(p.n2_chunk * ROW_BYTES * p.n2_chunks);
        const uint64_t chunk2_units = (uint64_t)((uint32_t)(p.n2_chunk * ROW_BYTES) >> 4);
        for (int kb = 0; kb < kb2; ++kb) {
          mbar_wait(w2_full_bar, (uint32_t)kb & 1u, failed);
          tc_fence_after();
          const uint64_t da_hi = make_smem_desc(smem_u32(smem + p.a3_offset + (size_t)kb * 2 * A_TILE_BYTES));
          const uint64_t da_lo = da_hi + (A_TILE_BYTES >> 4);
          const uint64_t db_hi = make_smem_desc(smem_u32(smem + p.w2_offset)), db_lo = db_hi + (w2_half >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t ko = (uint64_t)(k * 2);
            for (int c = 0; c < p.n2_chunks; ++c) {
              const uint64_t co = ko + c * chunk2_units;
              const uint32_t d = tmem_base + p.N + c * p.n2_chunk;   // second accumulator: columns after the first
              umma_elect<F16>(d, da_hi + ko, db_hi + co, idesc2, (kb | k) == 0 ? 0u : 1u, leader);
              umma_elect<F16>(d, da_lo + ko, db_hi + co, idesc2, 1u, leader);
              umma_elect<F16>(d, da_hi + ko, db_lo + co, idesc2, 1u, leader);
            }
          }
          umma_commit_elect(w2_empty_bar, leader);
        }
        umma_commit_elect(acc2_full_bar, leader);
      }
    }
  } else {
    // ===================== epilogue =====================
    // TMEM hands every thread one accumulator ROW (lane).  Writing rows straight to row-major global memory would
    // make each warp store touch 32 different sectors, so tiles go through shared memory (the idle pipeline
    // stages) and are written back with lane == COLUMN: every warp store is one contiguous 128-byte segment, and
    // the per-column vectors (bias, LayerNorm gamma/beta, positional encoding) become coalesced per-lane loads.
    // 16 epilogue warps: the 4 warps that share a TMEM lane group (warp id % 4) split the column chunks.
    const int lane_grp = warp & 3;                                   // TMEM lanes this warp may touch
    const int sub = (warp - 2) >> 2;                                 // 0..3 among the warps of this lane group
    const int slab_row0 = m_tile * BLOCK_M + lane_grp * 32;          // first global row of the 32-row slab
    const uint32_t trow = tmem_base + ((uint32_t)(lane_grp * 32) << 16);
    const int ncols_cta = p.n_chunk * p.n_chunks;
    mbar_wait(tmem_full_bar, 0, failed);
    tc_fence_after();
    // undoes the power-of-two pre-scaling of fp16 weights; from device memory when the weights were packed on the device
    // (read after the accumulator wait: everything this launch depends on is complete by then)
    const float sc = F16 ? (p.acc_scale_ptr ? __ldg(p.acc_scale_ptr) : p.acc_scale) : 1.f;
    if (tracing && threadIdx.x == 64) p.trace[3] = clock64();

    if (PRE == PRE_BIAS) {
      if (p.out_mask & OUT_NCHW) {
        // [b, n, hw] output: consecutive rows are consecutive hw, so the row-per-thread mapping IS the coalesced one
        const int m = slab_row0 + lane;
        const bool valid = m < p.M;
        const int hw = valid ? m % p.HW : 0, img = valid ? m / p.HW : 0;
        for (int j = sub * 16; j < ncols_cta; j += 16 * (EPI_WARPS / 4)) {
          const int n0 = n_base + j;
          if (n0 >= p.N) break;
          float v[16];
          if (p.dxsplit) {                   // combine the three column-shift accumulators (see the row-major path below)
            float vm[16], vp[16];
            tmem_ld16(trow + j, vm);
            tmem_ld16(trow + p.n_chunk + j, v);
            tmem_ld16(trow + 2 * p.n_chunk + j, vp);
            const int wcol = (slab_row0 + lane) % p.W;
            const bool has_l = wcol > 0, has_r = wcol < p.W - 1;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float l = __shfl_up_sync(0xffffffffu, vm[i], 1), r = __shfl_down_sync(0xffffffffu, vp[i], 1);
              v[i] += (has_l ? l : 0.f) + (has_r ? r : 0.f);
            }
          } else {
            tmem_ld16(trow + j, v);
          }
          if (!valid) continue;
          float* o = p.out_nchw + ((size_t)img * p.N + n0) * p.HW + hw;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (n0 + i < p.N) o[(size_t)i * p.HW] = fmaf(v[i], sc, p.bias ? __ldg(p.bias + n0 + i) : 0.f);
        }
      }
      if (p.out_mask & (OUT_F32 | OUT_HILO | OUT_HILO_CELU | OUT_HILO_RELU)) {
        // A. lane == row: accumulator (+ the two shifted neighbours in dx-split mode) + bias -> slab[row][col]
        const int pitch = ncols_cta + 4;                             // float4-aligned, conflict-free for 128-bit access
        float* slab = reinterpret_cast<float*>(smem) + lane_grp * (32 * pitch);
        const int bar_id = 1 + lane_grp;
        for (int j = sub * 16; j < ncols_cta; j += 16 * (EPI_WARPS / 4)) {
          float v[16];
          if (p.dxsplit) {
            // out[r] = P0[r] + P-1[r-1] (unless w == 0) + P+1[r+1] (unless w == W-1): neighbours are the adjacent
            // TMEM lanes = adjacent threads; slab edges coincide with image-row edges (32 % W == 0), where the term is 0
            float vm[16], vp[16];
            tmem_ld16(trow + j, vm);
            tmem_ld16(trow + p.n_chunk + j, v);
            tmem_ld16(trow + 2 * p.n_chunk + j, vp);
            const int wcol = (slab_row0 + lane) % p.W;
            const bool has_l = wcol > 0, has_r = wcol < p.W - 1;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float l = __shfl_up_sync(0xffffffffu, vm[i], 1), r = __shfl_down_sync(0xffffffffu, vp[i], 1);
              v[i] += (has_l ? l : 0.f) + (has_r ? r : 0.f);
            }
          } else {
            tmem_ld16(trow + j, v);
          }
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const int n = n_base + j + i;
            float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bias && n < p.N) bv = __ldg(reinterpret_cast<const float4*>(p.bias + n));
            *reinterpret_cast<float4*>(slab + lane * pitch + j + i) =
                make_float4(fmaf(v[i], sc, bv.x), fmaf(v[i + 1], sc, bv.y), fmaf(v[i + 2], sc, bv.z), fmaf(v[i + 3], sc, bv.w));
          }
        }
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        // B. warp `sub` owns rows sub*8..sub*8+7; a lane owns 4 consecutive columns: 128-bit smem reads, 128-bit
        //    fully coalesced global stores
        for (int c4 = lane * 4; c4 < ncols_cta; c4 += 128) {
          const int n = n_base + c4;
          if (n >= p.N) break;
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) {
            const int r = sub * 8 + rr, m = slab_row0 + r;
            if (m >= p.M) break;
            const float4 y = *reinterpret_cast<const float4*>(slab + r * pitch + c4);
            const float ys[4] = {y.x, y.y, y.z, y.w};
            const size_t o = (size_t)m * p.N + n;
            if (p.out_mask & OUT_F32) *reinterpret_cast<float4*>(out_f32 + o) = y;
            if (p.out_mask & (OUT_HILO | OUT_HILO_RELU)) {             // RELU: NN_net's activations (affine_coupling.py:77-78)
              float t[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) t[i] = (p.out_mask & OUT_HILO_RELU) ? fmaxf(ys[i], 0.f) : ys[i];
              store_hilo4<F16>(p.out_hi, p.out_lo, o, t);
            }
            if (p.out_mask & OUT_HILO_CELU) {                        // concat_elu: [elu(y) | elu(-y)], width 2N
              const size_t o2 = (size_t)m * 2 * p.N + n;
              float t[4], t2[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                t[i] = elu1(ys[i]);
                t2[i] = elu1(-ys[i]);
              }
              store_hilo4<F16>(p.out_hi, p.out_lo, o2, t);
              store_hilo4<F16>(p.out_hi, p.out_lo, o2 + p.N, t2);
            }
          }
        }
      }
    } else if (PRE == PRE_LSTM) {
      // ConvLSTM cell (mar_prior/convolutional_rnn/functional.py:30-52): the accumulator row holds the hidden-to-hidden
      // gate pre-activations [i | f | g | o] (hid columns each); res = the input-to-hidden gates of this step (with their
      // bias), bias = b_hh, gamma = c_{t-1} [M, hid] -> c_t = sig(f) c + sig(i) tanh(g), h_t = sig(o) tanh(c_t).
      // c_t goes to out_f32 [M, hid], h_t to the (hi, lo) operand pair [M, hid] the next step / layer consumes.
      // One thread per row (the first warp of each TMEM lane group), 8 hidden units at a time.
      const int hid = p.N >> 2;
      const int m = slab_row0 + lane;
      if (sub == 0 && m < p.M) {
        const float* gi = p.res + (size_t)m * p.N;
        const float* cp = p.gamma + (size_t)m * hid;
        for (int j = 0; j < hid; j += 8) {
          float acc[4][8];
#pragma unroll
          for (int gte = 0; gte < 4; ++gte) {
            tmem_ld8(trow + gte * hid + j, acc[gte]);
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gi + gte * hid + j));
            const float4 g1 = __ldg(reinterpret_cast<const float4*>(gi + gte * hid + j + 4));
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + gte * hid + j));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + gte * hid + j + 4));
            const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[gte][i] = fmaf(acc[gte][i], sc, bv[i]) + gv[i];
          }
          const float4 c0 = __ldg(reinterpret_cast<const float4*>(cp + j)), c1 = __ldg(reinterpret_cast<const float4*>(cp + j + 4));
          const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
          float cn[8], hn[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float ig = 1.f / (1.f + expf(-acc[0][i])), fg = 1.f / (1.f + expf(-acc[1][i]));
            const float gg = tanhf(acc[2][i]), og = 1.f / (1.f + expf(-acc[3][i]));
            cn[i] = fg * cv[i] + ig * gg;
            hn[i] = og * tanhf(cn[i]);
          }
          float* co = out_f32 + (size_t)m * hid + j;
          *reinterpret_cast<float4*>(co) = make_float4(cn[0], cn[1], cn[2], cn[3]);
          *reinterpret_cast<float4*>(co + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
          store_hilo4<F16>(p.out_hi, p.out_lo, (size_t)m * hid + j, hn);
          store_hilo4<F16>(p.out_hi, p.out_lo, (size_t)m * hid + j + 4, hn + 4);
        }
      }
    } else if (PRE == PRE_MAR_EMBED || PRE == PRE_MAR_LSTM) {
      // One thread per row; the four warps of a TMEM lane group take interleaved 8-column slices.  EMBED: y = D + bias
      // (conv_embed).  LSTM: D holds the gates of W_ih x_t + W_hh h_{t-1} (one GEMM over the [x | h] rows), bias =
      // b_ih + b_hh; c is updated in place (only this thread reads or writes its row).  The result (y, or h_t) goes as an
      // fp16 pair to dst 0 and, when given, dst 1.  TMEM loads are warp-uniform; rows past M only skip their memory accesses.
      const int m = slab_row0 + lane;
      const bool row_ok = m < p.M;
      const int hid = PRE == PRE_MAR_LSTM ? p.N >> 2 : p.N;
      for (int j = sub * 8; j < hid; j += 32) {
        __syncwarp();
        float hn[8];
        if (PRE == PRE_MAR_EMBED) {
          tmem_ld8(trow + j, hn);
#pragma unroll
          for (int i = 0; i < 8; ++i) hn[i] = fmaf(hn[i], sc, __ldg(p.bias + j + i));
        } else {
          float acc[4][8];
#pragma unroll
          for (int gte = 0; gte < 4; ++gte) {
            tmem_ld8(trow + gte * hid + j, acc[gte]);
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[gte][i] = fmaf(acc[gte][i], sc, __ldg(p.bias + gte * hid + j + i));
          }
          if (row_ok) {
            float* cp = p.cell + (size_t)m * hid + j;
            const float4 c0 = *reinterpret_cast<const float4*>(cp), c1 = *reinterpret_cast<const float4*>(cp + 4);
            const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
            float cn[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {            // the accurate forms of the PRE_LSTM cell above
              const float ig = 1.f / (1.f + expf(-acc[0][i])), fg = 1.f / (1.f + expf(-acc[1][i]));
              const float gg = tanhf(acc[2][i]), og = 1.f / (1.f + expf(-acc[3][i]));
              cn[i] = fg * cv[i] + ig * gg;
              hn[i] = og * tanhf(cn[i]);
            }
            *reinterpret_cast<float4*>(cp) = make_float4(cn[0], cn[1], cn[2], cn[3]);
            *reinterpret_cast<float4*>(cp + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
          }
        }
        if (row_ok) {
#pragma unroll
          for (int d = 0; d < 2; ++d) {
            if (!p.dst_hi[d]) continue;
            const size_t o = (size_t)m * p.dst_pitch[d] + p.dst_col[d] + j;
            store_hilo4_f16(reinterpret_cast<float*>(p.dst_hi[d]), reinterpret_cast<float*>(p.dst_lo[d]), o, hn);
            store_hilo4_f16(reinterpret_cast<float*>(p.dst_hi[d]), reinterpret_cast<float*>(p.dst_lo[d]), o + 4, hn + 4);
          }
        }
      }
    } else if (PRE == PRE_MAR_SAMPLE) {
      // conv_out1 over [x | h] with weights [0 | W_out]: columns (mean, log-std) of channel t, never stored.  The sample
      // noise * exp(logs) + mean (corr_prior.py:96-101, same operation order, accurate expf) goes to z[b, t, hw] and, as an
      // fp16 pair, to column dst_col of dst 0 (the next step's input rows).
      if (sub == 0) {
        float v[8];
        tmem_ld8(trow, v);
        const int m = slab_row0 + lane;
        if (m < p.M) {
          const float mean = fmaf(v[0], sc, __ldg(p.bias)), logs = fmaf(v[1], sc, __ldg(p.bias + 1));
          const float s = __fadd_rn(__fmul_rn(__ldg(p.noise + m), expf(logs)), mean);
          p.z[(size_t)(m / p.HW) * p.z_stride + m % p.HW] = s;
          unsigned short h, l;
          split_f16(s, h, l);
          const size_t o = (size_t)m * p.dst_pitch[0] + p.dst_col[0];
          reinterpret_cast<unsigned short*>(p.dst_hi[0])[o] = h;
          reinterpret_cast<unsigned short*>(p.dst_lo[0])[o] = l;
        }
      }
    } else {
      // GLU over the [a | b] halves, + residual, LayerNorm over C = N/2
      // (mixlogcdf_nn.py:92-101 ConvAttnBlock, :257-258 GatedConv gate, :149-151 GatedAttn gate)
      const int C = p.N >> 1;
      const int pitch = C + 4;
      float* slab = reinterpret_cast<float*>(smem) + lane_grp * (32 * pitch);      // shared by the 4 warps of the group
      const int bar_id = 1 + lane_grp;                               // named barrier of this lane group (128 threads)
      const int nv = (C + 127) / 128;
      float g[8][NV][4], pe[8][NV][4];
      float mean[8], rstd[8];
      bool normalized = false;                                       // true: the slab already holds LayerNorm(g) * gamma + beta
      if (NV == 1) {
        // C <= 128.  Everything row-wise happens in the TMEM-lane layout (lane == row): GLU, residual add, BOTH LayerNorm
        // statistics are thread-local sums over the <= 32 columns this thread owns, combined across the four warps of the
        // lane group through 2 x 128 floats of shared memory - no warp-shuffle reductions, no second pass over the slab.
        __shared__ float ln_part[2][4][4][32];                       // [statistic][lane group][warp of the group][lane]
        const int m_row = slab_row0 + lane;
        const bool row_ok = m_row < p.M;
        float gb[2][16];
        float psum = 0.f;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int j = sub * 16 + ci * 64;
          if (j < C) {
            float a[16], b[16];
            tmem_ld16(trow + j, a);
            tmem_ld16(trow + C + j, b);
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              const float4 ba = __ldg(reinterpret_cast<const float4*>(p.bias + j + i));
              const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + C + j + i));
              const float4 rs = row_ok ? __ldg(reinterpret_cast<const float4*>(p.res + (size_t)m_row * C + j + i))
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
              gb[ci][i] = fmaf(a[i], sc, ba.x) * sigmoid_fast(fmaf(b[i], sc, bb.x)) + rs.x;
              gb[ci][i + 1] = fmaf(a[i + 1], sc, ba.y) * sigmoid_fast(fmaf(b[i + 1], sc, bb.y)) + rs.y;
              gb[ci][i + 2] = fmaf(a[i + 2], sc, ba.z) * sigmoid_fast(fmaf(b[i + 2], sc, bb.z)) + rs.z;
              gb[ci][i + 3] = fmaf(a[i + 3], sc, ba.w) * sigmoid_fast(fmaf(b[i + 3], sc, bb.w)) + rs.w;
              psum += (gb[ci][i] + gb[ci][i + 1]) + (gb[ci][i + 2] + gb[ci][i + 3]);
            }
          }
        }
        ln_part[0][lane_grp][sub][lane] = psum;
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        const float mu = ((ln_part[0][lane_grp][0][lane] + ln_part[0][lane_grp][1][lane]) +
                          (ln_part[0][lane_grp][2][lane] + ln_part[0][lane_grp][3][lane])) / (float)C;
        float pvar = 0.f;
#pragma unroll
        for (int ci = 0; ci < 2; ++ci)
          if (sub * 16 + ci * 64 < C) {
#pragma unroll
            for (int i = 0; i < 16; ++i) pvar = fmaf(gb[ci][i] - mu, gb[ci][i] - mu, pvar);
          }
        ln_part[1][lane_grp][sub][lane] = pvar;
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        const float rs_ = rsqrtf(((ln_part[1][lane_grp][0][lane] + ln_part[1][lane_grp][1][lane]) +
                                  (ln_part[1][lane_grp][2][lane] + ln_part[1][lane_grp][3][lane])) / (float)C + 1e-5f);
        if (tracing && threadIdx.x == 64) p.trace[6] = clock64();
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          const int j = sub * 16 + ci * 64;
          if (j < C) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              const float4 ga = __ldg(reinterpret_cast<const float4*>(p.gamma + j + i));
              const float4 be = __ldg(reinterpret_cast<const float4*>(p.beta + j + i));
              *reinterpret_cast<float4*>(slab + lane * pitch + j + i) =
                  make_float4(fmaf((gb[ci][i] - mu) * rs_, ga.x, be.x), fmaf((gb[ci][i + 1] - mu) * rs_, ga.y, be.y),
                              fmaf((gb[ci][i + 2] - mu) * rs_, ga.z, be.z), fmaf((gb[ci][i + 3] - mu) * rs_, ga.w, be.w));
            }
          }
        }
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        if (tracing && threadIdx.x == 64) p.trace[7] = clock64();
        normalized = true;
        // warp `sub` owns rows sub*8..+7, a lane 4 consecutive columns: read the normalised rows back for the output forms
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          const int r = sub * 8 + rr, m = slab_row0 + r;
          const int c4 = lane * 4;
          float4 ps = make_float4(0.f, 0.f, 0.f, 0.f), gv = ps;
          if (c4 < C) {
            gv = *reinterpret_cast<const float4*>(slab + r * pitch + c4);
            if (((p.out_mask & OUT_HILO_POS) || (p.chain && p.pos)) && m < p.M)
              ps = __ldg(reinterpret_cast<const float4*>(p.pos + (size_t)(m % p.HW) * C + c4));
          }
          g[rr][0][0] = gv.x; g[rr][0][1] = gv.y; g[rr][0][2] = gv.z; g[rr][0][3] = gv.w;
          pe[rr][0][0] = ps.x; pe[rr][0][1] = ps.y; pe[rr][0][2] = ps.z; pe[rr][0][3] = ps.w;
          mean[rr] = 0.f;
          rstd[rr] = 1.f;
        }
      } else {
        // 128 < C <= 256: the same scheme with twice the columns per thread.  Everything row-wise happens in the TMEM-lane layout (lane == row): GLU, residual add, BOTH LayerNorm
        // statistics are thread-local sums over the <= 32 columns this thread owns, combined across the four warps of the
        // lane group through 2 x 128 floats of shared memory - no warp-shuffle reductions, no second pass over the slab.
        __shared__ float ln_part2[2][4][4][32];                       // [statistic][lane group][warp of the group][lane]
        const int m_row = slab_row0 + lane;
        const bool row_ok = m_row < p.M;
        float gb[4][16];
        float psum = 0.f;
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
          const int j = sub * 16 + ci * 64;
          if (j < C) {
            float a[16], b[16];
            tmem_ld16(trow + j, a);
            tmem_ld16(trow + C + j, b);
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              const float4 ba = __ldg(reinterpret_cast<const float4*>(p.bias + j + i));
              const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + C + j + i));
              const float4 rs = row_ok ? __ldg(reinterpret_cast<const float4*>(p.res + (size_t)m_row * C + j + i))
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
              gb[ci][i] = fmaf(a[i], sc, ba.x) * sigmoid_fast(fmaf(b[i], sc, bb.x)) + rs.x;
              gb[ci][i + 1] = fmaf(a[i + 1], sc, ba.y) * sigmoid_fast(fmaf(b[i + 1], sc, bb.y)) + rs.y;
              gb[ci][i + 2] = fmaf(a[i + 2], sc, ba.z) * sigmoid_fast(fmaf(b[i + 2], sc, bb.z)) + rs.z;
              gb[ci][i + 3] = fmaf(a[i + 3], sc, ba.w) * sigmoid_fast(fmaf(b[i + 3], sc, bb.w)) + rs.w;
              psum += (gb[ci][i] + gb[ci][i + 1]) + (gb[ci][i + 2] + gb[ci][i + 3]);
            }
          }
        }
        ln_part2[0][lane_grp][sub][lane] = psum;
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        const float mu = ((ln_part2[0][lane_grp][0][lane] + ln_part2[0][lane_grp][1][lane]) +
                          (ln_part2[0][lane_grp][2][lane] + ln_part2[0][lane_grp][3][lane])) / (float)C;
        float pvar = 0.f;
#pragma unroll
        for (int ci = 0; ci < 4; ++ci)
          if (sub * 16 + ci * 64 < C) {
#pragma unroll
            for (int i = 0; i < 16; ++i) pvar = fmaf(gb[ci][i] - mu, gb[ci][i] - mu, pvar);
          }
        ln_part2[1][lane_grp][sub][lane] = pvar;
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        const float rs_ = rsqrtf(((ln_part2[1][lane_grp][0][lane] + ln_part2[1][lane_grp][1][lane]) +
                                  (ln_part2[1][lane_grp][2][lane] + ln_part2[1][lane_grp][3][lane])) / (float)C + 1e-5f);
        if (tracing && threadIdx.x == 64) p.trace[6] = clock64();
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
          const int j = sub * 16 + ci * 64;
          if (j < C) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              const float4 ga = __ldg(reinterpret_cast<const float4*>(p.gamma + j + i));
              const float4 be = __ldg(reinterpret_cast<const float4*>(p.beta + j + i));
              *reinterpret_cast<float4*>(slab + lane * pitch + j + i) =
                  make_float4(fmaf((gb[ci][i] - mu) * rs_, ga.x, be.x), fmaf((gb[ci][i + 1] - mu) * rs_, ga.y, be.y),
                              fmaf((gb[ci][i + 2] - mu) * rs_, ga.z, be.z), fmaf((gb[ci][i + 3] - mu) * rs_, ga.w, be.w));
            }
          }
        }
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        if (tracing && threadIdx.x == 64) p.trace[7] = clock64();
        normalized = true;
        // (the normalised rows are read back from the slab where they are emitted: sixteen float4 per lane would not fit
        // the register budget)
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          mean[rr] = 0.f;
          rstd[rr] = 1.f;
        }
      }
      if (tracing && threadIdx.x == 64) p.trace[8] = clock64();
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c4 = v * 128 + lane * 4;
        if (v >= nv || c4 >= C) {
          // fp16 chain: the second GEMM's last 64-channel k-block is zero beyond C; the lanes that own no column write it
          if (F16 && p.chain && v < nv && c4 < ((C + 63) & ~63)) {
#pragma unroll
            for (int rr = 0; rr < 8; ++rr) {
              const int R = lane_grp * 32 + sub * 8 + rr;
              uint8_t* t = smem + p.a3_offset + (size_t)(c4 >> 6) * 2 * A_TILE_BYTES + R * 128 + ((((c4 & 63) >> 3) ^ (R & 7)) << 4) +
                           ((c4 & 7) << 1);
              *reinterpret_cast<uint2*>(t) = make_uint2(0u, 0u);
              *reinterpret_cast<uint2*>(t + A_TILE_BYTES) = make_uint2(0u, 0u);
            }
          }
          continue;
        }
        const float4 ga = __ldg(reinterpret_cast<const float4*>(p.gamma + c4));
        const float4 be = __ldg(reinterpret_cast<const float4*>(p.beta + c4));
        const float gs[4] = {ga.x, ga.y, ga.z, ga.w}, bs[4] = {be.x, be.y, be.z, be.w};
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          const int m = slab_row0 + sub * 8 + rr;
          if (m >= p.M) {
            if (p.chain) {
              const int R = lane_grp * 32 + sub * 8 + rr;
              if (F16) {
                uint8_t* t = smem + p.a3_offset + (size_t)(c4 >> 6) * 2 * A_TILE_BYTES + R * 128 +
                             ((((c4 & 63) >> 3) ^ (R & 7)) << 4) + ((c4 & 7) << 1);
                *reinterpret_cast<uint2*>(t) = make_uint2(0u, 0u);
                *reinterpret_cast<uint2*>(t + A_TILE_BYTES) = make_uint2(0u, 0u);
              } else {
                const int kb = c4 >> 5, chunk = (c4 & 31) >> 2;
                uint8_t* t = smem + p.a3_offset + (size_t)kb * 2 * A_TILE_BYTES + R * 128 + ((chunk ^ (R & 7)) << 4);
                *reinterpret_cast<float4*>(t) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(t + A_TILE_BYTES) = make_float4(0.f, 0.f, 0.f, 0.f);
              }
            }
            continue;
          }
          float y[4];
          if (NV == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) y[i] = normalized ? g[rr][v][i] : (g[rr][v][i] - mean[rr]) * rstd[rr] * gs[i] + bs[i];
          } else {                                     // wide rows: normalised segment and positional encoding from the slab / L2
            const float4 gv = *reinterpret_cast<const float4*>(slab + (sub * 8 + rr) * pitch + c4);
            float4 ps = make_float4(0.f, 0.f, 0.f, 0.f);
            if ((p.out_mask & OUT_HILO_POS) || (p.chain && p.pos))
              ps = __ldg(reinterpret_cast<const float4*>(p.pos + (size_t)(m % p.HW) * C + c4));
            y[0] = gv.x; y[1] = gv.y; y[2] = gv.z; y[3] = gv.w;
            pe[rr][v][0] = ps.x; pe[rr][v][1] = ps.y; pe[rr][v][2] = ps.z; pe[rr][v][3] = ps.w;
          }
          const size_t o = (size_t)m * C + c4;
          if (p.out_mask & OUT_F32) *reinterpret_cast<float4*>(out_f32 + o) = make_float4(y[0], y[1], y[2], y[3]);
          if (p.out_mask & (OUT_HILO | OUT_HILO_POS)) {
            float t[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) t[i] = y[i] + pe[rr][v][i];                      // pe == 0 unless OUT_HILO_POS
            store_hilo4<F16>(p.out_hi, p.out_lo, o, t);
          }
          if (p.out_mask & OUT_HILO_CELU) {
            const size_t o2 = (size_t)m * 2 * C + c4;
            float t[4], t2[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              t[i] = elu1(y[i]);
              t2[i] = elu1(-y[i]);
            }
            store_hilo4<F16>(p.out_hi, p.out_lo, o2, t);
            store_hilo4<F16>(p.out_hi, p.out_lo, o2 + C, t2);
          }
          if (p.chain) {
            // operand of the chained GEMM, written where the tensor core will read it: K-major tile of 128 rows x 128 B
            // per 32-column block, 16-byte chunks XOR-swizzled with (row % 8) - the layout a SWIZZLE_128B TMA load
            // would have produced
            const int R = lane_grp * 32 + sub * 8 + rr;
            if (F16) {                               // 64 channels per 128-byte row: this lane's 4 columns are half a 16-byte chunk
              unsigned short h[4], l[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) split_f16(y[i] + pe[rr][v][i], h[i], l[i]);
              uint8_t* t = smem + p.a3_offset + (size_t)(c4 >> 6) * 2 * A_TILE_BYTES + R * 128 +
                           ((((c4 & 63) >> 3) ^ (R & 7)) << 4) + ((c4 & 7) << 1);
              *reinterpret_cast<uint2*>(t) = make_uint2((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16));
              *reinterpret_cast<uint2*>(t + A_TILE_BYTES) =
                  make_uint2((uint32_t)l[0] | ((uint32_t)l[1] << 16), (uint32_t)l[2] | ((uint32_t)l[3] << 16));
            } else {
              const int kb = c4 >> 5, chunk = (c4 & 31) >> 2;
              float h[4], l[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) split_tf32(y[i] + pe[rr][v][i], h[i], l[i]);
              uint8_t* t = smem + p.a3_offset + (size_t)kb * 2 * A_TILE_BYTES + R * 128 + ((chunk ^ (R & 7)) << 4);
              *reinterpret_cast<float4*>(t) = make_float4(h[0], h[1], h[2], h[3]);
              *reinterpret_cast<float4*>(t + A_TILE_BYTES) = make_float4(l[0], l[1], l[2], l[3]);
            }
          }
        }
      }
      if (p.chain) {
        fence_proxy_async();                                         // generic-proxy smem writes -> visible to the MMA unit
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(a3_full_bar)) : "memory");
        if (tracing && threadIdx.x == 64) p.trace[9] = clock64();
        // ---- second epilogue: rows of the chained GEMM, fp32 [M, n2]
        mbar_wait(acc2_full_bar, 0, failed);
        tc_fence_after();
        if (tracing && threadIdx.x == 64) p.trace[10] = clock64();
        const int n2 = p.n2, pitch2 = n2 + 4;
        const float sc2 = F16 ? p.acc_scale2 : 1.f;
        float* slab2 = reinterpret_cast<float*>(smem) + lane_grp * (32 * pitch2);   // all smem is idle again
        for (int j = sub * 16; j < n2; j += 16 * (EPI_WARPS / 4)) {
          float v16[16];
          tmem_ld16(trow + p.N + j, v16);
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(slab2 + lane * pitch2 + j + i) =
                make_float4(v16[i] * sc2, v16[i + 1] * sc2, v16[i + 2] * sc2, v16[i + 3] * sc2);
        }
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        for (int c4 = lane * 4; c4 < n2; c4 += 128) {
#pragma unroll
          for (int rr = 0; rr < 8; ++rr) {
            const int r = sub * 8 + rr, m = slab_row0 + r;
            if (m >= p.M) break;
            *reinterpret_cast<float4*>(p.out2_f32 + (size_t)m * n2 + c4) = *reinterpret_cast<const float4*>(slab2 + r * pitch2 + c4);
          }
        }
      }
    }
  }
  if (tracing && threadIdx.x == 64) p.trace[4] = clock64();
  tc_fence_before();
  if (PAIR) cluster_sync_all();         // neither CTA of a pair may retire while the other still uses its memory
  else __syncthreads();
  if (tracing && threadIdx.x == 0) p.trace[5] = clock64();
  if (warp == 1) {
    if (PAIR) tmem_dealloc_pair(tmem_base, (uint32_t)p.tmem_cols);
    else tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
  if (threadIdx.x == 0 && *failed && p.status) *p.status = 1;
}

// --------------------------------------------------------------------------------------------------
// elementwise helpers around the GEMMs
// --------------------------------------------------------------------------------------------------
// NCHW slice -> NHWC hi/lo operand, channel dim zero-padded to c_pad (conditioner input, mixlogcdf_nn.py:66)
template <bool F16>
__global__ void __launch_bounds__(256) nchw_to_nhwc_hilo_kernel(const float* __restrict__ x, long long batch_stride, int c,
                                                               int hw, int c_pad, float* __restrict__ hi,
                                                               float* __restrict__ lo) {
  // 32 pixels x 32 channels per CTA, transposed through shared memory: reads coalesced along the pixels of the NCHW
  // source, writes coalesced along the channels of the NHWC operand pair.  grid = (pixel tiles, channel tiles, B)
  __shared__ float tile[32][33];
  griddep_launch();
  griddep_wait();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* src = x + (size_t)blockIdx.z * batch_stride;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int ch = c0 + ty + 8 * r, p = p0 + tx;
    tile[ty + 8 * r][tx] = (ch < c && p < hw) ? __ldg(src + (size_t)ch * hw + p) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int p = p0 + ty + 8 * r, ch = c0 + tx;
    if (p < hw && ch < c_pad) {
      const size_t o = ((size_t)blockIdx.z * hw + p) * c_pad + ch;
      if (F16) {
        unsigned short h, l;
        split_f16(tile[tx][ty + 8 * r], h, l);
        reinterpret_cast<unsigned short*>(hi)[o] = h;
        reinterpret_cast<unsigned short*>(lo)[o] = l;
      } else {
        float h, l;
        split_tf32(tile[tx][ty + 8 * r], h, l);
        hi[o] = h;
        lo[o] = l;
      }
    }
  }
}

// fp32 rows -> hi/lo operand pair (attention output -> gate GEMM)
template <bool F16>
__global__ void split_hilo_kernel(const float* __restrict__ x, float* __restrict__ hi, float* __restrict__ lo,
                                  long long total, float scale) {
  griddep_launch();
  griddep_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (F16) {
      unsigned short h, l;
      split_f16(x[i] * scale, h, l);
      reinterpret_cast<unsigned short*>(hi)[i] = h;
      reinterpret_cast<unsigned short*>(lo)[i] = l;
    } else {
      float h, l;
      split_tf32(x[i], h, l);
      hi[i] = h;
      lo[i] = l;
    }
  }
}

// --------------------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------------------
// `es` = element size: 4 (tf32 values in fp32 containers, 32 channels per box) or 2 (fp16, 64 channels per box); a box
// that reaches past C (C not a multiple of the block) is zero-filled by the TMA unit
static bool make_map_act(CUtensorMap* map, const float* base, int B, int H, int W, int C, int bt, int ht, int wt, int es) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * es, (cuuint64_t)W * C * es, (cuuint64_t)H * W * C * es};
  cuuint32_t box[4] = {(cuuint32_t)(ROW_BYTES / es), (cuuint32_t)wt, (cuuint32_t)ht, (cuuint32_t)bt};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return encode_fn()(map, es == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static bool make_map_w(CUtensorMap* map, const float* base, int N, int Ktot, int rows, int es) {
  cuuint64_t dims[2] = {(cuuint64_t)Ktot, (cuuint64_t)N};
  cuuint64_t strides[1] = {(cuuint64_t)Ktot * es};
  cuuint32_t box[2] = {(cuuint32_t)(ROW_BYTES / es), (cuuint32_t)rows};
  cuuint32_t estr[2] = {1, 1};
  return encode_fn()(map, es == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// split-K finish: out = sum_s partial[s][m][n] + bias[n], as fp32 rows [M, N] or NCHW [B, N, HW]; slices in index order.
// 32 x 32 (m, n) tiles: the partial rows are read coalesced along n, transposed through shared memory and written
// coalesced along the pixels of the NCHW destination (or straight back as rows).
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ bias,
                                                            float* __restrict__ out_f32, float* __restrict__ out_nchw,
                                                            int M, int N, int HW, int splits) {
  __shared__ float tile[32][33];
  griddep_wait();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int m0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
  const size_t slice = (size_t)M * N;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int m = m0 + ty + 8 * r, n = n0 + tx;
    float acc = 0.f;
    if (m < M && n < N) {
      const float* q = partial + (size_t)m * N + n;
      acc = bias ? bias[n] : 0.f;
      for (int s = 0; s < splits; ++s) acc += q[s * slice];
      if (out_f32) out_f32[(size_t)m * N + n] = acc;
    }
    tile[ty + 8 * r][tx] = acc;
  }
  if (!out_nchw) return;
  __syncthreads();
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int n = n0 + ty + 8 * r, m = m0 + tx;
    if (m < M && n < N) {
      const int b = m / HW, hw = m - b * HW;
      out_nchw[((size_t)b * N + n) * HW + hw] = tile[tx][ty + 8 * r];
    }
  }
}

// How many K slices flowk_conv_gemm would use for this layer given a workspace (1 = no split-K).  Split-K serves the
// latency of single-stream (training) steps: layers with few 128-row tiles and a long K loop (deep levels, the
// out_conv input-gradient with K = 9 * 98c) otherwise run on a handful of SMs.
static int plan_ksplit(int m_tiles, int n_tiles, int kpt, int taps) {
  const int ctas = m_tiles * n_tiles, num_kb = taps * kpt;
  if (ctas * 2 > 148 || num_kb < 32) return 1;
  int ks = 148 / ctas;
  if (ks > kpt) ks = kpt;
  if (ks > num_kb / 8) ks = num_kb / 8;
  return ks < 2 ? 1 : ks;
}

}  // namespace tc
}  // namespace flowk

using namespace flowk;
using namespace flowk::tc;

static int conv_gemm_impl(const flowk_conv_gemm_args* a, flowk_stream_t stream, int* plan_only);

extern "C" int flowk_conv_gemm(const flowk_conv_gemm_args* a, flowk_stream_t stream) {
  return conv_gemm_impl(a, stream, nullptr);
}

// Number of split-K slices flowk_conv_gemm will use for `args` IF args->splitk_ws is non-null (>= 1; the workspace
// must then hold slices * B*H*W * N floats).  Pointers in `args` are not dereferenced.
extern "C" int flowk_conv_gemm_splitk_slices(const flowk_conv_gemm_args* a) {
  int ks = 1;
  const int st = conv_gemm_impl(a, nullptr, &ks);
  return st == FLOWK_OK ? ks : 1;
}

static int conv_gemm_impl(const flowk_conv_gemm_args* a, flowk_stream_t stream, int* plan_only) {
  if (!a) return FLOWK_ERR_ARG;
  if (!plan_only && (!a->a_hi || !a->a_lo || !a->w_hi || !a->w_lo)) return FLOWK_ERR_ARG;
  const int B = a->B, H = a->H, W = a->W, Cin = a->Cin, N = a->N;
  const bool f16 = a->operand_format == FLOWK_OPERAND_F16;
  if (a->operand_format != FLOWK_OPERAND_TF32 && !f16) return FLOWK_ERR_ARG;
  const int es = f16 ? 2 : 4, bk = ROW_BYTES / es;            // channels per k-block
  if (B < 1 || H < 1 || W < 1 || N < 1) return FLOWK_ERR_SHAPE;
  if (f16 ? (Cin < 8 || Cin % 8) : (Cin < BLOCK_K || Cin % BLOCK_K)) return FLOWK_ERR_SHAPE;   // 16-byte row pitch / whole blocks
  if (f16 && !(a->acc_scale > 0.f)) return FLOWK_ERR_ARG;
  if (a->taps != 1 && a->taps != 9 && a->taps != 25) return FLOWK_ERR_ARG;
  const int dil = a->dilation > 0 ? a->dilation : 1;
  if (a->pre != PRE_BIAS && a->pre != PRE_GLU_RES_LN && a->pre != PRE_LSTM) return FLOWK_ERR_ARG;
  if (!plan_only && !encode_fn()) return FLOWK_ERR_ARG;      // planning is a pure host computation
  // M tile = bt images x ht rows x W columns = 128 positions
  int wt = W, ht, bt;
  if (W > BLOCK_M || BLOCK_M % W) return FLOWK_ERR_SHAPE;
  if (H * W >= BLOCK_M) {
    if ((H * W) % BLOCK_M) return FLOWK_ERR_SHAPE;
    ht = BLOCK_M / W;
    bt = 1;
  } else {
    if (BLOCK_M % (H * W)) return FLOWK_ERR_SHAPE;
    ht = H;
    bt = BLOCK_M / (H * W);
  }
  Params p{};
  p.M = B * H * W;
  p.N = N;
  p.HW = H * W;
  p.W = W;
  p.H = H;
  p.taps = a->taps;
  p.ksz = a->taps == 25 ? 5 : a->taps == 9 ? 3 : 1;
  p.dil = dil;
  p.kblocks_per_tap = (Cin + bk - 1) / bk;
  p.acc_scale = f16 ? a->acc_scale : 1.f;
  p.acc_scale_ptr = f16 ? a->acc_scale_ptr : nullptr;
  p.wt = wt;
  p.ht = ht;
  p.bt = bt;
  p.pre = a->pre;
  p.out_mask = a->out_mask;
  p.bias = a->bias;
  p.res = a->res;
  p.gamma = a->gamma;
  p.beta = a->beta;
  p.pos = a->pos;
  p.out_f32 = a->out_f32;
  p.out_hi = a->out_hi;
  p.out_lo = a->out_lo;
  p.out_nchw = a->out_nchw;
  p.status = a->status;
  p.trace = a->trace;
  p.out2_f32 = a->out2_f32;
  int n_tiles;
  if (a->pre == PRE_GLU_RES_LN) {
    const int C = N / 2;
    if ((N & 1) || C % 16 || C > 256 || !a->res || !a->gamma || !a->beta || !a->bias) return FLOWK_ERR_SHAPE;
    if (N <= 256) { p.n_chunk = N; p.n_chunks = 1; }
    else { p.n_chunk = C; p.n_chunks = 2; }
    n_tiles = 1;
  } else if (a->pre == PRE_LSTM) {
    // N = 4 * hid gate columns, all in one CTA (the cell update needs the four gates of a unit together)
    if (N % 32 || N > 256 || !a->res || !a->gamma || !a->bias || !a->out_f32 || !a->out_hi || !a->out_lo) return FLOWK_ERR_SHAPE;
    p.n_chunk = N;
    p.n_chunks = 1;
    n_tiles = 1;
  } else {
    // split N into tiles of <= 256 columns, multiple of 16 (rows past N are zero-filled by TMA)
    const int n16 = (N + 15) / 16 * 16;
    n_tiles = (n16 + 255) / 256;
    int per = (n16 / 16 + n_tiles - 1) / n_tiles * 16;
    p.n_chunk = per;
    p.n_chunks = 1;
    const int m_tiles = (B * H * W + BLOCK_M - 1) / BLOCK_M;
    if (n_tiles == 2 && !(a->out_mask & OUT_NCHW) && m_tiles * 2 > 148 && n16 <= 384) {   // (epilogue slab must fit)
      n_tiles = 1;                                       // 256 < N <= 512 on a full machine: one CTA, two accumulator
      p.n_chunks = 2;                                    // chunks -> one wave instead of two
    }
    if (a->taps == 9 && !(a->out_mask & OUT_NCHW) && W <= 32 && 32 % W == 0 && p.n_chunks == 1)
      while (3 * p.n_chunk > 512 && p.n_chunk % 32 == 0) { p.n_chunk /= 2; n_tiles *= 2; }
    // Few M tiles (deep levels, small batches): per-CTA time is bound by the ~32 B/clk an SM can pull from / push to
    // L2, so spread the output columns over the idle SMs - narrower weight tiles and narrower epilogues per CTA.
    while (p.n_chunks == 1 && p.n_chunk % 32 == 0 && p.n_chunk >= 64 && m_tiles * n_tiles * 2 <= 148) {
      p.n_chunk /= 2;
      n_tiles *= 2;
    }
    // 3x3 layers (long main loop bound by the ~45 B/clk one SM ingests through TMA; every CTA streams its slice of the
    // weights): take the finest split of N into equal multiples of 16 columns that still fits one wave - N = 96: 6 x 16
    // columns on 8 M tiles, 3 x 32 on 32 M tiles.
    if (a->taps == 9 && p.n_chunks == 1 && N % 16 == 0 && p.n_chunk * n_tiles == N) {
      const int units = N / 16;
      for (int d = units; d > n_tiles; --d)
        if (units % d == 0 && m_tiles * d <= 148) {
          n_tiles = d;
          p.n_chunk = N / d;
          break;
        }
    }
  }
  if (p.n_chunk % 16 || p.n_chunk > 256) return FLOWK_ERR_SHAPE;
  // split-K: only the plain bias epilogue with a single fp32 destination, and only when the caller lends a workspace
  p.ksplit = 1;
  if (a->pre == PRE_BIAS && p.n_chunks == 1 && (a->out_mask == OUT_NCHW || a->out_mask == OUT_F32) && !(N & 3) &&
      (plan_only || a->splitk_ws))
    p.ksplit = plan_ksplit((B * H * W + BLOCK_M - 1) / BLOCK_M, n_tiles, p.kblocks_per_tap, a->taps);
  if (plan_only) {
    *plan_only = p.ksplit;
    return FLOWK_OK;
  }
  if (p.ksplit > 1) {                 // partial rows [slice][M][N] into the workspace; the reduce kernel adds the bias
    p.out_mask = OUT_F32;
    p.out_f32 = a->splitk_ws;
    p.out_nchw = nullptr;
    p.bias = nullptr;
  }
  const int cols = p.n_chunk * p.n_chunks;
  p.tmem_cols = cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512;
  const int stage_bytes = 2 * A_TILE_BYTES + 2 * cols * ROW_BYTES;
  int stages = (int)((220 * 1024 - 2048) / stage_bytes);
  if (stages > 6) stages = 6;
  if (stages < 1) return FLOWK_ERR_SHAPE;
  // Co-residency: kernels whose accumulators fit 256 TMEM columns can share an SM with a second CTA (of the same launch
  // or of another stream's launch) if they also fit half of the shared memory; their prologues / epilogues, which are
  // latency-bound, then overlap the neighbour's main loop.  FLOWK_GEMM_SMEM_CAP_KB caps the pipeline depth accordingly.
  static int smem_cap_kb = -1;
  if (smem_cap_kb < 0) { const char* e = getenv("FLOWK_GEMM_SMEM_CAP_KB"); smem_cap_kb = e ? atoi(e) : 0; }
  if (smem_cap_kb > 0 && p.tmem_cols <= 256)
    while (stages > 1 && (size_t)stages * stage_bytes > (size_t)smem_cap_kb * 1024) --stages;
  // 3x3 dx-split mode: three accumulators (one per column shift) so that an activation tile serves three taps
  p.dxsplit = (a->taps == 9 && dil == 1 && a->pre == PRE_BIAS && W <= 32 && 32 % W == 0 && p.n_chunks == 1 &&
               3 * p.n_chunk <= 512 && p.ksplit == 1) ? 1 : 0;
  // CTA pairs (cta_group::2) for the dx-split 3x3 layers that fill the machine: the main loop of these is bound by the
  // bytes ONE SM ingests through TMA, most of them weights that every CTA streams in full - a pair shares them, each CTA
  // staging half of the rows.  Needs an even number of M tiles (the pair = M tiles 2i, 2i + 1) and fp16 operands.
  p.pair = 0;
  if (p.dxsplit && f16) {
    static int pair_env = -1, nmma_env = 0;
    if (pair_env < 0) {
      const char* e = getenv("FLOWK_PAIR");
      pair_env = e ? atoi(e) : 0;
      e = getenv("FLOWK_PAIR_NMMA");
      nmma_env = e ? atoi(e) : 0;
    }
    const int m_tiles = (p.M + BLOCK_M - 1) / BLOCK_M;
    const int n_total = 3 * p.n_chunk;
    int n_mma = (n_total + 255) / 256;
    if ((n_total / n_mma) % 16 || n_total % n_mma) n_mma = 3;
    if (nmma_env == 3) n_mma = p.pair_nmma = 3;
    const int half = n_total / n_mma / 2;
    int unit = half;                                             // largest box that tiles `half` without straddling a dx block
    while (unit > 0 && (half % unit || p.n_chunk % unit || unit % 8)) unit -= 8;
    if (pair_env && m_tiles % 2 == 0 && p.M % BLOCK_M == 0 && m_tiles * n_tiles >= 64 && (n_total / n_mma) % 16 == 0 &&
        half % 8 == 0 && unit >= 8) {
      p.pair = 1;
      p.w_unit = unit;
    }
  }
  if (p.dxsplit) {
    p.tmem_cols = 3 * p.n_chunk <= 256 ? 256 : 512;
    if (3 * p.n_chunk <= 128) p.tmem_cols = 128;
    const int w_slot_bytes = (p.pair ? 3 : 6) * cols * ROW_BYTES;   // 3 column shifts x (hi, lo); a pair's CTA holds half
    // narrow N tiles (deep levels): the activation tiles dominate the bytes, so give THEM the deeper ring
    p.a_slots = (220 * 1024 - 2048 - 4 * 2 * A_TILE_BYTES) / w_slot_bytes >= 3 ? 4 : 2;
    if (const char* e = getenv("FLOWK_A_SLOTS")) p.a_slots = atoi(e);   // tuning knob
    int ws = (int)((220 * 1024 - 2048 - p.a_slots * 2 * A_TILE_BYTES) / w_slot_bytes);
    p.w_slots = ws > 4 ? 4 : ws;
    if (p.w_slots < 2) p.dxsplit = 0;
  }
  // epilogue staging (reuses the pipeline stages once the accumulator is complete)
  size_t epi_bytes = (size_t)4 * 32 * (cols + 4) * sizeof(float);
  if (a->pre == PRE_GLU_RES_LN) epi_bytes = (size_t)4 * 32 * (N / 2 + 4) * sizeof(float);
  if ((p.out_mask & (OUT_F32 | OUT_HILO | OUT_HILO_POS | OUT_HILO_CELU | OUT_HILO_RELU)) && (N & 3)) return FLOWK_ERR_SHAPE;
  while (stages > 1 && (size_t)stages * stage_bytes + 2048 > 227 * 1024) --stages;
  size_t region = (size_t)stages * stage_bytes;
  if (p.dxsplit) region = (size_t)p.a_slots * 2 * A_TILE_BYTES + (size_t)p.w_slots * (p.pair ? 3 : 6) * cols * ROW_BYTES;
  if (epi_bytes > region) region = (epi_bytes + 1023) / 1024 * 1024;
  if (region + 2048 > 227 * 1024) return FLOWK_ERR_SHAPE;
  // chained second GEMM (gate -> in_proj): needs both accumulators in TMEM and the operand / weight tiles in smem
  p.chain = 0;
  if (a->w2_hi && a->w2_lo && a->out2_f32 && a->N2 > 0) {
    const int C = N / 2, n2 = a->N2;
    if (a->pre != PRE_GLU_RES_LN || p.n_chunks != 1 || C % (f16 ? 8 : BLOCK_K) || n2 % 16 || N + n2 > 512) return FLOWK_ERR_SHAPE;
    if (f16 && !(a->acc_scale2 > 0.f)) return FLOWK_ERR_ARG;
    const int kb2 = (C + bk - 1) / bk;                       // k-blocks of the second GEMM
    p.acc_scale2 = f16 ? a->acc_scale2 : 1.f;
    p.n2 = n2;
    p.n2_chunks = n2 <= 256 ? 1 : 2;
    p.n2_chunk = n2 / p.n2_chunks;
    if (p.n2_chunk % 16 || p.n2_chunk > 256) return FLOWK_ERR_SHAPE;
    const size_t slab = (size_t)4 * 32 * (C + 4) * sizeof(float);
    p.a3_offset = (int)((slab + 1023) / 1024 * 1024);
    p.w2_offset = p.a3_offset + kb2 * 2 * A_TILE_BYTES;
    const size_t chain_end = (size_t)p.w2_offset + (size_t)2 * n2 * ROW_BYTES;
    const size_t slab2 = (size_t)4 * 32 * (n2 + 4) * sizeof(float);
    if (chain_end > region) region = (chain_end + 1023) / 1024 * 1024;
    if (slab2 > region) region = (slab2 + 1023) / 1024 * 1024;
    if (region + 2048 > 227 * 1024) return FLOWK_ERR_SHAPE;
    p.tmem_cols = 512;
    p.chain = 1;
  }
  p.stages = stages;
  p.bar_offset = (int)region;
  const size_t smem_bytes = region + 1024 + 256;

  alignas(64) CUtensorMap ma_hi, ma_lo, mw_hi, mw_lo, mw2_hi, mw2_lo;
  const int Ktot = a->taps * p.kblocks_per_tap * bk;          // weights: every tap padded to whole k-blocks
  if (!make_map_act(&ma_hi, a->a_hi, B, H, W, Cin, bt, ht, wt, es) || !make_map_act(&ma_lo, a->a_lo, B, H, W, Cin, bt, ht, wt, es) ||
      !make_map_w(&mw_hi, a->w_hi, N, Ktot, p.pair ? p.w_unit : p.n_chunk, es) ||
      !make_map_w(&mw_lo, a->w_lo, N, Ktot, p.pair ? p.w_unit : p.n_chunk, es))
    return FLOWK_ERR_ARG;
  if (p.chain) {
    const int k2tot = f16 ? ((N / 2 + bk - 1) / bk) * bk : N / 2;          // fp16 weights: rows padded to whole 64-channel blocks
    if (!make_map_w(&mw2_hi, a->w2_hi, p.n2, k2tot, p.n2_chunk, es) || !make_map_w(&mw2_lo, a->w2_lo, p.n2, k2tot, p.n2_chunk, es))
      return FLOWK_ERR_ARG;
  } else {
    mw2_hi = mw_hi;
    mw2_lo = mw_lo;
  }

  dim3 grid((p.M + BLOCK_M - 1) / BLOCK_M, n_tiles, p.ksplit);
  // one launch helper per (epilogue, LayerNorm width, operand format) instantiation; each remembers the largest dynamic
  // shared-memory opt-in it has requested
#define FLOWK_LAUNCH_GEMM(PRE_, NV_, F16_, PAIR_)                                                                         \
  do {                                                                                                              \
    static size_t smem_set = 0;                                                                                     \
    if (smem_bytes > smem_set) {                                                                                    \
      FLOWK_CUDA_OK(cudaFuncSetAttribute(conv_gemm_kernel<PRE_, NV_, F16_, PAIR_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                         (int)smem_bytes));                                                         \
      smem_set = smem_bytes;                                                                                        \
    }                                                                                                               \
    FLOWK_CUDA_OK(launch_pdl_cluster(conv_gemm_kernel<PRE_, NV_, F16_, PAIR_>, grid, dim3(NUM_THREADS), smem_bytes, stream,          \
                                     PAIR_ ? 2 : 1, ma_hi, ma_lo, mw_hi, mw_lo, mw2_hi, mw2_lo, p));               \
  } while (0)
  if (a->pre == PRE_LSTM) {
    if (f16) FLOWK_LAUNCH_GEMM(PRE_LSTM, 1, true, false); else FLOWK_LAUNCH_GEMM(PRE_LSTM, 1, false, false);
  } else if (a->pre == PRE_GLU_RES_LN && N / 2 > 128) {
    if (f16) FLOWK_LAUNCH_GEMM(PRE_GLU_RES_LN, 2, true, false); else FLOWK_LAUNCH_GEMM(PRE_GLU_RES_LN, 2, false, false);
  } else if (a->pre == PRE_GLU_RES_LN) {
    if (f16) FLOWK_LAUNCH_GEMM(PRE_GLU_RES_LN, 1, true, false); else FLOWK_LAUNCH_GEMM(PRE_GLU_RES_LN, 1, false, false);
  } else if (p.pair) {
    FLOWK_LAUNCH_GEMM(PRE_BIAS, 1, true, true);
  } else {
    if (f16) FLOWK_LAUNCH_GEMM(PRE_BIAS, 1, true, false); else FLOWK_LAUNCH_GEMM(PRE_BIAS, 1, false, false);
  }
#undef FLOWK_LAUNCH_GEMM
  if (p.ksplit > 1) {
    FLOWK_CUDA_OK(launch_pdl(splitk_reduce_kernel, dim3((p.M + 31) / 32, (N + 31) / 32), dim3(256), 0, stream, (const float*)a->splitk_ws, a->bias,
                             a->out_mask == OUT_F32 ? a->out_f32 : (float*)nullptr,
                             a->out_mask == OUT_NCHW ? a->out_nchw : (float*)nullptr, p.M, N, p.HW, p.ksplit));
  }
  return launch_status();
}

// A destination (hi, lo, pitch, column) of `width` fp16 elements per row; 8-byte stores need pitch and column % 4.
static int check_mar_dst(const void* hi, const void* lo, int pitch, int col, int width) {
  if (!hi || !lo) return FLOWK_ERR_ARG;
  if (pitch < 1 || col < 0 || col + width > pitch || (width > 1 && (pitch % 4 || col % 4))) return FLOWK_ERR_SHAPE;
  return FLOWK_OK;
}

extern "C" int flowk_mar_step(const flowk_mar_step_args* a, flowk_stream_t stream) {
  if (!a) return FLOWK_ERR_ARG;
  const int mode = a->mode;
  if (mode != FLOWK_MAR_EMBED && mode != FLOWK_MAR_LSTM && mode != FLOWK_MAR_SAMPLE) return FLOWK_ERR_ARG;
  if (!a->a_hi || !a->a_lo || !a->w_hi || !a->w_lo || !a->bias) return FLOWK_ERR_ARG;
  if (mode == FLOWK_MAR_LSTM && !a->c) return FLOWK_ERR_ARG;
  if (mode == FLOWK_MAR_SAMPLE && (!a->noise || !a->z)) return FLOWK_ERR_ARG;
  if (a->taps != 1 && a->taps != 9 && a->taps != 25) return FLOWK_ERR_ARG;
  if (!(a->acc_scale > 0.f)) return FLOWK_ERR_ARG;
  const int B = a->B, H = a->H, W = a->W, Cin = a->Cin, hid = a->hid;
  if (B < 1 || H < 1 || W < 1 || Cin < 8 || Cin % 8) return FLOWK_ERR_SHAPE;
  if (hid < 8 || hid % 8 || 4 * hid > 256) return FLOWK_ERR_SHAPE;
  const int width = mode == FLOWK_MAR_SAMPLE ? 1 : hid;
  int st = check_mar_dst(a->dst0_hi, a->dst0_lo, a->dst0_pitch, a->dst0_col, width);
  if (st != FLOWK_OK) return st;
  const bool dst1 = mode == FLOWK_MAR_LSTM && (a->dst1_hi || a->dst1_lo);
  if (dst1 && (st = check_mar_dst(a->dst1_hi, a->dst1_lo, a->dst1_pitch, a->dst1_col, width)) != FLOWK_OK) return st;
  if (mode == FLOWK_MAR_SAMPLE && a->z_stride < (long long)H * W) return FLOWK_ERR_SHAPE;
  if (W > BLOCK_M || BLOCK_M % W) return FLOWK_ERR_SHAPE;
  if (H * W >= BLOCK_M ? (H * W) % BLOCK_M != 0 : BLOCK_M % (H * W) != 0) return FLOWK_ERR_SHAPE;
  if (!encode_fn()) return FLOWK_ERR_ARG;

  const int N = mode == FLOWK_MAR_LSTM ? 4 * hid : mode == FLOWK_MAR_EMBED ? hid : 2;
  constexpr int bk = 64;                                       // fp16 channels per k-block
  Params p{};
  p.M = B * H * W;
  p.N = N;
  p.HW = H * W;
  p.W = W;
  p.H = H;
  p.taps = a->taps;
  p.ksz = a->taps == 25 ? 5 : a->taps == 9 ? 3 : 1;
  p.dil = a->dilation > 0 ? a->dilation : 1;
  p.kblocks_per_tap = (Cin + bk - 1) / bk;
  p.wt = W;
  p.ht = H * W >= BLOCK_M ? BLOCK_M / W : H;
  p.bt = H * W >= BLOCK_M ? 1 : BLOCK_M / (H * W);
  p.n_chunk = (N + 15) / 16 * 16;                              // weight rows past N are zero-filled by TMA
  p.n_chunks = 1;
  p.ksplit = 1;
  p.pre = PRE_MAR_EMBED + mode;
  p.bias = a->bias;
  p.acc_scale = a->acc_scale;
  p.status = a->status;
  p.dst_hi[0] = a->dst0_hi;
  p.dst_lo[0] = a->dst0_lo;
  p.dst_pitch[0] = a->dst0_pitch;
  p.dst_col[0] = a->dst0_col;
  if (dst1) {
    p.dst_hi[1] = a->dst1_hi;
    p.dst_lo[1] = a->dst1_lo;
    p.dst_pitch[1] = a->dst1_pitch;
    p.dst_col[1] = a->dst1_col;
  }
  p.cell = a->c;
  p.noise = a->noise;
  p.z = a->z;
  p.z_stride = a->z_stride;
  p.tmem_cols = p.n_chunk <= 32 ? 32 : p.n_chunk <= 64 ? 64 : p.n_chunk <= 128 ? 128 : 256;
  const int stage_bytes = 2 * A_TILE_BYTES + 2 * p.n_chunk * ROW_BYTES;
  int stages = (220 * 1024 - 2048) / stage_bytes;
  if (stages > 6) stages = 6;
  p.stages = stages;
  p.bar_offset = stages * stage_bytes;                         // these epilogues stage nothing in shared memory
  const size_t smem_bytes = (size_t)p.bar_offset + 1024 + 256;

  alignas(64) CUtensorMap ma_hi, ma_lo, mw_hi, mw_lo;
  const int Ktot = p.taps * p.kblocks_per_tap * bk;
  if (!make_map_act(&ma_hi, (const float*)a->a_hi, B, H, W, Cin, p.bt, p.ht, p.wt, 2) ||
      !make_map_act(&ma_lo, (const float*)a->a_lo, B, H, W, Cin, p.bt, p.ht, p.wt, 2) ||
      !make_map_w(&mw_hi, (const float*)a->w_hi, N, Ktot, p.n_chunk, 2) ||
      !make_map_w(&mw_lo, (const float*)a->w_lo, N, Ktot, p.n_chunk, 2))
    return FLOWK_ERR_ARG;
  const dim3 grid((p.M + BLOCK_M - 1) / BLOCK_M, 1, 1);
#define FLOWK_LAUNCH_MAR(PRE_)                                                                                          \
  do {                                                                                                                  \
    static size_t smem_set = 0;                                                                                         \
    if (smem_bytes > smem_set) {                                                                                        \
      FLOWK_CUDA_OK(cudaFuncSetAttribute(conv_gemm_kernel<PRE_, 1, true, false>,                                        \
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));                \
      smem_set = smem_bytes;                                                                                            \
    }                                                                                                                   \
    FLOWK_CUDA_OK(launch_pdl_cluster(conv_gemm_kernel<PRE_, 1, true, false>, grid, dim3(NUM_THREADS), smem_bytes,       \
                                     stream, 1, ma_hi, ma_lo, mw_hi, mw_lo, mw_hi, mw_lo, p));                          \
  } while (0)
  if (mode == FLOWK_MAR_EMBED) FLOWK_LAUNCH_MAR(PRE_MAR_EMBED);
  else if (mode == FLOWK_MAR_LSTM) FLOWK_LAUNCH_MAR(PRE_MAR_LSTM);
  else FLOWK_LAUNCH_MAR(PRE_MAR_SAMPLE);
#undef FLOWK_LAUNCH_MAR
  return launch_status();
}

extern "C" int flowk_nchw_to_nhwc_hilo(const float* x, long long batch_stride, int B, int C, int HW, int C_pad,
                                       float* hi, float* lo, flowk_stream_t stream) {
  if (B < 0 || C < 1 || HW < 1 || C_pad < C) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!x || !hi || !lo) return FLOWK_ERR_ARG;
  if (B > 65535) return FLOWK_ERR_SHAPE;
  FLOWK_CUDA_OK(launch_pdl(nchw_to_nhwc_hilo_kernel<false>, dim3((HW + 31) / 32, (C_pad + 31) / 32, B), dim3(256), 0, stream, x,
                           batch_stride, C, HW, C_pad, hi, lo));
  return launch_status();
}

extern "C" int flowk_nchw_to_nhwc_hilo_f16(const float* x, long long batch_stride, int B, int C, int HW, int C_pad,
                                           void* hi, void* lo, flowk_stream_t stream) {
  if (B < 0 || C < 1 || HW < 1 || C_pad < C || C_pad % 8) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!x || !hi || !lo) return FLOWK_ERR_ARG;
  if (B > 65535) return FLOWK_ERR_SHAPE;
  FLOWK_CUDA_OK(launch_pdl(nchw_to_nhwc_hilo_kernel<true>, dim3((HW + 31) / 32, (C_pad + 31) / 32, B), dim3(256), 0, stream, x,
                           batch_stride, C, HW, C_pad, reinterpret_cast<float*>(hi), reinterpret_cast<float*>(lo)));
  return launch_status();
}

extern "C" int flowk_split_hilo(const float* x, float* hi, float* lo, long long n, flowk_stream_t stream) {
  if (n < 0) return FLOWK_ERR_SHAPE;
  if (n == 0) return FLOWK_OK;
  if (!x || !hi || !lo) return FLOWK_ERR_ARG;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  FLOWK_CUDA_OK(launch_pdl(split_hilo_kernel<false>, dim3(blocks), dim3(256), 0, stream, x, hi, lo, (long long)n, 1.f));
  return launch_status();
}

extern "C" int flowk_split_hilo_f16(const float* x, void* hi, void* lo, long long n, float scale, flowk_stream_t stream) {
  if (n < 0) return FLOWK_ERR_SHAPE;
  if (n == 0) return FLOWK_OK;
  if (!x || !hi || !lo) return FLOWK_ERR_ARG;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  FLOWK_CUDA_OK(launch_pdl(split_hilo_kernel<true>, dim3(blocks), dim3(256), 0, stream, x, reinterpret_cast<float*>(hi),
                           reinterpret_cast<float*>(lo), (long long)n, scale));
  return launch_status();
}
