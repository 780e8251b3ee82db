// Self-attention core of GatedAttn (flow_modules/mixlogcdf_nn.py:134-147) on the 5th-gen tensor cores, inference.
//
//   att[q, :] = softmax_k(q . k / sqrt(d)) v        per (image, head); seq = H*W in {128, 256}, d = C / heads <= 64
//
// One CTA per (image, head); its 128-query tiles run one after the other with K / V staged once:
//   1. all 16 warps stage Q (pre-scaled by log2(e) / sqrt(d)), K and V^T of the pair from the fp32 in_proj rows
//      (k | v | q column order) into shared memory as fp16 (hi, lo) operand tiles, written straight in the K-major
//      128-byte-swizzled layout tcgen05 reads (what a SWIZZLE_128B TMA load would have produced);
//   2. S = Q K^T: tcgen05.mma kind::f16, M = 128 queries, N = seq keys, accumulators in TMEM (seq columns); fp32
//      accuracy from the two-term split S = Qh Kh + Ql Kh + Qh Kl (same scheme as the conv GEMMs, csrc/tc_gemm.cu);
//   3. softmax: a thread owns half of one score row (TMEM lane): row maximum, p = 2^(s - max), row sum; P goes back
//      to shared memory as the (hi, lo) A operand of the second GEMM, over the dead Q / K tiles;
//   4. O = P V: M = 128, N = d (padded to 16), K = seq; O lands in the TMEM columns S no longer needs;
//   5. epilogue: O / rowsum -> the (hi, lo) operand pair of the gate GEMM, fp16 or TF32 containers.
// Nothing of size seq x seq touches HBM.  Replaces the mma.sync kernel (csrc/attention.cu) for seq in {128, 256}.
#include <cuda.h>
#include "common.cuh"
#include "umma.cuh"
#include "attention_tile.cuh"

namespace flowk {
namespace tc {

constexpr int ATT_THREADS = 512;                // 16 warps: 4 threads share a score row (TMEM lane), a quarter of the keys each

struct AttParams {
  const float* qkv;         // [B*HW, 3C], columns (k | v | q)
  float* out_hi;            // [B*HW, C] operand pair (fp16 when out_f16, else TF32 values in fp32 containers)
  float* out_lo;
  int out_f16;
  int HW, C, heads, D;      // D = C / heads (multiple of 8, <= 64)
  int dk;                   // D rounded up to 16: contraction length of S and MMA N of O
  float qscale;             // log2(e) / sqrt(D)
  int q_off, k_off, v_off, p_off, o_off;   // byte offsets of the tile groups in dynamic shared memory
  float acc_scale;          // fused in_proj (attention_tc_v2_kernel<.., true>): undoes the weights' power-of-two pre-scaling
  int kslices;              // fused in_proj: 32-channel K slices of the projection, ceil(C / 32)
  int* status;
  long long* trace;         // optional device [8]: clock64 stamps of CTA (0,0) (profiling), NULL in production
};

template <int KCH>           // KCH = dk / 8: 16-byte chunks per staged row the MMAs read (compile-time: index math without divisions)
__global__ void __launch_bounds__(ATT_THREADS, 1) attention_tc_kernel(const AttParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar_s[2], bar_o[2];
  __shared__ uint32_t tmem_slot;
  __shared__ int failed_flag;
  __shared__ float red_max[4][128], red_sum[2][4][128];
  volatile int* failed = &failed_flag;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pair = blockIdx.x, b = pair / p.heads, h = pair - b * p.heads;
  const int HW = p.HW, D = p.D, C = p.C, row_stride = 3 * C;
  const int tiles = HW >> 7;                    // 128-query tiles of this (image, head): all handled by this CTA, K / V staged once
  const int chunks = D >> 3;                    // 16-byte chunks of real data per row
  constexpr int kchunks = KCH;                  // chunks the MMAs read (a zero chunk pads D % 16 == 8)
  const int hw_shift = HW == 256 ? 8 : 7;
  const int tmem_cols = HW <= 128 ? 128 : 512;  // one S accumulator (HW columns) per query tile

  if (threadIdx.x == 0) {
    failed_flag = 0;
    mbar_init(&bar_s[0], 1);
    mbar_init(&bar_s[1], 1);
    mbar_init(&bar_o[0], 1);
    mbar_init(&bar_o[1], 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_slot, (uint32_t)tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const bool tracing = p.trace && blockIdx.x == 0 && threadIdx.x == 0;
  griddep_launch();
  griddep_wait();                               // the in_proj GEMM's rows are complete from here on
  if (tracing) p.trace[0] = clock64();

  // ---- 1. stage Q (all tiles), K (K-major rows) and V^T as fp16 (hi, lo) swizzled operand tiles ----------------------
  uint8_t* q_hi = smem + p.q_off;               // [HW rows][128 B]: query tile t = rows [128 t, 128 t + 128)
  uint8_t* q_lo = q_hi + HW * ROW_B;
  uint8_t* k_hi = smem + p.k_off;               // [HW rows][128 B]
  uint8_t* k_lo = k_hi + HW * ROW_B;
  const int vt_tile = 2 * p.dk * ROW_B;         // one 64-key block of V^T: [dk rows of hi | dk rows of lo][128 B]
  uint8_t* v_t = smem + p.v_off;                // [HW / 64 blocks][2 dk rows][128 B]
  {
    // One item = 8 consecutive floats (32 bytes) of one row of Q, K or V.  A thread issues the loads of six items before it
    // converts and scatters them (two L2 round trips for the whole staging phase).
    const float* base = p.qkv + (size_t)b * HW * row_stride + h * D;
    const int nk = HW * kchunks, total = 3 * nk;
    constexpr int MAXI = 6;
    for (int i0 = threadIdx.x; i0 < total; i0 += MAXI * ATT_THREADS) {
      float4 a[MAXI], c[MAXI];
#pragma unroll
      for (int u = 0; u < MAXI; ++u) {
        const int i = i0 + u * ATT_THREADS;
        a[u] = c[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total) {
          int r, ch, col;
          if (i < nk) { r = i / kchunks; ch = i % kchunks; col = 2 * C; }
          else if (i < 2 * nk) { r = (i - nk) / kchunks; ch = (i - nk) % kchunks; col = 0; }
          else { r = (i - 2 * nk) & (HW - 1); ch = (i - 2 * nk) >> hw_shift; col = C; }   // V: consecutive threads -> consecutive keys
          if (ch < chunks) {
            const float4* g = reinterpret_cast<const float4*>(base + (size_t)r * row_stride + col + ch * 8);
            a[u] = __ldg(g);
            c[u] = __ldg(g + 1);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < MAXI; ++u) {
        const int i = i0 + u * ATT_THREADS;
        if (i >= total) continue;
        if (i < 2 * nk) {                       // Q (scaled) and K: K-major rows as they lie
          const bool isq = i < nk;
          const int j = isq ? i : i - nk;
          const int r = j / kchunks, ch = j % kchunks;
          const float sc = isq ? p.qscale : 1.f;
          const float v[8] = {a[u].x * sc, a[u].y * sc, a[u].z * sc, a[u].w * sc, c[u].x * sc, c[u].y * sc, c[u].z * sc, c[u].w * sc};
          uint4 hi, lo;
          cvt8(v, hi, lo);
          *reinterpret_cast<uint4*>((isq ? q_hi : k_hi) + sw_off(r, ch)) = hi;
          *reinterpret_cast<uint4*>((isq ? q_lo : k_lo) + sw_off(r, ch)) = lo;
        } else {
          // V^T: rows = head dims, contraction (keys) along the 128-byte rows, 64 keys per block; the 8 dims of this key are
          // scattered to 8 rows of the transposed tile.  The lo rows of a block follow its hi rows, so [V_hi ; V_lo] is ONE
          // B operand of N = 2 dk rows.
          const int j = i - 2 * nk, key = j & (HW - 1), ch = j >> hw_shift;
          const float v[8] = {a[u].x, a[u].y, a[u].z, a[u].w, c[u].x, c[u].y, c[u].z, c[u].w};
          const int kb = key >> 6, kk = key & 63;
          uint8_t* tile = v_t + (size_t)kb * vt_tile;
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            const int dim = ch * 8 + jj;
            unsigned short hh, ll;
            split_f16(v[jj], hh, ll);
            *reinterpret_cast<unsigned short*>(tile + sw_off(dim, kk >> 3) + ((kk & 7) << 1)) = hh;
            *reinterpret_cast<unsigned short*>(tile + sw_off(p.dk + dim, kk >> 3) + ((kk & 7) << 1)) = ll;
          }
        }
      }
    }
  }
  fence_proxy_async();                          // generic-proxy smem writes -> visible to the tensor core
  __syncthreads();
  if (tracing) p.trace[1] = clock64();

  // ---- 2. S_t = Q_t K^T for every query tile, issued back to back (tile t into TMEM columns [t HW, t HW + HW)) ---------
  // (MMAs are issued by warp 0 as a whole with uniform operands, the instruction predicated on the elected lane: umma.cuh)
  const uint32_t leader = warp == 0 ? elect_one() : 0u;
  if (warp == 0) {
    tc_fence_after();
    const uint32_t idesc = make_idesc_f16(HW);
    const uint64_t dk_hi = make_smem_desc(smem_u32(k_hi)), dk_lo = make_smem_desc(smem_u32(k_lo));
    const int ksteps = p.dk >> 4;
    for (int t = 0; t < tiles; ++t) {
      const uint64_t dq_hi = make_smem_desc(smem_u32(q_hi + t * 128 * ROW_B)), dq_lo = make_smem_desc(smem_u32(q_lo + t * 128 * ROW_B));
      const uint32_t d = tmem_base + (uint32_t)(t * HW);
      for (int ks = 0; ks < ksteps; ++ks) {
        const uint64_t ko = (uint64_t)(ks * 2); // 32 bytes per K = 16 step, in 16-byte units
        umma_elect<true>(d, dq_hi + ko, dk_hi + ko, idesc, ks == 0 ? 0u : 1u, leader);
        umma_elect<true>(d, dq_lo + ko, dk_hi + ko, idesc, 1u, leader);
        umma_elect<true>(d, dq_hi + ko, dk_lo + ko, idesc, 1u, leader);
      }
      umma_commit_elect(&bar_s[t], leader);
    }
  }

  const int lane_grp = warp & 3, quarter = warp >> 2;
  const int row = lane_grp * 32 + lane;
  const int ncols = HW >> 2, c0 = quarter * ncols;
  uint8_t* p_hi = smem + p.p_off;               // [HW / 64 blocks][128 rows][128 B]: over the dead Q / K tiles
  uint8_t* p_lo = p_hi + (HW >> 6) * (128 * ROW_B);
  uint8_t* stage = smem + p.o_off;              // epilogue staging: [2 (hi, lo)][128 rows][chunks] 16-byte items

  // epilogue of tile t: O / rowsum -> operand pair.  fp16 output goes through shared memory so that global stores are 16-byte
  // chunks of whole head rows; TF32 output: direct pair stores.
  auto epilogue = [&](int t) {
    mbar_wait(&bar_o[t], 0, failed);
    tc_fence_after();
    const uint32_t trow = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)(t * HW);
    const float inv = 1.0f / ((red_sum[t][0][row] + red_sum[t][1][row]) + (red_sum[t][2][row] + red_sum[t][3][row]));
    const int q0 = t * 128;
    const size_t o0 = (size_t)(b * HW + q0 + row) * C + h * D;
    for (int ch = quarter; ch < chunks; ch += 4) {
      float a[8], c[8];
      tmem_ld8(trow + ch * 8, a);
      tmem_ld8(trow + p.dk + ch * 8, c);
#pragma unroll
      for (int i = 0; i < 8; ++i) c[i] = (a[i] + c[i]) * inv;
      if (p.out_f16) {
        uint4 hi, lo;
        cvt8(c, hi, lo);
        *reinterpret_cast<uint4*>(stage + ((size_t)row * chunks + ch) * 16) = hi;
        *reinterpret_cast<uint4*>(stage + ((size_t)(128 + row) * chunks + ch) * 16) = lo;
      } else {
#pragma unroll
        for (int i = 0; i < 8; i += 2) store_pair(p.out_hi, p.out_lo, o0 + ch * 8 + i, c[i], c[i + 1], 0);
      }
    }
    if (p.out_f16) {
      __syncthreads();
      const int items = 2 * 128 * chunks;
      for (int i = threadIdx.x; i < items; i += ATT_THREADS) {
        const int mat = i / (128 * chunks), rr = (i / chunks) % 128, ch = i % chunks;
        const uint4 v = *reinterpret_cast<const uint4*>(stage + (size_t)i * 16);
        unsigned short* dst = reinterpret_cast<unsigned short*>(mat ? p.out_lo : p.out_hi);
        *reinterpret_cast<uint4*>(dst + (size_t)(b * HW + q0 + rr) * C + h * D + ch * 8) = v;
      }
      __syncthreads();                          // the staging area is free again
    }
  };

  for (int t = 0; t < tiles; ++t) {
    const uint32_t trow = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)(t * HW);
    // ---- 3a. row maximum of S_t (thread = (row, quarter of the keys)); overlaps the previous tile's P V MMAs
    mbar_wait(&bar_s[t], 0, failed);
    tc_fence_after();
    if (tracing && t == 0) p.trace[2] = clock64();
    float mx = -INFINITY;
    for (int j = 0; j < ncols; j += 16) {
      float s[16];
      tmem_ld16(trow + c0 + j, s);
#pragma unroll
      for (int i = 0; i < 16; ++i) mx = fmaxf(mx, s[i]);
    }
    red_max[quarter][row] = mx;
    // P overwrites Q / K (tile 0: every S_t must have been computed) resp. the previous tile's P (its P V must be done)
    if (t == 0) mbar_wait(&bar_s[tiles - 1], 0, failed);
    else mbar_wait(&bar_o[t - 1], 0, failed);
    __syncthreads();
    if (tracing && t == 0) p.trace[3] = clock64();
    mx = fmaxf(fmaxf(red_max[0][row], red_max[1][row]), fmaxf(red_max[2][row], red_max[3][row]));
    // ---- 3b. p = 2^(s - max), row sums, P as the (hi, lo) A operand of the second GEMM
    float sum = 0.f;
    for (int j = 0; j < ncols; j += 16) {
      float s[16];
      tmem_ld16(trow + c0 + j, s);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        s[i] = ex2_fast(s[i] - mx);
        sum += s[i];
      }
      const int key = c0 + j, kb = key >> 6, ch = (key & 63) >> 3;       // two 8-key chunks
      uint4 hi, lo;
      cvt8(s, hi, lo);
      *reinterpret_cast<uint4*>(p_hi + kb * (128 * ROW_B) + sw_off(row, ch)) = hi;
      *reinterpret_cast<uint4*>(p_lo + kb * (128 * ROW_B) + sw_off(row, ch)) = lo;
      cvt8(s + 8, hi, lo);
      *reinterpret_cast<uint4*>(p_hi + kb * (128 * ROW_B) + sw_off(row, ch + 1)) = hi;
      *reinterpret_cast<uint4*>(p_lo + kb * (128 * ROW_B) + sw_off(row, ch + 1)) = lo;
    }
    red_sum[t][quarter][row] = sum;
    tc_fence_before();                          // our tcgen05.ld of S_t are complete before the MMAs overwrite those columns
    fence_proxy_async();
    __syncthreads();
    if (tracing && t == 0) p.trace[4] = clock64();

    // ---- 4. O_t = P V.  B operand = [V_hi ; V_lo] (N = 2 dk): P_hi [V_hi ; V_lo] fills columns [0, dk) and [dk, 2 dk) of S_t's
    //         (dead) leading columns in one MMA, P_lo V_hi adds to [0, dk); the epilogue sums the two column groups.
    if (warp == 0) {
      tc_fence_after();
      const uint32_t idesc2 = make_idesc_f16(2 * p.dk), idesc1 = make_idesc_f16(p.dk);
      const uint32_t d = tmem_base + (uint32_t)(t * HW);
      const int kblocks = HW >> 6;
      for (int kb = 0; kb < kblocks; ++kb) {
        const uint64_t dp_hi = make_smem_desc(smem_u32(p_hi + kb * (128 * ROW_B)));
        const uint64_t dp_lo = make_smem_desc(smem_u32(p_lo + kb * (128 * ROW_B)));
        const uint64_t dv = make_smem_desc(smem_u32(v_t + (size_t)kb * vt_tile));
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t ko = (uint64_t)(k * 2);
          umma_elect<true>(d, dp_hi + ko, dv + ko, idesc2, (kb | k) == 0 ? 0u : 1u, leader);
          umma_elect<true>(d, dp_lo + ko, dv + ko, idesc1, 1u, leader);
        }
      }
      umma_commit_elect(&bar_o[t], leader);
    }
    // ---- 5. the PREVIOUS tile's epilogue runs while this tile's P V MMAs execute
    if (t > 0) epilogue(t - 1);
  }
  if (tracing) p.trace[5] = clock64();
  epilogue(tiles - 1);
  tc_fence_before();
  __syncthreads();
  if (tracing) p.trace[6] = clock64();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
  if (threadIdx.x == 0 && failed_flag && p.status) *p.status = 1;
}

// ---------------------------------------------------------------------------------------------------------------------
// One-wave variant for head dims 24 and 32 (attention_tc_v2_kernel): 256 TMEM columns and < 110 KB of shared memory, so two
// CTAs share an SM and the 256 (image, head) CTAs of a level-1 launch at B = 64 run in ONE wave of 2 x 148 slots; each CTA's
// staging and softmax overlap its neighbour's MMAs.  Still one CTA per (image, head), 16 warps.  Differences to the kernel
// above:
//   * Q and K tiles have 64-byte SWIZZLE_64B rows (32 fp16 = dk) instead of 128-byte rows that are half zeros;
//   * keys are processed in blocks of 128: S_b = Q_t K_b^T fills ONE 128-column TMEM region, softmax gives p = 2^(s - m_b)
//     with the block's own row maximum m_b and row sum l_b, and P_b goes back into the same columns as packed fp16
//     (hi: columns [0, 64), lo: [64, 128)) from where O_b = P_b V_b reads it as the A operand (TS-mode MMA); no P tile in
//     shared memory.  The epilogue combines the blocks exactly: O = sum_b O_b 2^(m_b - m) / sum_b l_b 2^(m_b - m);
//   * O_b has dk columns: P_hi V_hi, P_lo V_hi and P_hi V_lo accumulate into the same N = dk accumulator (the three-product
//     scheme of the conv GEMMs);
//   * TMEM: [0, 128) S / P, then one dk-column O_b per (query tile, key block): 128 + 4 dk <= 256.
// Within a CTA the phases are serial (S -> softmax -> P V -> next S into the same columns); the second CTA on the SM
// fills the gaps.
//
// INPROJ = true (flowk_attention_inproj_tc) computes q, k, v in the CTA instead of reading the in_proj GEMM's fp32 rows:
//   * the input is the gate GEMM's normalised rows + positional encoding as an fp16 (hi, lo) pair [B*HW, C], and the in_proj
//     weight operand [3C, ceil64(C)] (k | v | q rows, pre-scaled like every fp16 weight operand, undone by acc_scale);
//   * warp 0 streams K slices of 32 channels through two stages: the image's HW rows of P (hi, lo) and this head's three
//     32-row groups of weight rows (k at h D, v at C + h D, q at 2C + h D; rows past D belong to the next head or are
//     zero-filled past 3C, their output columns are never read), all SWIZZLE_64B TMA boxes;
//   * per query tile, [k | v | q] = P W^T (N = 96, the three-product split) lands in TMEM columns [96 t, 96 t + 96);
//   * the drain turns those columns into the Q (pre-scaled), K and V^T operand tiles the staging loop writes in the
//     INPROJ = false kernel, over the stage buffers (every projection MMA has retired by then) and before the first S.
constexpr int V2_THREADS = 512;                 // 4 threads per score row (TMEM lane), 32 keys of a 128-key block each
constexpr int V2_TMEM_COLS = 256;
constexpr int V2_QTILE_B = 2 * 128 * V2_ROW_B;  // one 128-query tile of Q: hi rows, then lo rows
constexpr int PJ_N = 96;                        // projection MMA N: k, v, q groups of 32 columns
constexpr int PJ_W_B = PJ_N * V2_ROW_B;         // one K slice of the head's weight rows (hi or lo)
// one stage of the projection: [P_hi: HW rows | P_lo: HW rows | W_hi: 96 rows | W_lo: 96 rows] x 64 B
__host__ __device__ constexpr int pj_stage_bytes(int HW) { return 2 * HW * V2_ROW_B + 2 * PJ_W_B; }


// blockIdx.x, read anew at every use (the compiler may not keep values derived from it live across the kernel)
__device__ __forceinline__ int cta_index() {
  int r;
  asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(r));
  return r;
}

// INPROJ: the maps of the P pair (boxes of 32 channels x HW rows) and of the in_proj weight pair (32 channels x 32 rows);
// unused otherwise.
template <int KCH, int TILES, bool INPROJ>  // KCH = dk / 8 (4), TILES = seq / 128 (1 or 2)
__global__ void __launch_bounds__(V2_THREADS, 2)
attention_tc_v2_kernel(const AttParams p, const __grid_constant__ CUtensorMap map_p_hi,
                       const __grid_constant__ CUtensorMap map_p_lo, const __grid_constant__ CUtensorMap map_w_hi,
                       const __grid_constant__ CUtensorMap map_w_lo) {
  constexpr int DK = KCH * 8, tiles = TILES, HW = 128 * TILES;
  constexpr int TR = INPROJ ? 1 : 0;            // trace slot 1 is the projection's when INPROJ; the later stamps move up one
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t bar_s, bar_o;
  __shared__ uint64_t bar_full[2], bar_empty[2], bar_proj;   // INPROJ: projection stages and the last projection MMA
  __shared__ uint32_t tmem_slot;
  __shared__ int failed_flag;
  __shared__ float red_max[4][128], red_sum[4][128];
  volatile int* failed = &failed_flag;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pair = blockIdx.x, b = pair / p.heads, h = pair - b * p.heads;
  const int D = p.D, C = p.C, row_stride = 3 * C;
  const int chunks = D >> 3;                    // 16-byte chunks of real data per row
  constexpr int hw_shift = TILES == 2 ? 8 : 7;

  if (threadIdx.x == 0) {
    failed_flag = 0;
    mbar_init(&bar_s, 1);
    mbar_init(&bar_o, 1);
    if (INPROJ) {
      mbar_init(&bar_full[0], 1);
      mbar_init(&bar_full[1], 1);
      mbar_init(&bar_empty[0], 1);
      mbar_init(&bar_empty[1], 1);
      mbar_init(&bar_proj, 1);
    }
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&tmem_slot, (uint32_t)V2_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const bool tracing = p.trace && blockIdx.x == 0 && threadIdx.x == 0;
  if (INPROJ && threadIdx.x == 0) {
    prefetch_tmap(&map_p_hi);
    prefetch_tmap(&map_p_lo);
    prefetch_tmap(&map_w_hi);
    prefetch_tmap(&map_w_lo);
  }
  griddep_launch();
  griddep_wait();                               // the producing GEMM's rows are complete from here on
  if (tracing) p.trace[0] = clock64();

  // ---- 1. stage Q (scaled, all tiles), K and V^T as fp16 (hi, lo) operand tiles ------------------------------------------
  uint8_t* q_t = smem + p.q_off;                // [tiles][hi | lo][128 rows][64 B], SWIZZLE_64B
  uint8_t* k_hi = smem + p.k_off;               // [HW rows][64 B], SWIZZLE_64B
  uint8_t* k_lo = k_hi + HW * V2_ROW_B;
  constexpr int vt_tile = 2 * DK * ROW_B;       // one 64-key block of V^T: [DK rows of hi | DK rows of lo][128 B], SWIZZLE_128B
  uint8_t* v_t = smem + p.v_off;
  // V^T: rows = head dims, contraction (keys) along the 128-byte rows, 64 keys per block; dims [8 ch, 8 ch + 8) of `key`
  auto store_vt = [&](int key, int ch, const float* v) {
    const int kb = key >> 6, kk = key & 63;
    uint8_t* tile = v_t + (size_t)kb * vt_tile;
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      const int dim = ch * 8 + jj;
      unsigned short hh, ll;
      split_f16(v[jj], hh, ll);
      *reinterpret_cast<unsigned short*>(tile + sw_off(dim, kk >> 3) + ((kk & 7) << 1)) = hh;
      *reinterpret_cast<unsigned short*>(tile + sw_off(DK + dim, kk >> 3) + ((kk & 7) << 1)) = ll;
    }
  };
  if constexpr (INPROJ) {
    // ---- 1a. [k | v | q]_t = P_t W_h^T for both query tiles, K slices of 32 channels through two stages (warp 0) ----------
    constexpr int STAGE_B = pj_stage_bytes(HW);
    const int nsl = p.kslices;
    const uint32_t leader = warp == 0 ? elect_one() : 0u;
    auto load_slice = [&](int ks) {             // elected lane of warp 0
      uint8_t* st = smem + (ks & 1) * STAGE_B;
      uint64_t* bar = &bar_full[ks & 1];
      mbar_expect_tx(bar, (uint32_t)STAGE_B);
      tma_load_2d(st, &map_p_hi, bar, ks * 32, b * HW);
      tma_load_2d(st + HW * V2_ROW_B, &map_p_lo, bar, ks * 32, b * HW);
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        tma_load_2d(st + 2 * HW * V2_ROW_B + g * 32 * V2_ROW_B, &map_w_hi, bar, ks * 32, g * C + h * D);
        tma_load_2d(st + 2 * HW * V2_ROW_B + PJ_W_B + g * 32 * V2_ROW_B, &map_w_lo, bar, ks * 32, g * C + h * D);
      }
    };
    if (warp == 0) {
      if (leader) {
        load_slice(0);
        if (nsl > 1) load_slice(1);
      }
      const uint32_t idesc = make_idesc_f16(PJ_N);
      for (int ks = 0; ks < nsl; ++ks) {
        mbar_wait(&bar_full[ks & 1], (uint32_t)((ks >> 1) & 1), failed);
        tc_fence_after();
        const uint8_t* st = smem + (ks & 1) * STAGE_B;
        const uint64_t dw_hi = make_smem_desc_sw64(smem_u32(st + 2 * HW * V2_ROW_B));
        const uint64_t dw_lo = make_smem_desc_sw64(smem_u32(st + 2 * HW * V2_ROW_B + PJ_W_B));
#pragma unroll
        for (int t = 0; t < tiles; ++t) {
          const uint64_t dp_hi = make_smem_desc_sw64(smem_u32(st + t * 128 * V2_ROW_B));
          const uint64_t dp_lo = make_smem_desc_sw64(smem_u32(st + (HW + t * 128) * V2_ROW_B));
          const uint32_t d = tmem_base + (uint32_t)(t * PJ_N);
#pragma unroll
          for (int k = 0; k < 2; ++k) {         // K = 16 per MMA: two per 64-byte row
            const uint64_t ko = (uint64_t)(k * 2);
            umma_elect<true>(d, dp_hi + ko, dw_hi + ko, idesc, (ks | k) == 0 ? 0u : 1u, leader);
            umma_elect<true>(d, dp_lo + ko, dw_hi + ko, idesc, 1u, leader);
            umma_elect<true>(d, dp_hi + ko, dw_lo + ko, idesc, 1u, leader);
          }
        }
        umma_commit_elect(&bar_empty[ks & 1], leader);
        if (ks >= 1 && ks + 1 < nsl) {          // the other stage held slice ks - 1: refill it once its MMAs have read it
          mbar_wait(&bar_empty[(ks + 1) & 1], (uint32_t)(((ks - 1) >> 1) & 1), failed);
          if (leader) load_slice(ks + 1);
        }
      }
      umma_commit_elect(&bar_proj, leader);
    }
    mbar_wait(&bar_proj, 0, failed);            // every projection MMA has retired: the stage buffers are free
    tc_fence_after();
    if (tracing) p.trace[1] = clock64();
    // ---- 1b. drain: thread (row, quarter) takes 16-byte chunk `quarter` of the row's k, v and q; dims >= D are zero
    const int lane_grp = warp & 3, ch = warp >> 2;
    const int row = lane_grp * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(lane_grp * 32) << 16);
    const float sc = p.acc_scale;
#pragma unroll 1
    for (int t = 0; t < tiles; ++t) {
      const uint32_t col = lane_addr + (uint32_t)(t * PJ_N + ch * 8);
      const int key = t * 128 + row;
      float v[8];
      uint4 hi, lo;
      if (ch < chunks) {
        tmem_ld8(col, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] *= sc;
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = 0.f;
      }
      cvt8(v, hi, lo);
      *reinterpret_cast<uint4*>(k_hi + sw64_off(key, ch)) = hi;
      *reinterpret_cast<uint4*>(k_lo + sw64_off(key, ch)) = lo;
      if (ch < chunks) {
        tmem_ld8(col + 64, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = v[i] * sc * p.qscale;
      }
      cvt8(v, hi, lo);
      *reinterpret_cast<uint4*>(q_t + t * V2_QTILE_B + sw64_off(row, ch)) = hi;
      *reinterpret_cast<uint4*>(q_t + t * V2_QTILE_B + 128 * V2_ROW_B + sw64_off(row, ch)) = lo;
      if (ch < chunks) {
        tmem_ld8(col + 32, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] *= sc;
      }
      store_vt(key, ch, v);
    }
    tc_fence_before();                          // the drain's loads are complete before S overwrites those columns
  } else {
    const float* base = p.qkv + (size_t)b * HW * row_stride + h * D;
    const int nk = HW * KCH, total = 3 * nk;
    constexpr int MAXI = 3;                     // loads in flight per thread (the 64-register budget of two CTAs per SM)
    for (int i0 = threadIdx.x; i0 < total; i0 += MAXI * V2_THREADS) {
      float4 a[MAXI], c[MAXI];
#pragma unroll
      for (int u = 0; u < MAXI; ++u) {
        const int i = i0 + u * V2_THREADS;
        a[u] = c[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total) {
          int r, ch, col;
          if (i < nk) { r = i / KCH; ch = i % KCH; col = 2 * C; }
          else if (i < 2 * nk) { r = (i - nk) / KCH; ch = (i - nk) % KCH; col = 0; }
          else { r = (i - 2 * nk) & (HW - 1); ch = (i - 2 * nk) >> hw_shift; col = C; }   // V: consecutive threads -> keys
          if (ch < chunks) {
            const float4* g = reinterpret_cast<const float4*>(base + (size_t)r * row_stride + col + ch * 8);
            a[u] = __ldg(g);
            c[u] = __ldg(g + 1);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < MAXI; ++u) {
        const int i = i0 + u * V2_THREADS;
        if (i >= total) continue;
        if (i < 2 * nk) {                       // Q (scaled) and K: K-major rows as they lie
          const bool isq = i < nk;
          const int j = isq ? i : i - nk;
          const int r = j / KCH, ch = j % KCH;
          const float sc = isq ? p.qscale : 1.f;
          const float v[8] = {a[u].x * sc, a[u].y * sc, a[u].z * sc, a[u].w * sc, c[u].x * sc, c[u].y * sc, c[u].z * sc, c[u].w * sc};
          uint4 hi, lo;
          cvt8(v, hi, lo);
          uint8_t* dst_hi = isq ? q_t + (r >> 7) * V2_QTILE_B : k_hi;
          uint8_t* dst_lo = isq ? dst_hi + 128 * V2_ROW_B : k_lo;
          const int rr = isq ? (r & 127) : r;
          *reinterpret_cast<uint4*>(dst_hi + sw64_off(rr, ch)) = hi;
          *reinterpret_cast<uint4*>(dst_lo + sw64_off(rr, ch)) = lo;
        } else {                                // V^T: as in attention_tc_kernel, hi and lo rows of a block kept apart
          const int j = i - 2 * nk, key = j & (HW - 1), ch = j >> hw_shift;
          const float v[8] = {a[u].x, a[u].y, a[u].z, a[u].w, c[u].x, c[u].y, c[u].z, c[u].w};
          store_vt(key, ch, v);
        }
      }
    }
  }
  fence_proxy_async();                          // generic-proxy smem writes -> visible to the tensor core
  __syncthreads();
  if (tracing) p.trace[TR + 1] = clock64();

  // ---- 2. per (query tile t, key block kb): S -> softmax -> P (TMEM) -> O_{t,kb} += P V ---------------------------------
  const uint32_t leader = warp == 0 ? elect_one() : 0u;
  const int lane_grp = warp & 3, quarter = warp >> 2;
  const int row = lane_grp * 32 + lane;
  const uint32_t lane_addr = tmem_base + ((uint32_t)(lane_grp * 32) << 16);
  auto o_col = [&](int t, int kb) { return (uint32_t)(128 + (t * tiles + kb) * DK); };

  auto issue_s = [&](int t, int kb) {           // warp 0: S = Q_t K_kb^T into columns [0, 128)
    tc_fence_after();
    const uint32_t idesc = make_idesc_f16(128);
    const uint64_t dq_hi = make_smem_desc_sw64(smem_u32(q_t + t * V2_QTILE_B));
    const uint64_t dq_lo = make_smem_desc_sw64(smem_u32(q_t + t * V2_QTILE_B + 128 * V2_ROW_B));
    const uint64_t dk_hi = make_smem_desc_sw64(smem_u32(k_hi + kb * 128 * V2_ROW_B));
    const uint64_t dk_lo = make_smem_desc_sw64(smem_u32(k_lo + kb * 128 * V2_ROW_B));
#pragma unroll
    for (int ks = 0; ks < DK / 16; ++ks) {
      const uint64_t ko = (uint64_t)(ks * 2);  // 32 bytes per K = 16 step, in 16-byte units
      umma_elect<true>(tmem_base, dq_hi + ko, dk_hi + ko, idesc, ks == 0 ? 0u : 1u, leader);
      umma_elect<true>(tmem_base, dq_lo + ko, dk_hi + ko, idesc, 1u, leader);
      umma_elect<true>(tmem_base, dq_hi + ko, dk_lo + ko, idesc, 1u, leader);
    }
    umma_commit_elect(&bar_s, leader);
  };

  if (warp == 0) issue_s(0, 0);
  int it = 0;                                   // blocks done: phase of bar_s / bar_o
#pragma unroll 1
  for (int t = 0; t < tiles; ++t) {
    float m0 = 0.f, m1 = 0.f, l0 = 0.f, l1 = 0.f;  // per key block: row maximum and row sum
    for (int kb = 0; kb < tiles; ++kb, ++it) {
      // ---- 3a. this thread's 32 scores of the row (kept in registers: P overwrites them in place) and the block maximum
      mbar_wait(&bar_s, (uint32_t)(it & 1), failed);
      tc_fence_after();
      if (tracing && it == 0) p.trace[TR + 2] = clock64();
      float s[32];
      tmem_ld32(lane_addr + (uint32_t)(quarter * 32), s);
      float mx = s[0];
#pragma unroll
      for (int i = 1; i < 32; ++i) mx = fmaxf(mx, s[i]);
      red_max[quarter][row] = mx;
      tc_fence_before();                        // every load of S is complete before anyone writes P over it
      __syncthreads();
      tc_fence_after();
      if (tracing && it == 0) p.trace[TR + 3] = clock64();
      mx = fmaxf(fmaxf(red_max[0][row], red_max[1][row]), fmaxf(red_max[2][row], red_max[3][row]));
      // ---- 3b. p = 2^(s - m_b) as packed fp16 (hi, lo): keys (2i, 2i + 1) of the block in column i of each half
      float sum = 0.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {    // 16 keys -> 8 columns of P_hi and 8 of P_lo
        uint32_t ph[8], pl[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float e0 = ex2_fast(s[16 * half + 2 * i] - mx), e1 = ex2_fast(s[16 * half + 2 * i + 1] - mx);
          sum += e0 + e1;
          ph[i] = pack_h2(e0, e1);
          float a0, a1;
          unpack_h2(ph[i], a0, a1);
          pl[i] = pack_h2(e0 - a0, e1 - a1);
        }
        tmem_st8u(lane_addr + (uint32_t)(quarter * 16 + half * 8), ph);
        tmem_st8u(lane_addr + (uint32_t)(64 + quarter * 16 + half * 8), pl);
      }
      red_sum[quarter][row] = sum;
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncthreads();
      if (tracing && it == 0) p.trace[TR + 4] = clock64();
      const float l = (red_sum[0][row] + red_sum[1][row]) + (red_sum[2][row] + red_sum[3][row]);
      if (kb == 0) { m0 = mx; l0 = l; }
      else { m1 = mx; l1 = l; }

      // ---- 4. O_{t,kb} = P_hi V_hi + P_lo V_hi + P_hi V_lo (N = dk, K = 128 keys), then the next S into the freed columns
      if (warp == 0) {
        tc_fence_after();
        const uint32_t idesc = make_idesc_f16(DK);
        const uint32_t d = tmem_base + o_col(t, kb);
#pragma unroll
        for (int j = 0; j < 8; ++j) {           // K = 16 keys per step: 8 packed columns of P, 32 bytes of a V^T row
          const int key = kb * 128 + j * 16;
          const uint8_t* vb = v_t + (size_t)(key >> 6) * vt_tile;
          const uint64_t ko = (uint64_t)(((key & 63) >> 4) * 2);
          const uint64_t dv_hi = make_smem_desc(smem_u32(vb)) + ko, dv_lo = make_smem_desc(smem_u32(vb + DK * ROW_B)) + ko;
          const uint32_t a_hi = tmem_base + (uint32_t)(j * 8), a_lo = tmem_base + (uint32_t)(64 + j * 8);
          umma_f16_ts_elect(d, a_hi, dv_hi, idesc, j == 0 ? 0u : 1u, leader);
          umma_f16_ts_elect(d, a_lo, dv_hi, idesc, 1u, leader);
          umma_f16_ts_elect(d, a_hi, dv_lo, idesc, 1u, leader);
        }
        umma_commit_elect(&bar_o, leader);
        const int nt = kb + 1 < tiles ? t : t + 1, nkb = kb + 1 < tiles ? kb + 1 : 0;
        if (nt < tiles) {
          mbar_wait(&bar_o, (uint32_t)(it & 1), failed);   // P has been read
          issue_s(nt, nkb);
        }
      }
    }
    if (tracing && t == tiles - 1) p.trace[TR + 5] = clock64();

    // ---- 5. epilogue of tile t (overlaps the next tile's first S MMAs): exact combination of the key blocks
    mbar_wait(&bar_o, (uint32_t)((it - 1) & 1), failed);
    tc_fence_after();
    float w0 = 1.f, w1 = 0.f;
    if (tiles == 2) {
      const float m = fmaxf(m0, m1);
      w0 = ex2_fast(m0 - m);
      w1 = ex2_fast(m1 - m);
    }
    const float inv = 1.0f / (l0 * w0 + l1 * w1);
    w0 *= inv;
    w1 *= inv;
    const int q0 = t * 128;
    // the output offset of this (image, head) from a fresh read of the CTA index: keeping the image index in a register
    // from the prologue to here costs the fused in_proj variant a spill under its 64-register budget
    const size_t out0 = (size_t)(cta_index() / p.heads) * HW * C + (size_t)(cta_index() % p.heads) * D;
    const size_t o0 = out0 + (size_t)(q0 + row) * C;
    uint8_t* stage = q_t + t * V2_QTILE_B;      // Q_t is dead (every S of tile t is done): [2 (hi, lo)][128 rows][chunks] x 16 B
    for (int ch = quarter; ch < chunks; ch += 4) {
      float a[8], c[8];
      tmem_ld8(lane_addr + o_col(t, 0) + ch * 8, a);
      if (tiles == 2) tmem_ld8(lane_addr + o_col(t, 1) + ch * 8, c);
      else {
#pragma unroll
        for (int i = 0; i < 8; ++i) c[i] = 0.f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) c[i] = a[i] * w0 + c[i] * w1;
      if (p.out_f16) {
        uint4 hi, lo;
        cvt8(c, hi, lo);
        *reinterpret_cast<uint4*>(stage + ((size_t)row * chunks + ch) * 16) = hi;
        *reinterpret_cast<uint4*>(stage + ((size_t)(128 + row) * chunks + ch) * 16) = lo;
      } else {
#pragma unroll
        for (int i = 0; i < 8; i += 2) store_pair(p.out_hi, p.out_lo, o0 + ch * 8 + i, c[i], c[i + 1], 0);
      }
    }
    if (p.out_f16) {
      __syncthreads();
      const int items = 2 * 128 * chunks;
      for (int i = threadIdx.x; i < items; i += V2_THREADS) {
        const int mat = i / (128 * chunks), rr = (i / chunks) % 128, ch = i % chunks;
        const uint4 v = *reinterpret_cast<const uint4*>(stage + (size_t)i * 16);
        unsigned short* dst = reinterpret_cast<unsigned short*>(mat ? p.out_lo : p.out_hi);
        *reinterpret_cast<uint4*>(dst + out0 + (size_t)(q0 + rr) * C + ch * 8) = v;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tracing) p.trace[TR + 6] = clock64();
  if (warp == 0) tmem_dealloc(tmem_base, (uint32_t)V2_TMEM_COLS);
  if (threadIdx.x == 0 && failed_flag && p.status) *p.status = 1;
}

}  // namespace tc
}  // namespace flowk

using namespace flowk;
using namespace flowk::tc;

// Same contract as flowk_attention / flowk_attention_f16 (include/flowk.h); returns FLOWK_ERR_SHAPE for shapes this
// kernel does not take (the caller then uses the mma.sync kernel): seq must be 128 or 256, C / heads a multiple of 8, <= 64.
extern "C" int flowk_attention_tc(const float* qkv, void* out_hi, void* out_lo, int out_f16, int B, int HW, int C, int heads,
                                  int* status, long long* trace, flowk_stream_t stream) {
  if (B < 0 || HW < 1 || C < 1 || heads < 1 || C % heads) return FLOWK_ERR_SHAPE;
  const int D = C / heads;
  if ((HW != 128 && HW != 256) || D % 8 || D > 64 || C % 4) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!qkv || !out_hi || !out_lo) return FLOWK_ERR_ARG;
  if ((long long)B * heads > 0x7fffffffLL) return FLOWK_ERR_SHAPE;
  AttParams p{};
  p.qkv = qkv;
  p.out_hi = reinterpret_cast<float*>(out_hi);
  p.out_lo = reinterpret_cast<float*>(out_lo);
  p.out_f16 = out_f16;
  p.HW = HW;
  p.C = C;
  p.heads = heads;
  p.D = D;
  p.dk = (D + 15) / 16 * 16;
  p.qscale = 1.4426950408889634f / sqrtf((float)D);
  p.status = status;
  p.trace = trace;
  // shared memory: [P tiles of one query tile | over them: Q (all tiles), K], then V^T, then the epilogue staging area
  const int p_bytes = 2 * (HW / 64) * 128 * ROW_B;           // hi + lo
  const int qk_bytes = 2 * HW * ROW_B + 2 * HW * ROW_B;
  const int first = p_bytes > qk_bytes ? p_bytes : qk_bytes;
  p.p_off = 0;
  p.q_off = 0;
  p.k_off = 2 * HW * ROW_B;
  p.v_off = first;
  p.o_off = first + 2 * (HW / 64) * p.dk * ROW_B;
  const size_t smem = (size_t)p.o_off + (size_t)2 * 128 * (D / 8) * 16 + 1024;
  if (smem + 8 * 1024 > 227 * 1024) return FLOWK_ERR_SHAPE;   // (+ the kernel's static shared memory)
#define FLOWK_LAUNCH_ATT(KCH_)                                                                                          \
  do {                                                                                                                 \
    static size_t smem_set = 0;                                                                                        \
    if (smem > smem_set) {                                                                                             \
      FLOWK_CUDA_OK(cudaFuncSetAttribute(attention_tc_kernel<KCH_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      smem_set = smem;                                                                                                 \
    }                                                                                                                  \
    FLOWK_CUDA_OK(launch_pdl(attention_tc_kernel<KCH_>, dim3(B * heads), dim3(ATT_THREADS), smem, stream, p));          \
  } while (0)
  switch (p.dk >> 3) {
    case 2: FLOWK_LAUNCH_ATT(2); break;
    case 4: FLOWK_LAUNCH_ATT(4); break;
    case 6: FLOWK_LAUNCH_ATT(6); break;
    default: FLOWK_LAUNCH_ATT(8); break;
  }
#undef FLOWK_LAUNCH_ATT
  return launch_status();
}

namespace {
// Shared-memory plan of attention_tc_v2_kernel: Q (all tiles), K, V^T; the epilogue stages its output over the dead Q tile.
// With the fused in_proj, the two projection stages lie over the same region first.
bool attention_tc_v2_plan(int HW, int C, int heads, bool inproj, AttParams& p, size_t& smem) {
  if (HW != 128 && HW != 256) return false;
  if (heads < 1 || C < 1 || C % heads) return false;
  const int D = C / heads;
  if (D != 24 && D != 32) return false;         // dk = 32: one 64-byte swizzle row (dk = 16 would not keep 64 registers)
  p.HW = HW;
  p.C = C;
  p.heads = heads;
  p.D = D;
  p.dk = (D + 15) / 16 * 16;
  p.qscale = 1.4426950408889634f / sqrtf((float)D);
  p.q_off = 0;
  p.k_off = (HW / 128) * V2_QTILE_B;
  p.v_off = p.k_off + 2 * HW * V2_ROW_B;
  p.kslices = (C + 31) / 32;
  size_t bytes = (size_t)p.v_off + (size_t)2 * (HW / 64) * p.dk * ROW_B;
  if (inproj && (size_t)2 * pj_stage_bytes(HW) > bytes) bytes = (size_t)2 * pj_stage_bytes(HW);
  smem = bytes + 1024;                          // + alignment of the 1024-byte swizzle atoms
  return true;
}

template <int KCH, int TILES, bool INPROJ>
cudaError_t attention_tc_v2_prepare(size_t smem) {
  static size_t smem_set = 0;
  if (smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(attention_tc_v2_kernel<KCH, TILES, INPROJ>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(attention_tc_v2_kernel<KCH, TILES, INPROJ>, cudaFuncAttributePreferredSharedMemoryCarveout,
                             (int)cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    smem_set = smem;
  }
  return cudaSuccess;
}

template <bool INPROJ>
int attention_tc_v2_launch(const AttParams& p, int B, size_t smem, const CUtensorMap* maps, cudaStream_t stream) {
#define FLOWK_LAUNCH_ATT_V2(KCH_, TILES_)                                                                             \
  do {                                                                                                                 \
    FLOWK_CUDA_OK((attention_tc_v2_prepare<KCH_, TILES_, INPROJ>(smem)));                                               \
    FLOWK_CUDA_OK(launch_pdl(attention_tc_v2_kernel<KCH_, TILES_, INPROJ>, dim3(B * p.heads), dim3(V2_THREADS), smem,    \
                             stream, p, maps[0], maps[1], maps[2], maps[3]));                                          \
  } while (0)
  if (p.HW == 256) FLOWK_LAUNCH_ATT_V2(4, 2);
  else FLOWK_LAUNCH_ATT_V2(4, 1);
#undef FLOWK_LAUNCH_ATT_V2
  return launch_status();
}

}  // namespace

// One-wave kernel (two CTAs per SM) for C / heads in {24, 32}; same contract as flowk_attention_tc otherwise.
extern "C" int flowk_attention_tc_v2(const float* qkv, void* out_hi, void* out_lo, int out_f16, int B, int HW, int C,
                                     int heads, int* status, long long* trace, flowk_stream_t stream) {
  AttParams p{};
  size_t smem = 0;
  if (B < 0 || !attention_tc_v2_plan(HW, C, heads, false, p, smem)) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!qkv || !out_hi || !out_lo) return FLOWK_ERR_ARG;
  if ((long long)B * heads > 0x7fffffffLL) return FLOWK_ERR_SHAPE;
  p.qkv = qkv;
  p.out_hi = reinterpret_cast<float*>(out_hi);
  p.out_lo = reinterpret_cast<float*>(out_lo);
  p.out_f16 = out_f16;
  p.status = status;
  p.trace = trace;
  const CUtensorMap unused[4] = {};
  return attention_tc_v2_launch<false>(p, B, smem, unused, stream);
}

// The one-wave kernel with the in_proj GEMM fused in front (attention_tc_v2_kernel<.., true>): p_hi / p_lo [B*HW, C] fp16
// normalised rows + positional encoding, w_hi / w_lo the in_proj weight operand [3C, ceil64(C)] fp16 (k | v | q rows).
extern "C" int flowk_attention_inproj_tc(const void* p_hi, const void* p_lo, const void* w_hi, const void* w_lo,
                                         float acc_scale, void* out_hi, void* out_lo, int B, int HW, int C, int heads,
                                         int* status, long long* trace, flowk_stream_t stream) {
  AttParams p{};
  size_t smem = 0;
  if (B < 0 || !attention_tc_v2_plan(HW, C, heads, true, p, smem)) return FLOWK_ERR_SHAPE;
  if (B == 0) return FLOWK_OK;
  if (!p_hi || !p_lo || !w_hi || !w_lo || !out_hi || !out_lo || !(acc_scale > 0.f)) return FLOWK_ERR_ARG;
  if (!aligned16(p_hi) || !aligned16(p_lo) || !aligned16(w_hi) || !aligned16(w_lo)) return FLOWK_ERR_ALIGN;
  if ((long long)B * HW > 0x7fffffffLL) return FLOWK_ERR_SHAPE;
  p.out_hi = reinterpret_cast<float*>(out_hi);
  p.out_lo = reinterpret_cast<float*>(out_lo);
  p.out_f16 = 1;
  p.acc_scale = acc_scale;
  p.status = status;
  p.trace = trace;
  const long long rows = (long long)B * HW, kw = (C + 63) / 64 * 64;
  CUtensorMap maps[4];
  if (!make_map_sw64(&maps[0], p_hi, rows, C, HW) || !make_map_sw64(&maps[1], p_lo, rows, C, HW) ||
      !make_map_sw64(&maps[2], w_hi, 3LL * C, kw, 32) || !make_map_sw64(&maps[3], w_lo, 3LL * C, kw, 32))
    return FLOWK_ERR_ARG;
  return attention_tc_v2_launch<true>(p, B, smem, maps, stream);
}

// CTAs of flowk_attention_tc_v2's (or flowk_attention_inproj_tc's) kernel that one SM's registers, shared memory and thread
// slots hold at this shape; writes the dynamic shared memory per CTA to *smem_bytes when it is not NULL.  FLOWK_ERR_SHAPE
// for shapes it does not take.  (cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for every kernel that uses tcgen05
// instructions, whatever its resources, so the limits are applied here from the kernel's attributes and the device's.)
namespace {
template <int KCH, int TILES, bool INPROJ>
int attention_tc_v2_fit(size_t smem, int* blocks_per_sm) {
  FLOWK_CUDA_OK((attention_tc_v2_prepare<KCH, TILES, INPROJ>(smem)));
  cudaFuncAttributes fa;
  FLOWK_CUDA_OK(cudaFuncGetAttributes(&fa, attention_tc_v2_kernel<KCH, TILES, INPROJ>));
  int dev = 0, regs_sm = 0, smem_sm = 0, reserved = 0, threads_sm = 0;
  FLOWK_CUDA_OK(cudaGetDevice(&dev));
  FLOWK_CUDA_OK(cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev));
  FLOWK_CUDA_OK(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
  FLOWK_CUDA_OK(cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, dev));
  FLOWK_CUDA_OK(cudaDeviceGetAttribute(&threads_sm, cudaDevAttrMaxThreadsPerMultiProcessor, dev));
  const int warp_regs = (fa.numRegs * 32 + 255) / 256 * 256;            // registers are allocated per warp, 256 at a time
  const int by_regs = regs_sm / (warp_regs * (V2_THREADS / 32));
  const int by_smem = smem_sm / (int)(smem + fa.sharedSizeBytes + (size_t)reserved);
  const int by_threads = threads_sm / V2_THREADS;
  *blocks_per_sm = by_regs < by_smem ? (by_regs < by_threads ? by_regs : by_threads) : (by_smem < by_threads ? by_smem : by_threads);
  return FLOWK_OK;
}

template <bool INPROJ>
int attention_tc_v2_occupancy(int HW, int C, int heads, int* blocks_per_sm, int* smem_bytes) {
  AttParams p{};
  size_t smem = 0;
  if (!attention_tc_v2_plan(HW, C, heads, INPROJ, p, smem)) return FLOWK_ERR_SHAPE;
  if (!blocks_per_sm) return FLOWK_ERR_ARG;
  if (smem_bytes) *smem_bytes = (int)smem;
  return HW == 256 ? attention_tc_v2_fit<4, 2, INPROJ>(smem, blocks_per_sm) : attention_tc_v2_fit<4, 1, INPROJ>(smem, blocks_per_sm);
}
}  // namespace

extern "C" int flowk_attention_tc_v2_occupancy(int HW, int C, int heads, int* blocks_per_sm, int* smem_bytes) {
  return attention_tc_v2_occupancy<false>(HW, C, heads, blocks_per_sm, smem_bytes);
}

extern "C" int flowk_attention_inproj_tc_occupancy(int HW, int C, int heads, int* blocks_per_sm, int* smem_bytes) {
  return attention_tc_v2_occupancy<true>(HW, C, heads, blocks_per_sm, smem_bytes);
}
