// Weight gradient of the conditioner convolutions / linear layers on the 5th-gen tensor cores (training path).
//
//   dW[t][n][c] = sum_{b, p} gy[b, n, p] * x[b, c, p + shift(t)]        (taps = 1 or 3x3, zero "same" padding)
//
// The contraction runs over PIXELS, so the channel-major (NCHW) fp32 tensors autograd already holds are K-major
// operands as they lie: a k-block is 32 consecutive pixels of one image (one 128-byte swizzle row per channel),
// fetched by one TMA box per operand over the (H*W, C, B) view.  A row shift dy of a 3x3 tap is a coordinate offset
// of dy*W pixels - rows outside the image are out of bounds of the pixel dimension and zero-filled by the TMA unit.
// A column shift dx = +-1 cannot be a TMA coordinate (the innermost coordinate must be 16-byte aligned: measured,
// profiles/dbg/tma_box_probe.cu), so the caller passes two column-shifted copies of x (flowk_shift_columns, zero at
// the image border) and the tap picks its tensor map.
// NHWC rows (flowk_conv_wgrad_nhwc: the mAR prior's time-major [T*B*H*W, C] tensors, 3x3 / 5x5 taps at any dilation)
// need no copies: a k-block is a 5-D box (32 channels, bw columns, bh rows, bb images; bw * bh * bb = 32 pixels) whose
// W / H start coordinates carry the tap's (dx, dy) * dilation - the innermost dimension is the channel block, so every
// shift is aligned - and the TMA unit zero-fills pixels outside the image ("same" padding).  Per 32-channel block the
// tile is the [32 pixels x 128 B] MN-major tile of the row-major (Linear) mode, read with the same descriptors.
// No operand is pre-split in HBM: tcgen05 kind::tf32 ignores the 13 low mantissa bits of its fp32 containers
// (measured, profiles/trunc_probe.py), so the raw tile IS `hi`, and eight converter warps build
// lo = rna(x - trunc(x)) into a second tile (same swizzled offsets, pure elementwise) while the previous k-block's
// MMAs run.  D += G_hi X_hi + G_lo X_hi + G_hi X_lo, fp32 accumulators in TMEM.
// Split-K over CTAs: every (tile, split) CTA writes its own partial dW; the consumer (flowk_weight_norm_bwd_partials)
// adds the partials in index order, so the result is deterministic.
//
// warp roles: 0 = TMA producer, 1 = TMEM owner + MMA issuer, 2..9 = lo converters, 2..5 also the epilogue.
// Reference semantics: autograd of F.conv2d / F.linear in flow_modules/mixlogcdf_nn.py:12-29,124-152.
#include <cuda.h>
#include "common.cuh"
#include "umma.cuh"

namespace flowk {
namespace tc {

constexpr int WG_CONV_WARPS = 8;
constexpr int WG_THREADS = 64 + 32 * WG_CONV_WARPS;
constexpr int WG_MAX_STAGES = 4;

struct WgradParams {
  int N, Cin, taps;               // here N = channels of the A-side tensor, Cin = channels of the B-side tensor
  int shift_a;                    // 1: the A side is x (carries the tap shift), 0: the B side is
  int rows;                       // 1: row-major operands [M, C] (Linear layers): MN-major tiles of [32 rows x 32 channels]
                                  //    blocks, 3-D TMA boxes (32 ch, 32 rows, blocks), transposed UMMA descriptors
                                  // 2: NHWC rows [NB*H*W, C] of a k x k (dilated) convolution: the same tiles, fetched as
                                  //    5-D boxes (32 ch, bw, bh, bb, blocks) whose W / H coordinates carry the tap shift
  int g_tile_bytes;               // shared-memory bytes reserved for the A tile (its real rows, rounded to 8)
  int kblk;                       // pixels per k-block: 32 (128-byte swizzle rows) or 16 (64-byte rows, H*W == 16 maps)
  int W;                          // image width: a row shift is W pixels
  int kb_per_image, total_kb;     // k-block = 32 consecutive pixels of one image
  int g_rows, x_rows;             // TMA box rows (<= 128, <= c_tile)
  int c_tile, c_tiles, m_tiles;
  int stages, stage_bytes, tmem_cols;
  float* partial;                 // [splits][taps][N][Cin]
  int* status;
  int ksz, dil;                   // rows == 2: taps = ksz * ksz, tap (ky, kx) reads pixel + ((ky, kx) - ksz / 2) * dil
  int bw, bh, bb, kpi_w, kpi_h;   // rows == 2: k-block box (bw x bh pixels x bb images = 32), boxes per image row / column
};

__global__ void __launch_bounds__(WG_THREADS, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_x,
                  const __grid_constant__ CUtensorMap map_xm, const __grid_constant__ CUtensorMap map_xp, const WgradParams p) {
  // map_g: the un-shifted tensor (gy); map_x / map_xm / map_xp: x and its column-shifted copies.
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full_raw[WG_MAX_STAGES], full_lo[WG_MAX_STAGES], empty_bar[WG_MAX_STAGES], acc_full;
  __shared__ uint32_t tmem_slot;
  __shared__ int failed_flag;
  volatile int* failed = &failed_flag;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // tile decode: blockIdx.x = (m_tile, tap, c_tile)
  int tile = blockIdx.x;
  const int ct = tile % p.c_tiles;
  tile /= p.c_tiles;
  const int tap = tile % p.taps;
  const int mt = tile / p.taps;
  const int split = blockIdx.y, splits = gridDim.y;
  const int kb0 = (int)((long long)p.total_kb * split / splits), kb1 = (int)((long long)p.total_kb * (split + 1) / splits);
  const int dy = p.taps == 9 ? tap / 3 - 1 : 0, dx = p.taps == 9 ? tap % 3 - 1 : 0;
  const int row_bytes = p.kblk * 4;
  const int g_bytes = p.g_rows * row_bytes, x_bytes = p.x_rows * row_bytes;
  const int x_off = p.g_tile_bytes;                      // the MMA reads 128 A rows: rows past the tile are garbage
                                                         // that only reaches accumulator rows nobody stores
  const int lo_off = x_off + p.c_tile * row_bytes;       // lo tiles mirror the raw ones

  if (threadIdx.x == 0) {
    failed_flag = 0;
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_raw[s], 1);
      mbar_init(&full_lo[s], WG_CONV_WARPS);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&acc_full, 1);
    fence_barrier_init();
    prefetch_tmap(&map_g);
    prefetch_tmap(dx < 0 ? &map_xm : dx > 0 ? &map_xp : &map_x);
  }
  if (warp == 1) tmem_alloc(&tmem_slot, (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  griddep_wait();

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = kb0; kb < kb1; ++kb) {
        const int i = kb - kb0, s = i % p.stages;
        if (i >= p.stages) mbar_wait(&empty_bar[s], ((uint32_t)(i / p.stages) - 1u) & 1u, failed);
        const int b = kb / p.kb_per_image, p0 = (kb - b * p.kb_per_image) * p.kblk;
        uint8_t* st = smem + (size_t)s * p.stage_bytes;
        mbar_expect_tx(&full_raw[s], (uint32_t)(g_bytes + x_bytes));
        const CUtensorMap* mx = dx < 0 ? &map_xm : dx > 0 ? &map_xp : &map_x;
        if (p.rows == 2) {            // k-block = a (bw, bh, bb) box of pixels; out-of-image taps are zero-filled by TMA
          const int sy = (tap / p.ksz - p.ksz / 2) * p.dil, sx = (tap % p.ksz - p.ksz / 2) * p.dil;
          const int r = kb / p.kpi_w, w0 = (kb - r * p.kpi_w) * p.bw;
          const int h0 = (r % p.kpi_h) * p.bh, b0 = (r / p.kpi_h) * p.bb;
          const int ay = p.shift_a ? sy : 0, ax = p.shift_a ? sx : 0;
          tma_load_5d(st, p.shift_a ? &map_x : &map_g, &full_raw[s], 0, w0 + ax, h0 + ay, b0, mt * (BLOCK_M / 32));
          tma_load_5d(st + x_off, p.shift_a ? &map_g : &map_x, &full_raw[s], 0, w0 + sx - ax, h0 + sy - ay, b0,
                      ct * (p.c_tile / 32));
        } else if (p.rows) {          // k-block = rows [32 kb, 32 kb + 32); A side = map_g when !shift_a
          tma_load_3d(st, p.shift_a ? &map_x : &map_g, &full_raw[s], 0, kb * BLOCK_K, mt * (BLOCK_M / 32));
          tma_load_3d(st + x_off, p.shift_a ? &map_g : &map_x, &full_raw[s], 0, kb * BLOCK_K, ct * (p.c_tile / 32));
        } else if (p.shift_a) {
          tma_load_4d(st, mx, &full_raw[s], p0 + dy * p.W, mt * BLOCK_M, b, 0);
          tma_load_4d(st + x_off, &map_g, &full_raw[s], p0, ct * p.c_tile, b, 0);
        } else {
          tma_load_4d(st, &map_g, &full_raw[s], p0, mt * BLOCK_M, b, 0);
          tma_load_4d(st + x_off, mx, &full_raw[s], p0 + dy * p.W, ct * p.c_tile, b, 0);
        }
      }
    }
  } else if (warp == 1) {
    // the whole warp runs the loop with uniform operands; only the elected lane's tcgen05 instructions execute (umma.cuh)
    const uint32_t leader = elect_one();
    {
      const uint32_t idesc = p.rows ? make_idesc_mn(p.c_tile) : make_idesc(p.c_tile);
      for (int kb = kb0; kb < kb1; ++kb) {
        const int i = kb - kb0, s = i % p.stages;
        const uint32_t ph = (uint32_t)(i / p.stages) & 1u;
        mbar_wait(&full_raw[s], ph, failed);
        mbar_wait(&full_lo[s], ph, failed);
        tc_fence_after();
        const uint32_t base = smem_u32(smem + (size_t)s * p.stage_bytes);
        uint64_t dg_hi, dx_hi, dg_lo, dx_lo;
        if (p.rows) {
          dg_hi = make_smem_desc_mn(base, 4096), dx_hi = make_smem_desc_mn(base + x_off, 4096);
          dg_lo = make_smem_desc_mn(base + lo_off, 4096), dx_lo = make_smem_desc_mn(base + lo_off + x_off, 4096);
        } else if (p.kblk == 16) {
          dg_hi = make_smem_desc_sw64(base), dx_hi = make_smem_desc_sw64(base + x_off);
          dg_lo = make_smem_desc_sw64(base + lo_off), dx_lo = make_smem_desc_sw64(base + lo_off + x_off);
        } else {
          dg_hi = make_smem_desc(base), dx_hi = make_smem_desc(base + x_off);
          dg_lo = make_smem_desc(base + lo_off), dx_lo = make_smem_desc(base + lo_off + x_off);
        }
        const int ksteps = p.kblk / UMMA_K;
#pragma unroll 4
        for (int k = 0; k < ksteps; ++k) {
          // K-major: 32 bytes further inside the 128-byte row; MN-major: 8 rows = 1024 bytes further
          const uint64_t ko = p.rows ? (uint64_t)(k * 1024 >> 4) : (uint64_t)(k * UMMA_K * 4 >> 4);
          umma_elect<false>(tmem_base, dg_hi + ko, dx_hi + ko, idesc, (i | k) == 0 ? 0u : 1u, leader);
          umma_elect<false>(tmem_base, dg_lo + ko, dx_hi + ko, idesc, 1u, leader);
          umma_elect<false>(tmem_base, dg_hi + ko, dx_lo + ko, idesc, 1u, leader);
        }
        umma_commit_elect(&empty_bar[s], leader);
      }
      umma_commit_elect(&acc_full, leader);
    }
  } else {
    // ===================== converters: lo = rna(x - trunc(x)) at the same (swizzled) offsets =====================
    const int ctid = threadIdx.x - 64;
    const int vec_total = lo_off / 16;                   // float4 slots of (G tile + X tile)
    for (int kb = kb0; kb < kb1; ++kb) {
      const int i = kb - kb0, s = i % p.stages;
      mbar_wait(&full_raw[s], (uint32_t)(i / p.stages) & 1u, failed);
      const float4* src = reinterpret_cast<const float4*>(smem + (size_t)s * p.stage_bytes);
      float4* dst = reinterpret_cast<float4*>(smem + (size_t)s * p.stage_bytes + lo_off);
      for (int v = ctid; v < vec_total; v += 32 * WG_CONV_WARPS) {
        const float4 a = src[v];
        float4 l;
        l.x = rna_tf32(a.x - __uint_as_float(__float_as_uint(a.x) & 0xffffe000u));
        l.y = rna_tf32(a.y - __uint_as_float(__float_as_uint(a.y) & 0xffffe000u));
        l.z = rna_tf32(a.z - __uint_as_float(__float_as_uint(a.z) & 0xffffe000u));
        l.w = rna_tf32(a.w - __uint_as_float(__float_as_uint(a.w) & 0xffffe000u));
        dst[v] = l;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&full_lo[s])) : "memory");
      }
    }
    // ===================== epilogue: TMEM -> partial[split][tap][n][c] =====================
    if (warp < 6) {
      mbar_wait(&acc_full, 0u, failed);
      tc_fence_after();
      const int q = warp & 3;                              // TMEM lane quarter this warp may read
      const int n = mt * BLOCK_M + q * 32 + lane;
      float* row = p.partial + (((size_t)split * p.taps + tap) * p.N + (size_t)(n < p.N ? n : 0)) * p.Cin;
      const int c0 = ct * p.c_tile;
      const bool vec_ok = (p.Cin & 3) == 0;
      for (int col = 0; col < p.c_tile; col += 16) {
        float v[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col, v);
        if (n < p.N && kb1 > kb0) {
          if (vec_ok && c0 + col + 16 <= p.Cin) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              *reinterpret_cast<float4*>(row + c0 + col + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + col + j < p.Cin) row[c0 + col + j] = v[j];
          }
        } else if (n < p.N) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (c0 + col + j < p.Cin) row[c0 + col + j] = 0.f;
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  griddep_launch();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  if (threadIdx.x == 0 && failed_flag && p.status) *p.status = 1;
}

// channel-major operand [B, C, H*W] viewed by TMA as dims (H*W, C, B, 1); box (32 pixels, rows, 1, 1)
static bool make_map_cm(CUtensorMap* map, const float* base, int B, int C, int HW, int rows, int kblk = BLOCK_K) {
  cuuint64_t dims[4] = {(cuuint64_t)HW, (cuuint64_t)C, (cuuint64_t)B, 1};
  cuuint64_t strides[3] = {(cuuint64_t)HW * 4, (cuuint64_t)C * HW * 4, (cuuint64_t)B * C * HW * 4};
  cuuint32_t box[4] = {(cuuint32_t)kblk, (cuuint32_t)rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return encode_fn() && encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box,
                                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                    kblk == 16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct WgradPlan {
  bool ok;
  int kblk;                      // pixels per k-block (32, or 16 for 4x4 maps)
  int swap;                      // 1: A side = x (Cin rows), B side = gy (N columns): partial[s][t][c][n]
  int a_ch, b_ch, g_tile_bytes;
  int c_tile, c_tiles, m_tiles, splits, stages, stage_bytes, tmem_cols;
};

static WgradPlan plan_wgrad(int B, int H, int W, int Cin, int N, int taps) {
  WgradPlan pl = {};
  if (B < 1 || H < 1 || W < 4 || W % 4 || (H * W) % 16 || Cin < 1 || N < 1 || (taps != 1 && taps != 9)) return pl;
  pl.kblk = (H * W) % BLOCK_K ? 16 : BLOCK_K;
  const int row_bytes = pl.kblk * 4;
  // a K=8 MMA costs about the same whatever its N <= 256 (measured): put the side that fills 128-row tiles with the
  // fewest MMAs on the A side
  auto tiles_of = [](int a, int b) { return ((a + BLOCK_M - 1) / BLOCK_M) * ((b + 255) / 256); };
  pl.swap = tiles_of(Cin, N) < tiles_of(N, Cin) ? 1 : 0;
  pl.a_ch = pl.swap ? Cin : N;
  pl.b_ch = pl.swap ? N : Cin;
  pl.c_tiles = (pl.b_ch + 255) / 256;
  pl.c_tile = ((pl.b_ch + pl.c_tiles - 1) / pl.c_tiles + 15) / 16 * 16;
  pl.m_tiles = (pl.a_ch + BLOCK_M - 1) / BLOCK_M;
  const int a_rows = pl.a_ch < BLOCK_M ? (pl.a_ch + 7) / 8 * 8 : BLOCK_M;
  pl.g_tile_bytes = a_rows * row_bytes;
  pl.stage_bytes = 2 * (pl.g_tile_bytes + pl.c_tile * row_bytes);
  // the MMA always reads 128 A rows: keep (128 rows - tile) bytes of slack after the last stage inside the allocation
  pl.stages = (225 * 1024 - (BLOCK_M * row_bytes - pl.g_tile_bytes)) / pl.stage_bytes;
  if (pl.stages > WG_MAX_STAGES) pl.stages = WG_MAX_STAGES;
  if (pl.stages < 2) return pl;
  pl.tmem_cols = 32;
  while (pl.tmem_cols < pl.c_tile) pl.tmem_cols <<= 1;
  const long long total_kb = (long long)B * H * W / pl.kblk;
  const int tiles = pl.m_tiles * taps * pl.c_tiles;
  long long s = (148 + tiles / 2) / tiles;
  if (s > total_kb / 4) s = total_kb / 4;
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  pl.splits = (int)s;
  pl.ok = true;
  return pl;
}

}  // namespace tc
}  // namespace flowk

using namespace flowk;
using namespace flowk::tc;

// x_left[.., w] = x[.., w-1] (tap dx = -1), x_right[.., w] = x[.., w+1] (tap dx = +1), zero at the image border
__global__ void shift_columns_kernel(const float* __restrict__ x, float* __restrict__ xl, float* __restrict__ xr,
                                     long long total4, int W) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const long long e = i * 4;
    const int w0 = (int)(e % W);
    const float4 v = *reinterpret_cast<const float4*>(x + e);
    const float left = w0 > 0 ? x[e - 1] : 0.f, right = w0 + 4 < W ? x[e + 4] : 0.f;
    *reinterpret_cast<float4*>(xl + e) = make_float4(left, v.x, v.y, v.z);
    *reinterpret_cast<float4*>(xr + e) = make_float4(v.y, v.z, v.w, right);
  }
}

extern "C" int flowk_shift_columns(const float* x, float* x_left, float* x_right, long long total, int W,
                                   flowk_stream_t stream) {
  if (total < 0 || W < 4 || W % 4 || total % W) return FLOWK_ERR_SHAPE;
  if (total == 0) return FLOWK_OK;
  if (!x || !x_left || !x_right) return FLOWK_ERR_ARG;
  if (!aligned16(x) || !aligned16(x_left) || !aligned16(x_right)) return FLOWK_ERR_ALIGN;
  long long blocks = (total / 4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  shift_columns_kernel<<<(unsigned)blocks, 256, 0, stream>>>(x, x_left, x_right, total / 4, W);
  return launch_status();
}

static size_t g_wgrad_smem_attr = 0;      // largest dynamic shared memory opted into so far (both entry points)

// row-major operand [M, C] (C % 32 == 0) viewed by TMA as dims (32, M, C/32); box (32 channels, 32 rows, blocks):
// per 32-channel block a [32 rows x 128 B] tile, swizzled in 32-byte atoms as transposed tf32 operands need
static bool make_map_rows(CUtensorMap* map, const float* base, long long M, int C, int blocks) {
  cuuint64_t dims[3] = {32, (cuuint64_t)M, (cuuint64_t)(C / 32)};
  cuuint64_t strides[2] = {(cuuint64_t)C * 4, 128};
  cuuint32_t box[3] = {32, (cuuint32_t)BLOCK_K, (cuuint32_t)blocks};
  cuuint32_t estr[3] = {1, 1, 1};
  return encode_fn() && encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box,
                                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static WgradPlan plan_linear_wgrad(long long M, int K, int N) {
  WgradPlan pl = {};
  if (M < BLOCK_K || M % BLOCK_K || M > 0x7fffffff || K < 32 || K % 32 || N < 32 || N % 32) return pl;
  auto tiles_of = [](int a, int b) { return ((a + BLOCK_M - 1) / BLOCK_M) * ((b + 255) / 256); };
  pl.swap = tiles_of(K, N) < tiles_of(N, K) ? 1 : 0;
  pl.a_ch = pl.swap ? K : N;
  pl.b_ch = pl.swap ? N : K;
  pl.c_tiles = (pl.b_ch + 255) / 256;
  pl.c_tile = ((pl.b_ch + pl.c_tiles - 1) / pl.c_tiles + 31) / 32 * 32;
  pl.m_tiles = (pl.a_ch + BLOCK_M - 1) / BLOCK_M;
  pl.g_tile_bytes = (pl.a_ch < BLOCK_M ? pl.a_ch : BLOCK_M) / 32 * 4096;
  pl.stage_bytes = 2 * (pl.g_tile_bytes + pl.c_tile * 128);
  pl.stages = (225 * 1024 - (BLOCK_M * 128 - pl.g_tile_bytes)) / pl.stage_bytes;
  if (pl.stages > WG_MAX_STAGES) pl.stages = WG_MAX_STAGES;
  if (pl.stages < 2) return pl;
  pl.tmem_cols = 32;
  while (pl.tmem_cols < pl.c_tile) pl.tmem_cols <<= 1;
  const long long total_kb = M / BLOCK_K;
  const int tiles = pl.m_tiles * pl.c_tiles;
  long long s = (148 + tiles / 2) / tiles;
  if (s > total_kb / 4) s = total_kb / 4;
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  pl.splits = (int)s;
  pl.ok = true;
  return pl;
}

extern "C" int flowk_linear_wgrad_splits(long long M, int K, int N, int* transposed) {
  const WgradPlan pl = plan_linear_wgrad(M, K, N);
  if (transposed) *transposed = pl.ok ? pl.swap : 0;
  return pl.ok ? pl.splits : 0;
}

extern "C" int flowk_linear_wgrad(const float* x, const float* gy, float* partial, int* status, long long M, int K, int N,
                                  flowk_stream_t stream) {
  const WgradPlan pl = plan_linear_wgrad(M, K, N);
  if (!pl.ok) return FLOWK_ERR_SHAPE;
  if (!x || !gy || !partial) return FLOWK_ERR_ARG;
  if (!aligned16(x) || !aligned16(gy) || !aligned16(partial)) return FLOWK_ERR_ALIGN;
  WgradParams p = {};
  p.N = pl.a_ch;
  p.Cin = pl.b_ch;
  p.shift_a = pl.swap;
  p.rows = 1;
  p.kblk = BLOCK_K;
  p.g_tile_bytes = pl.g_tile_bytes;
  p.taps = 1;
  p.W = 32;
  p.kb_per_image = (int)(M / BLOCK_K);
  p.total_kb = p.kb_per_image;
  const int a_blocks = pl.g_tile_bytes / 4096, b_blocks = (pl.b_ch < pl.c_tile ? pl.b_ch : pl.c_tile) / 32;
  p.g_rows = a_blocks * 32;          // bytes per box = rows * 128 (32 rows x 128 B per block)
  p.x_rows = b_blocks * 32;
  p.c_tile = pl.c_tile;
  p.c_tiles = pl.c_tiles;
  p.m_tiles = pl.m_tiles;
  p.stages = pl.stages;
  p.stage_bytes = pl.stage_bytes;
  p.tmem_cols = pl.tmem_cols;
  p.partial = partial;
  p.status = status;
  CUtensorMap mg, mx;
  // map_g always describes gy, map_x always x; their box depths follow the side (A: 128 channels, B: c_tile) they feed
  if (!make_map_rows(&mg, gy, M, N, pl.swap ? b_blocks : a_blocks) || !make_map_rows(&mx, x, M, K, pl.swap ? a_blocks : b_blocks))
    return FLOWK_ERR_ARG;
  const size_t smem = (size_t)pl.stages * pl.stage_bytes + 1024 + (BLOCK_M * 128 - pl.g_tile_bytes);
  if (smem > g_wgrad_smem_attr) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    g_wgrad_smem_attr = smem;
  }
  FLOWK_CUDA_OK(launch_pdl(conv_wgrad_kernel, dim3(pl.m_tiles * pl.c_tiles, pl.splits), dim3(WG_THREADS), smem, stream, mg, mx,
                           mx, mx, p));
  return FLOWK_OK;
}

extern "C" int flowk_conv_wgrad_splits(int B, int H, int W, int Cin, int N, int taps, int* transposed) {
  const WgradPlan pl = plan_wgrad(B, H, W, Cin, N, taps);
  if (transposed) *transposed = pl.ok ? pl.swap : 0;
  return pl.ok ? pl.splits : 0;
}

extern "C" int flowk_conv_wgrad(const float* x, const float* x_left, const float* x_right, const float* gy, float* partial,
                                int* status, int B, int H, int W, int Cin, int N, int taps, flowk_stream_t stream) {
  const WgradPlan pl = plan_wgrad(B, H, W, Cin, N, taps);
  if (!pl.ok) return FLOWK_ERR_SHAPE;
  if (!x || !gy || !partial || (taps == 9 && (!x_left || !x_right))) return FLOWK_ERR_ARG;
  if (taps == 1) x_left = x_right = x;
  if (!aligned16(x) || !aligned16(x_left) || !aligned16(x_right) || !aligned16(gy) || !aligned16(partial))
    return FLOWK_ERR_ALIGN;
  WgradParams p = {};
  p.N = pl.a_ch;
  p.Cin = pl.b_ch;
  p.shift_a = pl.swap;
  p.g_tile_bytes = pl.g_tile_bytes;
  p.taps = taps;
  p.W = W;
  p.kblk = pl.kblk;
  p.kb_per_image = H * W / pl.kblk;
  p.total_kb = B * p.kb_per_image;
  p.g_rows = pl.a_ch < BLOCK_M ? pl.a_ch : BLOCK_M;
  p.x_rows = pl.b_ch < pl.c_tile ? pl.b_ch : pl.c_tile;
  p.c_tile = pl.c_tile;
  p.c_tiles = pl.c_tiles;
  p.m_tiles = pl.m_tiles;
  p.stages = pl.stages;
  p.stage_bytes = pl.stage_bytes;
  p.tmem_cols = pl.tmem_cols;
  p.partial = partial;
  p.status = status;
  CUtensorMap mg, mx, mxm, mxp;
  const int gy_rows = pl.swap ? p.x_rows : p.g_rows, xx_rows = pl.swap ? p.g_rows : p.x_rows;
  if (!make_map_cm(&mg, gy, B, N, H * W, gy_rows, pl.kblk) || !make_map_cm(&mx, x, B, Cin, H * W, xx_rows, pl.kblk) ||
      !make_map_cm(&mxm, x_left, B, Cin, H * W, xx_rows, pl.kblk) || !make_map_cm(&mxp, x_right, B, Cin, H * W, xx_rows, pl.kblk))
    return FLOWK_ERR_ARG;
  const size_t smem = (size_t)pl.stages * pl.stage_bytes + 1024 + (BLOCK_M * pl.kblk * 4 - pl.g_tile_bytes);
  if (smem > g_wgrad_smem_attr) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    g_wgrad_smem_attr = smem;
  }
  FLOWK_CUDA_OK(launch_pdl(conv_wgrad_kernel, dim3(pl.m_tiles * taps * pl.c_tiles, pl.splits), dim3(WG_THREADS), smem,
                           stream, mg, mx, mxm, mxp, p));
  return FLOWK_OK;
}

// NHWC rows [NB, H, W, C] (C % 32 == 0) viewed by TMA as dims (32, W, H, NB, C/32); box (32 channels, bw, bh, bb, blocks):
// per 32-channel block a [32 pixels x 128 B] tile laid out (and swizzled) exactly like make_map_rows' [32 rows x 128 B]
static bool make_map_nhwc(CUtensorMap* map, const float* base, int NB, int H, int W, int C, int bw, int bh, int bb,
                          int blocks) {
  cuuint64_t dims[5] = {32, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)NB, (cuuint64_t)(C / 32)};
  cuuint64_t strides[4] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4, 128};
  cuuint32_t box[5] = {32, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bb, (cuuint32_t)blocks};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  return encode_fn() && encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(base), dims, strides, box,
                                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct NhwcBox {
  int bw, bh, bb;
};

// The plan of plan_linear_wgrad over M = NB*H*W rows, with the split-K count re-balanced over taps x tiles CTAs and the
// k-block box: bw = min(W, 32) columns, bh rows, bb images (bw * bh * bb = 32; every box lies in whole images).
static WgradPlan plan_nhwc_wgrad(int NB, int H, int W, int Cin, int N, int taps, int dil, NhwcBox* box) {
  WgradPlan none = {};
  if (NB < 1 || H < 1 || W < 1 || dil < 1 || (taps != 1 && taps != 9 && taps != 25)) return none;
  if (W <= 32 ? 32 % W : W % 32) return none;
  const int bw = W < 32 ? W : 32, bh = H < 32 / bw ? H : 32 / bw;
  if (H % bh || 32 % (bw * bh)) return none;
  const int bb = 32 / (bw * bh);
  if (NB % bb || (long long)NB * H * W > 0x7fffffffLL) return none;
  WgradPlan pl = plan_linear_wgrad((long long)NB * H * W, Cin, N);
  if (!pl.ok) return pl;
  const long long total_kb = (long long)NB * H * W / BLOCK_K;
  const int tiles = pl.m_tiles * taps * pl.c_tiles;
  long long s = (148 + tiles / 2) / tiles;
  if (s > total_kb / 4) s = total_kb / 4;
  if (s > 64) s = 64;
  if (s < 1) s = 1;
  pl.splits = (int)s;
  if (box) *box = NhwcBox{bw, bh, bb};
  return pl;
}

extern "C" int flowk_conv_wgrad_nhwc_splits(int NB, int H, int W, int Cin, int N, int taps, int dilation, int* transposed) {
  const WgradPlan pl = plan_nhwc_wgrad(NB, H, W, Cin, N, taps, dilation, nullptr);
  if (transposed) *transposed = pl.ok ? pl.swap : 0;
  return pl.ok ? pl.splits : 0;
}

extern "C" int flowk_conv_wgrad_nhwc(const float* x, const float* gy, float* partial, int* status, int NB, int H, int W,
                                     int Cin, int N, int taps, int dilation, flowk_stream_t stream) {
  NhwcBox bx;
  const WgradPlan pl = plan_nhwc_wgrad(NB, H, W, Cin, N, taps, dilation, &bx);
  if (!pl.ok) return FLOWK_ERR_SHAPE;
  if (!x || !gy || !partial) return FLOWK_ERR_ARG;
  if (!aligned16(x) || !aligned16(gy) || !aligned16(partial)) return FLOWK_ERR_ALIGN;
  WgradParams p = {};
  p.N = pl.a_ch;
  p.Cin = pl.b_ch;
  p.shift_a = pl.swap;
  p.rows = 2;
  p.kblk = BLOCK_K;
  p.g_tile_bytes = pl.g_tile_bytes;
  p.taps = taps;
  p.ksz = taps == 25 ? 5 : taps == 9 ? 3 : 1;
  p.dil = dilation;
  p.W = W;
  p.bw = bx.bw;
  p.bh = bx.bh;
  p.bb = bx.bb;
  p.kpi_w = W / bx.bw;
  p.kpi_h = H / bx.bh;
  p.total_kb = (int)((long long)NB * H * W / BLOCK_K);
  p.kb_per_image = p.total_kb;
  const int a_blocks = pl.g_tile_bytes / 4096, b_blocks = (pl.b_ch < pl.c_tile ? pl.b_ch : pl.c_tile) / 32;
  p.g_rows = a_blocks * 32;
  p.x_rows = b_blocks * 32;
  p.c_tile = pl.c_tile;
  p.c_tiles = pl.c_tiles;
  p.m_tiles = pl.m_tiles;
  p.stages = pl.stages;
  p.stage_bytes = pl.stage_bytes;
  p.tmem_cols = pl.tmem_cols;
  p.partial = partial;
  p.status = status;
  CUtensorMap mg, mx;
  if (!make_map_nhwc(&mg, gy, NB, H, W, N, bx.bw, bx.bh, bx.bb, pl.swap ? b_blocks : a_blocks) ||
      !make_map_nhwc(&mx, x, NB, H, W, Cin, bx.bw, bx.bh, bx.bb, pl.swap ? a_blocks : b_blocks))
    return FLOWK_ERR_ARG;
  const size_t smem = (size_t)pl.stages * pl.stage_bytes + 1024 + (BLOCK_M * 128 - pl.g_tile_bytes);
  if (smem > g_wgrad_smem_attr) {
    FLOWK_CUDA_OK(cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    g_wgrad_smem_attr = smem;
  }
  FLOWK_CUDA_OK(launch_pdl(conv_wgrad_kernel, dim3(pl.m_tiles * taps * pl.c_tiles, pl.splits), dim3(WG_THREADS), smem, stream,
                           mg, mx, mx, mx, p));
  return FLOWK_OK;
}
