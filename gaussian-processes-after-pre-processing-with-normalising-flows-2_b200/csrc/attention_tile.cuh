// Operand-tile helpers shared by the tcgen05 attention kernels (attention_tc.cu, block_tail_tc.cu): fp16 (hi, lo) packing,
// K-major swizzled tile offsets, the TS-mode MMA and wide tensor-memory loads / stores (sm_100a).
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "umma.cuh"

namespace flowk {
namespace tc {

constexpr int ROW_B = 128;                      // bytes per swizzle row: 64 fp16

// byte offset of the 16-byte chunk `chunk` (0..7) of row `r` inside a K-major SWIZZLE_128B tile
__device__ __forceinline__ uint32_t sw_off(int r, int chunk) { return (uint32_t)(r * ROW_B + ((chunk ^ (r & 7)) << 4)); }

// 8 floats -> 8 fp16 hi + 8 fp16 lo (x = hi + lo), packed; |x| must be < 65504 (q, k, v and the softmax weights are)
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));      // low half = a
  return r;
}
__device__ __forceinline__ void unpack_h2(uint32_t v, float& a, float& b) {
  unsigned short lo16 = (unsigned short)(v & 0xffffu), hi16 = (unsigned short)(v >> 16);
  asm("cvt.f32.f16 %0, %1;" : "=f"(a) : "h"(lo16));
  asm("cvt.f32.f16 %0, %1;" : "=f"(b) : "h"(hi16));
}
__device__ __forceinline__ void cvt8(const float* v, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    h[i] = pack_h2(v[2 * i], v[2 * i + 1]);
    float a, b;
    unpack_h2(h[i], a, b);
    l[i] = pack_h2(v[2 * i] - a, v[2 * i + 1] - b);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

constexpr int V2_ROW_B = 64;                    // bytes per SWIZZLE_64B row of Q / K

// byte offset of the 16-byte chunk `chunk` (0..3) of row `r` inside a K-major SWIZZLE_64B tile (512-byte 8-row atoms)
__device__ __forceinline__ uint32_t sw64_off(int r, int chunk) {
  return (uint32_t)(r * V2_ROW_B + ((chunk ^ ((r >> 1) & 3)) << 4));
}
// kind::f16 MMA with the A operand in tensor memory (TS mode): 128 lanes = M rows, K = 16 fp16 packed in 8 columns
__device__ __forceinline__ void umma_f16_ts_elect(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
// 32 consecutive columns of this thread's lane, one wait
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// 8 packed columns into this thread's lane (no wait: the caller waits once for all its stores)
__device__ __forceinline__ void tmem_st8u(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

// K-major fp16 matrix [rows, cols] -> 2-D map with boxes of 32 columns (one 64-byte swizzle row) x box_rows rows
inline bool make_map_sw64(CUtensorMap* map, const void* base, long long rows, long long cols, int box_rows) {
  if (!encode_fn()) return false;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace tc
}  // namespace flowk
