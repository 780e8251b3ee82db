// tcgen05 / TMA / mbarrier PTX wrappers and UMMA descriptor builders shared by the tensor-core kernels (sm_100a).
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace flowk {
namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 32;                 // fp32 elements = one 128-byte swizzle row
constexpr int UMMA_K = 8;                   // tf32: 32 bytes per MMA along K

// --------------------------------------------------------------------------------------------------
// PTX wrappers
// --------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must never hang the GPU.  On timeout the CTA-wide `failed` flag is raised, every
// later wait returns at once, the kernel finishes (with garbage) and the host sees the flag in `status`.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, volatile int* failed) {
  if (*failed) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 400000000LL) {      // ~0.2 s
      *failed = 1;
      return;
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(smem)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_acc(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.u32 p, 1, 1;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc)
      : "memory");
}
// kind::f16 (fp16 operands, fp32 accumulate): K = 16 per instruction, twice the tf32 rate per dispatch
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
template <bool F16>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  if (F16) umma_f16(tmem_d, desc_a, desc_b, idesc, accumulate);
  else umma_tf32(tmem_d, desc_a, desc_b, idesc, accumulate);
}

// --- warp-uniform issue path -----------------------------------------------------------------------------------------
// When the MMA loop runs under `if (lane == 0)` the compiler sees divergent control flow, keeps the descriptors in
// per-thread registers and wraps every tcgen05.mma in a register -> uniform-register "waterfall" loop (~13 instructions
// with long-latency R2UR per MMA: measured 110-170 cycles per MMA, the bound of these kernels' main loops).  Here the WHOLE
// warp executes the loop with identical (uniform) operands and only the instruction itself is predicated on the lane
// elected once by elect.sync.
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred;
}
template <bool F16>
__device__ __forceinline__ void umma_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate, uint32_t leader) {
  if (F16)
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar)), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// --- CTA pairs (cta_group::2): two CTAs of a cluster, on the two SMs of one TPC, run ONE M = 256 MMA per instruction.
// Each CTA stages its own 128 activation rows and HALF of the weight rows (the tensor cores read both halves), so the
// weight bytes an SM has to pull through TMA halve; the accumulator of CTA r (rows 128 r .. 128 r + 127, all N columns)
// lands in that CTA's own TMEM, i.e. the epilogue is the single-CTA one.  The leader (cluster rank 0) issues the MMAs; the
// TMA loads of BOTH CTAs signal the leader's "full" barrier, the MMA commits are multicast to both CTAs' "empty" barriers.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `bar` (an address in this CTA's shared memory) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa_rank(const void* bar, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(bar)), "r"(rank));
  return r;
}
// `bytes` (a multiple of 16) from this CTA's shared memory to the shared::cluster address `dst` of another CTA of the
// cluster, completing as transaction bytes on the barrier at shared::cluster address `bar` (in the destination CTA)
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "r"(smem_u32(src)), "r"(bytes), "r"(bar)
               : "memory");
}
// one arrival on the barrier at shared::cluster address `bar` (possibly in another CTA of the cluster)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* smem, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1,
                                                 int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* smem, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols));
}
__device__ __forceinline__ void umma_f16_pair_elect(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                    uint32_t accumulate, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
// arrives on the barrier at `bar`'s offset in BOTH CTAs of the pair once the MMAs issued so far have retired
__device__ __forceinline__ void umma_commit_pair_elect(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t.reg .b16 m;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "mov.b16 m, 3;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
      ::"r"(smem_u32(bar)), "r"(leader)
      : "memory");
}
// kind::f16 instruction descriptor of a pair MMA: M = 256
__device__ __forceinline__ uint32_t make_idesc_f16_pair(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
      "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
      "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])),
      "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
      "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// K-major, 128-byte swizzle: 8-row groups of 1024 B (SBO), rows of 128 B; LBO unused.  (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                       // leading byte offset (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;             // stride byte offset: next 8-row group
  d |= (uint64_t)1 << 46;                       // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
  return d;
}
// K-major, 64-byte swizzle (rows of 16 fp32): 8-row groups of 512 B.  Used when a k-block can only be 16 elements long
// (weight gradients of 4x4 feature maps: 16 pixels per image).
__device__ __forceinline__ uint64_t make_smem_desc_sw64(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;                       // SWIZZLE_64B
  return d;
}
// MN-major tf32 operand (the contraction index is the ROW of the tile, 32 channels = 128 B are contiguous): tiles of
// [32 rows x 128 B] per 32-channel block, loaded by TMA with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B and described with the
// matching UMMA layout type 1 (SWIZZLE_128B_BASE32B): LBO = bytes between channel blocks, SBO = 512 B between groups of
// four rows; one K=8 MMA consumes 8 rows = 1024 B.  (Measured: profiles/dbg/umma_mn_probe.cu - the plain 128-byte
// swizzle, layout type 2, silently yields zeros for transposed tf32 operands.)
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t smem_addr, uint32_t block_stride_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((block_stride_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}
__device__ __forceinline__ uint32_t make_idesc_mn(int n) {       // both operands MN-major (bits 15, 16)
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(BLOCK_M >> 4) << 24);
}
// cute::UMMA::InstrDescriptor: c=F32 [4,6), a=TF32 [7,10), b=TF32 [10,13), K-major both, N>>3 [17,23), M>>4 [24,29)
__device__ __forceinline__ uint32_t make_idesc(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
}

// kind::f16 descriptor: c=F32 [4,6), a=F16 (0) [7,10), b=F16 (0) [10,13), K-major both, N>>3 [17,23), M>>4 [24,29)
__device__ __forceinline__ uint32_t make_idesc_f16(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
}
template <bool F16>
__device__ __forceinline__ uint32_t make_idesc_t(int n) { return F16 ? make_idesc_f16(n) : make_idesc(n); }

// four consecutive elements -> 8-byte stores into the hi / lo arrays (element offset `o`, o % 4 == 0)
__device__ __forceinline__ void store_hilo4_f16(float* out_hi, float* out_lo, size_t o, const float* v) {
  unsigned short h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) split_f16(v[i], h[i], l[i]);
  uint2 hv = make_uint2((uint32_t)h[0] | ((uint32_t)h[1] << 16), (uint32_t)h[2] | ((uint32_t)h[3] << 16));
  uint2 lv = make_uint2((uint32_t)l[0] | ((uint32_t)l[1] << 16), (uint32_t)l[2] | ((uint32_t)l[3] << 16));
  *reinterpret_cast<uint2*>(reinterpret_cast<unsigned short*>(out_hi) + o) = hv;
  *reinterpret_cast<uint2*>(reinterpret_cast<unsigned short*>(out_lo) + o) = lv;
}

// x = hi + lo with BOTH parts exactly representable in TF32 (round-to-nearest): the tensor core merely truncates
// its fp32 containers, which would otherwise bias every product by up to 2^-10 of the lo term.
__device__ __forceinline__ float rna_tf32(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = rna_tf32(x);
  lo = rna_tf32(x - hi);
}
__device__ __forceinline__ void store_hilo4_tf32(float* out_hi, float* out_lo, size_t o, const float* v) {
  float h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) split_tf32(v[i], h[i], l[i]);
  *reinterpret_cast<float4*>(out_hi + o) = make_float4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<float4*>(out_lo + o) = make_float4(l[0], l[1], l[2], l[3]);
}
template <bool F16>
__device__ __forceinline__ void store_hilo4(float* out_hi, float* out_lo, size_t o, const float* v) {
  if (F16) store_hilo4_f16(out_hi, out_lo, o, v);
  else store_hilo4_tf32(out_hi, out_lo, o, v);
}
// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

}  // namespace tc
}  // namespace flowk
