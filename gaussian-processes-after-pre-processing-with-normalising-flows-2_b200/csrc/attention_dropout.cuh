// Attention-weight dropout mask of the training attention kernels (attention_train.cu, attention_train_tc.cu): a
// counter-based hash of (seed, image*head, query, key), so the backward regenerates exactly the forward's mask and
// flowk_attention_dropout_mask can write it out for tests.  One definition, shared by every kernel that applies it.
#pragma once
#include "common.cuh"

namespace flowk {
namespace attn_train {

// dropout multiplier of attention weight (query q, key k) of pair `pair`: 0 with probability thresh / 2^32, else 1/(1-p)
__device__ __forceinline__ float drop_scale(uint32_t seed, uint32_t pair, uint32_t q, uint32_t k, uint32_t S, uint32_t thresh,
                                            float inv_keep) {
  uint32_t x = ((pair * S + q) * S + k) ^ seed;
  x *= 0x9E3779B1u; x ^= x >> 16;
  x *= 0x85EBCA6Bu; x ^= x >> 13;
  x *= 0xC2B2AE35u; x ^= x >> 16;
  return x >= thresh ? inv_keep : 0.f;
}
// the per-layer seed: the device-side step seed (read at run time, so a captured graph draws fresh masks per replay) x salt
__device__ __forceinline__ uint32_t layer_seed(const unsigned* seed_dev, unsigned salt) {
  return (seed_dev ? *seed_dev : 0u) * 0x01000193u ^ (salt * 0x9E3779B9u + 0x7F4A7C15u);
}

}  // namespace attn_train
}  // namespace flowk
