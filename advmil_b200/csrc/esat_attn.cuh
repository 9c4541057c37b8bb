// Shared between the FFMA (esat_kernels.cu) and the tcgen05 (esat_attn_tc.cu, esat_attn_bwd_tc.cu) attention kernels.
#pragma once
#include "common.cuh"

namespace advmil {

struct AttDrop {             // dropout on the attention probabilities of (bag, head, query, key)
  Drop drop;                 // counter generator (drop.mask unused)
  const uint8_t* mask;       // injected keep masks: per bag [heads, Rb, Rb] at mask_off[bag], or nullptr
  const int64_t* mask_off;
  int heads;
  __device__ __forceinline__ bool keep(int bag, int head, int q, int k, int Rb, int grow) const {
    if (!drop.active) return true;
    if (mask) return mask[mask_off[bag] + ((int64_t)head * Rb + q) * Rb + k] != 0;
    return drop.keep((uint32_t)grow * (uint32_t)heads + (uint32_t)head, (uint32_t)k);
  }
};

// tcgen05 forward (esat_attn_tc.cu): head widths 16 / 32 / 48 / 64; mx = the largest number of regions of a bag
bool mha_tcgen05_supported(int hd, int d);
int mha_fwd_tcgen05(const float* qkv, const int32_t* ro, int bags, int Rtot, int d, int heads, int mx, float scale, const AttDrop& ad,
                    float* ctx, float* lse, cudaStream_t st);

// tcgen05 backward (esat_attn_bwd_tc.cu): dQ pass + dK/dV pass, same head widths; Dq [heads, Rtot] scratch (D = dO . O)
int mha_bwd_tcgen05(const float* qkv, const float* ctx, const float* d_ctx, const float* lse, const int32_t* ro, int bags, int Rtot, int d,
                    int heads, int mx, float scale, const AttDrop& ad, float* d_qkv, float* Dq, cudaStream_t st);

}  // namespace advmil
