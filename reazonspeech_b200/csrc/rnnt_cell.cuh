// Device arithmetic shared by the fp32-accurate RNN-T paths (ALSD beam search, decode_alsd.cu; forced alignment, align.cu):
// the three-term bf16 split of activations that meet the tripled weights in the tcgen05 GEMM, and the LSTM cell.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace rs {

// x -> three bf16 values with hi + mid + lo == x to 24 mantissa bits
__device__ __forceinline__ void split3(float x, __nv_bfloat16& hi, __nv_bfloat16& mid, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(hi);
  mid = __float2bfloat16_rn(r1);
  lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
}

// LSTM cell, gate order i, f, g, o (biases already in the gates): (c_prev, gates) -> (h, c)
__device__ __forceinline__ void lstm_cell(float gi, float gf, float gg, float go, float c_prev, float& h, float& c) {
  const float ig = sigmoidf_accurate(gi), fg = sigmoidf_accurate(gf);
  const float cg = tanhf(gg), og = sigmoidf_accurate(go);
  c = fg * c_prev + ig * cg;
  h = og * tanhf(c);
}

}  // namespace rs
