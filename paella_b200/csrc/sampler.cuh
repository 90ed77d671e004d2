// Fused out_mapper + Gumbel-max draw (see sampler.cu).
#pragma once
#include "common.cuh"

namespace pb {
// rows the fp16 feature buffer must be able to hold for R token rows (whole 4*rs-row Philox blocks)
int64_t fused_sampler_rows_padded(int64_t R, int NL);
// a16: fp16 [R, Kc] guided features; w16: fp16 [NL, Kc] out_mapper weight; out: int64 [R]
int launch_fused_sampler(const __half* a16, int64_t R, int Kc, const __half* w16, int NL, float inv_t, uint64_t seed,
                         uint64_t offset, int64_t* out, cudaStream_t st);
// scratch of launch_fused_sampler_masked (the needed-slot list), 256-byte aligned
int64_t fused_sampler_mask_scratch_bytes(int64_t R, int NL);
// same draw as launch_fused_sampler, written only where mask[row] != 0 (uint8 [R]); other rows of tokens_inout keep their value
int launch_fused_sampler_masked(const __half* a16, int64_t R, int Kc, const __half* w16, int NL, float inv_t, uint64_t seed,
                                uint64_t offset, const uint8_t* mask, void* mask_scratch, int64_t* tokens_inout, cudaStream_t st);
}  // namespace pb
