// Fused out_mapper GEMM + temperature + multinomial draw: logits never reach HBM.
// Replaces ref/src/modules.py:184-187 (out_mapper 1x1 conv, 256 -> 8192) and ref/src/utils.py:45-50
// (CFG mix, /T, softmax, permute+reshape copy, torch.multinomial) — ~0.74 GB of HBM traffic per image-step in
// the reference, ~1 MB here (SURVEY.md §8d).
//
// The classifier-free-guidance mix is linear, so it is applied to the 256-wide LayerNorm'd features BEFORE the
// GEMM (one GEMM instead of two).  The draw is Gumbel-max in the log domain on torch's own random stream:
//     token = argmax_k ( l_k / T  -  log q_k ),   q_k = the Exp(1) variate torch.multinomial's
//                                                  exponential_() would hand to element (row, k)
// which equals argmax_k softmax(l/T)_k / q_k (what torch computes) up to fp32 rounding of near-ties.
//
// One CTA per 128 token rows, 320 threads:
//   warp 0     TMA: the 128 x c_out A tile once (resident), then W tiles [128 labels x 64] through a 6-deep ring
//   warp 1     tcgen05.mma issuer: 128x128 accumulators, double-buffered in TMEM
//   warps 2-9  epilogue: tcgen05.ld (thread = token row), Philox4x32-10 per element, running arg-max in registers
#include <cstdlib>

#include "gemm.cuh"
#include "sampler.cuh"

namespace pb {

constexpr int SMP_BN = 128;
constexpr int SMP_STAGES = 6;
constexpr int SMP_MAX_KB = 4;                 // c_out <= 256
constexpr int SMP_EPI_WARPS = 16;             // 4 per TMEM lane quarter: Philox is a long dependent chain, hide it with warps
constexpr int SMP_THREADS = 64 + 32 * SMP_EPI_WARPS;
constexpr int SMP_COLS_PER_WARP = SMP_BN / (SMP_EPI_WARPS / 4);
constexpr int SMP_A_BYTES = 128 * 64 * 2;     // one k-block of the A tile
constexpr int SMP_W_BYTES = SMP_BN * 64 * 2;
constexpr int SMP_SMEM = SMP_MAX_KB * SMP_A_BYTES + SMP_STAGES * SMP_W_BYTES + 1024 + 256 + (SMP_EPI_WARPS / 4) * 128 * 8;

// MASKED: only rows with mask[row] != 0 are written; a CTA whose 128 rows are all kept exits before its first TMA.
template <bool MASKED>
__global__ void __launch_bounds__(SMP_THREADS, 1)
fused_sampler_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, int R, int NL,
                     int Kc, float inv_t, TorchPhilox rng, const uint8_t* __restrict__ mask, int64_t* __restrict__ out) {
    if constexpr (MASKED) {
        const int r = blockIdx.x * 128 + (int)threadIdx.x;
        if (!__syncthreads_or(threadIdx.x < 128 && r < R && mask[r] != 0)) return;
    }
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t a_base = smem_base;
    const uint32_t w_base = smem_base + SMP_MAX_KB * SMP_A_BYTES;
    const uint32_t bar_base = w_base + SMP_STAGES * SMP_W_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (SMP_STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * SMP_STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * SMP_STAGES + 2 + s); };
    const uint32_t a_bar = bar_base + 8u * (2 * SMP_STAGES + 4);
    const uint32_t tmem_slot = bar_base + 8u * (2 * SMP_STAGES + 5);
    uint8_t* tail = smem_gen + (bar_base - smem_base) + 256;
    float* best_v = reinterpret_cast<float*>(tail);                // [slices-1][128] candidates of the other column slices
    int* best_i = reinterpret_cast<int*>(tail + (SMP_EPI_WARPS / 4) * 128 * 4);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int n_kb = (Kc + 63) / 64;
    const int n_chunks = (NL + SMP_BN - 1) / SMP_BN;
    const int m_idx = blockIdx.x * 128;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a);
        ptx::prefetch_tensormap(&tm_w);
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < SMP_STAGES; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
            for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), SMP_EPI_WARPS); }
            ptx::mbar_init(a_bar, 1);
            ptx::fence_barrier_init();
        }
        __syncwarp();
        ptx::tmem_alloc(tmem_slot, 256);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<uint32_t*>(smem_gen + (tmem_slot - smem_base));

    if (warp == 0) {
        if (ptx::elect_one()) {
            ptx::mbar_arrive_expect_tx(a_bar, n_kb * SMP_A_BYTES);
            for (int kb = 0; kb < n_kb; ++kb) ptx::tma_load_2d(&tm_a, a_bar, a_base + kb * SMP_A_BYTES, kb * 64, m_idx);
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = 0; ch < n_chunks; ++ch)
                for (int kb = 0; kb < n_kb; ++kb) {
                    ptx::mbar_wait(empty_bar(stage), phase ^ 1);
                    ptx::mbar_arrive_expect_tx(full_bar(stage), SMP_W_BYTES);
                    ptx::tma_load_2d(&tm_w, full_bar(stage), w_base + stage * SMP_W_BYTES, kb * 64, ch * SMP_BN);
                    if (++stage == SMP_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = ptx::umma_idesc_f16(128, SMP_BN, 0);
        ptx::mbar_wait(a_bar, 0);
        int stage = 0;
        uint32_t phase = 0;
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int as = ch & 1;
            ptx::mbar_wait(tempty_bar(as), ((ch >> 1) & 1) ^ 1);
            ptx::tc_fence_after();
            for (int kb = 0; kb < n_kb; ++kb) {
                ptx::mbar_wait(full_bar(stage), phase);
                ptx::tc_fence_after();
                if (ptx::elect_one()) {
                    const uint64_t da = ptx::umma_desc_kmajor_sw128(a_base + kb * SMP_A_BYTES);
                    const uint64_t db = ptx::umma_desc_kmajor_sw128(w_base + stage * SMP_W_BYTES);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        ptx::umma_f16(tmem_base + as * SMP_BN, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                    ptx::umma_commit(empty_bar(stage));
                    if (kb == n_kb - 1) ptx::umma_commit(tfull_bar(as));
                }
                __syncwarp();
                if (++stage == SMP_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;                  // TMEM lane quarter
        const int half = (warp - 2) >> 2;        // which slice of the chunk's 128 columns
        const int row_in_tile = q * 32 + lane;
        const int row = m_idx + row_in_tile;
        const bool row_ok = row < R;
        float bv = -INFINITY;
        int bidx = 0;
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int as = ch & 1;
            ptx::mbar_wait(tfull_bar(as), (ch >> 1) & 1);
            ptx::tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < SMP_COLS_PER_WARP; c += 32) {
                const int col0 = ch * SMP_BN + half * SMP_COLS_PER_WARP + c;
                float v[32];
                ptx::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * SMP_BN + half * SMP_COLS_PER_WARP + c), v);
                if (row_ok && col0 < NL) {
                    const uint64_t e0 = (uint64_t)row * (uint64_t)NL + (uint64_t)col0;
                    uint64_t j = e0 / rng.stride;
                    uint32_t tid = (uint32_t)(e0 - j * rng.stride);
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const uint4 r4 = torch_philox_call(rng, tid, j >> 2);
                        const uint32_t ln = (uint32_t)(j & 3);
                        const uint32_t bits = ln == 0 ? r4.x : ln == 1 ? r4.y : ln == 2 ? r4.z : r4.w;
                        const float qv = torch_exponential1(u32_to_uniform(bits));
                        const float gum = fmaf(v[i], inv_t, -__logf(qv));
                        if (col0 + i < NL && gum > bv) { bv = gum; bidx = col0 + i; }
                        if (++tid == rng.stride) { tid = 0; ++j; }
                    }
                }
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tempty_bar(as));
        }
        // combine the column slices of each row
        constexpr int NS = SMP_EPI_WARPS / 4;
        if (half > 0) { best_v[(half - 1) * 128 + row_in_tile] = bv; best_i[(half - 1) * 128 + row_in_tile] = bidx; }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * SMP_EPI_WARPS) : "memory");
        if (half == 0 && row_ok && (!MASKED || mask[row] != 0)) {
#pragma unroll
            for (int s = 0; s < NS - 1; ++s) {
                const float ov = best_v[s * 128 + row_in_tile];
                const int oi = best_i[s * 128 + row_in_tile];
                if (ov > bv || (ov == bv && oi < bidx)) { bv = ov; bidx = oi; }
            }
            out[row] = bidx;
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc(tmem_base, 256);
}

// =====================================================================================================================
// Shared-Philox variant.  torch's generator hands element (row, label) the lane (row / rs) % 4 of curand4 call number
// row / (4 rs) of thread (row % rs) * NL + label, rs = stride / NL (37 on a B200 for 8192 labels): the four rows
// r, r+rs, r+2rs, r+3rs of a 4rs-row block share ONE Philox4x32-10 evaluation per label.  To use all four outputs in
// one thread the product is computed TRANSPOSED — D[label, token] = W[labels, K] . F[tokens, K]^T — with the token
// tile ordered (jj, g) -> row 4rs*i + rs*g + jj0 + jj (a 4-D TMA box, g innermost).  A thread then owns one label of
// each 128-label chunk (TMEM lane) and 20 token columns = 5 Philox calls, keeps a running arg-max per column over the
// 64 chunks in registers, and the 128 lanes are reduced once at the end.  ~2.9x fewer instructions per logit.
//
// SPARSE (masked sampling): the unit of work is a slot (blk, jj) = the 4 rows sharing one Philox call per label.  Task t
// takes slots [20t, 20t+20) of the list masked_slot_list_kernel built (a slot is listed when any of its rows is masked)
// and loads each with a {64, 4, 1, 1} box of the same 4-D view into the shared-memory rows 4i..4i+3 -- the rows, and
// the 128B-swizzle phase (address bits 7-9), the dense box would give slot jj0 + i.  MMA, Philox and arg-max are the
// dense ones per column, so a masked row gets exactly the dense draw; only masked rows are written.
constexpr int SH_JJ = 20;                      // jj slots per task
constexpr int SH_N = 4 * SH_JJ;                // token columns per MMA tile (UMMA N = 80)
constexpr int SH_EPI_WARPS = 16;
constexpr int SH_THREADS = 64 + 32 * SH_EPI_WARPS;
constexpr int SH_STAGES = 6;
constexpr int SH_F_BYTES = SH_N * 128;         // one k-block of the token tile
constexpr int SH_W_BYTES = 128 * 128;          // 128 labels x 64 halves
constexpr int SH_SMEM = SMP_MAX_KB * SH_F_BYTES + SH_STAGES * SH_W_BYTES + 1024 + 256 + 4 * SH_N * 8;

__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    ptx::tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, float* v) {
    uint32_t r[4];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
    ptx::tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}

template <bool SPARSE>
__global__ void __launch_bounds__(SH_THREADS, 1)
fused_sampler_shared_kernel(const __grid_constant__ CUtensorMap tm_f, const __grid_constant__ CUtensorMap tm_w, int R, int NL,
                            int Kc, int rs, int tasks_per_block, float inv_t, TorchPhilox rng, const int* __restrict__ slots,
                            const int* __restrict__ n_slots, const uint8_t* __restrict__ mask, int64_t* __restrict__ out) {
    int ns = SH_JJ;                                                    // SPARSE: slots of this task
    if constexpr (SPARSE) {
        ns = min(SH_JJ, *n_slots - (int)blockIdx.x * SH_JJ);
        if (ns <= 0) return;                                           // dense task count launched; the list is shorter
    }
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t f_base = smem_base;
    const uint32_t w_base = smem_base + SMP_MAX_KB * SH_F_BYTES;
    const uint32_t bar_base = w_base + SH_STAGES * SH_W_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (SH_STAGES + s); };
    auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * SH_STAGES + s); };
    auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * SH_STAGES + 2 + s); };
    const uint32_t f_bar = bar_base + 8u * (2 * SH_STAGES + 4);
    const uint32_t tmem_slot = bar_base + 8u * (2 * SH_STAGES + 5);
    uint8_t* tail = smem_gen + (bar_base - smem_base) + 256;
    float* red_v = reinterpret_cast<float*>(tail);                    // [4 quarters][SH_N]
    int* red_i = reinterpret_cast<int*>(tail + 4 * SH_N * 4);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int n_kb = (Kc + 63) / 64;
    const int n_chunks = (NL + 127) / 128;
    const int blk = blockIdx.x / tasks_per_block;                      // 4rs-row block = Philox call index
    const int jj0 = (blockIdx.x - blk * tasks_per_block) * SH_JJ;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_f);
        ptx::prefetch_tensormap(&tm_w);
    }
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < SH_STAGES; ++s) { ptx::mbar_init(full_bar(s), 1); ptx::mbar_init(empty_bar(s), 1); }
            for (int s = 0; s < 2; ++s) { ptx::mbar_init(tfull_bar(s), 1); ptx::mbar_init(tempty_bar(s), SH_EPI_WARPS); }
            ptx::mbar_init(f_bar, 1);
            ptx::fence_barrier_init();
        }
        __syncwarp();
        ptx::tmem_alloc(tmem_slot, 256);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<uint32_t*>(smem_gen + (tmem_slot - smem_base));

    if (warp == 0) {
        if constexpr (SPARSE) {
            // one slot per lane; the coordinates reach the TMA issue through a shuffle, which keeps them warp-uniform
            const int nsw = __shfl_sync(0xffffffffu, ns, 0);
            const int s = lane < nsw ? slots[blockIdx.x * SH_JJ + lane] : 0;
            const int sb = s / rs, sj = s - sb * rs;
            if (ptx::elect_one()) ptx::mbar_arrive_expect_tx(f_bar, n_kb * nsw * 4 * 128);
            __syncwarp();
            for (int kb = 0; kb < n_kb; ++kb)
                for (int i = 0; i < nsw; ++i) {
                    const int bi_ = __shfl_sync(0xffffffffu, sb, i), ji_ = __shfl_sync(0xffffffffu, sj, i);
                    if (ptx::elect_one()) ptx::tma_load_4d(&tm_f, f_bar, f_base + kb * SH_F_BYTES + i * 4 * 128, kb * 64, 0, ji_, bi_);
                    __syncwarp();
                }
        }
        if (ptx::elect_one()) {
            if constexpr (!SPARSE) {
                ptx::mbar_arrive_expect_tx(f_bar, n_kb * SH_F_BYTES);
                for (int kb = 0; kb < n_kb; ++kb) ptx::tma_load_4d(&tm_f, f_bar, f_base + kb * SH_F_BYTES, kb * 64, 0, jj0, blk);
            }
            int stage = 0;
            uint32_t phase = 0;
            for (int ch = 0; ch < n_chunks; ++ch)
                for (int kb = 0; kb < n_kb; ++kb) {
                    ptx::mbar_wait(empty_bar(stage), phase ^ 1);
                    ptx::mbar_arrive_expect_tx(full_bar(stage), SH_W_BYTES);
                    ptx::tma_load_2d(&tm_w, full_bar(stage), w_base + stage * SH_W_BYTES, kb * 64, ch * 128);
                    if (++stage == SH_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = ptx::umma_idesc_f16(128, SH_N, 0);
        ptx::mbar_wait(f_bar, 0);
        int stage = 0;
        uint32_t phase = 0;
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int as = ch & 1;
            ptx::mbar_wait(tempty_bar(as), ((ch >> 1) & 1) ^ 1);
            ptx::tc_fence_after();
            for (int kb = 0; kb < n_kb; ++kb) {
                ptx::mbar_wait(full_bar(stage), phase);
                ptx::tc_fence_after();
                if (ptx::elect_one()) {
                    const uint64_t da = ptx::umma_desc_kmajor_sw128(w_base + stage * SH_W_BYTES);     // labels = M
                    const uint64_t db = ptx::umma_desc_kmajor_sw128(f_base + kb * SH_F_BYTES);        // tokens = N
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        ptx::umma_f16(tmem_base + as * 128, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                    ptx::umma_commit(empty_bar(stage));
                    if (kb == n_kb - 1) ptx::umma_commit(tfull_bar(as));
                }
                __syncwarp();
                if (++stage == SH_STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;                      // TMEM lane quarter -> labels 32q..32q+31 of the chunk
        const int sub = (warp - 2) >> 2;             // token columns [sub*20, sub*20+20): jj = sub*5 .. sub*5+4
        const int l = q * 32 + lane;
        float bv[SH_JJ];
        int bi[SH_JJ];
#pragma unroll
        for (int i = 0; i < SH_JJ; ++i) { bv[i] = -INFINITY; bi[i] = 0x7fffffff; }
        int sp_blk[SH_JJ / 4], sp_jj[SH_JJ / 4];                    // SPARSE: the (blk, jj) of this thread's 5 slots
        if constexpr (SPARSE) {
#pragma unroll
            for (int c4 = 0; c4 < SH_JJ / 4; ++c4) {
                const int i = sub * (SH_JJ / 4) + c4;
                const int s = i < ns ? slots[blockIdx.x * SH_JJ + i] : 0;
                sp_blk[c4] = s / rs;
                sp_jj[c4] = s - sp_blk[c4] * rs;
            }
        }
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int as = ch & 1;
            ptx::mbar_wait(tfull_bar(as), (ch >> 1) & 1);
            ptx::tc_fence_after();
            float v[SH_JJ];
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 128 + sub * SH_JJ);
            tmem_ld_x16(taddr, v);
            tmem_ld_x4(taddr + 16, v + 16);
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(tempty_bar(as));      // accumulator copied to registers: MMA may reuse it
            const int label = ch * 128 + l;
            if (label < NL) {
#pragma unroll
                for (int c4 = 0; c4 < SH_JJ / 4; ++c4) {
                    const int jj = SPARSE ? sp_jj[c4] : jj0 + sub * (SH_JJ / 4) + c4;
                    const int pb = SPARSE ? sp_blk[c4] : blk;
                    const uint4 r4 = torch_philox_call(rng, (uint64_t)jj * (uint64_t)NL + (uint64_t)label, (uint64_t)pb);
                    const uint32_t bits[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const float qv = torch_exponential1(u32_to_uniform(bits[g]));
                        const float gum = fmaf(v[c4 * 4 + g], inv_t, -__logf(qv));
                        if (gum > bv[c4 * 4 + g]) { bv[c4 * 4 + g] = gum; bi[c4 * 4 + g] = label; }
                    }
                }
            }
        }
        // reduce over the 32 labels of this warp, then over the 4 quarters through shared memory
#pragma unroll
        for (int i = 0; i < SH_JJ; ++i) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv[i], o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi[i], o);
                if (ov > bv[i] || (ov == bv[i] && oi < bi[i])) { bv[i] = ov; bi[i] = oi; }
            }
        }
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < SH_JJ; ++i) { red_v[q * SH_N + sub * SH_JJ + i] = bv[i]; red_i[q * SH_N + sub * SH_JJ + i] = bi[i]; }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * SH_EPI_WARPS) : "memory");
        const int t = threadIdx.x - 64;
        if (t < SH_N) {
            float best = red_v[t];
            int besti = red_i[t];
#pragma unroll
            for (int qq = 1; qq < 4; ++qq) {
                const float ov = red_v[qq * SH_N + t];
                const int oi = red_i[qq * SH_N + t];
                if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
            }
            if constexpr (SPARSE) {
                if (t / 4 < ns) {
                    const int s = slots[blockIdx.x * SH_JJ + t / 4];
                    const int sb = s / rs;
                    const int64_t row = (int64_t)sb * 4 * rs + (int64_t)(t & 3) * rs + (s - sb * rs);
                    if (row < R && mask[row] != 0) out[row] = besti;
                }
            } else {
                const int jj = jj0 + t / 4, g = t & 3;
                const int64_t row = (int64_t)blk * 4 * rs + (int64_t)g * rs + jj;
                if (jj < rs && row < R) out[row] = besti;
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) ptx::tmem_dealloc(tmem_base, 256);
}

// Masked sampling: lists the slots (blk, jj) with at least one masked row, in slot order within a CTA (the order across
// CTAs follows the atomics and does not affect the draws).  *count must be zero on entry.
__global__ void __launch_bounds__(256) masked_slot_list_kernel(const uint8_t* __restrict__ mask, int64_t R, int rs, int n_slots,
                                                                int* __restrict__ slots, int* __restrict__ count) {
    __shared__ int warp_n[8];
    __shared__ int base;
    const int s = blockIdx.x * 256 + threadIdx.x;
    bool need = false;
    if (s < n_slots) {
        const int blk = s / rs, jj = s - blk * rs;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int64_t row = (int64_t)blk * 4 * rs + (int64_t)g * rs + jj;
            need |= row < R && mask[row] != 0;
        }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bal = __ballot_sync(0xffffffffu, need);
    if (lane == 0) warp_n[warp] = __popc(bal);
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int w = 0; w < 8; ++w) { const int n = warp_n[w]; warp_n[w] = tot; tot += n; }
        base = tot ? atomicAdd(count, tot) : 0;
    }
    __syncthreads();
    if (need) slots[base + warp_n[warp] + __popc(bal & ((1u << lane) - 1u))] = s;
}

int64_t fused_sampler_rows_padded(int64_t R, int NL) {
    TorchPhilox rng = make_torch_philox(0, 0, R * (int64_t)NL);
    if (NL <= 0 || rng.stride % (uint32_t)NL != 0) return R;
    const int64_t rs = rng.stride / NL;
    return (R + 4 * rs - 1) / (4 * rs) * (4 * rs);
}

int64_t fused_sampler_mask_scratch_bytes(int64_t R, int NL) {
    // the slot count (256 bytes) + one int per slot: a slot covers 4 rows of the padded feature buffer
    return 256 + (fused_sampler_rows_padded(R, NL) + 255) / 256 * 256;
}

static int launch_fused_sampler_impl(const __half* a16, int64_t R, int Kc, const __half* w16, int NL, float inv_t,
                                     uint64_t seed, uint64_t offset, const uint8_t* mask, void* mask_scratch, int64_t* out,
                                     cudaStream_t st) {
    PB_CHECK(Kc % 8 == 0 && Kc <= 64 * SMP_MAX_KB, "fused sampler: c_out=%d unsupported (<= %d, multiple of 8)", Kc, 64 * SMP_MAX_KB);
    PB_CHECK(R * (int64_t)NL < (1ll << 31), "fused sampler: rows*labels >= 2^31 would split the torch kernel (unsupported)");
    PB_CHECK(offset % 4 == 0, "philox offset must be a multiple of 4");
    if (R == 0) return 0;
    {
        // shared-Philox path: needs stride % NL == 0 (rows of a lane group are whole rows).  The feature buffer must hold
        // fused_sampler_rows_padded(R, NL) rows (the caller's workspace does); rows >= R are never written to `out`.
        TorchPhilox rng = make_torch_philox(seed, offset, R * (int64_t)NL);
        static const bool no_shared = getenv("PB200_SAMPLER_GENERIC") != nullptr;
        if (!no_shared && rng.stride % (uint32_t)NL == 0 && (int64_t)rng.stride / NL < (1 << 24)) {
            const int rs = (int)(rng.stride / NL);
            const int n_blocks = (int)((R + 4 * (int64_t)rs - 1) / (4 * (int64_t)rs));
            const int tpb = (rs + SH_JJ - 1) / SH_JJ;
            int* count = nullptr;
            int* slots = nullptr;
            if (mask) {
                count = reinterpret_cast<int*>(mask_scratch);
                slots = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(mask_scratch) + 256);
                const int n_slots = n_blocks * rs;
                PB_CUDA(cudaMemsetAsync(count, 0, sizeof(int), st));
                masked_slot_list_kernel<<<ceil_div(n_slots, 256), 256, 0, st>>>(mask, R, rs, n_slots, slots, count);
                PB_LAUNCH_CHECK();
            }
            static DeviceOnce attr2;
            if (attr2.first()) {
                PB_CUDA(cudaFuncSetAttribute(fused_sampler_shared_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SH_SMEM));
                PB_CUDA(cudaFuncSetAttribute(fused_sampler_shared_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SH_SMEM));
    }
            ProfScope prof("fused_sampler", 2.0 * (double)R * (double)NL * (double)Kc, st);
            CUtensorMap tf, tw;
            const int64_t dims[4] = {Kc, 4, rs, n_blocks};
            const int64_t strides[3] = {(int64_t)rs * Kc * 2, (int64_t)Kc * 2, 4 * (int64_t)rs * Kc * 2};
            const int box[4] = {64, 4, mask ? 1 : SH_JJ, 1};
            PB_TRY(make_tmap_f16_nd(&tf, a16, 4, dims, strides, box));
            PB_TRY(make_tmap_f16_2d(&tw, w16, NL, Kc, Kc, 128));
            if (mask)
                fused_sampler_shared_kernel<true><<<n_blocks * tpb, SH_THREADS, SH_SMEM, st>>>(tf, tw, (int)R, NL, Kc, rs, tpb, inv_t, rng,
                                                                                             slots, count, mask, out);
            else
                fused_sampler_shared_kernel<false><<<n_blocks * tpb, SH_THREADS, SH_SMEM, st>>>(tf, tw, (int)R, NL, Kc, rs, tpb, inv_t, rng,
                                                                                              nullptr, nullptr, nullptr, out);
            PB_LAUNCH_CHECK();
            return 0;
        }
    }
    static DeviceOnce attr_set;
    if (attr_set.first()) {
        PB_CUDA(cudaFuncSetAttribute(fused_sampler_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMP_SMEM));
        PB_CUDA(cudaFuncSetAttribute(fused_sampler_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMP_SMEM));
    }
    ProfScope prof("fused_sampler", 2.0 * (double)R * (double)NL * (double)Kc, st);
    CUtensorMap ta, tw;
    PB_TRY(make_tmap_f16_2d(&ta, a16, R, Kc, Kc, 128));
    PB_TRY(make_tmap_f16_2d(&tw, w16, NL, Kc, Kc, SMP_BN));
    TorchPhilox rng = make_torch_philox(seed, offset, R * (int64_t)NL);
    if (mask)
        fused_sampler_kernel<true><<<ceil_div(R, 128), SMP_THREADS, SMP_SMEM, st>>>(ta, tw, (int)R, NL, Kc, inv_t, rng, mask, out);
    else
        fused_sampler_kernel<false><<<ceil_div(R, 128), SMP_THREADS, SMP_SMEM, st>>>(ta, tw, (int)R, NL, Kc, inv_t, rng, nullptr, out);
    PB_LAUNCH_CHECK();
    return 0;
}

int launch_fused_sampler(const __half* a16, int64_t R, int Kc, const __half* w16, int NL, float inv_t, uint64_t seed,
                         uint64_t offset, int64_t* out, cudaStream_t st) {
    return launch_fused_sampler_impl(a16, R, Kc, w16, NL, inv_t, seed, offset, nullptr, nullptr, out, st);
}

int launch_fused_sampler_masked(const __half* a16, int64_t R, int Kc, const __half* w16, int NL, float inv_t, uint64_t seed,
                                uint64_t offset, const uint8_t* mask, void* mask_scratch, int64_t* tokens_inout, cudaStream_t st) {
    PB_CHECK(mask != nullptr && mask_scratch != nullptr, "masked sampler: mask and scratch are required");
    return launch_fused_sampler_impl(a16, R, Kc, w16, NL, inv_t, seed, offset, mask, mask_scratch, tokens_inout, st);
}

}  // namespace pb
