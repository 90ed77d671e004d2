// Host-side executor of the Paella denoiser: layer plan, weight packing, conditioning cache, forward.
//   plan / parameter names   ref/src/modules.py:110-187 (ModuleList construction order == state-dict keys)
//   gen_c_embeddings         ref/src/modules.py:223-232, ref/utils/modules.py:228-235 (list clip_image)
//   forward                  ref/src/modules.py:263-275 (_down_encode :234-247, _up_decode :249-261)
// The x- and t-independent half of every AttnBlock (kv_mapper + K/V projection of the conditioning rows,
// ref/src/modules.py:77 + nn.MultiheadAttention in_proj rows [E:3E]) is hoisted into pb200_paella_prepare_cond.
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

#include "attention.cuh"
#include "gemm.cuh"
#include "ops.cuh"
#include "sampler.cuh"

namespace pb {

// ------------------------------------------------------------------ weight packing
enum PackKind { PK_COPY_F32, PK_CAST_F16, PK_DW, PK_CONV2, PK_CONVT2, PK_CLF_W, PK_CLF_B, PK_BIAS_REP4 };

__global__ void pack_kernel(const float* __restrict__ src, void* __restrict__ dst, int kind, int64_t n, int d0, int d1,
                            int d2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float* d32 = reinterpret_cast<float*>(dst);
    __half* d16 = reinterpret_cast<__half*>(dst);
    switch (kind) {
        case PK_COPY_F32: d32[i] = src[i]; break;
        case PK_CAST_F16: d16[i] = __float2half_rn(src[i]); break;
        case PK_DW: {       // src [c=d0, per=d1, k=d2, k] -> dst [k*k][per][c]
            const int c = d0, per = d1, k = d2;
            const int ch = (int)(i % c);
            const int j = (int)((i / c) % per);
            const int tap = (int)(i / ((int64_t)c * per));
            d32[i] = src[((int64_t)(ch * per + j) * k + tap / k) * k + tap % k];
            break;
        }
        case PK_CONV2: {    // src [Cout=d0, Cin=d1, 2, 2] -> dst fp16 [Cout][(dy,dx,Cin)]
            const int cin = d1;
            const int ci = (int)(i % cin);
            const int q = (int)((i / cin) % 4);
            const int co = (int)(i / (4 * (int64_t)cin));
            d16[i] = __float2half_rn(src[((int64_t)(co * cin + ci) * 2 + (q >> 1)) * 2 + (q & 1)]);
            break;
        }
        case PK_CONVT2: {   // src [Cin=d0, Cout=d1, 2, 2] -> dst fp16 [(dy,dx,Cout)][Cin]
            const int cin = d0, cout = d1;
            const int ci = (int)(i % cin);
            const int co = (int)((i / cin) % cout);
            const int q = (int)(i / ((int64_t)cin * cout));
            d16[i] = __float2half_rn(src[((int64_t)(ci * cout + co) * 2 + (q >> 1)) * 2 + (q & 1)]);
            break;
        }
        case PK_CLF_W: {    // src [c_out*4 (c*4+q), K=d1] -> dst fp16 [(q, c)][K]   (PixelShuffle(2) channel order)
            const int cout = d0, K = d1;
            const int k = (int)(i % K);
            const int c = (int)((i / K) % cout);
            const int q = (int)(i / ((int64_t)K * cout));
            d16[i] = __float2half_rn(src[(int64_t)(c * 4 + q) * K + k]);
            break;
        }
        case PK_CLF_B: {    // src [c_out*4] -> dst fp32 [(q, c)]
            const int cout = d0;
            d32[i] = src[(i % cout) * 4 + i / cout];
            break;
        }
        case PK_BIAS_REP4: d32[i] = src[i % d0]; break;
    }
}

// out[r] = sum_k fp32(w[r, k]) of a packed fp16 matrix (warp per row): the rowsum(W) of the folded LayerNorm
__global__ void __launch_bounds__(256) rowsum_f16_kernel(const __half* __restrict__ w, int rows, int cols, float* __restrict__ out) {
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= rows) return;
    float s = 0.f;
    for (int k = lane; k < cols; k += 32) s += __half2float(w[(int64_t)r * cols + k]);
    s = warp_sum(s);
    if (lane == 0) out[r] = s;
}

// out[n] = b2[n] + sum_k fp32(w2[n, k]) * beta[k]: the GlobalResponseNorm shift pushed through the Linear that follows it
// (GRN(h) W2^T + b2 = (h * s) W2^T + (W2 beta + b2)); warp per output row
__global__ void __launch_bounds__(256) fold_bias_kernel(const __half* __restrict__ w2, const float* __restrict__ beta,
                                                        const float* __restrict__ b2, int rows, int cols, float* __restrict__ out) {
    const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (r >= rows) return;
    float s = 0.f;
    for (int k = lane; k < cols; k += 32) s = fmaf(__half2float(w2[(int64_t)r * cols + k]), beta[k], s);
    s = warp_sum(s);
    if (lane == 0) out[r] = s + b2[r];
}

struct ParamSpec {
    std::string name;
    int64_t numel;      // reference tensor numel
    int kind;
    int64_t dst_off;    // bytes into the blob
    int64_t dst_numel;
    int d0, d1, d2;
    int64_t rowsum_off = -1;     // fp32 [rowsum_rows]: row sums of the packed fp16 matrix [rowsum_rows, rowsum_cols]
    int rowsum_rows = 0, rowsum_cols = 0;
    int fold_group = -1;         // index into pb200_paella::folds (channelwise.2.beta / .4.weight / .4.bias of one MLP)
};

// derived parameter of one ResBlock / FeedForwardBlock MLP: b2_fold = channelwise.4.bias + channelwise.4.weight . channelwise.2.beta
struct FoldGroup {
    int64_t w2, beta, b2, out;
    int c;
    int loaded = 0;              // parameters of the group seen by load_param since the blob was bound
};

enum BlockKind { BK_RES, BK_TIME, BK_ATTN, BK_FF, BK_DOWN, BK_UP, BK_SAVE };

struct BlockPlan {
    int kind, level, c, c_skip;
    int64_t dw_w = -1, dw_b = -1, w1 = -1, b1 = -1, gamma = -1, beta = -1, w2 = -1, b2 = -1;
    int64_t b2_fold = -1;           // fp32 [c]: b2 + W2 beta (GRN shift folded through the second Linear)
    int64_t film_off = -1;          // RES/FF: fused FiLM of the following TimestepBlock; TIME: own offset
    bool film_fused = false;        // TIME: already applied by the previous block's epilogue
    int64_t kvm_w = -1, kvm_b = -1, inproj_w = -1, inproj_b = -1, outproj_w = -1, outproj_b = -1;
    int64_t inproj_wsum = -1;       // ATTN: row sums of in_proj_weight (LayerNorm folded into the QKV GEMM)
    int attn_index = -1;
    int ln_fold_attn = -1;          // RES/FF: index of the AttnBlock that directly consumes this block's output, or -1
    int ln_shift_attn = -1;         // RES/FF (folded) and ATTN: index of the previous AttnBlock on the same residual stream,
                                    // whose input row means are the per-row shift of the folded LayerNorm; -1 = none
    int64_t rs_w = -1, rs_b = -1;
};

}  // namespace pb

using namespace pb;

struct pb200_paella {
    pb200_paella_config cfg;
    std::vector<ParamSpec> params;
    std::unordered_map<std::string, int> by_name;
    std::vector<BlockPlan> blocks;
    std::vector<FoldGroup> folds;
    int64_t weight_bytes = 0;
    uint8_t* blob = nullptr;
    int64_t emb_table = -1, emb_w = -1, emb_b = -1, byt5_w = -1, byt5_b = -1, clip_w = -1, clip_b = -1, clipimg_w = -1,
            clipimg_b = -1, clf_w = -1, clf_b = -1, out_w = -1, film_w = -1, film_b = -1;
    int film_total = 0, n_attn = 0, max_c = 0;
    std::map<std::tuple<const void*, int64_t, int64_t, int64_t, int>, CUtensorMap> tmaps;

    int64_t add_param(const std::string& name, int64_t numel, int kind, int64_t dst_numel, int elem_bytes, int d0 = 0,
                      int d1 = 0, int d2 = 0, int64_t forced_off = -1) {
        ParamSpec p;
        p.name = name; p.numel = numel; p.kind = kind; p.dst_numel = dst_numel; p.d0 = d0; p.d1 = d1; p.d2 = d2;
        if (forced_off >= 0) {
            p.dst_off = forced_off;
        } else {
            p.dst_off = weight_bytes;
            weight_bytes += (dst_numel * elem_bytes + 255) / 256 * 256;
        }
        by_name[name] = (int)params.size();
        params.push_back(p);
        return p.dst_off;
    }
    int64_t f32(const std::string& n, int64_t numel) { return add_param(n, numel, PK_COPY_F32, numel, 4); }
    int64_t f16(const std::string& n, int64_t numel) { return add_param(n, numel, PK_CAST_F16, numel, 2); }

    template <typename T>
    T* w(int64_t off) const { return reinterpret_cast<T*>(blob + off); }

    int tmap(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, const CUtensorMap** out) {
        auto key = std::make_tuple(ptr, rows, cols, ld, box_rows);
        auto it = tmaps.find(key);
        if (it == tmaps.end()) {
            CUtensorMap tm;
            PB_TRY(make_tmap_f16_2d(&tm, ptr, rows, cols, ld, box_rows));
            it = tmaps.emplace(key, tm).first;
        }
        *out = &it->second;
        return 0;
    }

    // C = A[M,K] . W[N,K]^T with W at blob offset w_off
    int gemm(const __half* A, int64_t lda, int64_t M, int64_t K, int64_t w_off, int64_t N, const pb200_gemm_epilogue& ep,
             cudaStream_t st) {
        const int bn = gemm_pick_block_n(M, N, K);
        const CUtensorMap *ta, *tb;
        PB_TRY(tmap(A, M, K, lda, GEMM_BLOCK_M, &ta));
        PB_TRY(tmap(w<__half>(w_off), N, K, K, bn / 2, &tb));     // W box = half a tile
        GemmTail tail{gemm_tail_block_n(M, N, bn), nullptr};
        if (tail.bn) PB_TRY(tmap(w<__half>(w_off), N, K, K, tail.bn / 2, &tail.tb));
        return gemm_launch(*ta, *tb, bn, ep, M, N, K, st, tail.bn ? &tail : nullptr);
    }
};

namespace pb {

static pb200_gemm_epilogue epi(int mode, const float* bias, void* out, int64_t ldo) {
    pb200_gemm_epilogue e;
    memset(&e, 0, sizeof(e));
    e.mode = mode; e.bias = bias; e.out = out; e.ldo = ldo; e.alpha = 1.0f;
    return e;
}

// ------------------------------------------------------------------ plan construction
static int build_plan(pb200_paella* m) {
    const pb200_paella_config& c = m->cfg;
    PB_CHECK(c.n_levels >= 1 && c.n_levels <= PB200_MAX_LEVELS, "n_levels %d out of range", c.n_levels);
    PB_CHECK(c.patch_size == 2, "patch_size %d unsupported (2 only)", c.patch_size);
    PB_CHECK(c.c_in % 8 == 0 && c.c_out % 8 == 0 && c.c_cond % 8 == 0 && c.byt5_embd % 8 == 0 && c.clip_embd % 8 == 0 &&
                 c.num_labels % 8 == 0, "channel counts must be multiples of 8");
    PB_CHECK(c.c_r % 4 == 0 && c.c_r >= 4, "c_r=%d must be a multiple of 4", c.c_r);
    for (int i = 0; i < c.n_levels; ++i) {
        PB_CHECK(c.c_hidden[i] % 8 == 0, "c_hidden[%d]=%d must be a multiple of 8", i, c.c_hidden[i]);
        m->max_c = c.c_hidden[i] > m->max_c ? c.c_hidden[i] : m->max_c;
    }
    const int ps2 = c.patch_size * c.patch_size;
    m->byt5_w = m->f16("byt5_mapper.weight", (int64_t)c.c_cond * c.byt5_embd);
    m->byt5_b = m->f32("byt5_mapper.bias", c.c_cond);
    m->clip_w = m->f16("clip_mapper.weight", (int64_t)c.c_cond * c.clip_seq_len * c.clip_embd);
    m->clip_b = m->f32("clip_mapper.bias", (int64_t)c.c_cond * c.clip_seq_len);
    m->clipimg_w = m->f16("clip_image_mapper.weight", (int64_t)c.c_cond * c.clip_seq_len * c.clip_embd);
    m->clipimg_b = m->f32("clip_image_mapper.bias", (int64_t)c.c_cond * c.clip_seq_len);
    m->emb_table = m->f32("in_mapper.0.weight", (int64_t)c.num_labels * c.c_in);
    m->emb_w = m->f16("embedding.1.weight", (int64_t)c.c_hidden[0] * c.c_in * ps2);
    m->emb_b = m->f32("embedding.1.bias", c.c_hidden[0]);
    m->clf_w = m->add_param("clf.1.weight", (int64_t)c.c_out * ps2 * c.c_hidden[0], PK_CLF_W,
                            (int64_t)c.c_out * ps2 * c.c_hidden[0], 2, c.c_out, c.c_hidden[0]);
    m->clf_b = m->add_param("clf.1.bias", (int64_t)c.c_out * ps2, PK_CLF_B, (int64_t)c.c_out * ps2, 4, c.c_out);
    m->out_w = m->f16("out_mapper.1.weight", (int64_t)c.num_labels * c.c_out);

    // first pass: count FiLM rows so the concatenated mapper matrix can be laid out
    int film_rows = 0;
    for (int pass = 0; pass < 2; ++pass)
        for (int i = 0; i < c.n_levels; ++i)
            for (const char* t = c.level_config[i]; *t; ++t)
                if (*t == 'T') film_rows += 2 * c.c_hidden[i] * c.blocks[i];
    m->film_total = film_rows;
    m->film_w = m->weight_bytes;
    m->weight_bytes += ((int64_t)film_rows * c.c_r * 4 + 255) / 256 * 256;
    m->film_b = m->weight_bytes;
    m->weight_bytes += ((int64_t)film_rows * 4 + 255) / 256 * 256;

    int film_cursor = 0;
    auto add_block = [&](const std::string& pre, char bt, int lvl, int c_skip) -> int {
        const int ch = c.c_hidden[lvl];
        BlockPlan b;
        b.level = lvl; b.c = ch; b.c_skip = c_skip;
        auto mlp = [&]() {
            b.w1 = m->f16(pre + "channelwise.0.weight", (int64_t)4 * ch * ch);
            b.b1 = m->f32(pre + "channelwise.0.bias", 4 * ch);
            b.gamma = m->f32(pre + "channelwise.2.gamma", 4 * ch);
            b.beta = m->f32(pre + "channelwise.2.beta", 4 * ch);
            b.w2 = m->f16(pre + "channelwise.4.weight", (int64_t)4 * ch * ch);
            b.b2 = m->f32(pre + "channelwise.4.bias", ch);
            b.b2_fold = m->weight_bytes;
            m->weight_bytes += ((int64_t)ch * 4 + 255) / 256 * 256;
            FoldGroup fg;
            fg.w2 = b.w2; fg.beta = b.beta; fg.b2 = b.b2; fg.out = b.b2_fold; fg.c = ch;
            for (const char* suffix : {"channelwise.2.beta", "channelwise.4.weight", "channelwise.4.bias"})
                m->params[m->by_name[pre + suffix]].fold_group = (int)m->folds.size();
            m->folds.push_back(fg);
        };
        if (bt == 'C') {
            b.kind = BK_RES;
            const int per = c_skip ? 2 : 1;
            PB_CHECK(c_skip == 0 || c_skip == ch, "skip width %d != %d unsupported", c_skip, ch);
            const int64_t n = (int64_t)ch * per * c.kernel_size * c.kernel_size;
            b.dw_w = m->add_param(pre + "depthwise.weight", n, PK_DW, n, 4, ch, per, c.kernel_size);
            b.dw_b = m->f32(pre + "depthwise.bias", ch);
            mlp();
        } else if (bt == 'F') {
            b.kind = BK_FF;
            mlp();
        } else if (bt == 'T') {
            b.kind = BK_TIME;
            b.film_off = film_cursor;
            m->add_param(pre + "mapper.weight", (int64_t)2 * ch * c.c_r, PK_COPY_F32, (int64_t)2 * ch * c.c_r, 4, 0, 0, 0,
                         m->film_w + (int64_t)film_cursor * c.c_r * 4);
            m->add_param(pre + "mapper.bias", 2 * ch, PK_COPY_F32, 2 * ch, 4, 0, 0, 0, m->film_b + (int64_t)film_cursor * 4);
            film_cursor += 2 * ch;
        } else if (bt == 'A') {
            b.kind = BK_ATTN;
            PB_CHECK(c.nhead[lvl] > 0 && ch % c.nhead[lvl] == 0, "level %d: nhead %d does not divide %d", lvl, c.nhead[lvl], ch);
            b.inproj_w = m->f16(pre + "attention.attn.in_proj_weight", (int64_t)3 * ch * ch);
            {   // derived: fp32 row sums of the fp16 matrix, filled when the parameter is loaded
                ParamSpec& ps = m->params.back();
                ps.rowsum_off = m->weight_bytes;
                ps.rowsum_rows = 3 * ch; ps.rowsum_cols = ch;
                m->weight_bytes += ((int64_t)3 * ch * 4 + 255) / 256 * 256;
                b.inproj_wsum = ps.rowsum_off;
            }
            b.inproj_b = m->f32(pre + "attention.attn.in_proj_bias", 3 * ch);
            b.outproj_w = m->f16(pre + "attention.attn.out_proj.weight", (int64_t)ch * ch);
            b.outproj_b = m->f32(pre + "attention.attn.out_proj.bias", ch);
            b.kvm_w = m->f16(pre + "kv_mapper.1.weight", (int64_t)ch * c.c_cond);
            b.kvm_b = m->f32(pre + "kv_mapper.1.bias", ch);
            b.attn_index = m->n_attn++;
        } else {
            PB_CHECK(false, "block type '%c' not supported", bt);
        }
        m->blocks.push_back(b);
        return 0;
    };

    const int L = c.n_levels;
    for (int i = 0; i < L; ++i) {
        int j = 0;
        if (i > 0) {
            const std::string pre = "down_blocks." + std::to_string(i) + "." + std::to_string(j) + ".";
            BlockPlan b;
            b.kind = BK_DOWN; b.level = i; b.c = c.c_hidden[i]; b.c_skip = 0;
            const int cin = c.c_hidden[i - 1], cout = c.c_hidden[i];
            b.rs_w = m->add_param(pre + "1.weight", (int64_t)cout * cin * 4, PK_CONV2, (int64_t)cout * cin * 4, 2, cout, cin);
            b.rs_b = m->f32(pre + "1.bias", cout);
            m->blocks.push_back(b);
            ++j;
        }
        for (int r = 0; r < c.blocks[i]; ++r)
            for (const char* t = c.level_config[i]; *t; ++t) {
                PB_TRY(add_block("down_blocks." + std::to_string(i) + "." + std::to_string(j) + ".", *t, i, 0));
                ++j;
            }
        BlockPlan s;
        s.kind = BK_SAVE; s.level = i; s.c = c.c_hidden[i]; s.c_skip = 0;
        m->blocks.push_back(s);
    }
    for (int ui = 0; ui < L; ++ui) {
        const int i = L - 1 - ui;
        int j = 0;
        for (int r = 0; r < c.blocks[i]; ++r) {
            int k = 0;
            for (const char* t = c.level_config[i]; *t; ++t, ++k) {
                const int skip = (i < L - 1 && r == 0 && k == 0) ? c.c_hidden[i] : 0;
                PB_TRY(add_block("up_blocks." + std::to_string(ui) + "." + std::to_string(j) + ".", *t, i, skip));
                ++j;
            }
        }
        if (i > 0) {
            const std::string pre = "up_blocks." + std::to_string(ui) + "." + std::to_string(j) + ".";
            BlockPlan b;
            b.kind = BK_UP; b.level = i; b.c = c.c_hidden[i]; b.c_skip = 0;
            const int cin = c.c_hidden[i], cout = c.c_hidden[i - 1];
            b.rs_w = m->add_param(pre + "1.weight", (int64_t)cin * cout * 4, PK_CONVT2, (int64_t)cin * cout * 4, 2, cin, cout);
            b.rs_b = m->add_param(pre + "1.bias", cout, PK_BIAS_REP4, (int64_t)4 * cout, 4, cout);
            m->blocks.push_back(b);
        }
    }
    PB_CHECK(film_cursor == film_rows / 2 || film_cursor == film_rows, "internal: FiLM row count mismatch");
    m->film_total = film_cursor;
    // (below, after the FiLM fusion:) a ResBlock/FeedForwardBlock whose output -- after its fused TimestepBlock, if any --
    // goes straight into an AttnBlock also produces that block's LayerNorm inputs (fp16 rows + row statistics)
    // fuse each TimestepBlock that directly follows a ResBlock/FeedForwardBlock into that block's GEMM epilogue
    for (size_t i = 0; i + 1 < m->blocks.size(); ++i) {
        BlockPlan& a = m->blocks[i];
        BlockPlan& t = m->blocks[i + 1];
        if ((a.kind == BK_RES || a.kind == BK_FF) && t.kind == BK_TIME && t.level == a.level) {
            a.film_off = t.film_off;
            t.film_fused = true;
        }
    }
    // Each AttnBlock's predecessor on the same residual stream (same level, no resampler in between; the deepest level's
    // SAVE is a no-op on the tensor): the row means that block saw are the shift of this block's folded LayerNorm.
    {
        int prev = -1, prev_level = -1;
        for (BlockPlan& b : m->blocks) {
            if (b.kind == BK_DOWN || b.kind == BK_UP || (b.kind == BK_SAVE && b.level != L - 1)) prev = -1;
            if (b.kind == BK_ATTN) {
                b.ln_shift_attn = (prev >= 0 && prev_level == b.level) ? prev : -1;
                prev = b.attn_index;
                prev_level = b.level;
            }
        }
    }
    // The LayerNorm fold rounds the producer's rows to fp16 before the mean is removed; it is only used where a shift close
    // to the row mean is available (every AttnBlock but the first of a stream segment), which keeps that rounding relative
    // to the row's spread (tests/test_oracle_lnfold.py; DESIGN.md "Numerics").
    static const bool no_fold = getenv("PB200_NO_LN_FOLD") != nullptr;      // A/B knob
    for (size_t i = 0; !no_fold && i + 1 < m->blocks.size(); ++i) {
        BlockPlan& a = m->blocks[i];
        if (a.kind != BK_RES && a.kind != BK_FF) continue;
        size_t j = i + 1;
        if (m->blocks[j].kind == BK_TIME && m->blocks[j].film_fused) ++j;
        if (j < m->blocks.size() && m->blocks[j].kind == BK_ATTN && m->blocks[j].level == a.level &&
            m->blocks[j].ln_shift_attn >= 0) {
            a.ln_fold_attn = m->blocks[j].attn_index;
            a.ln_shift_attn = m->blocks[j].ln_shift_attn;
        }
    }
    return 0;
}

// ------------------------------------------------------------------ scratch planning
struct Arena {
    uint8_t* base;
    int64_t off = 0;
    template <typename T>
    T* take(int64_t n) {
        const int64_t o = off;
        off += (n * (int64_t)sizeof(T) + 255) / 256 * 256;
        return reinterpret_cast<T*>(base ? base + o : nullptr);
    }
};

struct FeatWs {
    float* xd[PB200_MAX_LEVELS];
    float* xu[PB200_MAX_LEVELS];
    __half *a16, *h16, *qkv16, *o16;
    uint64_t *gsq, *gscale;      // GRN statistic ping/pong (2^-24 fixed point)
    float* grn_mult;             // GRN per-(sample, channel) multipliers [Bt, 4*max_c]
    int64_t* lnstat;             // folded LayerNorm: per AttnBlock [M][2] fixed-point row statistics
    int64_t lnstat_stride;       // int64 elements per AttnBlock
    float* lnmean;               // per AttnBlock [M]: mean of its input rows (the next folded LayerNorm's per-row shift)
    int64_t lnmean_stride;
    float *r_emb, *film, *y;
};

static void plan_features(const pb200_paella* m, int Bt, int H, int W, Arena& ar, FeatWs& ws) {
    const pb200_paella_config& c = m->cfg;
    const int ps = c.patch_size;
    int64_t max_mc = 0, P = (int64_t)(H / ps) * (W / ps);
    for (int l = 0; l < c.n_levels; ++l) {
        const int64_t M = (int64_t)Bt * (P >> (2 * l));
        ws.xd[l] = ar.take<float>(M * c.c_hidden[l]);
        ws.xu[l] = (l < c.n_levels - 1) ? ar.take<float>(M * c.c_hidden[l]) : nullptr;
        max_mc = M * c.c_hidden[l] > max_mc ? M * c.c_hidden[l] : max_mc;
    }
    const int64_t m0_emb = (int64_t)Bt * P * c.c_in * ps * ps;
    ws.a16 = ar.take<__half>(max_mc);
    ws.h16 = ar.take<__half>(4 * max_mc > m0_emb ? 4 * max_mc : m0_emb);
    ws.qkv16 = ar.take<__half>(3 * max_mc);
    ws.o16 = ar.take<__half>(max_mc);
    ws.gsq = ar.take<uint64_t>((int64_t)Bt * 4 * m->max_c);     // ping
    ws.gscale = ar.take<uint64_t>((int64_t)Bt * 4 * m->max_c);  // pong (second GRN statistic buffer)
    ws.grn_mult = ar.take<float>((int64_t)Bt * 4 * m->max_c);
    {
        int64_t max_m = 0;
        for (const BlockPlan& b : m->blocks)
            if (b.kind == BK_ATTN) { const int64_t M = (int64_t)Bt * (P >> (2 * b.level)); max_m = M > max_m ? M : max_m; }
        ws.lnstat_stride = 2 * max_m;
        ws.lnstat = ar.take<int64_t>(ws.lnstat_stride * (m->n_attn > 0 ? m->n_attn : 1));
        ws.lnmean_stride = max_m;
        ws.lnmean = ar.take<float>(ws.lnmean_stride * (m->n_attn > 0 ? m->n_attn : 1));
    }
    ws.r_emb = ar.take<float>((int64_t)Bt * c.c_r);
    ws.film = ar.take<float>((int64_t)Bt * (m->film_total > 0 ? m->film_total : 4));
    ws.y = ar.take<float>((int64_t)Bt * H * W * c.c_out);
}

struct CondWs {
    __half *byt5_16, *clip_16, *silu16, *kvm16;
    float* seq;
};

static void plan_cond(const pb200_paella* m, int B, int L, int S, Arena& ar, CondWs& ws) {
    const pb200_paella_config& c = m->cfg;
    ws.byt5_16 = ar.take<__half>((int64_t)B * L * c.byt5_embd);
    ws.clip_16 = ar.take<__half>((int64_t)B * c.clip_embd);
    ws.seq = ar.take<float>((int64_t)B * S * c.c_cond);
    ws.silu16 = ar.take<__half>((int64_t)B * S * c.c_cond);
    ws.kvm16 = ar.take<__half>((int64_t)B * S * m->max_c);
}

// cond cache: per attention block [Bt, s_max, 2c] fp16, then kv_len int32 [Bt]
static int64_t cond_block_off(const pb200_paella* m, int attn_index, int Bt, int s_max) {
    int64_t off = 0;
    for (const BlockPlan& b : m->blocks)
        if (b.kind == BK_ATTN) {
            if (b.attn_index == attn_index) return off;
            off += ((int64_t)Bt * s_max * 2 * b.c * 2 + 255) / 256 * 256;
        }
    return off;     // attn_index == n_attn: end of the K/V area (kv_len lives here)
}

__global__ void fill_int_kernel(int* p, int n, int v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace pb

// ====================================================================== C ABI
extern "C" {

int pb200_paella_create(const pb200_paella_config* cfg, pb200_paella** out) {
    PB_CHECK(cfg && out, "paella_create: null argument");
    pb200_paella* m = new pb200_paella();
    m->cfg = *cfg;
    for (int i = 0; i < PB200_MAX_LEVELS; ++i) m->cfg.level_config[i][7] = 0;
    if (build_plan(m)) {
        delete m;
        return 1;
    }
    *out = m;
    return 0;
}

void pb200_paella_destroy(pb200_paella* m) { delete m; }
int64_t pb200_paella_weight_bytes(const pb200_paella* m) { return m->weight_bytes; }

int pb200_paella_bind_weights(pb200_paella* m, void* blob) {
    PB_CHECK(((uintptr_t)blob & 255) == 0, "weight blob must be 256-byte aligned");
    m->blob = reinterpret_cast<uint8_t*>(blob);
    m->tmaps.clear();
    for (FoldGroup& g : m->folds) g.loaded = 0;
    return 0;
}

int pb200_paella_num_params(const pb200_paella* m) { return (int)m->params.size(); }
const char* pb200_paella_param_name(const pb200_paella* m, int i) {
    return (i >= 0 && i < (int)m->params.size()) ? m->params[i].name.c_str() : "";
}
int64_t pb200_paella_param_numel(const pb200_paella* m, int i) {
    return (i >= 0 && i < (int)m->params.size()) ? m->params[i].numel : -1;
}

int pb200_paella_load_param(pb200_paella* m, const char* name, const float* src, int64_t numel, void* stream) {
    PB_CHECK(m->blob != nullptr, "load_param: bind a weight blob first");
    auto it = m->by_name.find(name);
    PB_CHECK(it != m->by_name.end(), "load_param: '%s' is not a parameter of this plan", name);
    const ParamSpec& p = m->params[it->second];
    PB_CHECK(numel == p.numel, "load_param: '%s' has %lld elements, expected %lld", name, (long long)numel, (long long)p.numel);
    pack_kernel<<<ceil_div(p.dst_numel, 256), 256, 0, (cudaStream_t)stream>>>(src, m->blob + p.dst_off, p.kind, p.dst_numel,
                                                                             p.d0, p.d1, p.d2);
    PB_LAUNCH_CHECK();
    if (p.rowsum_off >= 0) {
        rowsum_f16_kernel<<<ceil_div(p.rowsum_rows, 8), 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const __half*>(m->blob + p.dst_off), p.rowsum_rows, p.rowsum_cols,
            reinterpret_cast<float*>(m->blob + p.rowsum_off));
        PB_LAUNCH_CHECK();
    }
    if (p.fold_group >= 0) {     // the derived bias is (re)computed whenever its three inputs are all present in the blob
        FoldGroup& g = m->folds[p.fold_group];
        if (++g.loaded >= 3) {
            fold_bias_kernel<<<ceil_div(g.c, 8), 256, 0, (cudaStream_t)stream>>>(m->w<__half>(g.w2), m->w<float>(g.beta), m->w<float>(g.b2),
                                                                              g.c, 4 * g.c, m->w<float>(g.out));
            PB_LAUNCH_CHECK();
        }
    }
    return 0;
}

int64_t pb200_paella_workspace_bytes(const pb200_paella* m, int batch_total, int h, int w, int s_max) {
    if (m == nullptr) { set_error("workspace_bytes: null model handle"); return -1; }
    Arena a{nullptr};
    FeatWs f;
    plan_features(m, batch_total, h, w, a, f);
    Arena b{nullptr};
    CondWs cw;
    plan_cond(m, batch_total, s_max, s_max, b, cw);
    // logits / sampling scratch: fp16 features for B*H*W rows
    // fp16 features of the sampler; the shared-Philox kernel reads whole 4*rs-row blocks (rs <= 1184*256/num_labels + 1)
    const int64_t pad_rows = 4 * ((int64_t)1184 * 256 / m->cfg.num_labels + 2);
    const int64_t samp_rows = (int64_t)batch_total * h * w + pad_rows;
    // + the needed-slot list of the masked sampler (pb200_paella_sample_tokens_masked)
    const int64_t samp = (samp_rows * m->cfg.c_out * 2 + 255) / 256 * 256 + 256 + (samp_rows + 255) / 256 * 256;
    int64_t need = a.off > b.off ? a.off : b.off;
    need = need > samp ? need : samp;
    return need + 256;
}

int64_t pb200_paella_cond_cache_bytes(const pb200_paella* m, int batch_total, int s_max) {
    if (m == nullptr) { set_error("cond_cache_bytes: null model handle"); return -1; }
    return cond_block_off(m, m->n_attn, batch_total, s_max) + ((int64_t)batch_total * 4 + 255) / 256 * 256;
}

// gen_c_embeddings into ws.seq (fp32 [B,S,c_cond], LayerNorm'd): ref/src/modules.py:223-232
static int cond_embed(pb200_paella* m, const pb200_cond* cond, int B, int L, int S, CondWs& ws, cudaStream_t st) {
    const pb200_paella_config& c = m->cfg;
    // byt5_mapper -> rows [b, 0:L)
    PB_TRY(launch_cast_f16(cond->byt5, (int64_t)B * L * c.byt5_embd, ws.byt5_16, st));
    {
        pb200_gemm_epilogue e = epi(PB200_EPI_F32, m->w<float>(m->byt5_b), ws.seq, c.c_cond);
        e.remap_in = L; e.remap_out = S;
        PB_TRY(m->gemm(ws.byt5_16, c.byt5_embd, (int64_t)B * L, c.byt5_embd, m->byt5_w, c.c_cond, e, st));
    }
    // clip / clip_image mappers -> clip_seq_len rows each, appended in order
    int row = L;
    auto map_clip = [&](const float* src, int64_t w_off, int64_t b_off) -> int {
        PB_TRY(launch_cast_f16(src, (int64_t)B * c.clip_embd, ws.clip_16, st));
        pb200_gemm_epilogue e = epi(PB200_EPI_F32, m->w<float>(b_off), ws.seq + (int64_t)row * c.c_cond, (int64_t)S * c.c_cond);
        PB_TRY(m->gemm(ws.clip_16, c.clip_embd, B, c.clip_embd, w_off, (int64_t)c.c_cond * c.clip_seq_len, e, st));
        row += c.clip_seq_len;
        return 0;
    };
    if (cond->clip) PB_TRY(map_clip(cond->clip, m->clip_w, m->clip_b));
    if (cond->clip_image)
        for (int i = 0; i < cond->n_clip_image; ++i)
            PB_TRY(map_clip(cond->clip_image + (int64_t)i * B * c.clip_embd, m->clipimg_w, m->clipimg_b));
    // seq_norm
    return launch_ln_rows(ws.seq, (int64_t)B * S, c.c_cond, 1.0f, 0.0f, nullptr, ws.seq, st);
}

int pb200_paella_r_embedding(const float* r, int batch, int c_r, float* out, void* stream) {
    return launch_r_embed(r, batch, c_r, out, (cudaStream_t)stream);
}

int pb200_paella_c_embeddings(pb200_paella* m, const pb200_cond* cond, int batch, float* out, void* workspace,
                              int64_t workspace_bytes, void* stream) {
    PB_CHECK(m->blob != nullptr, "c_embeddings: weights not bound");
    PB_CHECK(cond && cond->byt5 && cond->byt5_len > 0, "c_embeddings: byt5 embeddings are required");
    const pb200_paella_config& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const int L = cond->byt5_len;
    const int S = L + c.clip_seq_len * ((cond->clip ? 1 : 0) + (cond->clip_image ? cond->n_clip_image : 0));
    PB_CHECK(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    Arena ar{reinterpret_cast<uint8_t*>(workspace)};
    CondWs ws;
    plan_cond(m, batch, L, S, ar, ws);
    PB_CHECK(ar.off <= workspace_bytes, "c_embeddings: workspace too small");
    PB_TRY(cond_embed(m, cond, batch, L, S, ws, st));
    PB_CUDA(cudaMemcpyAsync(out, ws.seq, (size_t)batch * S * c.c_cond * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

int pb200_paella_prepare_cond(pb200_paella* m, const pb200_cond* cond, int batch, int batch_offset, int batch_total,
                              int s_max, void* cond_cache, void* workspace, int64_t workspace_bytes, void* stream) {
    PB_CHECK(m->blob != nullptr, "prepare_cond: weights not bound");
    PB_CHECK(cond && cond->byt5 && cond->byt5_len > 0, "prepare_cond: byt5 embeddings are required");
    const pb200_paella_config& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = batch, L = cond->byt5_len;
    const int n_extra = (cond->clip ? 1 : 0) + (cond->clip_image ? cond->n_clip_image : 0);
    const int S = L + c.clip_seq_len * n_extra;
    PB_CHECK(S <= s_max, "prepare_cond: sequence length %d exceeds s_max %d", S, s_max);
    PB_CHECK(batch_offset >= 0 && batch_offset + B <= batch_total, "prepare_cond: batch range out of bounds");
    PB_CHECK(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)cond_cache & 255) == 0, "buffers must be 256-byte aligned");
    Arena ar{reinterpret_cast<uint8_t*>(workspace)};
    CondWs ws;
    plan_cond(m, B, L, S, ar, ws);
    PB_CHECK(ar.off <= workspace_bytes, "prepare_cond: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)ar.off);
    PB_TRY(cond_embed(m, cond, B, L, S, ws, st));
    // the SiLU every kv_mapper starts with
    PB_TRY(launch_silu_cast_f16(ws.seq, (int64_t)B * S * c.c_cond, ws.silu16, st));

    uint8_t* cache = reinterpret_cast<uint8_t*>(cond_cache);
    for (const BlockPlan& b : m->blocks) {
        if (b.kind != BK_ATTN) continue;
        const int ch = b.c;
        pb200_gemm_epilogue e1 = epi(PB200_EPI_F16, m->w<float>(b.kvm_b), ws.kvm16, ch);
        PB_TRY(m->gemm(ws.silu16, c.c_cond, (int64_t)B * S, c.c_cond, b.kvm_w, ch, e1, st));
        __half* dst = reinterpret_cast<__half*>(cache + cond_block_off(m, b.attn_index, batch_total, s_max)) +
                      (int64_t)batch_offset * s_max * 2 * ch;
        pb200_gemm_epilogue e2 = epi(PB200_EPI_F16, m->w<float>(b.inproj_b) + ch, dst, 2 * ch);
        e2.remap_in = S; e2.remap_out = s_max;
        PB_TRY(m->gemm(ws.kvm16, ch, (int64_t)B * S, ch, b.inproj_w + (int64_t)ch * ch * 2, 2 * ch, e2, st));
    }
    int* kv_len = reinterpret_cast<int*>(cache + cond_block_off(m, m->n_attn, batch_total, s_max));
    fill_int_kernel<<<ceil_div(B, 128), 128, 0, st>>>(kv_len + batch_offset, B, S);
    PB_LAUNCH_CHECK();
    return 0;
}

int pb200_paella_features(pb200_paella* m, const int64_t* tokens, const float* r, int batch_total, int cfg_pairs, int h, int w,
                          const void* cond_cache, int cache_slots, const int* kv_slot, int s_max, const float* attn_weights,
                          int n_attn_weights,
                          int attn_weights_batch, float* features, void* workspace, int64_t workspace_bytes,
                          void* stream) {
    PB_CHECK(m->blob != nullptr, "features: weights not bound");
    const pb200_paella_config& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const int Bt = batch_total, ps = c.patch_size, L = c.n_levels;
    PB_CHECK(h % (ps << (L - 1)) == 0 && w % (ps << (L - 1)) == 0, "latent grid %dx%d not divisible by %d", h, w, ps << (L - 1));
    PB_CHECK(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    PB_CHECK(m->n_attn == 0 || cond_cache != nullptr, "features: conditioning cache required");
    Arena ar{reinterpret_cast<uint8_t*>(workspace)};
    FeatWs ws;
    plan_features(m, Bt, h, w, ar, ws);
    PB_CHECK(ar.off <= workspace_bytes, "features: workspace too small (%lld < %lld)", (long long)workspace_bytes, (long long)ar.off);
    const uint8_t* cache = reinterpret_cast<const uint8_t*>(cond_cache);
    PB_CHECK(cache_slots > 0 && (kv_slot != nullptr || cache_slots == Bt), "features: %d cache slots for %d samples need a slot map",
             cache_slots, Bt);
    const int* kv_len = reinterpret_cast<const int*>(cache + cond_block_off(m, m->n_attn, cache_slots, s_max));

    int gh[PB200_MAX_LEVELS], gw[PB200_MAX_LEVELS];
    for (int l = 0; l < L; ++l) { gh[l] = (h / ps) >> l; gw[l] = (w / ps) >> l; }

    // Classifier-free-guidance pairs: sample i and sample i + Bt/2 carry the same (tokens, r) and differ only in their
    // conditioning rows, which enter through the AttnBlocks alone.  Everything before the first AttnBlock (the whole
    // level-0 down stack of the reference config, 'CT') is therefore computed ONCE for Bt/2 samples and replicated
    // when the first AttnBlock is reached -- the same arithmetic on the same inputs, not an approximation.
    PB_CHECK(!cfg_pairs || Bt % 2 == 0, "features: cfg_pairs needs an even batch_total (got %d)", Bt);
    int Bc = cfg_pairs ? Bt / 2 : Bt;                   // samples currently carried by x

    // timestep embedding and every TimestepBlock's (a, b) at once
    PB_TRY(launch_r_embed(r, Bc, c.c_r, ws.r_emb, st));
    PB_TRY(launch_film_table(ws.r_emb, Bc, c.c_r, m->w<float>(m->film_w), m->w<float>(m->film_b), m->film_total, ws.film, st));
    if (Bc < Bt)
        PB_CUDA(cudaMemcpyAsync(ws.film + (size_t)Bc * m->film_total, ws.film, (size_t)Bc * m->film_total * sizeof(float),
                                cudaMemcpyDeviceToDevice, st));
    PB_CUDA(cudaMemsetAsync(ws.gsq, 0, (size_t)Bt * 4 * m->max_c * sizeof(uint64_t), st));
    if (Bc < Bt) PB_CUDA(cudaMemsetAsync(ws.gscale, 0, (size_t)Bt * 4 * m->max_c * sizeof(uint64_t), st));
    if (m->n_attn > 0) PB_CUDA(cudaMemsetAsync(ws.lnstat, 0, (size_t)ws.lnstat_stride * m->n_attn * sizeof(int64_t), st));
    int ln_ready = -1;             // AttnBlock index whose fp16 input rows (a16) + row statistics the last block produced
    uint64_t* grn_stat[2] = {ws.gsq, ws.gscale};      // ping-pong: the GRN kernel of block i zeroes the buffer of block i+1
    int grn_flip = 0;

    // in_mapper + embedding
    PB_TRY(launch_embed_tokens(tokens, m->w<float>(m->emb_table), c.num_labels, c.c_in, Bc, h, w, ps, ws.h16, st));
    {
        const int64_t M0 = (int64_t)Bc * gh[0] * gw[0];
        pb200_gemm_epilogue e = epi(PB200_EPI_F32, m->w<float>(m->emb_b), ws.xd[0], c.c_hidden[0]);
        PB_TRY(m->gemm(ws.h16, (int64_t)c.c_in * ps * ps, M0, (int64_t)c.c_in * ps * ps, m->emb_w, c.c_hidden[0], e, st));
        PB_TRY(launch_ln_rows(ws.xd[0], M0, c.c_hidden[0], 1.0f, 0.0f, nullptr, ws.xd[0], st));
    }

    float* x = ws.xd[0];
    bool up_phase = false;
    // replicate the shared prefix: x (= xd[l] on the down path) and every saved level output below it
    auto replicate = [&](int level, int attn_index) -> int {
        for (int q = 0; q <= level; ++q) {
            const size_t n = (size_t)Bc * gh[q] * gw[q] * c.c_hidden[q];
            PB_CUDA(cudaMemcpyAsync(ws.xd[q] + n, ws.xd[q], n * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
        if (attn_index >= 0 && ln_ready == attn_index) {   // the folded-LayerNorm inputs of the AttnBlock that starts here
            const size_t rows = (size_t)Bc * gh[level] * gw[level];
            PB_CUDA(cudaMemcpyAsync(ws.a16 + rows * c.c_hidden[level], ws.a16, rows * c.c_hidden[level] * sizeof(__half),
                                    cudaMemcpyDeviceToDevice, st));
            int64_t* stat = ws.lnstat + ws.lnstat_stride * ln_ready;
            PB_CUDA(cudaMemcpyAsync(stat + 2 * rows, stat, 2 * rows * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        }
        Bc = Bt;
        return 0;
    };
    for (size_t bi = 0; bi < m->blocks.size(); ++bi) {
        const BlockPlan& b = m->blocks[bi];
        const int l = b.level, ch = b.c, P = gh[l] * gw[l];
        // the prefix ends at the first AttnBlock, or where the up path starts (its tensors live outside xd[])
        if (Bc < Bt && (b.kind == BK_ATTN || b.kind == BK_UP || (b.kind == BK_SAVE && l == L - 1))) PB_TRY(replicate(l, b.kind == BK_ATTN ? b.attn_index : -1));
        const int64_t M = (int64_t)Bc * P;
        switch (b.kind) {
            case BK_SAVE:
                if (l == L - 1) up_phase = true;       // deepest level: the up path continues on the same tensor
                break;
            case BK_DOWN: {
                PB_TRY(launch_ln_patchify2(x, Bc, gh[l - 1], gw[l - 1], c.c_hidden[l - 1], ws.a16, st));
                pb200_gemm_epilogue e = epi(PB200_EPI_F32, m->w<float>(b.rs_b), ws.xd[l], ch);
                PB_TRY(m->gemm(ws.a16, 4 * (int64_t)c.c_hidden[l - 1], M, 4 * (int64_t)c.c_hidden[l - 1], b.rs_w, ch, e, st));
                x = ws.xd[l];
                break;
            }
            case BK_UP: {
                const int cout = c.c_hidden[l - 1];
                PB_TRY(launch_ln_rows(x, M, ch, 1.0f, 0.0f, ws.a16, nullptr, st));
                pb200_gemm_epilogue e = epi(PB200_EPI_UNPATCH_F32, m->w<float>(b.rs_b), ws.xu[l - 1], 0);
                e.up_h = gh[l]; e.up_w = gw[l]; e.up_cout = cout;
                PB_TRY(m->gemm(ws.a16, ch, M, ch, b.rs_w, 4 * (int64_t)cout, e, st));
                x = ws.xu[l - 1];
                break;
            }
            case BK_RES:
            case BK_FF: {
                if (b.kind == BK_RES) {
                    const float* skip = b.c_skip ? ws.xd[l] : nullptr;
                    PB_TRY(launch_dwconv_ln(x, skip, m->w<float>(b.dw_w), m->w<float>(b.dw_b), Bc, gh[l], gw[l], ch,
                                            c.kernel_size, ws.a16, st));
                } else {
                    PB_TRY(launch_ln_rows(x, M, ch, 1.0f, 0.0f, ws.a16, nullptr, st));
                }
                pb200_gemm_epilogue e1 = epi(PB200_EPI_GELU_F16, m->w<float>(b.b1), ws.h16, 4 * ch);
                uint64_t* stat = grn_stat[grn_flip];
                uint64_t* stat_next = grn_stat[grn_flip ^ 1];
                grn_flip ^= 1;
                e1.sqsum = stat; e1.rows_per_sample = P;
                PB_TRY(m->gemm(ws.a16, ch, M, ch, b.w1, 4 * (int64_t)ch, e1, st));
                // GlobalResponseNorm: folded into GEMM2's A operand where its tiles line up with the samples (multipliers only,
                // shift pushed into the bias), else applied to the hidden in place
                // Measured on B200 (profiles/r02_ab_notes.md): the fold removes the 168 MB GRN pass (-12.4 ms per bench step) but the
                // in-place rescale adds 32 KB of shared-memory traffic per k-block to a 2-SM main loop whose operand reads already
                // use ~3/4 of the 128 B/clk port: GEMM2 61 -> 89 us per level-1 launch (+17 ms per step).  Net loss: opt-in.
                static const bool fold_on = getenv("PB200_GRN_FOLD") != nullptr;
                const bool fold_grn = fold_on && gemm_can_scale_a(M, ch, 4 * (int64_t)ch, P);
                __half* grn_s16 = reinterpret_cast<__half*>(ws.grn_mult);
                if (fold_grn)
                    PB_TRY(launch_grn_scale_f16(Bc, 4 * ch, stat, stat_next, 4 * m->max_c, m->w<float>(b.gamma), grn_s16, st));
                else
                    PB_TRY(launch_grn_fused(ws.h16, Bc, P, 4 * ch, stat, stat_next, 4 * m->max_c, m->w<float>(b.gamma), m->w<float>(b.beta), ws.grn_mult, st));
                // the next AttnBlock's LayerNorm is folded into its QKV GEMM when this block feeds it directly
                const bool fold = b.ln_fold_attn >= 0;
                pb200_gemm_epilogue e2 = epi(fold ? PB200_EPI_RESID_LN_F32 : PB200_EPI_RESID_F32, m->w<float>(fold_grn ? b.b2_fold : b.b2), x, ch);
                if (fold_grn) { e2.a_scale = grn_s16; e2.a_scale_ld = 4 * (int64_t)ch; }
                e2.resid = x; e2.ldr = ch; e2.rows_per_sample = P;
                if (b.film_off >= 0) { e2.film = ws.film; e2.film_ld = m->film_total; e2.film_off = b.film_off; }
                if (fold) {
                    e2.out16 = ws.a16;
                    e2.ln_stat = ws.lnstat + ws.lnstat_stride * b.ln_fold_attn;
                    e2.ln_shift = ws.lnmean + ws.lnmean_stride * b.ln_shift_attn;
                    ln_ready = b.ln_fold_attn;
                }
                PB_TRY(m->gemm(ws.h16, 4 * (int64_t)ch, M, 4 * (int64_t)ch, b.w2, ch, e2, st));
                break;
            }
            case BK_TIME:
                if (!b.film_fused) PB_TRY(launch_film_apply(x, M, ch, P, ws.film, m->film_total, b.film_off, st));
                break;
            case BK_ATTN: {
                const bool folded = ln_ready == b.attn_index;
                pb200_gemm_epilogue e1 = epi(folded ? PB200_EPI_F16_LN : PB200_EPI_F16, m->w<float>(b.inproj_b), ws.qkv16, 3 * ch);
                float* mean_out = ws.lnmean + ws.lnmean_stride * b.attn_index;      // read by the next block's folded LayerNorm
                if (folded) {       // a16 = fp16(x - shift) and the row statistics came out of the previous GEMM's epilogue
                    e1.ln_stat = ws.lnstat + ws.lnstat_stride * b.attn_index;
                    e1.ln_wsum = m->w<float>(b.inproj_wsum);
                    e1.ln_c = ch;
                    e1.ln_shift = ws.lnmean + ws.lnmean_stride * b.ln_shift_attn;
                    e1.ln_mean_out = mean_out;
                } else {
                    PB_TRY(launch_ln_rows(x, M, ch, 1.0f, 0.0f, ws.a16, nullptr, st, mean_out));
                }
                PB_TRY(m->gemm(ws.a16, ch, M, ch, b.inproj_w, 3 * (int64_t)ch, e1, st));
                AttnParams ap;
                ap.qkv = ws.qkv16;
                ap.ckv = reinterpret_cast<const __half*>(cache + cond_block_off(m, b.attn_index, cache_slots, s_max));
                ap.kv_len = kv_len;
                ap.kv_slot = kv_slot;
                ap.n_slots = cache_slots;
                ap.out = ws.o16;
                ap.B = Bt; ap.P = P; ap.S_max = s_max; ap.E = ch; ap.nhead = c.nhead[l];
                ap.self_attn = c.self_attn;
                ap.scale_log2 = 1.4426950408889634f / sqrtf((float)(ch / c.nhead[l]));
                ap.attn_w = attn_weights; ap.n_w = n_attn_weights; ap.w_batch = attn_weights_batch;
                PB_TRY(launch_attention(ap, st));
                pb200_gemm_epilogue e2 = epi(PB200_EPI_RESID_F32, m->w<float>(b.outproj_b), x, ch);
                e2.resid = x; e2.ldr = ch; e2.rows_per_sample = P;
                PB_TRY(m->gemm(ws.o16, ch, M, ch, b.outproj_w, ch, e2, st));
                break;
            }
        }
    }
    (void)up_phase;
    // clf (LN2d, 1x1 conv, PixelShuffle) + out_mapper's LayerNorm2d
    {
        const int ch = c.c_hidden[0];
        const int64_t M0 = (int64_t)Bc * gh[0] * gw[0];
        PB_TRY(launch_ln_rows(x, M0, ch, 1.0f, 0.0f, ws.a16, nullptr, st));
        pb200_gemm_epilogue e = epi(PB200_EPI_UNPATCH_F32, m->w<float>(m->clf_b), ws.y, 0);
        e.up_h = gh[0]; e.up_w = gw[0]; e.up_cout = c.c_out;
        PB_TRY(m->gemm(ws.a16, ch, M0, ch, m->clf_w, 4 * (int64_t)c.c_out, e, st));
        PB_TRY(launch_ln_rows(ws.y, (int64_t)Bc * h * w, c.c_out, 1.0f, 0.0f, nullptr, features, st));
        if (Bc < Bt) {      // a model without any AttnBlock or up path: the two halves are identical to the end
            const size_t n = (size_t)Bc * h * w * c.c_out;
            PB_CUDA(cudaMemcpyAsync(features + n, features, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
        }
    }
    return 0;
}

int pb200_paella_logits(pb200_paella* m, const float* features, int batch, int hw, float* logits_nchw, void* workspace,
                        int64_t workspace_bytes, void* stream) {
    PB_CHECK(m->blob != nullptr, "logits: weights not bound");
    const pb200_paella_config& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = (int64_t)batch * hw;
    PB_CHECK(rows * c.c_out * 2 <= workspace_bytes, "logits: workspace too small");
    __half* a16 = reinterpret_cast<__half*>(workspace);
    PB_TRY(launch_cast_f16(features, rows * c.c_out, a16, st));
    pb200_gemm_epilogue e = epi(PB200_EPI_NCHW_F32, nullptr, logits_nchw, 0);
    e.rows_per_sample = hw;
    return m->gemm(a16, c.c_out, rows, c.c_out, m->out_w, c.num_labels, e, st);
}

int pb200_paella_sample_tokens(pb200_paella* m, const float* features, int batch, int hw, int cfg_on, double cfg,
                               double temperature, uint64_t seed, uint64_t offset, int64_t* tokens_out, void* workspace,
                               int64_t workspace_bytes, void* stream) {
    PB_CHECK(m->blob != nullptr, "sample_tokens: weights not bound");
    const pb200_paella_config& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = (int64_t)batch * hw;
    PB_CHECK(fused_sampler_rows_padded(rows, c.num_labels) * c.c_out * 2 <= workspace_bytes,
             "sample_tokens: workspace too small (use pb200_paella_workspace_bytes)");
    PB_CHECK(temperature > 0, "sample_tokens: temperature must be positive");
    __half* a16 = reinterpret_cast<__half*>(workspace);
    // classifier-free guidance is linear in the features: mix before the GEMM
    if (cfg_on)
        PB_TRY(launch_mix_cast_f16(features, features + rows * c.c_out, (float)cfg, (float)(1.0 - cfg), rows * c.c_out, a16, st));
    else
        PB_TRY(launch_cast_f16(features, rows * c.c_out, a16, st));
    return launch_fused_sampler(a16, rows, c.c_out, m->w<__half>(m->out_w), c.num_labels, 1.0f / (float)temperature, seed,
                                offset, tokens_out, st);
}

int pb200_paella_sample_tokens_masked(pb200_paella* m, const float* features, int batch, int hw, int cfg_on, double cfg,
                                      double temperature, uint64_t seed, uint64_t offset, const uint8_t* mask,
                                      int64_t* tokens_inout, void* workspace, int64_t workspace_bytes, void* stream) {
    PB_CHECK(m->blob != nullptr, "sample_tokens_masked: weights not bound");
    PB_CHECK(mask != nullptr, "sample_tokens_masked: mask is required");
    PB_CHECK(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    const pb200_paella_config& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t rows = (int64_t)batch * hw;
    const int64_t a16_bytes = (fused_sampler_rows_padded(rows, c.num_labels) * c.c_out * 2 + 255) / 256 * 256;
    PB_CHECK(a16_bytes + fused_sampler_mask_scratch_bytes(rows, c.num_labels) <= workspace_bytes,
             "sample_tokens_masked: workspace too small (use pb200_paella_workspace_bytes)");
    PB_CHECK(temperature > 0, "sample_tokens_masked: temperature must be positive");
    __half* a16 = reinterpret_cast<__half*>(workspace);
    // the CFG mix / fp16 cast stays dense: it is one pass over c_out-wide rows, the sampler is the 8192-wide part
    if (cfg_on)
        PB_TRY(launch_mix_cast_f16(features, features + rows * c.c_out, (float)cfg, (float)(1.0 - cfg), rows * c.c_out, a16, st));
    else
        PB_TRY(launch_cast_f16(features, rows * c.c_out, a16, st));
    return launch_fused_sampler_masked(a16, rows, c.c_out, m->w<__half>(m->out_w), c.num_labels, 1.0f / (float)temperature, seed,
                                       offset, mask, reinterpret_cast<uint8_t*>(workspace) + a16_bytes, tokens_inout, st);
}

}  // extern "C"
