// Host-side executor and small kernels of the f4 VQGAN codec.
//   VQModel blocks / parameter names   ref/src/vqgan.py:45-89
//   encode / decode / decode_indices   ref/src/vqgan.py:91-107
//   ResBlock                           ref/src/vqgan.py:6-42
// The MLPs of the ResBlocks are the tcgen05 GEMMs of gemm.cu; Conv2d(k4,s2,p1) and ConvTranspose2d(k4,s2,p1) are
// the same kernel with an im2col-free TMA gather of the A operand (ConvGeom); the 12/4-channel 1x1 convs at the
// image / latent ends are CUDA-core kernels (K or N of 4..12 cannot fill a tensor-core tile).
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

#include "gemm.cuh"
#include "ops.cuh"

namespace pb {

enum VqPack { VP_COPY_F32, VP_CAST_F16, VP_DW9, VP_CONV4, VP_CONVT4, VP_T12 };

__global__ void vq_pack_kernel(const float* __restrict__ src, void* __restrict__ dst, int kind, int64_t n, int d0, int d1,
                               int d2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float* d32 = reinterpret_cast<float*>(dst);
    __half* d16 = reinterpret_cast<__half*>(dst);
    switch (kind) {
        case VP_COPY_F32: d32[i] = src[i]; break;
        case VP_CAST_F16: d16[i] = __float2half_rn(src[i]); break;
        case VP_DW9: {      // src [c=d0, 1, 3, 3] -> dst [9][c]
            const int c = d0, ch = (int)(i % c), tap = (int)(i / c);
            d32[i] = src[(int64_t)ch * 9 + tap];
            break;
        }
        case VP_T12: {      // src [c0=d0, 12] -> dst [12][c0]: the in_block kernel's lanes read consecutive output channels
            const int c0 = d0, co = (int)(i % c0), k = (int)(i / c0);
            d32[i] = src[(int64_t)co * 12 + k];
            break;
        }
        case VP_CONV4: {    // src [Cout=d0, Cin=d1, 4, 4] -> dst fp16 [Cout][16][Cpad=d2] (zero padded channels)
            const int cin = d1, cpad = d2;
            const int c = (int)(i % cpad), tap = (int)((i / cpad) % 16), co = (int)(i / (16 * (int64_t)cpad));
            d16[i] = c < cin ? __float2half_rn(src[((int64_t)(co * cin + c) * 4 + (tap >> 2)) * 4 + (tap & 3)]) : __float2half_rn(0.f);
            break;
        }
        case VP_CONVT4: {   // src [Cin=d0, Cout=d1, 4, 4] -> dst fp16 [4 phases][Cout][4 taps][Cpad=d2]
            const int cin = d0, cout = d1, cpad = d2;
            const int c = (int)(i % cpad);
            const int tap = (int)((i / cpad) % 4);
            const int co = (int)((i / (4 * (int64_t)cpad)) % cout);
            const int ph = (int)(i / (4 * (int64_t)cpad * cout));
            const int py = ph >> 1, px = ph & 1, ty = tap >> 1, tx = tap & 1;
            const int ky = py == 0 ? (ty == 0 ? 1 : 3) : (ty == 0 ? 0 : 2);
            const int kx = px == 0 ? (tx == 0 ? 1 : 3) : (tx == 0 ? 0 : 2);
            d16[i] = c < cin ? __float2half_rn(src[((int64_t)(c * cout + co) * 4 + ky) * 4 + kx]) : __float2half_rn(0.f);
            break;
        }
    }
}

// ------------------------------------------------------------------ image-side / latent-side 1x1 convs (CUDA cores)
// in_block: PixelUnshuffle(2) + Conv2d(12 -> c0, k=1).  img NCHW [B,3,H,W] -> NHWC fp32 [B,H/2,W/2,c0].  w is packed [12][c0]
// (VP_T12): one coalesced float4 per input tap and channel quad.  Round 2 history: [c0][12] weights (48 loads per thread, each
// touching 32 lines per warp) took 4.7 ms for 64 images; a thread per (position, quad) with 12 scalar image loads + 12 weight
// loads per 48 FMA sat at 1.5 TB/s (ncu: L1 73 %); now:
// in_block, register-resident weights: a thread keeps the 12 x 4 weights of ITS channel quad and walks VQ_IN_PPT consecutive
// positions of a row (two 2-pixel-wide float2 loads per plane and position instead of 12 scalar loads + 12 weight loads)
constexpr int VQ_IN_PPT = 4;
__global__ void __launch_bounds__(192) vq_in_block_rw_kernel(const float* __restrict__ img, const float* __restrict__ w,
                                                             const float* __restrict__ bias, int B, int H, int W, int c0,
                                                             float* __restrict__ out) {
    const int h2 = H >> 1, w2 = W >> 1, nq = c0 >> 2;
    const int groups_x = (w2 + VQ_IN_PPT - 1) / VQ_IN_PPT;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * h2 * groups_x * nq) return;
    const int q = (int)(i % nq);
    const int64_t grp = i / nq;
    const int gx = (int)(grp % groups_x);
    const int64_t row = grp / groups_x;                 // b * h2 + y
    const int b = (int)(row / h2), y = (int)(row - (int64_t)b * h2);
    float4 wv[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) wv[k] = __ldg(reinterpret_cast<const float4*>(w + (int64_t)k * c0) + q);
    const float4 bv = __ldg(reinterpret_cast<const float4*>(bias) + q);
#pragma unroll
    for (int pi = 0; pi < VQ_IN_PPT; ++pi) {
        const int x = gx * VQ_IN_PPT + pi;
        if (x >= w2) break;
        float in[12];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int dy = 0; dy < 2; ++dy) {
                const float2 v = *reinterpret_cast<const float2*>(img + (((int64_t)b * 3 + c) * H + 2 * y + dy) * W + 2 * x);
                in[c * 4 + dy * 2] = v.x; in[c * 4 + dy * 2 + 1] = v.y;
            }
        float4 acc = bv;
#pragma unroll
        for (int k = 0; k < 12; ++k) {
            acc.x = fmaf(in[k], wv[k].x, acc.x); acc.y = fmaf(in[k], wv[k].y, acc.y);
            acc.z = fmaf(in[k], wv[k].z, acc.z); acc.w = fmaf(in[k], wv[k].w, acc.w);
        }
        *reinterpret_cast<float4*>(out + ((row * w2) + x) * c0 + q * 4) = acc;
    }
}

// out_block: Conv2d(c0 -> 12, k=1) + PixelShuffle(2).  x NHWC fp32 [B,h2,w2,c0] -> img NCHW [B,3,2h2,2w2]; warp per position.
// MODE (include/paella_b200.h PB200_IMG_*): 0 raw fp32 NCHW, 1 clamp(0,1) fp32 NCHW, 2 uint8 NHWC [B,2h2,2w2,3] with
// save_image's rounding -- the callers' clamp / byte conversion passes fused into the store.
// COMPOSITE (pb200_vqgan_decode_composite): where pmask [B,2h2,2w2] is 0 the pixel is orig (fp32 NCHW, same size) instead of
// the decoded value, put through the same MODE conversion.
template <int MODE, bool COMPOSITE = false>
__global__ void __launch_bounds__(256) vq_out_block_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                           const float* __restrict__ bias, int B, int h2, int w2, int c0,
                                                           void* __restrict__ img_out, const float* __restrict__ orig = nullptr,
                                                           const uint8_t* __restrict__ pmask = nullptr) {
    const int lane = threadIdx.x & 31;
    const int64_t pos = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pos >= (int64_t)B * h2 * w2) return;
    float acc[12];
#pragma unroll
    for (int o = 0; o < 12; ++o) acc[o] = 0.f;
    for (int c = lane; c < c0; c += 32) {
        const float v = x[pos * c0 + c];
#pragma unroll
        for (int o = 0; o < 12; ++o) acc[o] = fmaf(v, __ldg(w + o * c0 + c), acc[o]);
    }
#pragma unroll
    for (int o = 0; o < 12; ++o) acc[o] = warp_sum(acc[o]);
    if (lane < 12) {
        float v = 0.f;
#pragma unroll
        for (int o = 0; o < 12; ++o) v = lane == o ? acc[o] : v;
        const int b = (int)(pos / ((int64_t)h2 * w2));
        const int rem = (int)(pos - (int64_t)b * h2 * w2);
        const int y = rem / w2, xx = rem - y * w2;
        const int c = lane >> 2, d = lane & 3;
        v += bias[lane];
        if constexpr (COMPOSITE) {
            const int64_t px = ((int64_t)b * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1);
            if (pmask[px] == 0) v = orig[(((int64_t)b * 3 + c) * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1)];
        }
        if (MODE != 0) v = fminf(fmaxf(v, 0.f), 1.f);
        if (MODE == 2) {
            uint8_t* img = reinterpret_cast<uint8_t*>(img_out);
            img[(((int64_t)b * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1)) * 3 + c] =
                (uint8_t)fminf(__fadd_rn(__fmul_rn(v, 255.0f), 0.5f), 255.0f);      // mul then add, two roundings like the torch ops (no FMA)
        } else {
            float* img = reinterpret_cast<float*>(img_out);
            img[(((int64_t)b * 3 + c) * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1)] = v;
        }
    }
}

// out_block, thread per position (c0 % 32 == 0): the warp-per-position kernel above issues 72 weight loads and 60 shuffles per
// lane and position (ncu: LSU 63 %, 0.96 TB/s).  Here a thread owns a position: it pulls its row in 128-byte pieces (eight 16-byte
// loads, consumed at once) and multiplies against the 12 x c0 weights staged in shared memory as [c/4][12] float4 (warp-wide
// broadcast reads) -- 1.5 global loads + 18 shared loads per 72 FFMA.  Summation order: channels ascending per output.
template <int MODE, bool COMPOSITE = false>
__global__ void __launch_bounds__(128) vq_out_block_tp_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                              const float* __restrict__ bias, int B, int h2, int w2, int c0,
                                                              void* __restrict__ img_out, const float* __restrict__ orig = nullptr,
                                                              const uint8_t* __restrict__ pmask = nullptr) {
    extern __shared__ float4 w_s[];                      // [c0/4][12]: the 4 channel weights of output o
    const int nj = c0 >> 2;
    for (int i = threadIdx.x; i < nj * 12; i += blockDim.x) {
        const int j = i / 12, o = i - j * 12;
        w_s[i] = *reinterpret_cast<const float4*>(w + (int64_t)o * c0 + 4 * j);
    }
    __syncthreads();
    const int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= (int64_t)B * h2 * w2) return;
    float acc[12];
#pragma unroll
    for (int o = 0; o < 12; ++o) acc[o] = __ldg(bias + o);
    const float4* xr = reinterpret_cast<const float4*>(x + pos * c0);
    for (int j0 = 0; j0 < nj; j0 += 8) {
        float4 v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = xr[j0 + t];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
#pragma unroll
            for (int o = 0; o < 12; ++o) {
                const float4 ww = w_s[(j0 + t) * 12 + o];
                acc[o] = fmaf(v[t].w, ww.w, fmaf(v[t].z, ww.z, fmaf(v[t].y, ww.y, fmaf(v[t].x, ww.x, acc[o]))));
            }
        }
    }
    const int b = (int)(pos / ((int64_t)h2 * w2));
    const int rem = (int)(pos - (int64_t)b * h2 * w2);
    const int y = rem / w2, xx = rem - y * w2;
#pragma unroll
    for (int o = 0; o < 12; ++o) {
        float v = acc[o];
        const int c = o >> 2, d = o & 3;
        if constexpr (COMPOSITE) {
            const int64_t px = ((int64_t)b * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1);
            if (pmask[px] == 0) v = orig[(((int64_t)b * 3 + c) * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1)];
        }
        if (MODE != 0) v = fminf(fmaxf(v, 0.f), 1.f);
        if (MODE == 2) {
            uint8_t* img = reinterpret_cast<uint8_t*>(img_out);
            img[(((int64_t)b * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1)) * 3 + c] =
                (uint8_t)fminf(__fadd_rn(__fmul_rn(v, 255.0f), 0.5f), 255.0f);      // mul then add, two roundings like the torch ops (no FMA)
        } else {
            float* img = reinterpret_cast<float*>(img_out);
            img[(((int64_t)b * 3 + c) * (2 * h2) + 2 * y + (d >> 1)) * (2 * w2) + 2 * xx + (d & 1)] = v;
        }
    }
}

// latent head: Conv2d(c1 -> cl, k=1, no bias) + BatchNorm2d(eval).  x [M,c1] -> lat [M,cl] (cl <= 8); warp per position
__global__ void __launch_bounds__(256) vq_latent_head_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                             const float* __restrict__ bn_w, const float* __restrict__ bn_b,
                                                             const float* __restrict__ bn_mean, const float* __restrict__ bn_var,
                                                             int64_t M, int c1, int cl, float* __restrict__ lat) {
    const int lane = threadIdx.x & 31;
    const int64_t pos = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pos >= M) return;
    float acc[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = 0.f;
    for (int c = lane; c < c1; c += 32) {
        const float v = x[pos * c1 + c];
#pragma unroll
        for (int o = 0; o < 8; ++o)
            if (o < cl) acc[o] = fmaf(v, __ldg(w + o * c1 + c), acc[o]);
    }
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = warp_sum(acc[o]);
    if (lane < cl) {
        float v = 0.f;
#pragma unroll
        for (int o = 0; o < 8; ++o) v = lane == o ? acc[o] : v;
        const float sc = bn_w[lane] / sqrtf(bn_var[lane] + 1e-5f);
        lat[pos * cl + lane] = (v - bn_mean[lane]) * sc + bn_b[lane];
    }
}

// decoder head: Conv2d(cl -> c1, k=1).  z [M,cl] -> x [M,c1]
__global__ void __launch_bounds__(256) vq_dec_head_kernel(const float* __restrict__ z, const float* __restrict__ w,
                                                          const float* __restrict__ bias, int64_t M, int cl, int c1,
                                                          float* __restrict__ out) {
    const int nq = c1 >> 2;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * nq) return;
    const int q = (int)(i % nq);
    const int64_t pos = i / nq;
    float zi[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) zi[k] = k < cl ? z[pos * cl + k] : 0.f;
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int co = q * 4 + j;
        float acc = bias[co];
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < cl) acc = fmaf(zi[k], __ldg(w + co * cl + k), acc);
        o[j] = acc;
    }
    *reinterpret_cast<float4*>(out + pos * c1 + q * 4) = make_float4(o[0], o[1], o[2], o[3]);
}

// the same for cl == 4 (the f4 codec): z and each output channel's weights are ONE 16-byte load -- 5 loads per thread instead of
// 40 (ncu, round 2: the scalar version sat at 63 % `lg_throttle` stalls, 213 us for a 100 MB store)
__global__ void __launch_bounds__(256) vq_dec_head4_kernel(const float* __restrict__ z, const float* __restrict__ w,
                                                           const float* __restrict__ bias, int64_t M, int c1,
                                                           float* __restrict__ out) {
    const int nq = c1 >> 2;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * nq) return;
    const int q = (int)(i % nq);
    const int64_t pos = i / nq;
    const float4 zv = *(reinterpret_cast<const float4*>(z) + pos);
    const float4 bv = __ldg(reinterpret_cast<const float4*>(bias) + q);
    const float4* wr = reinterpret_cast<const float4*>(w) + q * 4;          // rows 4q .. 4q+3 of w [c1, 4]
    const float4 w0 = __ldg(wr), w1 = __ldg(wr + 1), w2 = __ldg(wr + 2), w3 = __ldg(wr + 3);
    auto dot = [&](float b, const float4& ww) { return fmaf(zv.w, ww.w, fmaf(zv.z, ww.z, fmaf(zv.y, ww.y, fmaf(zv.x, ww.x, b)))); };
    *reinterpret_cast<float4*>(out + pos * c1 + q * 4) = make_float4(dot(bv.x, w0), dot(bv.y, w1), dot(bv.z, w2), dot(bv.w, w3));
}

// ResBlock middle: x += (depthwise3x3(ReplicationPad(xt)) + bias) * g2; xt, x NHWC fp32; w9 [9][c]
__global__ void __launch_bounds__(256) vq_dw_residual_kernel(const float* __restrict__ xt, float* __restrict__ x,
                                                             const float* __restrict__ w9, const float* __restrict__ bias,
                                                             float g2, int B, int h, int w, int c) {
    const int nq = c >> 2;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * h * w * nq) return;
    const int q = (int)(i % nq);
    const int64_t pos = i / nq;
    const int b = (int)(pos / ((int64_t)h * w));
    const int rem = (int)(pos - (int64_t)b * h * w);
    const int y = rem / w, xx = rem - y * w;
    float4 acc = __ldg(reinterpret_cast<const float4*>(bias) + q);
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int iy = min(max(y + ky - 1, 0), h - 1);
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
            const int ix = min(max(xx + kx - 1, 0), w - 1);
            const float4 v = *reinterpret_cast<const float4*>(xt + (((int64_t)b * h + iy) * w + ix) * c + q * 4);
            const float4 ww = __ldg(reinterpret_cast<const float4*>(w9 + (int64_t)(ky * 3 + kx) * c) + q);
            acc.x = fmaf(v.x, ww.x, acc.x); acc.y = fmaf(v.y, ww.y, acc.y);
            acc.z = fmaf(v.z, ww.z, acc.z); acc.w = fmaf(v.w, ww.w, acc.w);
        }
    }
    float4* xo = reinterpret_cast<float4*>(x + pos * c) + q;
    float4 r = *xo;
    r.x = fmaf(acc.x, g2, r.x); r.y = fmaf(acc.y, g2, r.y); r.z = fmaf(acc.z, g2, r.z); r.w = fmaf(acc.w, g2, r.w);
    *xo = r;
}

struct VqParam {
    std::string name;
    int64_t numel, dst_off, dst_numel;
    int kind, d0, d1, d2;
    float* host_copy;    // gammas: also mirrored on the host
};

struct VqResBlock {
    int c;
    int64_t dw_w, dw_b, w1, b1, w2, b2;
    float gam[6];
};

}  // namespace pb

using namespace pb;

struct pb200_vqgan {
    pb200_vqgan_config cfg;
    int c0, c1;                                    // level widths: c_hidden/2, c_hidden (levels == 2)
    std::vector<VqParam> params;
    std::unordered_map<std::string, int> by_name;
    int64_t weight_bytes = 0;
    uint8_t* blob = nullptr;
    int64_t in_w, in_b, down_w, down_b, lat_w, bn_w, bn_b, bn_mean, bn_var, codebook, dec_w, dec_b, up_w, up_b, out_w, out_b;
    int cpad0, cpad1;
    VqResBlock enc0, enc1, dec_last;
    std::vector<VqResBlock> bottleneck;
    bool host_params_stale = true;                 // the gammas' host mirror has not been read from the bound blob yet
    std::map<std::tuple<const void*, int64_t, int64_t, int64_t, int>, CUtensorMap> tmaps;

    int64_t add(const std::string& name, int64_t numel, int kind, int64_t dst_numel, int eb, int d0 = 0, int d1 = 0, int d2 = 0,
                float* host = nullptr) {
        VqParam p;
        p.name = name; p.numel = numel; p.kind = kind; p.dst_numel = dst_numel; p.d0 = d0; p.d1 = d1; p.d2 = d2;
        p.host_copy = host;
        p.dst_off = weight_bytes;
        weight_bytes += (dst_numel * eb + 255) / 256 * 256;
        by_name[name] = (int)params.size();
        params.push_back(p);
        return p.dst_off;
    }
    int64_t f32(const std::string& n, int64_t numel) { return add(n, numel, VP_COPY_F32, numel, 4); }
    int64_t f16(const std::string& n, int64_t numel) { return add(n, numel, VP_CAST_F16, numel, 2); }
    template <typename T>
    T* w(int64_t off) const { return reinterpret_cast<T*>(blob + off); }

    void add_resblock(const std::string& pre, int c, VqResBlock& rb) {
        rb.c = c;
        rb.dw_w = add(pre + "depthwise.1.weight", (int64_t)c * 9, VP_DW9, (int64_t)c * 9, 4, c);
        rb.dw_b = f32(pre + "depthwise.1.bias", c);
        rb.w1 = f16(pre + "channelwise.0.weight", (int64_t)4 * c * c);
        rb.b1 = f32(pre + "channelwise.0.bias", 4 * c);
        rb.w2 = f16(pre + "channelwise.2.weight", (int64_t)4 * c * c);
        rb.b2 = f32(pre + "channelwise.2.bias", c);
        for (int i = 0; i < 6; ++i) rb.gam[i] = 0.f;
        add(pre + "gammas", 6, VP_COPY_F32, 6, 4, 0, 0, 0, rb.gam);
    }

    int tmap2d(const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, const CUtensorMap** out) {
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
    int gemm(const __half* A, int64_t lda, int64_t M, int64_t K, int64_t w_off, int64_t N, const pb200_gemm_epilogue& ep,
             cudaStream_t st) {
        const int bn = gemm_pick_block_n(M, N, K);
        const CUtensorMap *ta, *tb;
        PB_TRY(tmap2d(A, M, K, lda, GEMM_BLOCK_M, &ta));
        PB_TRY(tmap2d(w<__half>(w_off), N, K, K, bn / 2, &tb));     // W box = half a tile
        return gemm_launch(*ta, *tb, bn, ep, M, N, K, st);
    }
};

namespace pb {

static pb200_gemm_epilogue vepi(int mode, const float* bias, void* out, int64_t ldo) {
    pb200_gemm_epilogue e;
    memset(&e, 0, sizeof(e));
    e.mode = mode; e.bias = bias; e.out = out; e.ldo = ldo; e.alpha = 1.0f;
    return e;
}

struct VqWs {
    float *xa, *xb, *tmp32, *lat, *zq;
    __half *a16, *h16;
    int64_t* idx;
};

static void vq_plan(const pb200_vqgan* m, int B, int H, int W, uint8_t* base, int64_t& off, VqWs& ws) {
    auto take = [&](int64_t bytes) -> uint8_t* {
        const int64_t o = off;
        off += (bytes + 255) / 256 * 256;
        return base ? base + o : nullptr;
    };
    const int64_t M0 = (int64_t)B * (H / 2) * (W / 2), M1 = (int64_t)B * (H / 4) * (W / 4);
    const int64_t big = M0 * m->c0 > M1 * m->c1 ? M0 * m->c0 : M1 * m->c1;
    ws.xa = (float*)take(big * 4);
    ws.xb = (float*)take(big * 4);
    ws.tmp32 = (float*)take(big * 4);
    ws.a16 = (__half*)take(big * 2);
    ws.h16 = (__half*)take(big * 4 * 2);
    ws.lat = (float*)take(M1 * m->cfg.c_latent * 4);
    ws.zq = (float*)take(M1 * m->cfg.c_latent * 4);
    ws.idx = (int64_t*)take(M1 * 8);
}

// The part of a codec ResBlock (ref/src/vqgan.py:36-42) before its MLP: x' = x + g2 * dw3x3(pad(LN(x)(1+g0)+g1)), then
// a16 = fp16(LN(x')(1+g3)+g4).  x: NHWC fp32 [B,h,w,c].  *resid = where x' lives: `tmp32` on the fused path (one patch kernel +
// a statistics pre-pass, ops.cu::launch_vq_front_fused; `scratch` = B*h*w float2), x itself (updated in place) on the three-launch
// path that narrow widths (tiny test codecs) and in_place = true (the fused-MLP experiment) take.
static int resblock_front(float* x, int B, int h, int w, int c, const float* dw_w9, const float* dw_b, const float* gam,
                          float* tmp32, __half* a16, void* scratch, bool in_place, const float** resid, cudaStream_t st) {
    const int64_t M = (int64_t)B * h * w;
    static const bool unfused = getenv("PB200_VQ_FRONT_UNFUSED") != nullptr;      // A/B knob
    if (!in_place && !unfused && vq_front_fused_ok(c, h, w)) {
        *resid = tmp32;
        return launch_vq_front_fused(x, B, h, w, c, dw_w9, dw_b, gam, reinterpret_cast<float2*>(scratch), tmp32, a16, st);
    }
    *resid = x;
    PB_TRY(launch_ln_rows(x, M, c, 1.0f + gam[0], gam[1], nullptr, tmp32, st));
    {
        ProfScope prof("vq_dwconv", (double)M * c * 12.0, st);
        vq_dw_residual_kernel<<<ceil_div(M * (c / 4), 256), 256, 0, st>>>(tmp32, x, dw_w9, dw_b, gam[2], B, h, w, c);
        PB_LAUNCH_CHECK();
    }
    return launch_ln_rows(x, M, c, 1.0f + gam[3], gam[4], a16, nullptr, st);
}

// x: NHWC fp32 [B,h,w,c], updated in place (ref/src/vqgan.py:36-42)
static int run_resblock(pb200_vqgan* m, const VqResBlock& rb, float* x, int B, int h, int w, VqWs& ws, cudaStream_t st) {
    const int c = rb.c;
    const int64_t M = (int64_t)B * h * w;
    static const bool fused = getenv("PB200_VQ_MLP_FUSED") != nullptr;      // experiment knob: see vq_mlp.cu (measured slower)
    const float* resid = x;
    // (h16 is idle until GEMM1 writes it: it lends its first bytes to the row statistics)
    PB_TRY(resblock_front(x, B, h, w, c, m->w<float>(rb.dw_w), m->w<float>(rb.dw_b), rb.gam, ws.tmp32, ws.a16, ws.h16, fused, &resid, st));
    if (fused) {    // Linear -> GELU -> Linear -> x + g5 * (.) in one kernel, the 4c hidden never leaves the SM
        const int rc = launch_vq_mlp_fused(ws.a16, M, c, m->w<__half>(rb.w1), m->w<float>(rb.b1), m->w<__half>(rb.w2), m->w<float>(rb.b2), x,
                                           rb.gam[5], st);
        if (rc >= 0) return rc;
    }
    pb200_gemm_epilogue e1 = vepi(PB200_EPI_GELU_F16, m->w<float>(rb.b1), ws.h16, 4 * c);
    PB_TRY(m->gemm(ws.a16, c, M, c, rb.w1, 4 * (int64_t)c, e1, st));
    pb200_gemm_epilogue e2 = vepi(PB200_EPI_RESID_F32, m->w<float>(rb.b2), x, c);
    e2.resid = resid; e2.ldr = c; e2.alpha = rb.gam[5];
    PB_TRY(m->gemm(ws.h16, 4 * (int64_t)c, M, 4 * (int64_t)c, rb.w2, c, e2, st));
    return 0;
}

static void conv_tile(int gw, int& tw, int& th) {
    tw = 128;
    while (tw > gw && tw > 8) tw >>= 1;
    th = 128 / tw;
}

}  // namespace pb

extern "C" {

int64_t pb200_vqgan_resblock_workspace_bytes(int batch, int h, int w, int c) {
    const int64_t M = (int64_t)batch * h * w;
    auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
    return up(M * c * 4) + up(M * c * 2) + up(M * 4 * c * 2) + 256;
}

int pb200_vqgan_resblock(float* x_nhwc, int batch, int h, int w, int c, const float* dw_w9, const float* dw_bias, const void* w1_f16,
                         const float* b1, const void* w2_f16, const float* b2, const float* gammas_host, void* workspace,
                         int64_t workspace_bytes, void* stream) {
    PB_CHECK(x_nhwc && dw_w9 && dw_bias && w1_f16 && b1 && w2_f16 && b2 && gammas_host, "vqgan_resblock: null pointer");
    PB_CHECK(c % 8 == 0, "vqgan_resblock: c=%d must be a multiple of 8", c);
    PB_CHECK(((uintptr_t)workspace & 255) == 0 && workspace_bytes >= pb200_vqgan_resblock_workspace_bytes(batch, h, w, c),
             "vqgan_resblock: workspace too small or misaligned");
    if (batch == 0 || h == 0 || w == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t M = (int64_t)batch * h * w;
    auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
    uint8_t* base = reinterpret_cast<uint8_t*>(workspace);
    float* tmp32 = reinterpret_cast<float*>(base);
    __half* a16 = reinterpret_cast<__half*>(base + up(M * c * 4));
    __half* h16 = reinterpret_cast<__half*>(base + up(M * c * 4) + up(M * c * 2));
    const float* resid = x_nhwc;
    PB_TRY(resblock_front(x_nhwc, batch, h, w, c, dw_w9, dw_bias, gammas_host, tmp32, a16, h16, false, &resid, st));
    pb200_gemm_epilogue e1 = vepi(PB200_EPI_GELU_F16, b1, h16, 4 * c);
    PB_TRY(gemm_f16(a16, c, w1_f16, c, M, 4 * (int64_t)c, c, e1, st));
    pb200_gemm_epilogue e2 = vepi(PB200_EPI_RESID_F32, b2, x_nhwc, c);
    e2.resid = resid; e2.ldr = c; e2.alpha = gammas_host[5];
    return gemm_f16(h16, 4 * (int64_t)c, w2_f16, 4 * (int64_t)c, M, c, 4 * (int64_t)c, e2, st);
}

int pb200_vq_mlp_fused(const void* a16, int64_t rows, int c, const void* w1_f16, const float* b1, const void* w2_f16, const float* b2,
                       float* x, float alpha, void* stream) {
    PB_CHECK(a16 && w1_f16 && b1 && w2_f16 && b2 && x, "vq_mlp_fused: null pointer");
    const int rc = launch_vq_mlp_fused(reinterpret_cast<const __half*>(a16), rows, c, reinterpret_cast<const __half*>(w1_f16), b1,
                                       reinterpret_cast<const __half*>(w2_f16), b2, x, alpha, (cudaStream_t)stream);
    PB_CHECK(rc >= 0, "vq_mlp_fused: built for c in {384, 192} and rows >= 256 only (got c=%d, rows=%lld)", c, (long long)rows);
    return rc;
}

int pb200_vqgan_create(const pb200_vqgan_config* cfg, pb200_vqgan** out) {
    PB_CHECK(cfg && out, "vqgan_create: null argument");
    PB_CHECK(cfg->levels == 2, "vqgan: levels=%d unsupported (the f4 codec has 2)", cfg->levels);
    PB_CHECK(cfg->c_hidden % 16 == 0 && cfg->c_latent >= 1 && cfg->c_latent <= 8, "vqgan: bad widths");
    pb200_vqgan* m = new pb200_vqgan();
    m->cfg = *cfg;
    m->c1 = cfg->c_hidden;
    m->c0 = cfg->c_hidden / 2;
    m->cpad0 = (m->c0 + 63) / 64 * 64;
    m->cpad1 = (m->c1 + 63) / 64 * 64;
    const int c0 = m->c0, c1 = m->c1, cl = cfg->c_latent;
    m->in_w = m->add("in_block.1.weight", (int64_t)c0 * 12, VP_T12, (int64_t)c0 * 12, 4, c0);
    m->in_b = m->f32("in_block.1.bias", c0);
    m->add_resblock("down_blocks.0.", c0, m->enc0);
    m->down_w = m->add("down_blocks.1.weight", (int64_t)c1 * c0 * 16, VP_CONV4, (int64_t)c1 * 16 * m->cpad0, 2, c1, c0, m->cpad0);
    m->down_b = m->f32("down_blocks.1.bias", c1);
    m->add_resblock("down_blocks.2.", c1, m->enc1);
    m->lat_w = m->f32("down_blocks.3.0.weight", (int64_t)cl * c1);
    m->bn_w = m->f32("down_blocks.3.1.weight", cl);
    m->bn_b = m->f32("down_blocks.3.1.bias", cl);
    m->bn_mean = m->f32("down_blocks.3.1.running_mean", cl);
    m->bn_var = m->f32("down_blocks.3.1.running_var", cl);
    m->codebook = m->f32("vquantizer.codebook.weight", (int64_t)cfg->codebook_size * cl);
    m->dec_w = m->f32("up_blocks.0.0.weight", (int64_t)c1 * cl);
    m->dec_b = m->f32("up_blocks.0.0.bias", c1);
    m->bottleneck.resize(cfg->bottleneck_blocks);
    int j = 1;
    for (int i = 0; i < cfg->bottleneck_blocks; ++i, ++j) m->add_resblock("up_blocks." + std::to_string(j) + ".", c1, m->bottleneck[i]);
    m->up_w = m->add("up_blocks." + std::to_string(j) + ".weight", (int64_t)c1 * c0 * 16, VP_CONVT4, (int64_t)4 * c0 * 4 * m->cpad1, 2,
                     c1, c0, m->cpad1);
    m->up_b = m->f32("up_blocks." + std::to_string(j) + ".bias", c0);
    ++j;
    m->add_resblock("up_blocks." + std::to_string(j) + ".", c0, m->dec_last);
    m->out_w = m->f32("out_block.0.weight", (int64_t)12 * c0);
    m->out_b = m->f32("out_block.0.bias", 12);
    *out = m;
    return 0;
}

void pb200_vqgan_destroy(pb200_vqgan* m) { delete m; }
int64_t pb200_vqgan_weight_bytes(const pb200_vqgan* m) { return m->weight_bytes; }
int pb200_vqgan_bind_weights(pb200_vqgan* m, void* blob) {
    PB_CHECK(((uintptr_t)blob & 255) == 0, "weight blob must be 256-byte aligned");
    m->blob = reinterpret_cast<uint8_t*>(blob);
    m->tmaps.clear();
    m->host_params_stale = true;
    return 0;
}

int pb200_vqgan_sync_params(pb200_vqgan* m, void* stream) {
    PB_CHECK(m->blob != nullptr, "sync_params: bind a weight blob first");
    cudaStream_t st = (cudaStream_t)stream;
    for (const VqParam& p : m->params)
        if (p.host_copy)
            PB_CUDA(cudaMemcpyAsync(p.host_copy, m->blob + p.dst_off, p.numel * sizeof(float), cudaMemcpyDeviceToHost, st));
    PB_CUDA(cudaStreamSynchronize(st));
    m->host_params_stale = false;
    return 0;
}
int pb200_vqgan_num_params(const pb200_vqgan* m) { return (int)m->params.size(); }
const char* pb200_vqgan_param_name(const pb200_vqgan* m, int i) {
    return (i >= 0 && i < (int)m->params.size()) ? m->params[i].name.c_str() : "";
}
int64_t pb200_vqgan_param_numel(const pb200_vqgan* m, int i) {
    return (i >= 0 && i < (int)m->params.size()) ? m->params[i].numel : -1;
}

int pb200_vqgan_load_param(pb200_vqgan* m, const char* name, const float* src, int64_t numel, void* stream) {
    PB_CHECK(m->blob != nullptr, "load_param: bind a weight blob first");
    auto it = m->by_name.find(name);
    PB_CHECK(it != m->by_name.end(), "load_param: '%s' is not a parameter of this plan", name);
    const VqParam& p = m->params[it->second];
    PB_CHECK(numel == p.numel, "load_param: '%s' has %lld elements, expected %lld", name, (long long)numel, (long long)p.numel);
    cudaStream_t st = (cudaStream_t)stream;
    vq_pack_kernel<<<ceil_div(p.dst_numel, 256), 256, 0, st>>>(src, m->blob + p.dst_off, p.kind, p.dst_numel, p.d0, p.d1, p.d2);
    PB_LAUNCH_CHECK();
    if (p.host_copy) m->host_params_stale = true;      // the 6 ResBlock gammas are kernel arguments: re-read lazily
    return 0;
}

int64_t pb200_vqgan_workspace_bytes(const pb200_vqgan* m, int batch, int img_h, int img_w) {
    int64_t off = 0;
    VqWs ws;
    vq_plan(m, batch, img_h, img_w, nullptr, off, ws);
    return off + 256;
}

int pb200_vqgan_encode(pb200_vqgan* m, const float* img, int batch, int img_h, int img_w, float* latents_nchw,
                       float* quantised_nchw, int64_t* indices, void* workspace, int64_t workspace_bytes, void* stream) {
    PB_CHECK(m->blob != nullptr, "encode: weights not bound");
    if (m->host_params_stale) PB_TRY(pb200_vqgan_sync_params(m, stream));
    PB_CHECK(img_h % 4 == 0 && img_w % 4 == 0, "encode: image %dx%d not divisible by 4", img_h, img_w);
    PB_CHECK(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int B = batch, c0 = m->c0, c1 = m->c1, cl = m->cfg.c_latent;
    const int h0 = img_h / 2, w0 = img_w / 2, h1 = img_h / 4, w1 = img_w / 4;
    int64_t off = 0;
    VqWs ws;
    vq_plan(m, B, img_h, img_w, reinterpret_cast<uint8_t*>(workspace), off, ws);
    PB_CHECK(off <= workspace_bytes, "encode: workspace too small");
    const int64_t M0 = (int64_t)B * h0 * w0, M1 = (int64_t)B * h1 * w1;
    {
        ProfScope prof("vq_in_block", (double)M0 * (48.0 + c0 * 4.0), st);
        const int64_t n_thr = (int64_t)B * h0 * ceil_div(w0, VQ_IN_PPT) * (c0 / 4);
        vq_in_block_rw_kernel<<<ceil_div(n_thr, 192), 192, 0, st>>>(img, m->w<float>(m->in_w), m->w<float>(m->in_b), B, img_h, img_w,
                                                                    c0, ws.xa);
        PB_LAUNCH_CHECK();
    }
    PB_TRY(run_resblock(m, m->enc0, ws.xa, B, h0, w0, ws, st));
    // Conv2d(c0 -> c1, k=4, s=2, p=1): fp16 NHWC copy, then the TMA-gather GEMM
    PB_TRY(launch_cast_f16(ws.xa, M0 * c0, ws.a16, st));
    {
        ConvGeom g;
        memset(&g, 0, sizeof(g));
        g.mode = 1; g.batch = B; g.gh = h1; g.gw = w1; g.cin = c0; g.n_cchunk = m->cpad0 / 64;
        conv_tile(w1, g.tw, g.th);
        g.tiles_x = ceil_div(w1, g.tw); g.tiles_y = ceil_div(h1, g.th);
        g.oh = h1; g.ow = w1; g.sy = 1; g.sx = 1; g.py = 0; g.px = 0;
        const int64_t N = c1, K = 16 * (int64_t)m->cpad0;
        const int bn = gemm_pick_block_n((int64_t)B * g.tiles_x * g.tiles_y * 128, N, K, false);
        CUtensorMap ta;
        const int64_t dims[5] = {2 * (int64_t)c0, w0 / 2, 2, h0 / 2, B};
        const int64_t strides[4] = {2 * (int64_t)c0 * 2, (int64_t)w0 * c0 * 2, 2 * (int64_t)w0 * c0 * 2, (int64_t)h0 * w0 * c0 * 2};
        const int box[5] = {64, g.tw, 1, g.th, 1};
        PB_TRY(make_tmap_f16_nd(&ta, ws.a16, 5, dims, strides, box));
        const CUtensorMap* tb;
        PB_TRY(m->tmap2d(m->w<__half>(m->down_w), N, K, K, bn / 2, &tb));
        pb200_gemm_epilogue e = vepi(PB200_EPI_F32, m->w<float>(m->down_b), ws.xb, c1);
        PB_TRY(gemm_conv_launch(ta, *tb, bn, e, g, N, K, st));
    }
    PB_TRY(run_resblock(m, m->enc1, ws.xb, B, h1, w1, ws, st));
    {
        ProfScope prof("vq_latent_head", (double)M1 * c1 * 4.0, st);
        vq_latent_head_kernel<<<ceil_div(M1, 8), 256, 0, st>>>(ws.xb, m->w<float>(m->lat_w), m->w<float>(m->bn_w), m->w<float>(m->bn_b),
                                                              m->w<float>(m->bn_mean), m->w<float>(m->bn_var), M1, c1, cl, ws.lat);
        PB_LAUNCH_CHECK();
    }
    {
        ProfScope prof("vq_nearest", (double)M1 * (cl * 4.0 + 8.0), st);
        PB_TRY(pb200_vq_nearest(ws.lat, M1, cl, m->w<float>(m->codebook), m->cfg.codebook_size, indices ? indices : ws.idx, st));
    }
    if (latents_nchw) PB_TRY(launch_nhwc_to_nchw(ws.lat, B, cl, h1 * w1, latents_nchw, st));
    if (quantised_nchw) {
        PB_TRY(pb200_vq_gather(indices ? indices : ws.idx, M1, m->w<float>(m->codebook), m->cfg.codebook_size, cl, ws.zq, st));
        PB_TRY(launch_nhwc_to_nchw(ws.zq, B, cl, h1 * w1, quantised_nchw, st));
    }
    return 0;
}

int pb200_vqgan_decode(pb200_vqgan* m, const int64_t* indices, const float* latents_nchw, int batch, int h, int w, float* img,
                       void* workspace, int64_t workspace_bytes, void* stream) {
    return pb200_vqgan_decode_ex(m, indices, latents_nchw, batch, h, w, img, PB200_IMG_F32_NCHW, workspace, workspace_bytes, stream);
}

// orig / pmask non-null: the last kernel composites (pb200_vqgan_decode_composite)
static int vq_decode_impl(pb200_vqgan* m, const int64_t* indices, const float* latents_nchw, int batch, int h, int w, void* img,
                          int img_mode, const float* orig, const uint8_t* pmask, void* workspace, int64_t workspace_bytes,
                          void* stream) {
    PB_CHECK(m->blob != nullptr, "decode: weights not bound");
    PB_CHECK(img_mode >= 0 && img_mode <= 2, "decode: unknown image mode %d", img_mode);
    if (m->host_params_stale) PB_TRY(pb200_vqgan_sync_params(m, stream));
    PB_CHECK((indices != nullptr) != (latents_nchw != nullptr), "decode: pass indices or latents, not both");
    PB_CHECK(((uintptr_t)workspace & 255) == 0, "workspace must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int B = batch, c0 = m->c0, c1 = m->c1, cl = m->cfg.c_latent;
    const int h1 = h, w1 = w, h0 = 2 * h, w0 = 2 * w;
    int64_t off = 0;
    VqWs ws;
    vq_plan(m, B, 4 * h, 4 * w, reinterpret_cast<uint8_t*>(workspace), off, ws);
    PB_CHECK(off <= workspace_bytes, "decode: workspace too small");
    const int64_t M0 = (int64_t)B * h0 * w0, M1 = (int64_t)B * h1 * w1;
    if (indices)
        PB_TRY(pb200_vq_gather(indices, M1, m->w<float>(m->codebook), m->cfg.codebook_size, cl, ws.zq, st));
    else
        PB_TRY(launch_nchw_to_nhwc(latents_nchw, B, cl, h1 * w1, ws.zq, st));
    {
        ProfScope prof("vq_dec_head", (double)M1 * c1 * 4.0, st);
        if (cl == 4)
            vq_dec_head4_kernel<<<ceil_div(M1 * (c1 / 4), 256), 256, 0, st>>>(ws.zq, m->w<float>(m->dec_w), m->w<float>(m->dec_b), M1, c1, ws.xb);
        else
            vq_dec_head_kernel<<<ceil_div(M1 * (c1 / 4), 256), 256, 0, st>>>(ws.zq, m->w<float>(m->dec_w), m->w<float>(m->dec_b), M1, cl, c1,
                                                                            ws.xb);
        PB_LAUNCH_CHECK();
    }
    for (const VqResBlock& rb : m->bottleneck) PB_TRY(run_resblock(m, rb, ws.xb, B, h1, w1, ws, st));
    // ConvTranspose2d(c1 -> c0, k=4, s=2, p=1) as 4 sub-pixel phases of 2x2 taps
    PB_TRY(launch_cast_f16(ws.xb, M1 * c1, ws.a16, st));
    {
        ConvGeom g;
        memset(&g, 0, sizeof(g));
        g.mode = 2; g.batch = B; g.gh = h1; g.gw = w1; g.cin = c1; g.n_cchunk = m->cpad1 / 64;
        conv_tile(w1, g.tw, g.th);
        g.tiles_x = ceil_div(w1, g.tw); g.tiles_y = ceil_div(h1, g.th);
        g.oh = h0; g.ow = w0; g.sy = 2; g.sx = 2;
        const int64_t N = c0, K = 4 * (int64_t)m->cpad1;
        const int bn = gemm_pick_block_n((int64_t)B * g.tiles_x * g.tiles_y * 128, N, K, false);
        CUtensorMap ta;
        const int64_t dims[4] = {c1, w1, h1, B};
        const int64_t strides[3] = {(int64_t)c1 * 2, (int64_t)w1 * c1 * 2, (int64_t)h1 * w1 * c1 * 2};
        const int box[4] = {64, g.tw, g.th, 1};
        PB_TRY(make_tmap_f16_nd(&ta, ws.a16, 4, dims, strides, box));
        for (int ph = 0; ph < 4; ++ph) {
            g.py = ph >> 1; g.px = ph & 1;
            const CUtensorMap* tb;
            PB_TRY(m->tmap2d(m->w<__half>(m->up_w) + (int64_t)ph * N * K, N, K, K, bn / 2, &tb));
            pb200_gemm_epilogue e = vepi(PB200_EPI_F32, m->w<float>(m->up_b), ws.xa, c0);
            PB_TRY(gemm_conv_launch(ta, *tb, bn, e, g, N, K, st));
        }
    }
    PB_TRY(run_resblock(m, m->dec_last, ws.xa, B, h0, w0, ws, st));
    {
        ProfScope prof("vq_out_block", (double)M0 * (c0 * 4.0 + 48.0), st);
        const float *ow = m->w<float>(m->out_w), *ob = m->w<float>(m->out_b);
        if (pmask) {
            if (c0 % 32 == 0 && c0 <= 768) {
                const size_t sm = (size_t)c0 * 48;
                const unsigned g = (unsigned)ceil_div(M0, 128);
                if (img_mode == PB200_IMG_U8_NHWC) vq_out_block_tp_kernel<2, true><<<g, 128, sm, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img, orig, pmask);
                else if (img_mode == PB200_IMG_F32_NCHW_CLAMP01) vq_out_block_tp_kernel<1, true><<<g, 128, sm, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img, orig, pmask);
                else vq_out_block_tp_kernel<0, true><<<g, 128, sm, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img, orig, pmask);
            } else if (img_mode == PB200_IMG_U8_NHWC) vq_out_block_kernel<2, true><<<ceil_div(M0, 8), 256, 0, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img, orig, pmask);
            else if (img_mode == PB200_IMG_F32_NCHW_CLAMP01) vq_out_block_kernel<1, true><<<ceil_div(M0, 8), 256, 0, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img, orig, pmask);
            else vq_out_block_kernel<0, true><<<ceil_div(M0, 8), 256, 0, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img, orig, pmask);
        } else if (c0 % 32 == 0 && c0 <= 768) {         // thread per position, weights in shared memory
            const size_t sm = (size_t)c0 * 48;
            const unsigned g = (unsigned)ceil_div(M0, 128);
            if (img_mode == PB200_IMG_U8_NHWC) vq_out_block_tp_kernel<2><<<g, 128, sm, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img);
            else if (img_mode == PB200_IMG_F32_NCHW_CLAMP01) vq_out_block_tp_kernel<1><<<g, 128, sm, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img);
            else vq_out_block_tp_kernel<0><<<g, 128, sm, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img);
        } else if (img_mode == PB200_IMG_U8_NHWC) vq_out_block_kernel<2><<<ceil_div(M0, 8), 256, 0, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img);
        else if (img_mode == PB200_IMG_F32_NCHW_CLAMP01) vq_out_block_kernel<1><<<ceil_div(M0, 8), 256, 0, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img);
        else vq_out_block_kernel<0><<<ceil_div(M0, 8), 256, 0, st>>>(ws.xa, ow, ob, B, h0, w0, c0, img);
        PB_LAUNCH_CHECK();
    }
    return 0;
}

int pb200_vqgan_decode_ex(pb200_vqgan* m, const int64_t* indices, const float* latents_nchw, int batch, int h, int w, void* img,
                          int img_mode, void* workspace, int64_t workspace_bytes, void* stream) {
    return vq_decode_impl(m, indices, latents_nchw, batch, h, w, img, img_mode, nullptr, nullptr, workspace, workspace_bytes, stream);
}

int pb200_vqgan_decode_composite(pb200_vqgan* m, const int64_t* indices, int batch, int h, int w, const float* orig_img,
                                 const uint8_t* pixel_mask, void* img, int img_mode, void* workspace, int64_t workspace_bytes,
                                 void* stream) {
    PB_CHECK(indices != nullptr && orig_img != nullptr && pixel_mask != nullptr,
             "decode_composite: indices, orig_img and pixel_mask are required");
    return vq_decode_impl(m, indices, nullptr, batch, h, w, img, img_mode, orig_img, pixel_mask, workspace, workspace_bytes, stream);
}

}  // extern "C"
