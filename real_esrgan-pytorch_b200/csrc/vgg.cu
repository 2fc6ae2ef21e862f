// VGG19 content loss of the RealESRGAN generator step (reference ContentLoss, model.py:278-335): torchvision's
// Normalize, the conv / ReLU / max-pool stack of vgg19().features up to the deepest requested node, one L1 (mean) per node
// between the SR and the GT features, and the gradient of those losses with respect to SR. The weights are frozen: there
// are no weight gradients. See DESIGN.md §8.
//
// Every convolution runs on the tcgen05 kernels of conv3x3_tc.cu / conv3x3_pair.cu (fp16 operands forward, bf16 data
// gradients backward, as the generator). Those hold a layer's weights resident in shared memory, which bounds Cin at 256;
// a 512-channel input is split into two 256-channel halves: the first writes an fp32 partial with the bias, the second
// reads the channels at offset 256 and adds the partial as its residual (EP_SKIP, zero bias) before ReLU / mask.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "../../include/resr.h"
#include "conv3x3.cuh"
#include "errors.h"
#include "gen_internal.cuh"

#define RESR_TRY(expr) do { const int rc__ = (expr); if (rc__ != RESR_OK) return rc__; } while (0)

namespace resr {
namespace {

constexpr int kVggConvs = 16;
constexpr int kFeature[kVggConvs] = {0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34};
constexpr int kCin[kVggConvs] = {3, 64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512};
constexpr int kCout[kVggConvs] = {64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512};
// a 2x2 / stride 2 max-pool follows conv i (features.4 / 9 / 18 / 27); the pool after conv 15 (features.36) is never needed
constexpr bool kPoolAfter[kVggConvs] = {false, true, false, true, false, false, false, true,
                                        false, false, false, true, false, false, false, false};
constexpr int kHalf = 256;        // input channels of one split-K half (the kernels' resident-weight limit)
constexpr int kInPad = 8;         // channels per pixel of the normalized 16-bit input (3 real, zero-padded)
constexpr int kLossBlocks = 296;  // fixed grid of the L1 partial sums: the summation order never depends on the device

struct PackRef {
    size_t off;                // byte offset in the pack buffer
    int nout, nslices, nchunks;
};

size_t pack_bytes(int nout, int nslices, int nchunks) { return static_cast<size_t>(nslices) * nchunks * 3 * (3 * nout) * 128; }

struct Layout {   // parameter and pack offsets of the 16 convolutions
    size_t p_off[kVggConvs];          // weight offset in the flat fp32 vector (the bias follows)
    PackRef fwd[kVggConvs][2];        // forward packs: [1] used when Cin == 512
    PackRef bwd[kVggConvs][2];        // data-gradient packs: [1] used when Cout == 512
    size_t b_off[kVggConvs];          // float offset of the padded bias
    size_t n_params, fwd_bytes, bwd_bytes, bias_floats;
    Layout() {
        size_t p = 0, f = 0, b = 0, t = 0;
        for (int i = 0; i < kVggConvs; ++i) {
            p_off[i] = p;
            p += static_cast<size_t>(kCout[i]) * kCin[i] * 9 + kCout[i];
            const int fh = kCin[i] > kHalf ? 2 : 1, bh = kCout[i] > kHalf ? 2 : 1;
            for (int h = 0; h < fh; ++h) {
                fwd[i][h] = {f, 32, kCout[i] / 32, (kCin[i] / fh + 63) / 64};
                f += pack_bytes(32, fwd[i][h].nslices, fwd[i][h].nchunks);
            }
            const int tnout = kCin[i] >= 32 ? 32 : 16;
            for (int h = 0; h < bh; ++h) {
                bwd[i][h] = {t, tnout, (kCin[i] + tnout - 1) / tnout, (kCout[i] / bh + 63) / 64};
                t += pack_bytes(tnout, bwd[i][h].nslices, bwd[i][h].nchunks);
            }
            b_off[i] = b;
            b += kCout[i];
        }
        n_params = p; fwd_bytes = f; bwd_bytes = t; bias_floats = b;
    }
};
const Layout& layout() {
    static Layout L;
    return L;
}

size_t up1k(size_t v) { return (v + 1023) / 1024 * 1024; }

// Workspace of one (N, H, W) call up to conv `deepest`. Forward maps hold the 2N batch (SR images first, then GT).
struct VggWs {
    size_t xin, act[kVggConvs], pool[kVggConvs], partial, g[2], sums, total;
    int h[kVggConvs], w[kVggConvs];   // resolution of conv i
};
VggWs vgg_ws(size_t N, int H, int W, int deepest) {
    VggWs L;
    memset(&L, 0, sizeof(L));
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = up1k(o + bytes); return at; };
    int h = H, w = W;
    size_t partial = 0, g = 0;
    L.xin = take(2 * N * H * W * kInPad * 2);
    for (int i = 0; i <= deepest; ++i) {
        L.h[i] = h; L.w[i] = w;
        const size_t P = N * h * w;
        L.act[i] = take(2 * P * kCout[i] * 2);
        if (kCin[i] > kHalf) partial = std::max(partial, 2 * P * kCout[i] * 4);   // forward: fp32 partial of the 2N batch
        if (kCout[i] > kHalf) partial = std::max(partial, P * kCin[i] * 4);       // backward: fp32 partial of the N batch
        g = std::max(g, P * kCout[i] * 2);
        if (i > 0) g = std::max(g, P * kCin[i] * 2);
        if (kPoolAfter[i] && i < deepest) {
            h /= 2; w /= 2;
            L.pool[i] = take(2 * N * h * w * kCout[i] * 2);
        }
    }
    L.partial = partial ? take(partial) : 0;
    L.g[0] = take(g);
    L.g[1] = take(g);
    L.sums = take(static_cast<size_t>(kVggConvs) * kLossBlocks * sizeof(double));
    L.total = o;
    return L;
}

// ------------------------------------------------------------------------------------------------------------ kernels

// transforms.Normalize + layout: sr / gt NCHW fp32 [N,3,H,W] -> one NHWC fp16 [2N,H,W,8] batch, x' = (x - mean) / std
// rounded as torch rounds it (fp32 subtract, fp32 divide), channels 3..7 zero.
__global__ void __launch_bounds__(256) vgg_normalize_kernel(const float* __restrict__ sr, const float* __restrict__ gt,
                                                           uint16_t* __restrict__ out, int N, int HW, float m0, float m1,
                                                           float m2, float s0, float s1, float s2) {
    const size_t total = 2 * static_cast<size_t>(N) * HW;
    for (size_t pix = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; pix < total;
         pix += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t n = pix / HW, r = pix % HW;
        const float* src = n < static_cast<size_t>(N) ? sr + n * 3 * HW : gt + (n - N) * 3 * HW;
        const float v0 = __fdiv_rn(__fsub_rn(src[r], m0), s0);
        const float v1 = __fdiv_rn(__fsub_rn(src[HW + r], m1), s1);
        const float v2 = __fdiv_rn(__fsub_rn(src[2 * static_cast<size_t>(HW) + r], m2), s2);
        const __half2 a = __floats2half2_rn(v0, v1), b = __floats2half2_rn(v2, 0.f);
        reinterpret_cast<uint4*>(out)[pix] =
            make_uint4(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b), 0u, 0u);
    }
}

// 2x2 / stride 2 max-pool (floor) of NHWC fp16 maps [B,H,W,C] -> [B,H/2,W/2,C]; one thread per 8 channels of an output pixel.
__global__ void __launch_bounds__(256) vgg_maxpool_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, int B, int H,
                                                         int W, int C) {
    const int ho = H / 2, wo = W / 2, c8 = C / 8;
    const size_t total = static_cast<size_t>(B) * ho * wo * c8;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int g = static_cast<int>(idx % c8);
        size_t t = idx / c8;
        const int xo = static_cast<int>(t % wo);
        t /= wo;
        const int yo = static_cast<int>(t % ho);
        const size_t n = t / ho;
        const uint4* p = reinterpret_cast<const uint4*>(in + ((n * H + 2 * yo) * W + 2 * xo) * C) + g;
        const size_t row = static_cast<size_t>(W) * c8;
        uint4 q[4] = {p[0], p[c8], p[row], p[row + c8]};
        uint4 m = q[0];
        __half2* mh = reinterpret_cast<__half2*>(&m);
#pragma unroll
        for (int k = 1; k < 4; ++k) {
            const __half2* qh = reinterpret_cast<const __half2*>(&q[k]);
#pragma unroll
            for (int j = 0; j < 4; ++j) mh[j] = __hmax2(mh[j], qh[j]);
        }
        reinterpret_cast<uint4*>(out)[idx] = m;
    }
}

__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

// Gradient at the output of conv i (before its ReLU), one thread per 8 channels of a pixel of conv i's output [N,H,W,C]:
//   g = [(pool ? (first max of its 2x2 window ? g_in[pooled pixel] : 0) : g_in) + w * sign(a_sr - a_gt) / numel] * relu'
// g_in: bf16 gradient at the next layer's input (null: none); act: the saved fp16 outputs of conv i, SR batch then GT
// batch; gw: device pointer to the upstream gradient of this node's loss (null: conv i is not a node); mask: multiply by
// (a_sr > 0) -- the ReLU after conv i. torchvision's ReLU(inplace=True) rewrites a node's tensor when the next layer runs,
// so a node other than the deepest is the post-ReLU value and its term is inside the mask. Pool ties go to the first
// element in row-major order, as max_pool2d's backward does.
__global__ void __launch_bounds__(256) vgg_node_bwd_kernel(const uint16_t* __restrict__ gin, const uint16_t* __restrict__ act,
                                                          const float* __restrict__ gw, float inv_numel, int mask, int pool,
                                                          uint16_t* __restrict__ gout, int N, int H, int W, int C) {
    const int c8 = C / 8;
    const size_t total = static_cast<size_t>(N) * H * W * c8;
    const size_t gt_off = static_cast<size_t>(N) * H * W * C;
    const float wk = gw ? __ldg(gw) * inv_numel : 0.f;
    const int ho = H / 2, wo = W / 2;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int g8 = static_cast<int>(idx % c8);
        const size_t pix = idx / c8;
        const int x = static_cast<int>(pix % W);
        const size_t r = pix / W;
        const int y = static_cast<int>(r % H);
        const size_t n = r / H;
        float a[8], v[8];
        {
            const uint4 q = reinterpret_cast<const uint4*>(act)[idx];
            const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
            for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(h[j]); a[2 * j] = f.x; a[2 * j + 1] = f.y; }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = 0.f;
        if (gin && !pool) {
            const uint4 q = reinterpret_cast<const uint4*>(gin)[idx];
            const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) { v[2 * j] = bf16_lo(w4[j]); v[2 * j + 1] = bf16_hi(w4[j]); }
        } else if (gin && (y >> 1) < ho && (x >> 1) < wo) {
            const int y0 = y & ~1, x0 = x & ~1, me = ((y & 1) << 1) | (x & 1);
            float win[4][8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const size_t pk = (n * H + y0 + (k >> 1)) * W + x0 + (k & 1);
                const uint4 q = reinterpret_cast<const uint4*>(act + pk * C)[g8];
                const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
                for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(h[j]); win[k][2 * j] = f.x; win[k][2 * j + 1] = f.y; }
            }
            const uint4 q = reinterpret_cast<const uint4*>(gin + ((n * ho + (y >> 1)) * wo + (x >> 1)) * C)[g8];
            const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                int arg = 0;
                float m = win[0][e];
#pragma unroll
                for (int k = 1; k < 4; ++k)
                    if (win[k][e] > m) { m = win[k][e]; arg = k; }
                const float gp = (e & 1) ? bf16_hi(w4[e >> 1]) : bf16_lo(w4[e >> 1]);
                v[e] = arg == me ? gp : 0.f;
            }
        }
        if (gw) {
            const uint4 q = reinterpret_cast<const uint4*>(act + gt_off)[idx];
            const __half2* h = reinterpret_cast<const __half2*>(&q);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = __half22float2(h[j]);
                const float d0 = a[2 * j] - f.x, d1 = a[2 * j + 1] - f.y;
                v[2 * j] += d0 > 0.f ? wk : (d0 < 0.f ? -wk : 0.f);
                v[2 * j + 1] += d1 > 0.f ? wk : (d1 < 0.f ? -wk : 0.f);
            }
        }
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float lo = (mask && !(a[2 * j] > 0.f)) ? 0.f : v[2 * j];
            const float hi = (mask && !(a[2 * j + 1] > 0.f)) ? 0.f : v[2 * j + 1];
            const __nv_bfloat162 b = __floats2bfloat162_rn(lo, hi);
            pk[j] = *reinterpret_cast<const uint32_t*>(&b);
        }
        reinterpret_cast<uint4*>(gout)[idx] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

// Sum |a_sr - a_gt| over one node's maps (fp16, SR batch of `half` elements then GT batch): a fixed grid of kLossBlocks
// blocks, each writing one fp64 partial, so the result does not depend on scheduling (bit-reproducible).
__global__ void __launch_bounds__(256) vgg_l1_partial_kernel(const uint16_t* __restrict__ act, size_t half, double* __restrict__ out) {
    __shared__ double red[8];
    const size_t n8 = half / 8;
    const uint4* a = reinterpret_cast<const uint4*>(act);
    const uint4* b = reinterpret_cast<const uint4*>(act + half);
    double local = 0.0;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n8; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const uint4 qa = a[i], qb = b[i];
        const __half2* ha = reinterpret_cast<const __half2*>(&qa);
        const __half2* hb = reinterpret_cast<const __half2*>(&qb);
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 fa = __half22float2(ha[j]), fb = __half22float2(hb[j]);
            s += fabsf(fa.x - fb.x) + fabsf(fa.y - fb.y);
        }
        local += s;
    }
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < 8; ++i) s += red[i];
        out[blockIdx.x] = s;
    }
}

struct NodeNumel { double inv[kVggConvs]; };
__global__ void vgg_l1_finish_kernel(const double* __restrict__ sums, float* __restrict__ losses, int count, NodeNumel nn) {
    for (int k = threadIdx.x; k < count; k += blockDim.x) {
        double s = 0.0;
        for (int b = 0; b < kLossBlocks; ++b) s += sums[static_cast<size_t>(k) * kLossBlocks + b];
        losses[k] = static_cast<float>(s * nn.inv[k]);
    }
}

// d/d sr of Normalize: the gradient at the normalized input divided by std (in place on the NCHW fp32 result).
__global__ void __launch_bounds__(256) vgg_input_grad_kernel(float* __restrict__ g, int N, int HW, float s0, float s1, float s2) {
    const size_t total = static_cast<size_t>(N) * 3 * HW;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>((i / HW) % 3);
        g[i] = __fdiv_rn(g[i], c == 0 ? s0 : (c == 1 ? s1 : s2));
    }
}

// Input channels [c0, c0 + cn) of an OIHW weight as a contiguous [cout, cn, 3, 3] tensor (a split-K half before packing).
__global__ void __launch_bounds__(256) vgg_cin_slice_kernel(const float* __restrict__ w, float* __restrict__ out, int cout, int cin,
                                                           int c0, int cn) {
    const size_t total = static_cast<size_t>(cout) * cn * 9;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t co = i / (static_cast<size_t>(cn) * 9), rem = i % (static_cast<size_t>(cn) * 9);
        out[i] = w[co * cin * 9 + static_cast<size_t>(c0) * 9 + rem];
    }
}

}  // namespace
}  // namespace resr

using namespace resr;

struct resr_vgg {
    int nodes[kVggConvs];     // conv index of each requested node, in the caller's order
    int nnodes = 0;
    int deepest = -1;
    int node_pos[kVggConvs];  // position of conv i in `nodes`, or -1
    float mean[3], stdv[3];
    int device = -1, num_sms = 148;
    uint8_t* wpack = nullptr;   // forward packs (fp16)
    uint8_t* wpack_t = nullptr; // data-gradient packs (bf16)
    float* bias = nullptr;
    float* zero_bias = nullptr; // second split-K halves and the data-gradient convolutions
    float* slice = nullptr;     // fp32 scratch of one split-K weight half
    bool loaded = false;
    // the forward whose activations the workspace holds (the backward must match it)
    const void* fwd_ws = nullptr;
    int fwd_shape[3] = {0, 0, 0};
};

namespace {

int check_shape(const resr_vgg* v, int n, int h, int w) {
    if (n < 1 || h < 1 || w < 1) return set_error(RESR_E_INVALID, "content loss: empty or negative n / h / w (%d, %d, %d)", n, h, w);
    int pools = 0;
    for (int i = 0; i < v->deepest; ++i) pools += kPoolAfter[i];
    if ((h >> pools) < 1 || (w >> pools) < 1)
        return set_error(RESR_E_INVALID, "content loss: %d x %d leaves no pixel at features.%d (needs at least %d x %d)", h, w,
                         kFeature[v->deepest], 1 << pools, 1 << pools);
    return RESR_OK;
}

int check_device(const resr_vgg* v) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return set_error(RESR_E_CUDA, "content loss: no CUDA device"); }
    if (dev != v->device) return set_error(RESR_E_INVALID, "content loss: handle loaded on device %d, current device is %d", v->device, dev);
    return RESR_OK;
}

int launch_end(const char* what) {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? RESR_OK : set_error(RESR_E_CUDA, "content loss %s: %s", what, cudaGetErrorString(e));
}

// Convolution `i` (forward: fp16 in, fp16 out of the 2N batch; backward: its data gradient, bf16 in and out of the N batch).
// in16 / in_c: the input map and its channel stride. The forward writes out16 (ReLU unless `relu` is 0); the backward
// writes out16 (bf16, ReLU' mask of `mask16` when non-null) or, for conv 0, the NCHW fp32 input gradient out_nchw.
int run_conv(const resr_vgg* v, int i, bool backward, int B, int H, int W, const uint16_t* in16, uint16_t* out16, int relu,
             const uint16_t* mask16, float* out_nchw, float* partial, cudaStream_t s) {
    const Layout& L = layout();
    const int cin = backward ? kCout[i] : kCin[i];
    const int cout = backward ? kCin[i] : kCout[i];
    const PackRef* pk = backward ? L.bwd[i] : L.fwd[i];
    const uint8_t* base = backward ? v->wpack_t : v->wpack;
    const Geo q{H, W};
    ConvIO io;
    io.in16 = in16; io.in_c = i == 0 && !backward ? kInPad : cin;
    io.fmt = backward ? 1 : 0;
    io.nout = pk[0].nout; io.nslices = pk[0].nslices;
    io.out16_fmt = backward ? 1 : 0;
    io.out16_c = cout;
    const bool split = cin > kHalf;
    if (split) {   // first half: fp32 partial (+ bias) of input channels [0, 256)
        ConvIO h0 = io;
        h0.wpack = base + pk[0].off; h0.nchunks = pk[0].nchunks; h0.kvalid = kHalf;
        h0.bias = backward ? v->zero_bias : v->bias + L.b_off[i];
        h0.outf = partial; h0.outf_c = cout;
        RESR_TRY(launch_conv_io(v->num_sms, q, B, h0, s));
        io.in16 = in16 + kHalf;
        io.ep_mode = EP_SKIP; io.res1 = partial; io.res1_c = cout;
    }
    const PackRef& p = pk[split ? 1 : 0];
    io.wpack = base + p.off; io.nchunks = p.nchunks; io.kvalid = split ? kHalf : cin;
    io.bias = backward || split ? v->zero_bias : v->bias + L.b_off[i];
    if (out_nchw) {
        io.out_nchw = out_nchw; io.out_nchw_c = cout;
    } else {
        io.out16 = out16;
        io.relu = relu;
        if (mask16) { io.mask16 = mask16; io.mask16_c = cout; io.mask16_relu = 1; }
    }
    return launch_conv_io(v->num_sms, q, B, io, s);
}

}  // namespace

extern "C" {

size_t resr_vgg_num_params(void) { return layout().n_params; }

int resr_vgg_create(resr_vgg_t** out, const int* features_host, int count, const float* mean_host, const float* std_host) {
    if (!out || !features_host || !mean_host || !std_host) return set_error(RESR_E_INVALID, "content loss: null argument");
    if (count < 1 || count > kVggConvs) return set_error(RESR_E_INVALID, "content loss: 1 to 16 nodes (got %d)", count);
    resr_vgg v;
    for (int i = 0; i < kVggConvs; ++i) v.node_pos[i] = -1;
    for (int k = 0; k < count; ++k) {
        int conv = -1;
        for (int i = 0; i < kVggConvs; ++i)
            if (kFeature[i] == features_host[k]) conv = i;
        if (conv < 0) return set_error(RESR_E_INVALID, "content loss: features.%d is not a VGG19 convolution output", features_host[k]);
        if (v.node_pos[conv] >= 0) return set_error(RESR_E_INVALID, "content loss: features.%d requested twice", features_host[k]);
        v.node_pos[conv] = k;
        v.nodes[k] = conv;
        if (conv > v.deepest) v.deepest = conv;
    }
    v.nnodes = count;
    for (int c = 0; c < 3; ++c) {
        if (!(std_host[c] != 0.f) || !std::isfinite(std_host[c]) || !std::isfinite(mean_host[c]))
            return set_error(RESR_E_INVALID, "content loss: normalize mean must be finite and std finite and non-zero");
        v.mean[c] = mean_host[c];
        v.stdv[c] = std_host[c];
    }
    *out = new resr_vgg(v);
    return RESR_OK;
}

void resr_vgg_destroy(resr_vgg_t* v) {
    if (!v) return;
    cudaFree(v->wpack);
    cudaFree(v->wpack_t);
    cudaFree(v->bias);
    cudaFree(v->zero_bias);
    cudaFree(v->slice);
    delete v;
}

int resr_vgg_load_params(resr_vgg_t* v, const float* flat_params, void* stream) {
    if (!v || !flat_params) return set_error(RESR_E_INVALID, "content loss: null argument");
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        cudaGetLastError();
        return set_error(RESR_E_CUDA, "content loss: no CUDA device");
    }
    if (prop.major != 10) return set_error(RESR_E_CUDA, "libresr needs an sm_100a device (found sm_%d%d)", prop.major, prop.minor);
    const Layout& L = layout();
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (v->device != dev) {   // first load, or the caller moved the parameters to another device
        if (v->device >= 0) cudaStreamSynchronize(s);
        cudaFree(v->wpack); cudaFree(v->wpack_t); cudaFree(v->bias); cudaFree(v->zero_bias); cudaFree(v->slice);
        v->wpack = v->wpack_t = nullptr; v->bias = v->zero_bias = v->slice = nullptr;
        v->loaded = false;
        v->fwd_ws = nullptr;
        if (cudaMalloc(&v->wpack, L.fwd_bytes) != cudaSuccess || cudaMalloc(&v->wpack_t, L.bwd_bytes) != cudaSuccess ||
            cudaMalloc(&v->bias, L.bias_floats * 4) != cudaSuccess || cudaMalloc(&v->zero_bias, 512 * 4) != cudaSuccess ||
            cudaMalloc(&v->slice, static_cast<size_t>(512) * kHalf * 9 * 4) != cudaSuccess) {
            cudaGetLastError();
            return set_error(RESR_E_CUDA, "content loss: cudaMalloc of the packed weights failed");
        }
        cudaMemsetAsync(v->zero_bias, 0, 512 * 4, s);
        v->device = dev;
        v->num_sms = prop.multiProcessorCount;
    }
    for (int i = 0; i < kVggConvs; ++i) {
        const float* w = flat_params + L.p_off[i];
        const float* b = w + static_cast<size_t>(kCout[i]) * kCin[i] * 9;
        if (kCin[i] <= kHalf) {
            const PackRef& p = L.fwd[i][0];
            launch_pack_conv(w, b, reinterpret_cast<uint16_t*>(v->wpack + p.off), v->bias + L.b_off[i], kCin[i], kCout[i], p.nout,
                             p.nslices, p.nchunks, 0, 0, s);
        } else {
            for (int h = 0; h < 2; ++h) {   // the scratch is reused: stream order serialises slice -> pack -> next slice
                const PackRef& p = L.fwd[i][h];
                const size_t n = static_cast<size_t>(kCout[i]) * kHalf * 9;
                vgg_cin_slice_kernel<<<grid_for(n, 256), 256, 0, s>>>(w, v->slice, kCout[i], kCin[i], h * kHalf, kHalf);
                launch_pack_conv(v->slice, h == 0 ? b : nullptr, reinterpret_cast<uint16_t*>(v->wpack + p.off),
                                 h == 0 ? v->bias + L.b_off[i] : nullptr, kHalf, kCout[i], p.nout, p.nslices, p.nchunks, 0, 0, s);
            }
        }
        // data-gradient packs: Cout halves of an OIHW weight are contiguous blocks of output channels
        const int bh = kCout[i] > kHalf ? 2 : 1;
        for (int h = 0; h < bh; ++h) {
            const PackRef& p = L.bwd[i][h];
            const int co = kCout[i] / bh;
            launch_pack_conv(w + static_cast<size_t>(h) * co * kCin[i] * 9, nullptr, reinterpret_cast<uint16_t*>(v->wpack_t + p.off),
                             nullptr, kCin[i], co, p.nout, p.nslices, p.nchunks, 1, 1, s);
        }
    }
    RESR_TRY(launch_end("weight packing"));
    v->loaded = true;
    return RESR_OK;
}

size_t resr_vgg_workspace_bytes(const resr_vgg_t* v, int n, int h, int w) {
    if (!v || check_shape(v, n, h, w) != RESR_OK) return 0;
    return vgg_ws(n, h, w, v->deepest).total;
}

int resr_vgg_forward(resr_vgg_t* v, const float* sr, const float* gt, float* losses, int n, int h, int w, void* workspace,
                     size_t workspace_bytes, void* stream) {
    if (!v || !sr || !gt || !losses || !workspace) return set_error(RESR_E_INVALID, "content loss: null argument");
    RESR_TRY(check_shape(v, n, h, w));
    const VggWs L = vgg_ws(n, h, w, v->deepest);
    if (workspace_bytes < L.total)
        return set_error(RESR_E_INVALID, "content loss: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    if (reinterpret_cast<uintptr_t>(workspace) % 1024 != 0) return set_error(RESR_E_INVALID, "content loss: workspace must be 1024-byte aligned");
    if (!v->loaded) return set_error(RESR_E_INVALID, "content loss: resr_vgg_load_params has not run");
    RESR_TRY(check_device(v));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* base = static_cast<uint8_t*>(workspace);
    auto buf16 = [&](size_t off) { return reinterpret_cast<uint16_t*>(base + off); };
    float* partial = reinterpret_cast<float*>(base + L.partial);
    double* sums = reinterpret_cast<double*>(base + L.sums);
    const int B = 2 * n;
    v->fwd_ws = nullptr;   // a failure below leaves no forward for a backward to use

    const size_t npix = static_cast<size_t>(B) * h * w;
    vgg_normalize_kernel<<<grid_for(npix, 256), 256, 0, s>>>(sr, gt, buf16(L.xin), n, h * w, v->mean[0], v->mean[1], v->mean[2],
                                                            v->stdv[0], v->stdv[1], v->stdv[2]);
    RESR_TRY(launch_end("normalize"));
    const uint16_t* in = buf16(L.xin);
    NodeNumel nn;
    for (int i = 0; i <= v->deepest; ++i) {
        const int H = L.h[i], W = L.w[i];
        uint16_t* act = buf16(L.act[i]);
        RESR_TRY(run_conv(v, i, false, B, H, W, in, act, i != v->deepest, nullptr, nullptr, partial, s));
        const int k = v->node_pos[i];
        if (k >= 0) {
            const size_t half = static_cast<size_t>(n) * H * W * kCout[i];
            vgg_l1_partial_kernel<<<kLossBlocks, 256, 0, s>>>(act, half, sums + static_cast<size_t>(k) * kLossBlocks);
            RESR_TRY(launch_end("node loss"));
            nn.inv[k] = 1.0 / static_cast<double>(half);
        }
        in = act;
        if (kPoolAfter[i] && i < v->deepest) {
            uint16_t* pooled = buf16(L.pool[i]);
            const size_t total = static_cast<size_t>(B) * (H / 2) * (W / 2) * (kCout[i] / 8);
            vgg_maxpool_kernel<<<grid_for(total, 256), 256, 0, s>>>(act, pooled, B, H, W, kCout[i]);
            RESR_TRY(launch_end("max-pool"));
            in = pooled;
        }
    }
    vgg_l1_finish_kernel<<<1, 32, 0, s>>>(sums, losses, v->nnodes, nn);
    RESR_TRY(launch_end("loss"));
    v->fwd_ws = workspace;
    v->fwd_shape[0] = n; v->fwd_shape[1] = h; v->fwd_shape[2] = w;
    return RESR_OK;
}

int resr_vgg_backward(resr_vgg_t* v, const float* grad_losses, float* grad_sr, int n, int h, int w, void* workspace,
                      size_t workspace_bytes, void* stream) {
    if (!v || !grad_losses || !grad_sr || !workspace) return set_error(RESR_E_INVALID, "content loss: null argument");
    RESR_TRY(check_shape(v, n, h, w));
    const VggWs L = vgg_ws(n, h, w, v->deepest);
    if (workspace_bytes < L.total)
        return set_error(RESR_E_INVALID, "content loss: workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
    if (v->fwd_ws != workspace || v->fwd_shape[0] != n || v->fwd_shape[1] != h || v->fwd_shape[2] != w)
        return set_error(RESR_E_INVALID, "content loss: the workspace holds no forward of this handle at %d x 3 x %d x %d", n, h, w);
    RESR_TRY(check_device(v));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* base = static_cast<uint8_t*>(workspace);
    auto buf16 = [&](size_t off) { return reinterpret_cast<uint16_t*>(base + off); };
    float* partial = reinterpret_cast<float*>(base + L.partial);
    uint16_t* g[2] = {buf16(L.g[0]), buf16(L.g[1])};
    int cur = 0;

    auto node_bwd = [&](int i, const uint16_t* gin, int pool, uint16_t* gout) {
        const int k = v->node_pos[i];
        const int H = L.h[i], W = L.w[i];
        const size_t total = static_cast<size_t>(n) * H * W * (kCout[i] / 8);
        const float inv = k >= 0 ? static_cast<float>(1.0 / (static_cast<double>(n) * H * W * kCout[i])) : 0.f;
        vgg_node_bwd_kernel<<<grid_for(total, 256), 256, 0, s>>>(gin, buf16(L.act[i]), k >= 0 ? grad_losses + k : nullptr, inv,
                                                                 i != v->deepest, pool, gout, n, H, W, kCout[i]);
        return launch_end("node backward");
    };
    // the deepest node: its loss term alone (no ReLU follows it)
    RESR_TRY(node_bwd(v->deepest, nullptr, 0, g[cur]));
    for (int i = v->deepest; i >= 0; --i) {
        const int H = L.h[i], W = L.w[i];
        if (i == 0) {
            RESR_TRY(run_conv(v, 0, true, n, H, W, g[cur], nullptr, 0, nullptr, grad_sr, partial, s));
            const size_t total = static_cast<size_t>(n) * 3 * H * W;
            vgg_input_grad_kernel<<<grid_for(total, 256), 256, 0, s>>>(grad_sr, n, H * W, v->stdv[0], v->stdv[1], v->stdv[2]);
            return launch_end("input gradient");
        }
        const int prev = i - 1;
        if (!kPoolAfter[prev] && v->node_pos[prev] < 0) {
            // ReLU' of conv i-1 fused into the data-gradient epilogue (the SR half of its saved output is the mask)
            RESR_TRY(run_conv(v, i, true, n, H, W, g[cur], g[1 - cur], 0, buf16(L.act[prev]), nullptr, partial, s));
            cur = 1 - cur;
        } else {
            RESR_TRY(run_conv(v, i, true, n, H, W, g[cur], g[1 - cur], 0, nullptr, nullptr, partial, s));
            RESR_TRY(node_bwd(prev, g[1 - cur], kPoolAfter[prev], g[cur]));
        }
    }
    return RESR_OK;
}

}  // extern "C"
