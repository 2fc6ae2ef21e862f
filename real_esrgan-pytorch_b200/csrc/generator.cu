// RRDBNet x4 generator forward: host orchestration + layout / weight-packing kernels + C ABI.
// Reference: /root/reference/model.py:64-132 (RDB, RRDB), :206-275 (Generator). See DESIGN.md §3-4.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/resr.h"
#include "conv3x3.cuh"
#include "errors.h"
#include "gen_internal.cuh"

namespace resr {

// ------------------------------------------------------------------------------------------- small kernels

// OIHW fp32 -> [slice][chunk][dx][n = dy*NOUT + co][64 ch] 16-bit with the 128B shared-memory swizzle applied, so a
// plain bulk copy drops a ready-to-use UMMA B operand into shared memory.
__device__ __forceinline__ void pack_conv_body(const float* __restrict__ w, const float* __restrict__ bias, uint16_t* __restrict__ wp,
                                               float* __restrict__ bp, int cin, int cout, int nout, int nslices, int nchunks, int fmt,
                                               int transposed, size_t first, size_t stride) {
    const int NT = 3 * nout;
    const size_t total = static_cast<size_t>(nslices) * nchunks * 3 * NT * 64;
    for (size_t idx = first; idx < total; idx += stride) {   // (a layer's pack has < 2^32 elements: 32-bit index decoding)
        const int k = static_cast<int>(idx & 63);
        unsigned t = static_cast<unsigned>(idx >> 6);
        const int n = t % NT;
        t /= NT;
        const int dx = t % 3;
        t /= 3;
        const int chunk = t % nchunks;
        const int slice = static_cast<int>(t / nchunks);
        const int co = slice * nout + n % nout;
        const int dy = n / nout;
        const int ci = chunk * 64 + k;
        float v = 0.f;
        if (!transposed) {
            if (co < cout && ci < cin) v = w[((static_cast<size_t>(co) * cin + ci) * 3 + dy) * 3 + dx];
        } else {
            // data-gradient convolution: its output channel `co` is a forward INPUT channel, its input channel `ci` a
            // forward OUTPUT channel, taps flipped
            if (co < cin && ci < cout) v = w[((static_cast<size_t>(ci) * cin + co) * 3 + (2 - dy)) * 3 + (2 - dx)];
        }
        uint16_t bits;
        if (fmt == 1) {
            __nv_bfloat16 h = __float2bfloat16_rn(v);
            bits = *reinterpret_cast<uint16_t*>(&h);
        } else {
            __half h = __float2half_rn(v);
            bits = *reinterpret_cast<uint16_t*>(&h);
        }
        const size_t tile = ((static_cast<size_t>(slice) * nchunks + chunk) * 3 + dx) * NT * 64;  // elements
        const size_t off = tile + static_cast<size_t>(n) * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7));
        wp[off] = bits;
    }
    const int nb = nslices * nout;
    if (bp)
        for (size_t i = first; i < static_cast<size_t>(nb); i += stride) bp[i] = (i < static_cast<size_t>(cout) && bias) ? bias[i] : 0.f;
}

__global__ void pack_conv_kernel(const float* __restrict__ w, const float* __restrict__ bias, uint16_t* __restrict__ wp,
                                 float* __restrict__ bp, int cin, int cout, int nout, int nslices, int nchunks, int fmt,
                                 int transposed) {
    pack_conv_body(w, bias, wp, bp, cin, cout, nout, nslices, nchunks, fmt, transposed,
                   blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x, static_cast<size_t>(gridDim.x) * blockDim.x);
}

// All layers in one launch (blockIdx.y = layer): the repack after every optimizer step is 2 launches instead of 701.
struct PackJob {
    unsigned long long p_off, w_off, b_off;  // floats into the flat parameter vector, bytes into the pack, floats into the bias
    int cin, cout, nout, nslices, nchunks, fmt;
};
__global__ void __launch_bounds__(256) pack_all_kernel(const float* __restrict__ flat, const PackJob* __restrict__ jobs,
                                                       uint8_t* __restrict__ wpack, float* __restrict__ bias, int transposed) {
    const PackJob j = jobs[blockIdx.y];
    const float* w = flat + j.p_off;
    const float* b = w + static_cast<size_t>(j.cout) * j.cin * 9;
    pack_conv_body(w, transposed ? nullptr : b, reinterpret_cast<uint16_t*>(wpack + j.w_off), transposed ? nullptr : bias + j.b_off,
                   j.cin, j.cout, j.nout, j.nslices, j.nchunks, j.fmt, transposed,
                   blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x, static_cast<size_t>(gridDim.x) * blockDim.x);
}

// Data-gradient packs of a dense block in "mirrored dense block" form (train.cu backward): step b (4, 3, 2, 1, 0) maps
//     dYcat' = [dY5 (64) | dY4 (32) | dY3 | dY2 | dY1]   (its first 64 + 32 * (4 - b) channels = the layers AFTER block b)
// to the gradient of concat-buffer block b (b = 0: the block input x, 64 channels; b >= 1: out_b, 32 channels):
//     W'_b[co'][ci'][dy][dx] = W_l[co_l][cin_index(b, co')][2 - dy][2 - dx],   (l, co_l) = the layer / channel ci' belongs to.
// Step b has exactly the shape of forward layer conv(5 - b) (Cin 64 / 96 / 128 / 160 / 192, Cout 32 / 32 / 32 / 32 / 64), so
// its tiles are stored at that layer's pack offset in a second pack buffer. blockIdx.y = step, blockIdx.z = dense block.
__global__ void __launch_bounds__(256) pack_rdb_bwd_kernel(const float* __restrict__ flat, const PackJob* __restrict__ jobs,
                                                          uint8_t* __restrict__ wpack) {
    const int r = blockIdx.z, b = 4 - static_cast<int>(blockIdx.y);     // blockIdx.y = 0..4 <-> b = 4..0 <-> forward shape conv1..conv5
    const PackJob shape = jobs[1 + 5 * r + blockIdx.y];                 // pack geometry (offset, nout, nslices, nchunks) of that shape
    const int cin_p = 64 + 32 * (4 - b);                                // channels of dYcat' this step reads
    const int cout_p = b == 0 ? 64 : 32;
    const int NT = 3 * shape.nout;
    uint16_t* wp = reinterpret_cast<uint16_t*>(wpack + shape.w_off);
    const size_t total = static_cast<size_t>(shape.nslices) * shape.nchunks * 3 * NT * 64;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int k = static_cast<int>(idx & 63);
        unsigned t = static_cast<unsigned>(idx >> 6);   // (a layer's pack has < 2^32 elements: 32-bit index decoding)
        const int n = t % NT;
        t /= NT;
        const int dx = t % 3;
        t /= 3;
        const int chunk = t % shape.nchunks;
        const int slice = static_cast<int>(t / shape.nchunks);
        const int co = slice * shape.nout + n % shape.nout;   // channel inside concat block b
        const int dy = n / shape.nout;
        const int ci = chunk * 64 + k;                          // channel of dYcat'
        float v = 0.f;
        if (co < cout_p && ci < cin_p) {
            const int l = ci < 64 ? 5 : 4 - (ci - 64) / 32;     // forward layer (1..5) whose output gradient this channel is
            const int co_l = ci < 64 ? ci : (ci - 64) % 32;
            const int cin_l = 64 + 32 * (l - 1);
            const int cin_idx = b == 0 ? co : 64 + 32 * (b - 1) + co;   // input channel of layer l that is block b's channel co
            const PackJob lay = jobs[1 + 5 * r + (l - 1)];
            v = flat[lay.p_off + ((static_cast<size_t>(co_l) * cin_l + cin_idx) * 3 + (2 - dy)) * 3 + (2 - dx)];
        }
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        const size_t tile = ((static_cast<size_t>(slice) * shape.nchunks + chunk) * 3 + dx) * NT * 64;  // elements
        wp[tile + static_cast<size_t>(n) * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7))] = *reinterpret_cast<const uint16_t*>(&h);
    }
}

// NCHW fp32 -> NHWC 16-bit with channels zero-padded to c_pad (multiple of 8).
__global__ void nchw_to_nhwc16_kernel(const float* __restrict__ x, uint16_t* __restrict__ out, int N, int C, int H, int W,
                                      int c_pad, int fmt) {
    const size_t npix = static_cast<size_t>(N) * H * W;
    const int groups = c_pad / 8;
    const size_t total = npix * groups;
    const size_t plane = static_cast<size_t>(H) * W;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int gch = idx % groups;
        const size_t pix = idx / groups;
        const size_t n = pix / plane, rem = pix % plane;
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = gch * 8 + 2 * j + e;
                v[e] = c < C ? x[(n * C + c) * plane + rem] : 0.f;
            }
            if (fmt == 1) {
                __nv_bfloat162 h = __floats2bfloat162_rn(v[0], v[1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&h);
            } else {
                __half2 h = __floats2half2_rn(v[0], v[1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&h);
            }
        }
        reinterpret_cast<uint4*>(out + pix * c_pad)[gch] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

// NHWC u8 image -> NHWC 16-bit with channels zero-padded to c_pad: image_to_tensor (imgproc.py:1557: to_tensor = / 255 in
// fp32) fused with the layout change of the first convolution's input.
__global__ void u8nhwc_to_nhwc16_kernel(const unsigned char* __restrict__ x, uint16_t* __restrict__ out, size_t npix, int C, int c_pad,
                                        int fmt) {
    const int groups = c_pad / 8;
    const size_t total = npix * groups;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int gch = idx % groups;
        const size_t pix = idx / groups;
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float v[2];
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = gch * 8 + 2 * j + e;
                v[e] = c < C ? __fdiv_rn(static_cast<float>(x[pix * C + c]), 255.f) : 0.f;
            }
            if (fmt == 1) {
                __nv_bfloat162 h = __floats2bfloat162_rn(v[0], v[1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&h);
            } else {
                __half2 h = __floats2half2_rn(v[0], v[1]);
                pk[j] = *reinterpret_cast<uint32_t*>(&h);
            }
        }
        reinterpret_cast<uint4*>(out + pix * c_pad)[gch] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

// imgproc.tensor_to_image (imgproc.py:1570-1596) on the device: NCHW float -> HWC u8 of image 0.
__global__ void tensor_to_image_kernel(const float* __restrict__ x, unsigned char* __restrict__ out, int C, size_t HW, int range_norm,
                                       int half) {
    const size_t total = HW * C;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int c = idx % C;
        const size_t p = idx / C;
        float v = x[static_cast<size_t>(c) * HW + p];
        if (range_norm) v = __fdiv_rn(__fadd_rn(v, 1.f), 2.f);            // imgproc.py:1587-1588
        if (half) {                                                        // :1591-1592: the arithmetic then runs in fp16
            const __half h = __hmul(__float2half_rn(v), __float2half_rn(255.f));
            v = fminf(fmaxf(__half2float(h), 0.f), 255.f);
        } else {
            v = fminf(fmaxf(__fmul_rn(v, 255.f), 0.f), 255.f);              // :1594
        }
        out[idx] = static_cast<unsigned char>(v);                           // astype("uint8"): truncation
    }
}

// ------------------------------------------------------------------------------------------- packed canvas
// resr_generator_forward_many runs a list of differently sized images as ONE N = 1 forward over a canvas that holds
// them side by side with at least one zero LR pixel between neighbours (DESIGN.md §3.2). Every convolution writes 0 at
// each canvas pixel outside an image (ConvArgs::vmask), so the gutters act as each image's own zero padding.

// One image of a canvas call (device table in the workspace, sorted by (y0, x0): shelf by shelf, left to right).
struct CanvasImage {
    const void* src;   // fp32 NCHW [3, h, w] or u8 NHWC [h, w, 3]
    void* dst;         // fp32 NCHW [3, 4h, 4w] or u8 NHWC [4h, 4w, 3]
    int x0, y0, h, w;  // LR rectangle on the canvas
};

// Index of the image covering LR canvas pixel (x, y), or -1. Relies on the shelf layout of canvas_pack: the images of a
// shelf share y0 and every later shelf starts below the bottom of every earlier image.
__device__ __forceinline__ int canvas_owner(const CanvasImage* __restrict__ im, int count, int x, int y) {
    int lo = 0, hi = count;   // first image with y0 > y
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (im[mid].y0 <= y) lo = mid + 1; else hi = mid;
    }
    if (lo == 0) return -1;
    const int sy = im[lo - 1].y0;   // the shelf that may hold row y
    int a = 0, b = lo;              // first image after (sy, x) in (y0, x0) order
    while (a < b) {
        const int mid = (a + b) >> 1;
        if (im[mid].y0 < sy || (im[mid].y0 == sy && im[mid].x0 <= x)) a = mid + 1; else b = mid;
    }
    const int i = a - 1;
    if (i < 0) return -1;
    const CanvasImage& c = im[i];
    return (x >= c.x0 && x < c.x0 + c.w && y >= c.y0 && y < c.y0 + c.h) ? i : -1;
}

__device__ __forceinline__ uint32_t pack2_16(float a, float b, int fmt) {
    if (fmt == 1) {
        __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    }
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

// Canvas input: every LR canvas pixel gets its 64-channel 16-bit NHWC value -- the image's 3 channels converted as
// nchw_to_nhwc16_kernel (fp32) / u8nhwc_to_nhwc16_kernel (u8: / 255 in fp32) do, zero in the gutters and margins -- and
// the valid-pixel bitmap the convolution epilogues read. cw % 32 == 0 and the stride is a multiple of 32, so a warp
// always covers 32 pixels of one row and its ballot is one bitmap word.
__global__ void canvas_gather_kernel(const CanvasImage* __restrict__ im, int count, int cw, size_t npix, int u8, int fmt,
                                     uint16_t* __restrict__ xin, uint32_t* __restrict__ vmask) {
    for (size_t p = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; p < npix;
         p += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int y = static_cast<int>(p / cw), x = static_cast<int>(p % cw);
        const int i = canvas_owner(im, count, x, y);
        float v[3] = {0.f, 0.f, 0.f};
        if (i >= 0) {
            const CanvasImage c = im[i];
            const size_t q = static_cast<size_t>(y - c.y0) * c.w + (x - c.x0);
            if (u8) {
                const unsigned char* s = static_cast<const unsigned char*>(c.src) + q * 3;
#pragma unroll
                for (int k = 0; k < 3; ++k) v[k] = __fdiv_rn(static_cast<float>(s[k]), 255.f);
            } else {
                const float* s = static_cast<const float*>(c.src) + q;
                const size_t plane = static_cast<size_t>(c.h) * c.w;
#pragma unroll
                for (int k = 0; k < 3; ++k) v[k] = s[k * plane];
            }
        }
        uint4* o = reinterpret_cast<uint4*>(xin + p * 64);
        o[0] = make_uint4(pack2_16(v[0], v[1], fmt), pack2_16(v[2], 0.f, fmt), 0u, 0u);
#pragma unroll
        for (int k = 1; k < 8; ++k) o[k] = make_uint4(0u, 0u, 0u, 0u);
        const unsigned word = __ballot_sync(0xffffffffu, i >= 0);
        if ((threadIdx.x & 31) == 0) vmask[p >> 5] = word;
    }
}

// Canvas output -> each image's own tensor: its 4h x 4w region of conv4's fp32 NCHW [1, 3, 4ch, 4cw] or u8 NHWC
// [4ch, 4cw, 3] canvas. blockIdx.y = image.
__global__ void canvas_scatter_kernel(const CanvasImage* __restrict__ im, const void* __restrict__ canvas, int ch, int cw, int u8) {
    const CanvasImage c = im[blockIdx.y];
    const int H4 = 4 * c.h, W4 = 4 * c.w;
    const size_t W4c = static_cast<size_t>(4) * cw;
    const size_t total = static_cast<size_t>(H4) * W4 * 3;
    for (size_t e = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; e < total;
         e += static_cast<size_t>(gridDim.x) * blockDim.x) {
        if (u8) {
            const size_t pix = e / 3;
            const int k = static_cast<int>(e % 3);
            const size_t yy = pix / W4, xx = pix % W4;
            static_cast<unsigned char*>(c.dst)[e] =
                static_cast<const unsigned char*>(canvas)[((4 * static_cast<size_t>(c.y0) + yy) * W4c + 4 * static_cast<size_t>(c.x0) + xx) * 3 + k];
        } else {
            const size_t xx = e % W4, t = e / W4;
            const size_t yy = t % H4, k = t / H4;
            static_cast<float*>(c.dst)[e] =
                static_cast<const float*>(canvas)[(k * 4 * ch + 4 * static_cast<size_t>(c.y0) + yy) * W4c + 4 * static_cast<size_t>(c.x0) + xx];
        }
    }
}

// Shelf packer of resr_canvas_pack: images tallest first (ties: wider first, then input order), left to right on shelves
// that are as tall as their first image. Neighbours keep one zero pixel between them, to the right and below; the canvas
// edge needs none (the convolutions' tensor maps zero-fill outside the tensor). max_width <= 0 picks a near-square canvas.
// The canvas size is rounded up to multiples of kCanvasRows x kCanvasCols, so varied lists share a few plans.
static const int kCanvasRows = 16, kCanvasCols = 128, kCanvasMaxSide = 16384;
static int canvas_pack(const int* hs, const int* ws, int count, int max_width, int* x0, int* y0, int* canvas_h, int* canvas_w) {
    if (!hs || !ws || !x0 || !y0 || !canvas_h || !canvas_w || count <= 0) return set_error(RESR_E_INVALID, "canvas_pack: bad argument");
    long long area = 0;
    int wmax = 0;
    for (int i = 0; i < count; ++i) {
        if (hs[i] <= 0 || ws[i] <= 0 || hs[i] > kCanvasMaxSide || ws[i] > kCanvasMaxSide)
            return set_error(RESR_E_INVALID, "canvas_pack: image %d has size %dx%d (1..%d per side)", i, hs[i], ws[i], kCanvasMaxSide);
        area += static_cast<long long>(hs[i] + 1) * (ws[i] + 1);
        wmax = std::max(wmax, ws[i]);
    }
    long long limit = max_width;
    if (max_width <= 0) {
        limit = std::max<long long>(static_cast<long long>(std::ceil(std::sqrt(static_cast<double>(area)))), wmax);
        limit = (limit + kCanvasCols - 1) / kCanvasCols * kCanvasCols;   // the whole bucket is computed anyway
    } else if (wmax > max_width) {
        return set_error(RESR_E_INVALID, "canvas_pack: an image is %d wide, the width limit is %d", wmax, max_width);
    }
    std::vector<int> order(count);
    for (int i = 0; i < count; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return hs[a] != hs[b] ? hs[a] > hs[b] : ws[a] > ws[b]; });
    long long x = 0, y = 0, shelf_h = 0, used_w = 0;
    for (int i : order) {
        if (x > 0 && x + ws[i] > limit) {   // next shelf, one gutter row below the tallest image of this one
            y += shelf_h + 1;
            x = 0;
            shelf_h = 0;
        }
        x0[i] = static_cast<int>(x);
        y0[i] = static_cast<int>(y);
        shelf_h = std::max<long long>(shelf_h, hs[i]);
        used_w = std::max(used_w, x + ws[i]);
        x += ws[i] + 1;
    }
    const long long H = (y + shelf_h + kCanvasRows - 1) / kCanvasRows * kCanvasRows;
    const long long W = (used_w + kCanvasCols - 1) / kCanvasCols * kCanvasCols;
    if (H > kCanvasMaxSide || W > kCanvasMaxSide)
        return set_error(RESR_E_INVALID, "canvas_pack: canvas %lldx%lld exceeds %d per side; split the list", H, W, kCanvasMaxSide);
    *canvas_h = static_cast<int>(H);
    *canvas_w = static_cast<int>(W);
    return RESR_OK;
}

int grid_for(size_t total, int block) {
    size_t g = (total + block - 1) / block;
    if (g > 148 * 16) g = 148 * 16;
    if (g < 1) g = 1;
    return static_cast<int>(g);
}

// Packs every layer from the flat parameter vector: forward packs (+ padded biases) or the transposed data-gradient packs.
int launch_pack_all(resr_generator* g, const float* flat, int transposed, cudaStream_t s) {
    const Table& T = table();
    PackJob** slot = reinterpret_cast<PackJob**>(transposed ? &g->pack_jobs_t : &g->pack_jobs);
    if (!*slot) {
        std::vector<PackJob> h(kNumConvs);
        for (int k = 0; k < kNumConvs; ++k) {
            const ConvSpec& c = T.c[k];
            PackJob& j = h[k];
            j.p_off = c.p_off;
            j.cin = c.cin; j.cout = c.cout;
            if (!transposed) {
                j.w_off = c.w_off; j.b_off = c.b_off; j.nout = c.nout; j.nslices = c.nslices; j.nchunks = c.nchunks;
                j.fmt = g->precision == 1 ? 1 : c.fmt;
            } else {
                j.w_off = c.wt_off; j.b_off = 0; j.nout = 32; j.nslices = c.t_nslices; j.nchunks = c.t_nchunks; j.fmt = 1;
            }
        }
        if (cudaMalloc(slot, kNumConvs * sizeof(PackJob)) != cudaSuccess) return -1;
        cudaMemcpyAsync(*slot, h.data(), kNumConvs * sizeof(PackJob), cudaMemcpyHostToDevice, s);
        cudaStreamSynchronize(s);  // h is a local
    }
    // conv 0 (3 -> 64) never needs its input gradient: the transposed table is launched from layer 1
    const int first = transposed ? 1 : 0;
    pack_all_kernel<<<dim3(24, kNumConvs - first), 256, 0, s>>>(flat, *slot + first, transposed ? g->wpack_t : g->wpack, g->bias,
                                                                transposed);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

// The mirrored dense-block data-gradient packs of all 69 blocks (needs the forward pack-job table on the device).
int launch_pack_rdb_bwd(resr_generator* g, const float* flat, uint8_t* wpack_t2, cudaStream_t s) {
    if (!g->pack_jobs) return -1;  // built by the forward pack (load_params always runs first)
    pack_rdb_bwd_kernel<<<dim3(8, 5, kNumRRDB * 3), 256, 0, s>>>(flat, static_cast<const PackJob*>(g->pack_jobs), wpack_t2);
    return cudaGetLastError() == cudaSuccess ? 0 : -2;
}

void launch_pack_conv(const float* w, const float* bias, uint16_t* wp, float* bp, int cin, int cout, int nout, int nslices,
                      int nchunks, int fmt, int transposed, cudaStream_t s) {
    const size_t total = static_cast<size_t>(nslices) * nchunks * 3 * (3 * nout) * 64;
    pack_conv_kernel<<<grid_for(total, 256), 256, 0, s>>>(w, bias, wp, bp, cin, cout, nout, nslices, nchunks, fmt, transposed);
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WsLayout {
    size_t xin, c[3], f0, m[4], t1, t2, t3, t4, total;
};
static WsLayout ws_layout(size_t N, size_t H, size_t W, int precision = 0) {
    const size_t P = N * H * W;
    WsLayout L;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o = align_up(o + bytes, 1024);
        return at;
    };
    L.xin = take(P * 64 * 2);
    for (int i = 0; i < 3; ++i) L.c[i] = take(P * 192 * 2);
    L.f0 = take(P * 64 * 4);
    for (int i = 0; i < 4; ++i) L.m[i] = precision == 1 ? take(P * 64 * 4) : 0;  // bf16 recipe: fp32 masters of the residual stream
    L.t1 = take(4 * P * 64 * 2);
    L.t2 = take(16 * P * 64 * 2);
    L.t3 = take(16 * P * 64 * 2);
    L.t4 = take(16 * P * 64 * 2);
    L.total = o;
    return L;
}

// vmask: valid-pixel bitmap of a packed canvas (N == 1, W % 32 == 0; W / 32 words per LR row), or null
static int build_plan(resr_generator* g, Plan& p, int N, int H, int W, void* ws, const uint32_t* vmask, cudaStream_t s) {
    p.valid = false;
    p.steps.clear();
    p.N = N; p.H = H; p.W = W; p.ws = ws;
    p.pair_policy = conv3x3_set_pair_policy(-1);
    const int prec = g->precision;
    const WsLayout L = ws_layout(N, H, W, prec);
    uint8_t* base = static_cast<uint8_t*>(ws);
    uint16_t* xin = reinterpret_cast<uint16_t*>(base + L.xin);
    // three 192-channel concat buffers: [0] holds the RRDB input (and receives the RRDB output in place), [1] / [2] the
    // inputs of its second / third dense block; F0 = fp32 copy of conv1's output for the global skip (model.py:261-262)
    uint16_t* cbuf[3];
    for (int i = 0; i < 3; ++i) cbuf[i] = reinterpret_cast<uint16_t*>(base + L.c[i]);
    float* F0 = reinterpret_cast<float*>(base + L.f0);
    float* M[4];
    for (int i = 0; i < 4; ++i) M[i] = reinterpret_cast<float*>(base + L.m[i]);
    uint16_t* t1 = reinterpret_cast<uint16_t*>(base + L.t1);
    uint16_t* t2 = reinterpret_cast<uint16_t*>(base + L.t2);
    uint16_t* t3 = reinterpret_cast<uint16_t*>(base + L.t3);
    uint16_t* t4 = reinterpret_cast<uint16_t*>(base + L.t4);
    p.xin = xin;

    // (one-time hygiene: no layer reads a channel that has not been written, the activation tensor maps end at Cin).
    // Issued on the CALLER's stream: ordered after whatever forward is still in flight on this workspace and capturable
    // into a CUDA graph (the legacy default stream is neither).
    for (int i = 0; i < 3; ++i) cudaMemsetAsync(cbuf[i], 0, static_cast<size_t>(N) * H * W * 192 * 2, s);

    const Table& T = table();
    int map_rc = 0;
    // in16: source activations [N, H<<s, W<<s, cin_total]
    auto make_step = [&](int conv, int s, const void* in16, int cin_total) {
        const ConvSpec& cs = T.c[conv];
        Step st;
        memset(&st, 0, sizeof(st));
        st.conv = conv;
        ConvArgs& a = st.a;
        conv3x3_init_geometry(&a, N, H << s, W << s, cs.cin, -1);
        a.nchunks = cs.nchunks;
        a.fmt_in = prec == 1 ? 1 : cs.fmt;
        a.wpack = g->wpack + cs.w_off;
        a.bias = g->bias + cs.b_off;
        if (vmask) { a.vmask = vmask; a.vmask_words = W / 32; a.vmask_shift = s; }
        // the input's channels past cs.cin are zeros this library wrote: the map may end at the next multiple of 8
        map_rc |= conv3x3_make_tmap_act(&st.maps.a, in16, N, a.H, a.W, cin_total, a.mode, a.BW, a.BN, (cs.cin + 7) / 8 * 8);
        return st;
    };
    auto set_out16 = [&](Step& st, void* dst, int c_total, int choff, int fmt, int up2) {
        const ConvArgs& a = st.a;
        st.a.has_out16 = 1; st.a.out16_fmt = prec == 1 ? 1 : fmt; st.a.out16_choff = choff; st.a.out16_up2 = up2;
        map_rc |= conv3x3_make_tmap_out16(&st.maps.o16, dst, N, a.H, a.W, c_total, T.c[st.conv].nout, a.BW, a.BN, up2);
    };
    auto set_outf = [&](Step& st, float* dst) {
        const ConvArgs& a = st.a;
        st.a.has_outf = 1; st.a.outf_choff = 0; st.a.outf = static_cast<float*>(dst); st.a.outf_cstride = 64;
        map_rc |= conv3x3_make_tmap_f32(&st.maps.of, dst, N, a.H, a.W, 64, a.BW, a.BN);
    };
    auto set_res1 = [&](Step& st, const float* src) {
        st.a.has_res1 = 1; st.a.res_choff = 0; st.a.res1 = src; st.a.res1_cstride = 64;
    };
    auto push = [&](Step& st) {
        if (!conv3x3_choose(&st.a, T.c[st.conv].nout, T.c[st.conv].nslices, &st.cfg)) map_rc |= 1 << 20;
        // serpentine order: every other pair-kernel launch walks its rows / column groups back to front, so that it starts
        // on what the previous layer touched last (L2-resident) instead of on what it touched first (long evicted)
        st.a.reverse = st.cfg.pair ? static_cast<int>(p.steps.size() & 1) : 0;
        p.steps.push_back(st);
    };

    // 16-bit residual: the trunk's residual stream is the fp16 conv input itself (channels [0, 64) of a concat buffer)
    auto set_res16 = [&](Step& st, const uint16_t* src) {
        st.a.has_res1 = 1; st.a.res_choff = 0; st.a.res1 = src; st.a.res1_cstride = 192;
        st.a.res16 = 1; st.a.res16_fmt = 0;
    };
    int conv = 0;
    {   // conv1: model.py:258
        Step st = make_step(conv, 0, xin, 64);
        st.a.ep_mode = EP_PLAIN;
        set_outf(st, F0);
        set_out16(st, cbuf[0], 192, 0, 0, 0);
        push(st);
        ++conv;
    }
    for (int i = 0; i < kNumRRDB; ++i) {
        for (int j = 0; j < 3; ++j) {
            uint16_t* cin_buf = cbuf[j];
            for (int k = 0; k < 4; ++k) {  // model.py:90-93
                Step st = make_step(conv, 0, cin_buf, 192);
                st.a.ep_mode = EP_PLAIN; st.a.lrelu = 1;
                set_out16(st, cin_buf, 192, 64 + 32 * k, 0, 0);
                push(st);
                ++conv;
            }
            Step st = make_step(conv, 0, cin_buf, 192);  // model.py:94-96 (+ :129-130 for the third RDB)
            st.a.ep_mode = j < 2 ? EP_RDB : EP_RRDB;
            if (prec == 1) {
                // bf16 recipe (north_star): the residual stream is kept in fp32 masters next to the bf16 operands. Dense
                // block t reads master t % 4 (conv1's fp32 output for t = 0) and writes master (t + 1) % 4; the RRDB skip
                // reads the master of the RRDB input, which no block of the same RRDB overwrites.
                const int t = i * 3 + j;
                set_res1(st, t == 0 ? F0 : M[t % 4]);
                if (j == 2) { st.a.res2 = i == 0 ? F0 : M[(3 * i) % 4]; st.a.res2_cstride = 64; }
                set_outf(st, M[(t + 1) % 4]);
            } else {
                set_res16(st, cin_buf);
                if (j == 2) { st.a.res2 = cbuf[0]; st.a.res2_cstride = 192; }
            }
            set_out16(st, cbuf[(j + 1) % 3], 192, 0, 0, 0);
            push(st);
            ++conv;
        }
    }
    {   // conv2 + skip (model.py:260-262), written nearest-upsampled x2 (model.py:264) in fp16
        Step st = make_step(conv, 0, cbuf[0], 192);
        st.a.ep_mode = EP_SKIP;
        set_res1(st, F0);
        set_out16(st, t1, 64, 0, 0, 1);
        push(st);
        ++conv;
    }
    {   // upsampling1 conv + LeakyReLU (model.py:264), output written upsampled x2 again (model.py:265)
        Step st = make_step(conv, 1, t1, 64);
        st.a.lrelu = 1;
        set_out16(st, t2, 64, 0, 0, 1);
        push(st);
        ++conv;
    }
    {   // upsampling2 conv + LeakyReLU (model.py:265)
        Step st = make_step(conv, 2, t2, 64);
        st.a.lrelu = 1;
        set_out16(st, t3, 64, 0, 0, 0);
        push(st);
        ++conv;
    }
    {   // conv3 + LeakyReLU (model.py:267)
        Step st = make_step(conv, 2, t3, 64);
        st.a.lrelu = 1;
        set_out16(st, t4, 64, 0, 0, 0);
        push(st);
        ++conv;
    }
    {   // conv4 + clamp (model.py:268-270): fp32 NCHW result, pointer patched per call
        Step st = make_step(conv, 2, t4, 64);
        st.a.clamp01 = 1;
        st.a.out_nchw = nullptr; st.a.out_nchw_c = 3;
        push(st);
        ++conv;
    }
    if (map_rc != 0) return set_error(RESR_E_CUDA, "tensor map / shared memory planning failed (%d)", map_rc);
    if (cudaGetLastError() != cudaSuccess) return set_error(RESR_E_CUDA, "workspace init failed");
    p.valid = true;
    return RESR_OK;
}

}  // namespace resr

using namespace resr;

extern "C" {

int resr_version(void) { return 1; }

size_t resr_generator_num_params(void) { return table().n_params; }
int resr_generator_num_tensors(void) { return 2 * kNumConvs; }
int resr_generator_launches_per_forward(void) { return 1 + kNumConvs; }

int resr_set_conv_pair_policy(int policy) { return conv3x3_set_pair_policy(policy); }

int resr_generator_tensor_span(int index, size_t* offset, size_t* count) {
    if (index < 0 || index >= 2 * kNumConvs || !offset || !count) return set_error(RESR_E_INVALID, "bad tensor index");
    const ConvSpec& c = table().c[index / 2];
    const size_t wn = static_cast<size_t>(c.cout) * c.cin * 9;
    if (index % 2 == 0) { *offset = c.p_off; *count = wn; }
    else { *offset = c.p_off + wn; *count = c.cout; }
    return RESR_OK;
}

int resr_generator_create(resr_generator_t** out, int in_channels, int out_channels, int upscale_factor) {
    if (!out) return set_error(RESR_E_INVALID, "null out");
    if (in_channels != 3 || out_channels != 3 || upscale_factor != 4)
        return set_error(RESR_E_INVALID, "only Generator(3, 3, 4) is implemented (got %d, %d, %d)", in_channels,
                         out_channels, upscale_factor);
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return set_error(RESR_E_CUDA, "no CUDA device: %s", cudaGetErrorString(cudaGetLastError()));
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return set_error(RESR_E_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10) return set_error(RESR_E_CUDA, "libresr needs an sm_100a device (found sm_%d%d)", prop.major, prop.minor);
    resr_generator* g = new resr_generator();
    g->num_sms = prop.multiProcessorCount;
    if (cudaMalloc(&g->wpack, table().pack_bytes) != cudaSuccess || cudaMalloc(&g->bias, table().bias_floats * 4) != cudaSuccess) {
        delete g;
        return set_error(RESR_E_CUDA, "cudaMalloc of packed weights failed");
    }
    *out = g;
    return RESR_OK;
}

void resr_generator_destroy(resr_generator_t* g) {
    if (!g) return;
    cudaFree(g->wpack);
    cudaFree(g->bias);
    cudaFree(g->wpack_t);
    cudaFree(g->wpack_t2);
    cudaFree(g->pack_jobs);
    cudaFree(g->pack_jobs_t);
    cudaFree(g->zero_bias);
    if (g->step_exec) cudaGraphExecDestroy(g->step_exec);
    if (g->h2d_stream) cudaStreamDestroy(g->h2d_stream);
    if (g->d2h_stream) cudaStreamDestroy(g->d2h_stream);
    for (int i = 0; i < 2; ++i) {
        if (g->ev_h2d[i]) cudaEventDestroy(g->ev_h2d[i]);
        if (g->ev_fwd[i]) cudaEventDestroy(g->ev_fwd[i]);
        if (g->ev_d2h[i]) cudaEventDestroy(g->ev_d2h[i]);
    }
    if (g->side_stream) cudaStreamDestroy(g->side_stream);
    if (g->ev_fork) cudaEventDestroy(g->ev_fork);
    if (g->ev_dy) cudaEventDestroy(g->ev_dy);
    if (g->ev_join) cudaEventDestroy(g->ev_join);
    for (int i = 0; i < 3; ++i)
        if (g->ev_dyc[i]) cudaEventDestroy(g->ev_dyc[i]);
    for (int i = 0; i < 4; ++i)
        if (g->ev_bucket[i]) cudaEventDestroy(g->ev_bucket[i]);
    delete g;
}

int resr_generator_load_params(resr_generator_t* g, const float* flat, void* stream) {
    if (!g || !flat) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const Table& T = table();
    if (launch_pack_all(g, flat, 0, s) != 0) return set_error(RESR_E_CUDA, "weight packing failed");
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "pack kernels: %s", cudaGetErrorString(e));
    g->loaded = true;
    g->packed_t = false;
    g->flat_params = flat;
    ensure_transposed_packs(g, s, false);  // training handles keep the data-gradient packs in step with the weights
    return RESR_OK;
}

size_t resr_generator_workspace_bytes(int n, int h, int w) {
    if (n <= 0 || h <= 0 || w <= 0) return 0;
    return ws_layout(n, h, w).total;
}

size_t resr_generator_workspace_bytes_for(const resr_generator_t* g, int n, int h, int w) {
    if (!g || n <= 0 || h <= 0 || w <= 0) return 0;
    return ws_layout(n, h, w, g->precision).total;
}

int resr_generator_set_precision(resr_generator_t* g, int precision) {
    if (!g) return set_error(RESR_E_INVALID, "null argument");
    if (precision != 0 && precision != 1) return set_error(RESR_E_INVALID, "precision must be 0 (fp16) or 1 (bf16 + fp32 residual masters)");
    if (g->precision != precision) {
        g->precision = precision;
        g->loaded = false;        // the packed weights are in the old operand format: the caller reloads its parameters
        g->plan.valid = false;
        g->canvas_plans.clear();
        cudaFree(g->pack_jobs);   // the batched pack table carries the operand format
        g->pack_jobs = nullptr;
        // the captured training step launches the old recipe's kernels: capture it again under the new one
        if (g->step_exec) cudaGraphExecDestroy(g->step_exec);
        g->step_exec = nullptr;
        memset(g->step_key, 0, sizeof(g->step_key));
        memset(g->step_shape, 0, sizeof(g->step_shape));
        g->step_precision = -1;
        g->step_graph_failed = false;
    }
    return RESR_OK;
}

static int forward_any(resr_generator_t* g, const float* x, const unsigned char* x_u8, float* y, unsigned char* y_u8, int n, int h, int w,
                       void* workspace, size_t workspace_bytes, void* stream);

// The 352 launches of a plan after its input layout kernel; conv4 writes y (fp32 NCHW) or y_u8 (u8 NHWC).
static int run_plan(resr_generator_t* g, Plan& p, float* y, unsigned char* y_u8, cudaStream_t s) {
    for (size_t i = 0; i < p.steps.size(); ++i) {
        Step& st = p.steps[i];
        if (i + 1 == p.steps.size()) { st.a.out_nchw = y; st.a.out_u8 = y_u8; }
        const cudaError_t e = conv3x3_run(st.maps, st.a, st.cfg, g->num_sms, s);
        if (e != cudaSuccess) return set_error(RESR_E_CUDA, "conv %d launch: %s", st.conv, cudaGetErrorString(e));
    }
    return RESR_OK;
}

int resr_generator_forward(resr_generator_t* g, const float* x, float* y, int n, int h, int w, void* workspace,
                           size_t workspace_bytes, void* stream) {
    if (!x || !y) return set_error(RESR_E_INVALID, "null argument");
    return forward_any(g, x, nullptr, y, nullptr, n, h, w, workspace, workspace_bytes, stream);
}

int resr_generator_forward_u8(resr_generator_t* g, const unsigned char* x_u8, unsigned char* y_u8, int n, int h, int w, void* workspace,
                              size_t workspace_bytes, void* stream) {
    if (!x_u8 || !y_u8) return set_error(RESR_E_INVALID, "null argument");
    return forward_any(g, nullptr, x_u8, nullptr, y_u8, n, h, w, workspace, workspace_bytes, stream);
}

int resr_generator_forward_u8_host(resr_generator_t* g, const unsigned char* x_host, unsigned char* y_host, int n, int h, int w,
                                   void* workspace, size_t workspace_bytes, void* stream) {
    if (!g || !x_host || !y_host) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t in_bytes = static_cast<size_t>(n) * 3 * h * w, out_bytes = in_bytes * 16;
    const size_t need = resr_generator_workspace_bytes_for(g, n, h, w);
    const size_t off_x = (need + 1023) / 1024 * 1024, off_y = off_x + (in_bytes + 1023) / 1024 * 1024;
    if (workspace_bytes < off_y + out_bytes) return set_error(RESR_E_NOMEM, "workspace too small for u8 host staging (need %zu)", off_y + out_bytes);
    unsigned char* xd = static_cast<unsigned char*>(workspace) + off_x;
    unsigned char* yd = static_cast<unsigned char*>(workspace) + off_y;
    if (cudaMemcpyAsync(xd, x_host, in_bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) return set_error(RESR_E_CUDA, "H2D failed");
    const int rc = resr_generator_forward_u8(g, xd, yd, n, h, w, workspace, need, stream);
    if (rc != RESR_OK) return rc;
    if (cudaMemcpyAsync(y_host, yd, out_bytes, cudaMemcpyDeviceToHost, s) != cudaSuccess) return set_error(RESR_E_CUDA, "D2H failed");
    const cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "forward_u8_host: %s", cudaGetErrorString(e));
    return RESR_OK;
}

int resr_tensor_to_image_u8(const float* x, unsigned char* out_hwc, int c, int h, int w, int range_norm, int half, void* stream) {
    if (!x || !out_hwc || c <= 0 || h <= 0 || w <= 0) return set_error(RESR_E_INVALID, "bad argument");
    const size_t HW = static_cast<size_t>(h) * w;
    tensor_to_image_kernel<<<grid_for(HW * c, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, out_hwc, c, HW, range_norm, half);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "tensor_to_image: %s", cudaGetErrorString(e));
    return RESR_OK;
}

static int forward_any(resr_generator_t* g, const float* x, const unsigned char* x_u8, float* y, unsigned char* y_u8, int n, int h, int w,
                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!g || !workspace) return set_error(RESR_E_INVALID, "null argument");
    if (n <= 0 || h <= 0 || w <= 0) return set_error(RESR_E_INVALID, "bad shape %dx3x%dx%d", n, h, w);
    if (!g->loaded) return set_error(RESR_E_INVALID, "resr_generator_load_params has not been called");
    if (workspace_bytes < resr_generator_workspace_bytes_for(g, n, h, w)) return set_error(RESR_E_NOMEM, "workspace too small");
    if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return set_error(RESR_E_INVALID, "workspace must be 1024-byte aligned");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Plan& p = g->plan;
    if (!p.valid || p.N != n || p.H != h || p.W != w || p.ws != workspace || p.pair_policy != conv3x3_set_pair_policy(-1)) {
        const int rc = build_plan(g, p, n, h, w, workspace, nullptr, s);
        if (rc != RESR_OK) return rc;
    }
    const size_t total = static_cast<size_t>(n) * h * w * 8;
    if (x_u8) u8nhwc_to_nhwc16_kernel<<<grid_for(total, 256), 256, 0, s>>>(x_u8, p.xin, static_cast<size_t>(n) * h * w, 3, 64, g->precision == 1 ? 1 : 0);
    else nchw_to_nhwc16_kernel<<<grid_for(total, 256), 256, 0, s>>>(x, p.xin, n, 3, h, w, 64, g->precision == 1 ? 1 : 0);
    return run_plan(g, p, y, y_u8, s);
}

// Workspace of a canvas call: the N = 1 forward of the canvas, then conv4's canvas output (fp32 NCHW; the u8 output
// takes a quarter of it), the valid-pixel bitmap and the per-image table.
struct ManyLayout {
    int ch, cw;
    size_t out, vmask, table, total;
};
static int many_layout(const resr_generator_t* g, const int* hs, const int* ws, int count, int* x0, int* y0, ManyLayout* L) {
    const int rc = canvas_pack(hs, ws, count, 0, x0, y0, &L->ch, &L->cw);
    if (rc != RESR_OK) return rc;
    const size_t P = static_cast<size_t>(L->ch) * L->cw;
    size_t o = ws_layout(1, L->ch, L->cw, g->precision).total;
    L->out = o;
    o = align_up(o + P * 48 * 4, 1024);
    L->vmask = o;
    o = align_up(o + P / 8, 1024);
    L->table = o;
    L->total = align_up(o + static_cast<size_t>(count) * sizeof(CanvasImage), 1024);
    return RESR_OK;
}

static const int kCanvasPlans = 8;      // canvas plans a handle keeps (each ~0.4 MB of host memory)
static const int kCanvasMaxImages = 65535;

static int forward_many_any(resr_generator_t* g, const void* const* xs, void* const* ys, const int* hs, const int* ws, int count,
                            int u8, void* workspace, size_t workspace_bytes, void* stream) {
    if (!g || !workspace || !xs || !ys || !hs || !ws) return set_error(RESR_E_INVALID, "null argument");
    if (count <= 0 || count > kCanvasMaxImages) return set_error(RESR_E_INVALID, "forward_many: count %d (1..%d)", count, kCanvasMaxImages);
    for (int i = 0; i < count; ++i)
        if (!xs[i] || !ys[i]) return set_error(RESR_E_INVALID, "forward_many: null image pointer %d", i);
    if (!g->loaded) return set_error(RESR_E_INVALID, "resr_generator_load_params has not been called");
    if ((reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) return set_error(RESR_E_INVALID, "workspace must be 1024-byte aligned");
    std::vector<int> x0(count), y0(count);
    ManyLayout L;
    const int rc = many_layout(g, hs, ws, count, x0.data(), y0.data(), &L);
    if (rc != RESR_OK) return rc;
    if (workspace_bytes < L.total) return set_error(RESR_E_NOMEM, "workspace too small (need %zu)", L.total);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint8_t* base = static_cast<uint8_t*>(workspace);
    uint32_t* vmask = reinterpret_cast<uint32_t*>(base + L.vmask);
    CanvasImage* table_d = reinterpret_cast<CanvasImage*>(base + L.table);

    // plans are cached by canvas geometry next to the single-shape plan (g->plan)
    const int policy = conv3x3_set_pair_policy(-1);
    Plan* p = nullptr;
    for (Plan& c : g->canvas_plans)
        if (c.valid && c.H == L.ch && c.W == L.cw && c.ws == workspace && c.pair_policy == policy) p = &c;
    if (!p) {
        if (static_cast<int>(g->canvas_plans.size()) >= kCanvasPlans) g->canvas_plans.erase(g->canvas_plans.begin());
        g->canvas_plans.emplace_back();
        p = &g->canvas_plans.back();
        const int brc = build_plan(g, *p, 1, L.ch, L.cw, workspace, vmask, s);
        if (brc != RESR_OK) {
            g->canvas_plans.pop_back();
            return brc;
        }
    }

    std::vector<CanvasImage> tab(count);
    size_t most = 0;
    for (int i = 0; i < count; ++i) {
        tab[i] = CanvasImage{xs[i], ys[i], x0[i], y0[i], hs[i], ws[i]};
        most = std::max(most, static_cast<size_t>(hs[i]) * ws[i] * 48);
    }
    std::sort(tab.begin(), tab.end(), [](const CanvasImage& a, const CanvasImage& b) { return a.y0 != b.y0 ? a.y0 < b.y0 : a.x0 < b.x0; });
    // (pageable source: the copy is staged before the call returns, so `tab` may go out of scope)
    if (cudaMemcpyAsync(table_d, tab.data(), tab.size() * sizeof(CanvasImage), cudaMemcpyHostToDevice, s) != cudaSuccess)
        return set_error(RESR_E_CUDA, "forward_many: table copy failed");
    const size_t npix = static_cast<size_t>(L.ch) * L.cw;
    canvas_gather_kernel<<<grid_for(npix, 256), 256, 0, s>>>(table_d, count, L.cw, npix, u8, g->precision == 1 ? 1 : 0, p->xin, vmask);
    const int rrc = run_plan(g, *p, u8 ? nullptr : reinterpret_cast<float*>(base + L.out), u8 ? base + L.out : nullptr, s);
    if (rrc != RESR_OK) return rrc;
    const int gx = static_cast<int>(std::min<size_t>(128, (most + 2047) / 2048));
    canvas_scatter_kernel<<<dim3(gx, count), 256, 0, s>>>(table_d, base + L.out, L.ch, L.cw, u8);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "forward_many: %s", cudaGetErrorString(e));
    return RESR_OK;
}

int resr_canvas_pack(const int* hs, const int* ws, int count, int max_width, int* x0, int* y0, int* canvas_h, int* canvas_w) {
    return canvas_pack(hs, ws, count, max_width, x0, y0, canvas_h, canvas_w);
}

size_t resr_generator_forward_many_workspace_bytes(const resr_generator_t* g, const int* hs, const int* ws, int count) {
    if (!g || !hs || !ws || count <= 0 || count > kCanvasMaxImages) return 0;
    std::vector<int> x0(count), y0(count);
    ManyLayout L;
    return many_layout(g, hs, ws, count, x0.data(), y0.data(), &L) == RESR_OK ? L.total : 0;
}

int resr_generator_forward_many(resr_generator_t* g, const float* const* xs, float* const* ys, const int* hs, const int* ws, int count,
                                void* workspace, size_t workspace_bytes, void* stream) {
    return forward_many_any(g, reinterpret_cast<const void* const*>(xs), reinterpret_cast<void* const*>(ys), hs, ws, count, 0, workspace,
                            workspace_bytes, stream);
}

int resr_generator_forward_many_u8(resr_generator_t* g, const unsigned char* const* xs, unsigned char* const* ys, const int* hs,
                                   const int* ws, int count, void* workspace, size_t workspace_bytes, void* stream) {
    return forward_many_any(g, reinterpret_cast<const void* const*>(xs), reinterpret_cast<void* const*>(ys), hs, ws, count, 1, workspace,
                            workspace_bytes, stream);
}

int resr_generator_forward_host(resr_generator_t* g, const float* x_host, float* y_host, int n, int h, int w,
                                void* workspace, size_t workspace_bytes, void* stream) {
    if (!x_host || !y_host) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t in_bytes = static_cast<size_t>(n) * 3 * h * w * 4, out_bytes = in_bytes * 16;
    const size_t need = resr_generator_workspace_bytes_for(g, n, h, w);
    // device staging for x and y lives at the end of the caller's workspace
    const size_t off_x = (need + 1023) / 1024 * 1024, off_y = off_x + (in_bytes + 1023) / 1024 * 1024;
    if (workspace_bytes < off_y + out_bytes) return set_error(RESR_E_NOMEM, "workspace too small for host staging (need %zu)", off_y + out_bytes);
    float* xd = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + off_x);
    float* yd = reinterpret_cast<float*>(static_cast<uint8_t*>(workspace) + off_y);
    if (cudaMemcpyAsync(xd, x_host, in_bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) return set_error(RESR_E_CUDA, "H2D failed");
    const int rc = resr_generator_forward(g, xd, yd, n, h, w, workspace, need, stream);
    if (rc != RESR_OK) return rc;
    if (cudaMemcpyAsync(y_host, yd, out_bytes, cudaMemcpyDeviceToHost, s) != cudaSuccess) return set_error(RESR_E_CUDA, "D2H failed");
    const cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "forward_host: %s", cudaGetErrorString(e));
    return RESR_OK;
}

int resr_generator_forward_host_async(resr_generator_t* g, const float* x_host, float* y_host, int n, int h, int w,
                                      void* workspace, size_t workspace_bytes, void* stream) {
    if (!g || !x_host || !y_host) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t in_bytes = static_cast<size_t>(n) * 3 * h * w * 4, out_bytes = in_bytes * 16;
    const size_t need = resr_generator_workspace_bytes_for(g, n, h, w);
    const size_t in_al = (in_bytes + 1023) / 1024 * 1024, out_al = (out_bytes + 1023) / 1024 * 1024;
    const size_t off0 = (need + 1023) / 1024 * 1024;
    if (workspace_bytes < off0 + 2 * (in_al + out_al))
        return set_error(RESR_E_NOMEM, "workspace too small for two host staging slots (need %zu)", off0 + 2 * (in_al + out_al));
    if (!g->h2d_stream) {
        if (cudaStreamCreateWithFlags(&g->h2d_stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&g->d2h_stream, cudaStreamNonBlocking) != cudaSuccess)
            return set_error(RESR_E_CUDA, "cannot create copy streams");
        for (int i = 0; i < 2; ++i) {
            cudaEventCreateWithFlags(&g->ev_h2d[i], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&g->ev_fwd[i], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&g->ev_d2h[i], cudaEventDisableTiming);
        }
    }
    if (g->host_calls > 0 && (g->host_shape[0] != n || g->host_shape[1] != h || g->host_shape[2] != w || g->host_ws != workspace)) {
        // a different shape (or workspace) moves the staging slots: drain every queued copy / forward before they are reused
        cudaStreamSynchronize(g->h2d_stream);
        cudaStreamSynchronize(s);
        cudaStreamSynchronize(g->d2h_stream);
        g->host_calls = 0;
    }
    g->host_shape[0] = n; g->host_shape[1] = h; g->host_shape[2] = w; g->host_ws = workspace;
    const int slot = static_cast<int>(g->host_calls & 1);
    const bool reused = g->host_calls >= 2;  // this slot has been through a full cycle before
    uint8_t* base = static_cast<uint8_t*>(workspace) + off0 + static_cast<size_t>(slot) * (in_al + out_al);
    float* xd = reinterpret_cast<float*>(base);
    float* yd = reinterpret_cast<float*>(base + in_al);
    // H2D into the slot once the forward that last read it is done
    if (reused) cudaStreamWaitEvent(g->h2d_stream, g->ev_fwd[slot], 0);
    if (cudaMemcpyAsync(xd, x_host, in_bytes, cudaMemcpyHostToDevice, g->h2d_stream) != cudaSuccess) return set_error(RESR_E_CUDA, "H2D failed");
    cudaEventRecord(g->ev_h2d[slot], g->h2d_stream);
    // forward once the input has landed and the slot's previous result has left the device
    cudaStreamWaitEvent(s, g->ev_h2d[slot], 0);
    if (reused) cudaStreamWaitEvent(s, g->ev_d2h[slot], 0);
    const int rc = resr_generator_forward(g, xd, yd, n, h, w, workspace, need, stream);
    if (rc != RESR_OK) return rc;
    cudaEventRecord(g->ev_fwd[slot], s);
    cudaStreamWaitEvent(g->d2h_stream, g->ev_fwd[slot], 0);
    if (cudaMemcpyAsync(y_host, yd, out_bytes, cudaMemcpyDeviceToHost, g->d2h_stream) != cudaSuccess) return set_error(RESR_E_CUDA, "D2H failed");
    cudaEventRecord(g->ev_d2h[slot], g->d2h_stream);
    ++g->host_calls;
    return RESR_OK;
}

int resr_generator_host_sync(resr_generator_t* g) {
    if (!g) return set_error(RESR_E_INVALID, "null argument");
    if (!g->d2h_stream) return RESR_OK;
    cudaError_t e = cudaStreamSynchronize(g->h2d_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->d2h_stream);
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "host_sync: %s", cudaGetErrorString(e));
    return RESR_OK;
}

int resr_nchw_to_nhwc16(const float* x, void* out16, int n, int c, int h, int w, int c_pad, int fmt, void* stream) {
    if (!x || !out16 || c_pad % 8 != 0 || c > c_pad) return set_error(RESR_E_INVALID, "bad argument");
    const size_t total = static_cast<size_t>(n) * h * w * (c_pad / 8);
    nchw_to_nhwc16_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        x, static_cast<uint16_t*>(out16), n, c, h, w, c_pad, fmt);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "nchw_to_nhwc16: %s", cudaGetErrorString(e));
    return RESR_OK;
}

// The one planning path of resr_conv3x3 and resr_conv3x3_plan: checks every field of `d`, then fills `a` (geometry,
// epilogue flags and pointers; no tensor maps, no weight pack) and `cfg` exactly as the launch will use them. Host only.
// Returns nullptr, or what is wrong with `d` (RESR_E_INVALID).
static const char* conv_desc_plan(const resr_conv_desc* d, int num_sms, ConvArgs* a, ConvLaunchCfg* cfg, resr_conv_plan* out) {
    if (!d || !d->in16 || !d->weight) return "null argument";
    if (num_sms < 1) return "num_sms must be positive";
    if (d->n < 1 || d->h < 1 || d->w < 1 || d->cin < 1 || d->cout < 1) return "empty or negative n / h / w / cin / cout";
    if (d->cin > d->c_total || d->c_total % 8 != 0) return "bad channel counts: cin <= c_total, c_total % 8 == 0";
    const int nchunks = (d->cin + 63) / 64;
    if (static_cast<long long>(nchunks) * 64 > d->c_total) return "c_total must cover cin rounded up to 64";
    if (d->fmt_in != 0 && d->fmt_in != 1) return "fmt_in must be 0 (fp16) or 1 (bf16)";
    if (d->mode < -1 || d->mode > 1) return "mode must be -1, 0 or 1";
    if (d->ep_mode < EP_PLAIN || d->ep_mode > EP_ADD2) return "ep_mode must be 0..4";
    const bool mode_res1 = d->ep_mode == EP_RDB || d->ep_mode == EP_RRDB || d->ep_mode == EP_SKIP;
    const bool mode_res2 = d->ep_mode == EP_RRDB || d->ep_mode == EP_ADD2;
    if ((mode_res1 && !d->res1) || (mode_res2 && !d->res2)) return "ep_mode needs a residual that is NULL";
    if (d->res16 != 0 && d->res16 != 1) return "res16 must be 0 or 1";
    if (d->res16_fmt != 0 && d->res16_fmt != 1) return "res16_fmt must be 0 or 1";
    if (d->ep_mode == EP_ADD2 && d->res16) return "ep_mode 4 reads fp32 residuals";
    // one launch slice is 32 output channels (16 for the RGB convolution); NHWC stores and residual loads cover whole slices
    const int nout = d->cout >= 32 ? 32 : 16;
    const int nslices = (d->cout + nout - 1) / nout;
    if ((d->out16 || d->outf) && d->cout % 32 != 0)
        return "an NHWC output (out16 / outf) needs cout % 32 == 0: the stores write whole 32-channel slices";
    if (nout == 16 && (d->res1 || d->res2)) return "cout < 32 takes no residual";
    if ((d->out_nchw || d->out_nchw_raw || d->out_u8) && d->out_nchw_c != d->cout) return "out_nchw_c must equal cout";
    const long long span = static_cast<long long>(nslices) * nout;  // channels a residual / mask read covers
    if (d->out16) {
        if (d->out16_fmt != 0 && d->out16_fmt != 1) return "out16_fmt must be 0 or 1";
        if (d->out16_up2 != 0 && d->out16_up2 != 1) return "out16_up2 must be 0 or 1";
        if (d->out16_cstride < 1 || d->out16_cstride % 8 != 0) return "out16_cstride must be a positive multiple of 8";
        if (d->out16_choff < 0 || d->out16_choff + (d->out16_slice_fixed ? 32ll : span) > d->out16_cstride)
            return "out16 channels [choff, choff + cout) must lie inside out16_cstride";
    }
    if (d->outf) {
        if (d->outf_cstride < 1 || d->outf_cstride % 4 != 0) return "outf_cstride must be a positive multiple of 4";
        if (d->outf_choff < 0 || d->outf_choff + span > d->outf_cstride) return "outf channels [choff, choff + cout) must lie inside outf_cstride";
    }
    const int res_align = d->res16 ? 8 : 4;   // 16-byte vector loads
    const int res2_cstride = d->res2_cstride ? d->res2_cstride : d->res_cstride;
    if ((d->res1 || d->res2) && (d->res_choff < 0 || d->res_choff % res_align != 0))
        return "res_choff must be a non-negative multiple of 8 (16-bit) / 4 (fp32) channels";
    if (d->res1 && (d->res_cstride % res_align != 0 || d->res_choff + span > d->res_cstride))
        return "res1: res_cstride must be a multiple of 8 (16-bit) / 4 (fp32) and hold res_choff + cout channels";
    if (d->res2 && (res2_cstride % res_align != 0 || d->res_choff + span > res2_cstride))
        return "res2: res2_cstride must be a multiple of 8 (16-bit) / 4 (fp32) and hold res_choff + cout channels";
    if (d->mask16 && d->out16 && (d->mask16_cstride % 8 != 0 || d->mask16_choff < 0 || d->mask16_choff % 8 != 0 ||
                                  d->mask16_choff + span > d->mask16_cstride))
        return "mask16: stride and offset must be multiples of 8 holding mask16_choff + cout channels";
    if (d->vmask && (d->vmask_shift < 0 || d->vmask_shift > 15 || d->vmask_words < 1 ||
                     static_cast<long long>(d->vmask_words) * 32 <= ((d->w - 1) >> d->vmask_shift)))
        return "vmask: vmask_shift must be 0..15 and vmask_words cover every column";

    memset(a, 0, sizeof(*a));
    conv3x3_init_geometry(a, d->n, d->h, d->w, d->cin, d->mode);
    a->nchunks = nchunks;
    a->fmt_in = d->fmt_in;
    a->ep_mode = d->ep_mode; a->lrelu = d->lrelu; a->clamp01 = d->clamp01;
    a->reverse = d->reverse != 0;
    if (d->out16) {
        a->has_out16 = 1; a->out16_fmt = d->out16_fmt; a->out16_choff = d->out16_choff; a->out16_up2 = d->out16_up2;
        a->out16_slice_fixed = d->out16_slice_fixed; a->slice_no16_mask = d->slice_no16_mask;
        a->mask16 = d->mask16; a->mask16_cstride = d->mask16_cstride; a->mask16_choff = d->mask16_choff;
        a->out16_scale = d->out16_scale;
    }
    if (d->outf) {
        a->has_outf = 1; a->outf_choff = d->outf_choff; a->outf = d->outf; a->outf_cstride = d->outf_cstride;
        a->slice_noutf_mask = d->slice_noutf_mask;
    }
    if (d->res1) {
        a->has_res1 = 1; a->res_choff = d->res_choff; a->res1 = d->res1; a->res1_cstride = d->res_cstride;
        a->slice_nores_mask = d->slice_nores_mask;
    }
    a->res16 = d->res16; a->res16_fmt = d->res16_fmt;
    a->res2 = d->res2; a->res2_cstride = res2_cstride; a->res2_scale = d->res2_scale;
    if (d->res2 && !d->res1) a->res_choff = d->res_choff;
    a->out_nchw = d->out_nchw; a->out_nchw_raw = d->out_nchw_raw; a->out_u8 = d->out_u8; a->out_nchw_c = d->out_nchw_c;
    a->vmask = d->vmask; a->vmask_words = d->vmask_words; a->vmask_shift = d->vmask_shift;
    if (!conv3x3_choose(a, nout, nslices, cfg))
        return "the weights of cin input channels and the output staging do not fit in shared memory";
    const long long units = cfg->pair ? static_cast<long long>((a->ncg + 1) / 2) * a->H : a->rows_total;
    const long long clusters = conv3x3_clusters(units, cfg->pair ? 2 : 1, cfg->nslices, num_sms);
    if (units * (clusters + 1) >= (1ll << 31)) return "too many rows for the kernels' 32-bit strip arithmetic";
    if (out) {
        out->pair = cfg->pair; out->nout = cfg->nout; out->nslices = cfg->nslices;
        out->bw = a->BW; out->bn = a->BN; out->mode = a->mode; out->nxs = a->nxs; out->ncg = a->ncg;
        out->tail_ksteps = a->tail_ksteps;
        out->nepi = a->nepi; out->epi_bufs = a->epi_bufs; out->nstages = a->nstages;
        out->masked = a->vmask != nullptr;
        out->units = units; out->clusters = clusters;
    }
    return nullptr;
}

int resr_conv3x3_plan(const resr_conv_desc* d, int num_sms, resr_conv_plan* plan) {
    if (!plan) return set_error(RESR_E_INVALID, "null argument");
    ConvArgs a;
    ConvLaunchCfg cfg;
    const char* bad = conv_desc_plan(d, num_sms, &a, &cfg, plan);
    if (bad) return set_error(RESR_E_INVALID, "resr_conv3x3: %s", bad);
    return RESR_OK;
}

int resr_conv3x3(const resr_conv_desc* d, void* stream) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // the SM count only sizes the grid; without a device the descriptor is still checked (and a bad one rejected)
    int dev = 0, sms = 0;
    const bool have_dev = cudaGetDevice(&dev) == cudaSuccess &&
                          cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0;
    if (!have_dev) { cudaGetLastError(); sms = 1; }
    ConvArgs a;
    ConvLaunchCfg cfg;
    const char* bad = conv_desc_plan(d, sms, &a, &cfg, nullptr);
    if (bad) return set_error(RESR_E_INVALID, "resr_conv3x3: %s", bad);
    if (!have_dev) return set_error(RESR_E_CUDA, "resr_conv3x3: no CUDA device");
    const int nout = d->cout >= 32 ? 32 : 16;   // the weight pack's slice width (a pair launch takes two 32-slices)
    const int nslices = (d->cout + nout - 1) / nout;
    const size_t pack_bytes = static_cast<size_t>(nslices) * a.nchunks * 3 * (3 * nout) * 128;
    uint8_t* wp = nullptr;
    float* bp = nullptr;
    if (cudaMalloc(&wp, pack_bytes) != cudaSuccess) return set_error(RESR_E_CUDA, "cudaMalloc failed");
    if (cudaMalloc(&bp, nslices * nout * 4) != cudaSuccess) {
        cudaFree(wp);
        return set_error(RESR_E_CUDA, "cudaMalloc failed");
    }
    launch_pack_conv(d->weight, d->bias, reinterpret_cast<uint16_t*>(wp), bp, d->cin, d->cout, nout, nslices, a.nchunks,
                     d->fmt_in, 0, s);
    cudaStreamSynchronize(s);  // the conv prefetches its weights before the programmatic grid dependency resolves
    a.wpack = wp; a.bias = bp;
    ConvMaps maps;
    memset(&maps, 0, sizeof(maps));
    int rc = conv3x3_make_tmap_act(&maps.a, d->in16, d->n, d->h, d->w, d->c_total, a.mode, a.BW, a.BN, d->cin);
    if (d->out16) rc |= conv3x3_make_tmap_out16(&maps.o16, d->out16, d->n, d->h, d->w, d->out16_cstride, nout, a.BW, a.BN, d->out16_up2);
    if (d->outf) rc |= conv3x3_make_tmap_f32(&maps.of, d->outf, d->n, d->h, d->w, d->outf_cstride, a.BW, a.BN);
    cudaError_t e = cudaSuccess;
    if (rc == 0) e = conv3x3_run(maps, a, cfg, sms, s);
    const cudaError_t e2 = cudaStreamSynchronize(s);
    cudaFree(wp);
    cudaFree(bp);
    if (rc != 0) return set_error(RESR_E_CUDA, "tensor map encoding failed (%d)", rc);
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "conv launch: %s", cudaGetErrorString(e));
    if (e2 != cudaSuccess) return set_error(RESR_E_CUDA, "conv run: %s", cudaGetErrorString(e2));
    return RESR_OK;
}

}  // extern "C"
