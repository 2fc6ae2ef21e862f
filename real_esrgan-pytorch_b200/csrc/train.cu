// Training path of the generator: forward that keeps every activation, L1 loss, and the full backward pass
// (data gradients through the same tcgen05 convolution kernel with transposed weights, weight gradients through
// wgrad_tc.cu). Reference: autograd of /root/reference/model.py:64-132, 206-275 and nn.L1Loss
// (train_realesrnet.py:190-194, 383-388). See DESIGN.md §6.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/resr.h"
#include "conv3x3.cuh"
#include "errors.h"
#include "gen_internal.cuh"
#include "wgrad.cuh"

namespace resr {

// ================================================================================================ small kernels

// NHWC 16-bit [P][cstride], channels [c0, c0 + C) -> channels-first bf16 [Cpad][P]; rows C..Cpad-1 are zero-filled.
// SHIFT3 additionally writes the copies shifted by one pixel along x (zero at the row ends),
//     out[dx][c][n][y][x] = in[n][y][x - dx + 1][c]   (dx = 0, 1, 2; zero when x - dx + 1 is outside [0, W)),
// because the weight-gradient kernel pairs X[.., x + dx - 1] with dY[.., x] and TMA cannot start a box at an odd 2-byte
// offset of the innermost (pixel) dimension; and, when db is given, accumulates the bias gradient
// db[c] += sum_p in[p][c] in the same pass (db zeroed by the caller).
// One block = 32 channels x 256 pixels; all global traffic is 16-byte vectors (requires W % 8 == 0, c0 % 8 == 0,
// cstride % 8 == 0).
template <bool SHIFT3>
__global__ void __launch_bounds__(256) nhwc16_to_cf_kernel(const uint16_t* __restrict__ in, int cstride, int c0, int C, int Cpad,
                                                          size_t P, int W, int fmt_in, uint16_t* __restrict__ out,
                                                          float* __restrict__ db) {
    constexpr int kRow = 272;                   // halo pixel -1 at index 7, pixels 0..255 at 8..263, halo 256 at 264
    __shared__ __align__(16) uint16_t tile[32][kRow];
    const int cb = blockIdx.y * 32;
    const long long p0 = static_cast<long long>(blockIdx.x) * 256;
    for (int idx = threadIdx.x; idx < 258 * 4; idx += 256) {
        const int px = idx >> 2, q = idx & 3;   // px 0..257 <-> pixel p0 - 1 + px
        const long long p = p0 - 1 + px;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (p >= 0 && p < static_cast<long long>(P) && cb + q * 8 < C)
            v = *reinterpret_cast<const uint4*>(in + static_cast<size_t>(p) * cstride + c0 + cb + q * 8);
        const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            uint16_t e = static_cast<uint16_t>(w4[j >> 1] >> ((j & 1) * 16));
            if (fmt_in == 0) {  // fp16 -> bf16
                const __half h = *reinterpret_cast<const __half*>(&e);
                const __nv_bfloat16 bb = __float2bfloat16_rn(__half2float(h));
                e = *reinterpret_cast<const uint16_t*>(&bb);
            }
            if (cb + q * 8 + j >= C) e = 0;
            tile[q * 8 + j][7 + px] = e;
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t plane = static_cast<size_t>(Cpad) * P;
    for (int c = warp; c < 32; c += 8) {
        if (cb + c >= Cpad) break;
        const long long p = p0 + 8 * lane;      // this lane's 8 pixels (never straddle an image row: W % 8 == 0)
        const uint4 cur = *reinterpret_cast<const uint4*>(&tile[c][8 + 8 * lane]);
        float bs = 0.f;
        if (p < static_cast<long long>(P)) {
            uint16_t* row = out + static_cast<size_t>(cb + c) * P + p;
            if (!SHIFT3) {
                *reinterpret_cast<uint4*>(row) = cur;
            } else {
                const uint32_t prev = *reinterpret_cast<const uint32_t*>(&tile[c][6 + 8 * lane]);   // pixels -2, -1
                const uint32_t next = *reinterpret_cast<const uint32_t*>(&tile[c][16 + 8 * lane]);  // pixels 8, 9
                const int x = static_cast<int>(p % W);
                uint4 lo, hi;  // lo: out[dx=0][p + i] = in[p + i + 1];  hi: out[dx=2][p + i] = in[p + i - 1]
                lo.x = __funnelshift_r(cur.x, cur.y, 16);
                lo.y = __funnelshift_r(cur.y, cur.z, 16);
                lo.z = __funnelshift_r(cur.z, cur.w, 16);
                lo.w = __funnelshift_r(cur.w, next, 16);
                hi.x = __funnelshift_r(prev, cur.x, 16);
                hi.y = __funnelshift_r(cur.x, cur.y, 16);
                hi.z = __funnelshift_r(cur.y, cur.z, 16);
                hi.w = __funnelshift_r(cur.z, cur.w, 16);
                if (x + 8 == W) lo.w &= 0x0000FFFFu;  // last pixel of an image row has no right neighbour
                if (x == 0) hi.x &= 0xFFFF0000u;      // first pixel has no left neighbour
                *reinterpret_cast<uint4*>(row) = lo;
                *reinterpret_cast<uint4*>(row + plane) = cur;
                *reinterpret_cast<uint4*>(row + 2 * plane) = hi;
            }
            if (SHIFT3 && db) {
                const uint32_t w4[4] = {cur.x, cur.y, cur.z, cur.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) bs += __uint_as_float(w4[j] << 16) + __uint_as_float(w4[j] & 0xFFFF0000u);
            }
        }
        if (SHIFT3 && db) {
            for (int o = 16; o > 0; o >>= 1) bs += __shfl_down_sync(0xffffffffu, bs, o);
            if (lane == 0 && cb + c < C) atomicAdd(db + cb + c, bs);
        }
    }
}

__global__ void __launch_bounds__(256) scale_f32_to_bf16_kernel(const float* __restrict__ a, float sa, const float* __restrict__ b,
                                                               float sb, uint16_t* __restrict__ out, size_t n) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        float v = sa * a[i];
        if (b) v += sb * b[i];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        out[i] = *reinterpret_cast<const uint16_t*>(&h);
    }
}

// Backward of nearest x2 upsampling (model.py:264-265): out[n,y,x,c] = sum of the 2x2 block of in[n,2y+a,2x+b,c].
// in: bf16 [N,2H,2W,64]; outputs (either may be null): fp32 and bf16 [N,H,W,64].
__global__ void __launch_bounds__(256) sum2x2_kernel(const uint16_t* __restrict__ in, float* __restrict__ outf,
                                                    uint16_t* __restrict__ out16, int N, int H, int W) {
    const size_t total = static_cast<size_t>(N) * H * W * 32;  // one thread per channel pair
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total; idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int cp = static_cast<int>(idx & 31);
        const size_t pix = idx >> 5;
        size_t rowi, n;   // 32-bit divisions whenever the index fits (64-bit ones are ~100-instruction subroutines)
        int x, y;
        if (pix <= 0xffffffffull) {
            const unsigned p32 = static_cast<unsigned>(pix), r32 = p32 / static_cast<unsigned>(W);
            x = static_cast<int>(p32 % static_cast<unsigned>(W)); y = static_cast<int>(r32 % static_cast<unsigned>(H)); n = r32 / static_cast<unsigned>(H);
        } else {
            rowi = pix / W; x = static_cast<int>(pix % W); y = static_cast<int>(rowi % H); n = rowi / H;
        }
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const size_t pi = (n * 2 * H + 2 * y + (k >> 1)) * (2 * W) + 2 * x + (k & 1);
            const uint32_t v = reinterpret_cast<const uint32_t*>(in + pi * 64)[cp];
            s0 += __uint_as_float(v << 16);
            s1 += __uint_as_float(v & 0xFFFF0000u);
        }
        if (outf) { outf[pix * 64 + 2 * cp] = s0; outf[pix * 64 + 2 * cp + 1] = s1; }
        if (out16) {
            const __nv_bfloat162 h = __floats2bfloat162_rn(s0, s1);
            reinterpret_cast<uint32_t*>(out16 + pix * 64)[cp] = *reinterpret_cast<const uint32_t*>(&h);
        }
    }
}

// Gradient of the network output. mode 0: L1 loss vs hr (train_realesrnet.py:190-194, 385): g = sign(clamp(v) - hr) / numel,
// loss accumulated in double; mode 1: g = upstream gradient `ref`. Both are gated by the clamp (model.py:270): the
// gradient passes where 0 <= v <= 1. Writes the NHWC bf16 operand of conv4's backward ([pixels][64], channels >= 3 zero).
__global__ void __launch_bounds__(256) out_grad_kernel(const float* __restrict__ raw, const float* __restrict__ ref,
                                                      uint16_t* __restrict__ dy, double* __restrict__ loss_sum, int N, size_t HW,
                                                      float inv_numel, int mode) {
    __shared__ double red[8];
    const size_t total = static_cast<size_t>(N) * HW;
    double local = 0.0;
    for (size_t pix = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; pix < total; pix += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t n = pix / HW, r = pix % HW;
        float g[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const size_t o = (n * 3 + c) * HW + r;
            const float v = raw[o];
            float gv;
            if (mode == 0) {
                const float d = fminf(fmaxf(v, 0.f), 1.f) - ref[o];
                local += fabs(static_cast<double>(d));
                gv = d > 0.f ? inv_numel : (d < 0.f ? -inv_numel : 0.f);
            } else {
                gv = ref[o];
            }
            g[c] = (v < 0.f || v > 1.f) ? 0.f : gv;
        }
        uint4* dst = reinterpret_cast<uint4*>(dy + pix * 64);
        const __nv_bfloat162 h01 = __floats2bfloat162_rn(g[0], g[1]);
        const __nv_bfloat162 h23 = __floats2bfloat162_rn(g[2], 0.f);
        dst[0] = make_uint4(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23), 0u, 0u);
#pragma unroll
        for (int i = 1; i < 8; ++i) dst[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (mode == 0) {
        for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0;
            for (int i = 0; i < 8; ++i) s += red[i];
            atomicAdd(loss_sum, s);
        }
    }
}

__global__ void finish_loss_kernel(const double* __restrict__ sum, float* __restrict__ loss, double inv_numel) {
    *loss = static_cast<float>(*sum * inv_numel);
}

static int egrid(size_t total) {
    size_t g = (total + 255) / 256;
    if (g > 148 * 32) g = 148 * 32;
    return static_cast<int>(g < 1 ? 1 : g);
}

// ================================================================================================ conv launcher

struct Geo { int H, W; };  // resolution of one convolution

struct ConvIO {
    const void* in16 = nullptr; int in_c = 64;
    const uint8_t* wpack = nullptr; const float* bias = nullptr;
    int nout = 32, nslices = 1, nchunks = 1, fmt = 1;
    int kvalid = 0;  // real input channels (0: every chunk is full)
    void* out16 = nullptr; int out16_c = 64, out16_choff = 0, out16_fmt = 1, out16_up2 = 0, out16_fixed = 0; unsigned no16_mask = 0;
    float* outf = nullptr; int outf_c = 64, outf_choff = 0; unsigned noutf_mask = 0;
    const float* res1 = nullptr; int res1_c = 64, res_choff = 0; unsigned nores_mask = 0;
    const float* res2 = nullptr; int res2_c = 64; float res2_scale = 1.f;
    const void* mask16 = nullptr; int mask16_c = 64, mask16_choff = 0;
    int ep_mode = EP_PLAIN, lrelu = 0, clamp01 = 0;
    float out16_scale = 0.f;
    float* out_nchw = nullptr; float* out_nchw_raw = nullptr; int out_nchw_c = 3;
};

static int launch_conv_io(const resr_generator* g, const Geo& q, int N, const ConvIO& io, cudaStream_t s) {
    ConvArgs a;
    ConvMaps m;
    memset(&a, 0, sizeof(a));
    memset(&m, 0, sizeof(m));
    conv3x3_init_geometry(&a, N, q.H, q.W, io.kvalid, -1);
    a.nchunks = io.nchunks;
    a.fmt_in = io.fmt;
    a.wpack = io.wpack; a.bias = io.bias;
    a.ep_mode = io.ep_mode; a.lrelu = io.lrelu; a.clamp01 = io.clamp01;
    // channels past kvalid are zeros this library wrote: the map may end at the next multiple of 8
    int rc = conv3x3_make_tmap_act(&m.a, io.in16, N, a.H, a.W, io.in_c, a.mode, a.BW, a.BN, (io.kvalid + 7) / 8 * 8);
    if (io.out16) {
        a.has_out16 = 1; a.out16_fmt = io.out16_fmt; a.out16_choff = io.out16_choff; a.out16_up2 = io.out16_up2;
        a.out16_slice_fixed = io.out16_fixed; a.slice_no16_mask = io.no16_mask;
        rc |= conv3x3_make_tmap_out16(&m.o16, io.out16, N, a.H, a.W, io.out16_c, io.nout, a.BW, a.BN, io.out16_up2);
    }
    if (io.outf) {
        a.has_outf = 1; a.outf_choff = io.outf_choff; a.slice_noutf_mask = io.noutf_mask;
        a.outf = io.outf; a.outf_cstride = io.outf_c;
        rc |= conv3x3_make_tmap_f32(&m.of, io.outf, N, a.H, a.W, io.outf_c, a.BW, a.BN);
    }
    if (io.res1) {
        a.has_res1 = 1; a.res_choff = io.res_choff; a.slice_nores_mask = io.nores_mask;
        a.res1 = io.res1; a.res1_cstride = io.res1_c;
    }
    a.res2 = io.res2; a.res2_cstride = io.res2_c; a.res2_scale = io.res2_scale;
    a.out16_scale = io.out16_scale;
    a.mask16 = io.mask16; a.mask16_cstride = io.mask16_c; a.mask16_choff = io.mask16_choff;
    a.out_nchw = io.out_nchw; a.out_nchw_raw = io.out_nchw_raw; a.out_nchw_c = io.out_nchw_c;
    ConvLaunchCfg cfg;  // CTA-pair kernel whenever two column groups can be paired (conv3x3_pair.cu)
    if (!conv3x3_choose(&a, io.nout, io.nslices, &cfg)) rc |= 1 << 20;
    if (rc != 0) return set_error(RESR_E_CUDA, "conv planning failed (%d)", rc);
    const cudaError_t e = conv3x3_run(m, a, cfg, g->num_sms, s);
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "conv launch: %s", cudaGetErrorString(e));
    return RESR_OK;
}

// ================================================================================================ workspace

static size_t up1k(size_t v) { return (v + 1023) / 1024 * 1024; }

struct TrainWs {
    size_t xin, c[70], f[4], t1, t2, t3, t4, yraw;       // forward
    size_t dycat[3], dbcat;
    size_t g, dya, dyb, dx[3], dskip, biga, bigb, mida, midb, xt, dyt, partial, loss;  // backward
    size_t total;
};

static TrainWs train_layout(size_t N, size_t H, size_t W, int num_sms) {
    const size_t P = N * H * W;
    TrainWs L;
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = up1k(o + bytes); return at; };
    L.xin = take(P * 64 * 2);
    for (int i = 0; i < 70; ++i) L.c[i] = take(P * 192 * 2);
    for (int i = 0; i < 4; ++i) L.f[i] = take(P * 64 * 4);
    L.t1 = take(4 * P * 64 * 2);
    L.t2 = take(16 * P * 64 * 2);
    L.t3 = take(16 * P * 64 * 2);
    L.t4 = take(16 * P * 64 * 2);
    L.yraw = take(16 * P * 3 * 4);
    L.g = take(P * 192 * 4);
    for (int i = 0; i < 3; ++i) L.dycat[i] = take(P * 192 * 2);
    L.dbcat = take(192 * 4);
    L.dya = take(P * 64 * 2);
    L.dyb = take(P * 64 * 2);
    for (int i = 0; i < 3; ++i) L.dx[i] = take(P * 64 * 4);
    L.dskip = take(P * 64 * 4);
    L.biga = take(16 * P * 64 * 2);
    L.bigb = take(16 * P * 64 * 2);
    L.mida = take(4 * P * 64 * 2);
    L.midb = take(4 * P * 64 * 2);
    L.xt = take(16 * P * 64 * 2 > P * 192 * 2 ? 16 * P * 64 * 2 : P * 192 * 2);
    L.dyt = take(3 * 16 * P * 64 * 2);  // also holds the three 192-channel copies of a dense block's dYcat (3 * 192 * P)
    {
        const size_t pa = wgrad_partial_bytes(num_sms), pb = wgrad_mn_workspace_bytes(num_sms);
        L.partial = take(pa > pb ? pa : pb);
    }
    L.loss = take(64);
    L.total = o;
    return L;
}

void ensure_transposed_packs(resr_generator* g, cudaStream_t s, bool force) {
    const Table& T = table();
    if (!g->wpack_t) {
        if (!force) return;  // inference-only handle
        cudaMalloc(&g->wpack_t, T.packt_bytes);
        cudaMalloc(&g->wpack_t2, T.pack_bytes);
        cudaMalloc(&g->zero_bias, 256 * sizeof(float));
        cudaMemsetAsync(g->zero_bias, 0, 256 * sizeof(float), s);
    }
    if (g->packed_t || !g->flat_params) return;
    launch_pack_all(g, g->flat_params, 1, s);
    launch_pack_rdb_bwd(g, g->flat_params, g->wpack_t2, s);
    g->packed_t = true;
}

}  // namespace resr

using namespace resr;

namespace {

struct Bufs {
    uint16_t *dycat[3];
    float* dbcat;
    uint16_t *xin, *c[70], *t1, *t2, *t3, *t4, *dya, *dyb, *biga, *bigb, *mida, *midb, *xt, *dyt;
    float *f[4], *yraw, *g, *dx[3], *dskip, *partial;
    double* loss;
};

Bufs carve(void* ws, const TrainWs& L) {
    uint8_t* b = static_cast<uint8_t*>(ws);
    Bufs B;
    B.xin = reinterpret_cast<uint16_t*>(b + L.xin);
    for (int i = 0; i < 70; ++i) B.c[i] = reinterpret_cast<uint16_t*>(b + L.c[i]);
    for (int i = 0; i < 4; ++i) B.f[i] = reinterpret_cast<float*>(b + L.f[i]);
    B.t1 = reinterpret_cast<uint16_t*>(b + L.t1); B.t2 = reinterpret_cast<uint16_t*>(b + L.t2);
    B.t3 = reinterpret_cast<uint16_t*>(b + L.t3); B.t4 = reinterpret_cast<uint16_t*>(b + L.t4);
    B.yraw = reinterpret_cast<float*>(b + L.yraw);
    B.g = reinterpret_cast<float*>(b + L.g);
    for (int i = 0; i < 3; ++i) B.dycat[i] = reinterpret_cast<uint16_t*>(b + L.dycat[i]);
    B.dbcat = reinterpret_cast<float*>(b + L.dbcat);
    B.dya = reinterpret_cast<uint16_t*>(b + L.dya); B.dyb = reinterpret_cast<uint16_t*>(b + L.dyb);
    for (int i = 0; i < 3; ++i) B.dx[i] = reinterpret_cast<float*>(b + L.dx[i]);
    B.dskip = reinterpret_cast<float*>(b + L.dskip);
    B.biga = reinterpret_cast<uint16_t*>(b + L.biga); B.bigb = reinterpret_cast<uint16_t*>(b + L.bigb);
    B.mida = reinterpret_cast<uint16_t*>(b + L.mida); B.midb = reinterpret_cast<uint16_t*>(b + L.midb);
    B.xt = reinterpret_cast<uint16_t*>(b + L.xt); B.dyt = reinterpret_cast<uint16_t*>(b + L.dyt);
    B.partial = reinterpret_cast<float*>(b + L.partial);
    B.loss = reinterpret_cast<double*>(b + L.loss);
    return B;
}

#define RESR_TRY(expr) do { const int rc__ = (expr); if (rc__ != RESR_OK) return rc__; } while (0)

// forward conv of layer `k` with the inference packs
ConvIO fwd_io(const resr_generator* g, int k) {
    const ConvSpec& c = table().c[k];
    ConvIO io;
    io.wpack = g->wpack + c.w_off; io.bias = g->bias + c.b_off;
    io.nout = c.nout; io.nslices = c.nslices; io.nchunks = c.nchunks; io.kvalid = c.cin;
    // forward activations are stored in the operand format of every consumer: fp16 (default recipe) or bf16 (precision 1;
    // the residual stream is fp32 in both, B.f[])
    io.fmt = g->precision == 1 ? 1 : c.fmt;
    io.out16_fmt = g->precision == 1 ? 1 : 0;
    return io;
}

int forward_train(resr_generator* g, const float* x, float* y, int N, int H, int W, const Bufs& B, cudaStream_t s) {
    const Geo g0{H, W}, g1{2 * H, 2 * W}, g2{4 * H, 4 * W};
    // (no clearing of the concat buffers: a layer's activation tensor map ends at its last input channel, the rest of
    // the tail chunk is zero-filled by TMA, so never-written growth channels are never read)
    RESR_TRY(resr_nchw_to_nhwc16(x, B.xin, N, 3, H, W, 64, g->precision == 1 ? 1 : 0, s));
    int k = 0;
    {
        ConvIO io = fwd_io(g, k++);
        io.in16 = B.xin; io.in_c = 64;
        io.outf = B.f[0]; io.out16 = B.c[0]; io.out16_c = 192;
        RESR_TRY(launch_conv_io(g, g0, N, io, s));
    }
    for (int i = 0; i < kNumRRDB; ++i) {
        float* X0 = (i == 0) ? B.f[0] : B.f[3];
        for (int j = 0; j < 3; ++j) {
            const int r = 3 * i + j;
            float* xm = (j == 0) ? X0 : B.f[j];
            for (int q = 0; q < 4; ++q) {
                ConvIO io = fwd_io(g, k++);
                io.in16 = B.c[r]; io.in_c = 192; io.lrelu = 1;
                io.out16 = B.c[r]; io.out16_c = 192; io.out16_choff = 64 + 32 * q;
                RESR_TRY(launch_conv_io(g, g0, N, io, s));
            }
            ConvIO io = fwd_io(g, k++);
            io.in16 = B.c[r]; io.in_c = 192;
            io.res1 = xm;
            if (j < 2) { io.ep_mode = EP_RDB; io.outf = B.f[j + 1]; }
            else { io.ep_mode = EP_RRDB; io.res2 = X0; io.res2_c = 64; io.outf = B.f[3]; }
            io.out16 = B.c[r + 1]; io.out16_c = 192;
            RESR_TRY(launch_conv_io(g, g0, N, io, s));
        }
    }
    {   // conv2 + skip, stored nearest-upsampled x2 (fp16)
        ConvIO io = fwd_io(g, k++);
        io.in16 = B.c[69]; io.in_c = 192; io.ep_mode = EP_SKIP; io.res1 = B.f[0];
        io.out16 = B.t1; io.out16_c = 64; io.out16_up2 = 1;
        RESR_TRY(launch_conv_io(g, g0, N, io, s));
    }
    {
        ConvIO io = fwd_io(g, k++);
        io.in16 = B.t1; io.lrelu = 1; io.out16 = B.t2; io.out16_up2 = 1;
        RESR_TRY(launch_conv_io(g, g1, N, io, s));
    }
    {
        ConvIO io = fwd_io(g, k++);
        io.in16 = B.t2; io.lrelu = 1; io.out16 = B.t3;
        RESR_TRY(launch_conv_io(g, g2, N, io, s));
    }
    {
        ConvIO io = fwd_io(g, k++);
        io.in16 = B.t3; io.lrelu = 1; io.out16 = B.t4;
        RESR_TRY(launch_conv_io(g, g2, N, io, s));
    }
    {
        ConvIO io = fwd_io(g, k++);
        io.in16 = B.t4; io.clamp01 = 1; io.out_nchw = y; io.out_nchw_raw = B.yraw; io.out_nchw_c = 3;
        RESR_TRY(launch_conv_io(g, g2, N, io, s));
    }
    return RESR_OK;
}

// weight + bias gradient of layer k. x16: NHWC input activations of the layer (first cin channels of a c_stride-wide
// tensor, format fmt_x); dy16: NHWC bf16 output gradient (64-channel buffer). Both are transposed to channels-first.
// The weight-gradient chain (transposes, split-K GEMM, reduction) of a layer only consumes the layer's dY and saved
// input, nothing downstream on the data-gradient chain waits for it: it runs on a second stream (a parallel branch of
// the captured graph) and fills the SMs the short data-gradient kernels leave idle. RESR_TRAIN_ONE_STREAM=1 disables it.
cudaStream_t wgrad_stream(resr_generator* g, cudaStream_t s) {
    static const bool one = getenv("RESR_TRAIN_ONE_STREAM") != nullptr;
    if (one) return s;
    if (!g->side_stream) {
        if (cudaStreamCreateWithFlags(&g->side_stream, cudaStreamNonBlocking) != cudaSuccess) { g->side_stream = nullptr; return s; }
        cudaEventCreateWithFlags(&g->ev_fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g->ev_dy, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g->ev_join, cudaEventDisableTiming);
        for (int i = 0; i < 3; ++i) cudaEventCreateWithFlags(&g->ev_dyc[i], cudaEventDisableTiming);
    }
    return g->side_stream;
}
// side stream continues from the current point of the main stream
void fork_to(resr_generator* g, cudaStream_t s, cudaStream_t w) {
    if (w == s) return;
    cudaEventRecord(g->ev_fork, s);
    cudaStreamWaitEvent(w, g->ev_fork, 0);
}

int layer_wgrad(resr_generator* g, int k, const uint16_t* x16, int x_cstride, int fmt_x, bool x_already_transposed, int xt_rows,
                const uint16_t* dy16, int N, const Geo& q, const Bufs& B, float* grads, cudaStream_t s) {
    const ConvSpec& c = table().c[k];
    const size_t P = static_cast<size_t>(N) * q.H * q.W;
    cudaStream_t w = wgrad_stream(g, s);
    fork_to(g, s, w);  // dY of this layer (and everything before it) is complete on the main stream
    if (g->precision == 1) {
        // bf16 recipe: X and dY share one operand format, the MN-major kernel reads both NHWC buffers in place
        WgradMnTable tb;
        float* dw = grads + c.p_off;
        for (int cs = 0; cs < 6; ++cs) {
            tb.dw[cs] = dw; tb.db[cs] = dw + static_cast<size_t>(c.cout) * c.cin * 9;
            tb.cin[cs] = c.cin; tb.cout[cs] = c.cout; tb.co_base[cs] = cs * 32;
        }
        const int dyc = (c.cout + 7) / 8 * 8 > 64 ? 64 : (c.cout + 7) / 8 * 8;
        int units[2][3] = {{0, 0, 64}, {128, 0, 64}};
        const int rc = wgrad_mn_launch(x16, x_cstride, c.cin, dy16, 64, dyc, N, q.H, q.W, units, c.cin > 128 ? 2 : 1, tb, true, B.partial,
                                       g->num_sms, w);
        if (rc != 0) return set_error(RESR_E_CUDA, "wgrad (nhwc) of layer %d failed (%d)", k, rc);
        if (w != s) {  // the main stream overwrites this dY buffer two layers later: wait for its reader here
            cudaEventRecord(g->ev_dy, w);
            cudaStreamWaitEvent(s, g->ev_dy, 0);
        }
        return RESR_OK;
    }
    if (!x_already_transposed) {
        xt_rows = (c.cin + 31) / 32 * 32;
        nhwc16_to_cf_kernel<false><<<dim3(static_cast<unsigned>((P + 255) / 256), xt_rows / 32), 256, 0, w>>>(x16, x_cstride, 0, c.cin, xt_rows, P, q.W,
                                                                                                               fmt_x, B.xt, nullptr);
    }
    const int dy_rows = (c.cout + 31) / 32 * 32;
    float* dw = grads + c.p_off;
    float* db = dw + static_cast<size_t>(c.cout) * c.cin * 9;  // zeroed with the whole gradient vector at the start of the backward
    nhwc16_to_cf_kernel<true><<<dim3(static_cast<unsigned>((P + 255) / 256), dy_rows / 32), 256, 0, w>>>(dy16, 64, 0, c.cout, dy_rows, P, q.W, 1, B.dyt, db);
    if (w != s) {  // the main stream may overwrite the dY buffer once its channels-first copies exist
        cudaEventRecord(g->ev_dy, w);
        cudaStreamWaitEvent(s, g->ev_dy, 0);
    }
    const int rc = wgrad_launch(B.xt, xt_rows, B.dyt, dy_rows, N, q.H, q.W, c.cin, c.cout, B.partial, dw, nullptr, g->num_sms, w);
    if (rc != 0) return set_error(RESR_E_CUDA, "wgrad of layer %d failed (%d)", k, rc);
    return RESR_OK;
}

// data-gradient convolution of layer k: ConvIO preset with the transposed packs
ConvIO bwd_io(const resr_generator* g, int k) {
    const ConvSpec& c = table().c[k];
    ConvIO io;
    io.wpack = g->wpack_t + c.wt_off; io.bias = g->zero_bias;
    io.nout = 32; io.nslices = c.t_nslices; io.nchunks = c.t_nchunks; io.fmt = 1; io.kvalid = c.cout;
    return io;
}

// Gradient buckets for data-parallel training (SURVEY.md §8e: the all-reduce overlapped with the backward). The backward
// finishes gradients tail first, then trunk.22 ... trunk.0, conv1 -- in the flat vector (state_dict order) that is from
// the END towards the front, so "everything from RRDB i on" is one contiguous suffix. Bucket 0 = [trunk.17, end),
// 1 = [trunk.11, trunk.17), 2 = [trunk.5, trunk.11), 3 = [0, trunk.5) (complete when the step itself is).
static const int kBucketRRDB[3] = {17, 11, 5};

static void record_bucket(resr_generator* g, int i, cudaStream_t st) {
    if (!g->ev_bucket[i] && cudaEventCreateWithFlags(&g->ev_bucket[i], cudaEventDisableTiming) != cudaSuccess) { g->ev_bucket[i] = nullptr; return; }
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    cudaEventRecordWithFlags(g->ev_bucket[i], st, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
}

// Common backward: B.biga holds conv4's output gradient (NHWC bf16 [16P][64], 3 channels used).
int backward_common(resr_generator* g, float* grads, int N, int H, int W, const Bufs& B, cudaStream_t s) {
    const Geo g0{H, W}, g1{2 * H, 2 * W}, g2{4 * H, 4 * W};
    const size_t P = static_cast<size_t>(N) * H * W;
    ensure_transposed_packs(g, s, true);
    g->ev_dyc_valid[0] = g->ev_dyc_valid[1] = g->ev_dyc_valid[2] = false;
    cudaMemsetAsync(grads, 0, table().n_params * sizeof(float), s);  // bias gradients are accumulated with atomics
    cudaMemsetAsync(B.dya, 0, P * 64 * 2, s);
    cudaMemsetAsync(B.dyb, 0, P * 64 * 2, s);
    const int kConv2 = 346, kUp1 = 347, kUp2 = 348, kConv3 = 349, kConv4 = 350;

    // ---- tail (model.py:264-270 backwards)
    RESR_TRY(layer_wgrad(g, kConv4, B.t4, 64, g->precision, false, 0, B.biga, N, g2, B, grads, s));
    {   // d(T4) masked by LeakyReLU'(conv3 out) -> conv3's dY
        ConvIO io = bwd_io(g, kConv4);
        io.in16 = B.biga; io.out16 = B.bigb; io.mask16 = B.t4;
        RESR_TRY(launch_conv_io(g, g2, N, io, s));
    }
    RESR_TRY(layer_wgrad(g, kConv3, B.t3, 64, g->precision, false, 0, B.bigb, N, g2, B, grads, s));
    {
        ConvIO io = bwd_io(g, kConv3);
        io.in16 = B.bigb; io.out16 = B.biga; io.mask16 = B.t3;
        RESR_TRY(launch_conv_io(g, g2, N, io, s));
    }
    RESR_TRY(layer_wgrad(g, kUp2, B.t2, 64, g->precision, false, 0, B.biga, N, g2, B, grads, s));
    {   // d(T2) at 4x, masked by LeakyReLU'(up1 out) (T2 holds its upsampled copy), then the 2x2 sum of nearest x2
        ConvIO io = bwd_io(g, kUp2);
        io.in16 = B.biga; io.out16 = B.bigb; io.mask16 = B.t2;
        RESR_TRY(launch_conv_io(g, g2, N, io, s));
        sum2x2_kernel<<<egrid(4 * P * 32), 256, 0, s>>>(B.bigb, nullptr, B.mida, N, 2 * H, 2 * W);
    }
    RESR_TRY(layer_wgrad(g, kUp1, B.t1, 64, g->precision, false, 0, B.mida, N, g1, B, grads, s));
    {   // d(T1) at 2x (no activation on the skip sum), 2x2 sum -> d(out) at LR: fp32 (skip branch) + bf16 (conv2's dY)
        ConvIO io = bwd_io(g, kUp1);
        io.in16 = B.mida; io.out16 = B.midb;
        RESR_TRY(launch_conv_io(g, g1, N, io, s));
        sum2x2_kernel<<<egrid(P * 32), 256, 0, s>>>(B.midb, B.dskip, B.dya, N, H, W);
    }
    RESR_TRY(layer_wgrad(g, kConv2, B.c[69], 192, g->precision, false, 0, B.dya, N, g0, B, grads, s));
    {   // d(trunk output), fp32, and its bf16 copy x 0.2 x 0.2 = dY5 of the last dense block (trunk.22.rdb3)
        ConvIO io = bwd_io(g, kConv2);
        io.in16 = B.dya; io.outf = B.dx[0];
        io.out16 = B.dycat[(3 * kNumRRDB - 1) % 3]; io.out16_c = 192; io.out16_choff = 0; io.out16_fmt = 1; io.out16_scale = 0.2f * 0.2f;
        RESR_TRY(launch_conv_io(g, g0, N, io, s));
    }

    // ---- trunk, RRDB 22 .. 0 (model.py:123-132 and 87-98 backwards)
    for (int i = kNumRRDB - 1; i >= 0; --i) {
        // d(out) of this RRDB is in dx[0]; rdb3 sees 0.2 * d(out)
        const float* dbuf[3] = {B.dx[0], B.dx[1], B.dx[2]};
        float* dxin[3] = {B.dx[1], B.dx[2], B.dx[1]};
        const float dscale[3] = {0.2f, 1.f, 1.f};
        for (int jj = 0; jj < 3; ++jj) {
            const int j = 2 - jj;          // rdb3, rdb2, rdb1
            const int r = 3 * i + j;       // concat buffer / RDB index
            const float* D = dbuf[jj];
            // Data gradient of the block as a MIRRORED DENSE BLOCK. The five output gradients live side by side in ONE
            // 192-channel buffer, latest layer first,
            //     dYcat' = [dY5 (64) | dY4 (32) | dY3 | dY2 | dY1]
            // (three buffers rotate across blocks). The gradient of out_b needs every later layer's dY, which is exactly a
            // channel PREFIX of dYcat': step b = 4, 3, 2, 1 is a convolution 64 / 96 / 128 / 160 -> 32 with the
            // mirrored packs (generator.cu pack_rdb_bwd_kernel), masked by LeakyReLU'(out_b) and written in place as
            // the next 32 channels; step 0 is 192 -> 64 and yields d(block input). Same launch shapes as the forward
            // block, all accumulation over layers happens in the MMA's K dimension: the fp32 gradient buffer that
            // round 1 read and re-wrote once per layer (210 MB per block) and its 20 K = 32 / 64 output slices are gone.
            // dY5 = 0.2 * d(xout) is already in channels 0..63 of this block's buffer: the convolution that produced
            // d(xout) (the previous block's step 0, or conv2's data gradient for the first block) stored it as its scaled
            // 16-bit output. Three buffers rotate, so a buffer's previous reader (the weight gradient of block r + 3) is long done.
            uint16_t* dyc = B.dycat[r % 3];
            cudaStream_t wst = wgrad_stream(g, s);
            for (int b = 4; b >= 0; --b) {
                const ConvSpec& shape = table().c[1 + 5 * r + (4 - b)];   // step b has the shape of forward conv(5 - b)
                ConvIO io;
                io.wpack = g->wpack_t2 + shape.w_off; io.bias = g->zero_bias;
                io.nout = shape.nout; io.nslices = shape.nslices; io.nchunks = shape.nchunks; io.fmt = 1;
                io.kvalid = 64 + 32 * (4 - b);
                io.in16 = dyc; io.in_c = 192;
                if (b > 0) {   // dY_b = LeakyReLU'(out_b) * (sum over later layers), bf16, next 32 channels of dYcat'
                    io.out16 = dyc; io.out16_c = 192; io.out16_choff = 64 + 32 * (4 - b); io.out16_fmt = 1;
                    io.mask16 = B.c[r]; io.mask16_c = 192; io.mask16_choff = 64 + 32 * (b - 1);
                } else {       // d(xin) = sum over the five layers + d(xout) * (1 or 0.2)   (model.py:94-96, 129-130)
                    io.ep_mode = EP_ADD2;
                    io.res2 = D; io.res2_c = 64; io.res2_scale = dscale[jj];
                    io.outf = dxin[jj]; io.outf_c = 64;
                    if (jj == 2) {   // rdb1: d(x0) = d(rdb1 input) + d(out) (model.py:129-130) accumulated in place into dx[0]
                        io.res1 = B.dx[0]; io.res1_c = 64;
                        io.outf = B.dx[0];
                    }
                    if (r > 0) {     // ... and the next block's dY5 = 0.2 * (its d(xout)) [* 0.2 for an rdb3], bf16
                        const int rn = (r - 1) % 3;
                        if (wst != s && g->ev_dyc_valid[rn]) cudaStreamWaitEvent(s, g->ev_dyc[rn], 0);   // its previous reader is done
                        io.out16 = B.dycat[rn]; io.out16_c = 192; io.out16_choff = 0; io.out16_fmt = 1;
                        io.out16_scale = jj == 2 ? 0.2f * 0.2f : 0.2f;
                    }
                }
                RESR_TRY(launch_conv_io(g, g0, N, io, s));
            }
            {   // weight + bias gradients of the five layers (side stream): dYcat is complete once conv2's launch is done
                fork_to(g, s, wst);
                if (g->precision == 1) {
                    // bf16 recipe: ONE MN-major GEMM straight from the concat buffer and dYcat' (no transposed copies).
                    // Units (128 ci x n co'): [0,128) x [0,128), [0,128) x [128,192), [128,192(+64 zero rows)) x [0,128);
                    // the reduction keeps ci < cin of the layer owning each 32-channel slice of dYcat'.
                    WgradMnTable tb;
                    for (int cs = 0; cs < 6; ++cs) {
                        const int kl = 1 + 5 * r + (cs < 2 ? 4 : 5 - cs);
                        const ConvSpec& c = table().c[kl];
                        tb.dw[cs] = grads + c.p_off;
                        tb.db[cs] = grads + c.p_off + static_cast<size_t>(c.cout) * c.cin * 9;
                        tb.cin[cs] = c.cin; tb.cout[cs] = c.cout;
                        tb.co_base[cs] = cs < 2 ? cs * 32 : 0;
                    }
                    const int units[3][3] = {{0, 0, 128}, {0, 128, 64}, {128, 0, 128}};
                    const int rc = wgrad_mn_launch(B.c[r], 192, 192, dyc, 192, 192, N, H, W, units, 3, tb, true, B.partial, g->num_sms, wst);
                    if (rc != 0) return set_error(RESR_E_CUDA, "dense-block wgrad (nhwc) failed (%d)", rc);
                    if (wst != s) {
                        cudaEventRecord(g->ev_dyc[r % 3], wst);
                        g->ev_dyc_valid[r % 3] = true;
                    }
                    continue;
                }
                const dim3 tg(static_cast<unsigned>((P + 255) / 256), 6);
                nhwc16_to_cf_kernel<false><<<tg, 256, 0, wst>>>(B.c[r], 192, 0, 192, 192, P, W, 0, B.xt, nullptr);
                cudaMemsetAsync(B.dbcat, 0, 192 * sizeof(float), wst);
                nhwc16_to_cf_kernel<true><<<tg, 256, 0, wst>>>(dyc, 192, 0, 192, 192, P, W, 1, B.dyt, B.dbcat);
                if (wst != s) {
                    cudaEventRecord(g->ev_dyc[r % 3], wst);
                    g->ev_dyc_valid[r % 3] = true;
                }
                WgradRdbTable tb;
                for (int cs = 0; cs < 6; ++cs) {   // slices of dYcat': conv5 (two halves), conv4, conv3, conv2, conv1
                    const int kl = 1 + 5 * r + (cs < 2 ? 4 : 5 - cs);
                    const ConvSpec& c = table().c[kl];
                    tb.dw[cs] = grads + c.p_off;
                    tb.cin[cs] = c.cin;
                    tb.co_base[cs] = cs < 2 ? cs * 32 : 0;
                    tb.db[cs] = grads + c.p_off + static_cast<size_t>(c.cout) * c.cin * 9 + tb.co_base[cs];
                }
                tb.dbcat = B.dbcat;
                // (giving the two chains disjoint SM subsets instead of letting them interleave was tried: 22.6 - 24.4 ms
                // against 21.5 ms, profiles/r02_train_sm_partition_ab.txt)
                const int rc = wgrad_launch_rdb(B.xt, B.dyt, N, H, W, B.partial, tb, g->num_sms, wst);
                if (rc != 0) return set_error(RESR_E_CUDA, "dense-block wgrad failed (%d)", rc);
            }
        }
        for (int bi = 0; bi < 3; ++bi)   // every gradient from RRDB i upwards has been enqueued on the weight-gradient stream
            if (i == kBucketRRDB[bi]) record_bucket(g, bi, wgrad_stream(g, s));
        // (d(x0) = d(rdb1 input) + d(out), model.py:129-130, was accumulated in place by rdb1's last convolution)
    }
    // ---- conv1 (model.py:258): dY = d(trunk input) + d(skip)
    scale_f32_to_bf16_kernel<<<egrid(P * 64), 256, 0, s>>>(B.dx[0], 1.f, B.dskip, 1.f, B.dya, P * 64);
    RESR_TRY(layer_wgrad(g, 0, B.xin, 64, g->precision, false, 0, B.dya, N, g0, B, grads, s));
    if (g->side_stream && wgrad_stream(g, s) != s) {  // join: the gradient vector is complete when the main stream continues
        cudaEventRecord(g->ev_join, g->side_stream);
        cudaStreamWaitEvent(s, g->ev_join, 0);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "backward: %s", cudaGetErrorString(e));
    return RESR_OK;
}

int check_train_args(resr_generator_t* g, int n, int h, int w, void* ws, size_t ws_bytes) {
    if (!g || !ws) return set_error(RESR_E_INVALID, "null argument");
    if (n <= 0 || h <= 0 || w <= 0) return set_error(RESR_E_INVALID, "bad shape");
    if (g->precision != 1 && w % 8 != 0)
        return set_error(RESR_E_INVALID, "the fp16 training recipe needs W %% 8 == 0 (channels-first TMA strides), got %d; the bf16 recipe has no such limit", w);
    if (!g->loaded || !g->flat_params) return set_error(RESR_E_INVALID, "resr_generator_load_params has not been called");
    if (ws_bytes < resr_generator_train_workspace_bytes(n, h, w)) return set_error(RESR_E_NOMEM, "training workspace too small");
    if ((reinterpret_cast<uintptr_t>(ws) & 1023) != 0) return set_error(RESR_E_INVALID, "workspace must be 1024-byte aligned");
    return RESR_OK;
}

}  // namespace

extern "C" {

size_t resr_generator_train_workspace_bytes(int n, int h, int w) {
    if (n <= 0 || h <= 0 || w <= 0) return 0;
    return train_layout(n, h, w, 160).total;
}

int resr_generator_forward_train(resr_generator_t* g, const float* x, float* y, int n, int h, int w, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    RESR_TRY(check_train_args(g, n, h, w, workspace, workspace_bytes));
    if (!x || !y) return set_error(RESR_E_INVALID, "null argument");
    const Bufs B = carve(workspace, train_layout(n, h, w, 160));
    return forward_train(g, x, y, n, h, w, B, static_cast<cudaStream_t>(stream));
}

int resr_generator_backward_l1(resr_generator_t* g, const float* hr, float* grads_flat, float* loss_out, int n, int h, int w,
                               void* workspace, size_t workspace_bytes, void* stream) {
    RESR_TRY(check_train_args(g, n, h, w, workspace, workspace_bytes));
    if (!hr || !grads_flat) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const Bufs B = carve(workspace, train_layout(n, h, w, 160));
    const size_t HW = static_cast<size_t>(16) * h * w;
    const double numel = static_cast<double>(n) * 3 * HW;
    cudaMemsetAsync(B.loss, 0, sizeof(double), s);
    out_grad_kernel<<<egrid(static_cast<size_t>(n) * HW), 256, 0, s>>>(B.yraw, hr, B.biga, B.loss, n, HW, static_cast<float>(1.0 / numel), 0);
    if (loss_out) finish_loss_kernel<<<1, 1, 0, s>>>(B.loss, loss_out, 1.0 / numel);
    return backward_common(g, grads_flat, n, h, w, B, s);
}

int resr_generator_backward(resr_generator_t* g, const float* dy, float* grads_flat, int n, int h, int w, void* workspace,
                            size_t workspace_bytes, void* stream) {
    RESR_TRY(check_train_args(g, n, h, w, workspace, workspace_bytes));
    if (!dy || !grads_flat) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const Bufs B = carve(workspace, train_layout(n, h, w, 160));
    const size_t HW = static_cast<size_t>(16) * h * w;
    out_grad_kernel<<<egrid(static_cast<size_t>(n) * HW), 256, 0, s>>>(B.yraw, dy, B.biga, nullptr, n, HW, 0.f, 1);
    return backward_common(g, grads_flat, n, h, w, B, s);
}

int resr_generator_train_step_l1(resr_generator_t* g, const float* x, const float* hr, float* y, float* grads_flat, float* loss_out,
                                 int n, int h, int w, void* workspace, size_t workspace_bytes, void* stream) {
    RESR_TRY(check_train_args(g, n, h, w, workspace, workspace_bytes));
    if (!x || !hr || !y || !grads_flat) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const void* key[6] = {x, hr, y, grads_flat, loss_out, workspace};
    const bool same = g->step_exec && memcmp(key, g->step_key, sizeof(key)) == 0 && g->step_shape[0] == n && g->step_shape[1] == h &&
                      g->step_shape[2] == w && g->step_precision == g->precision;
    if (same) {
        const cudaError_t e = cudaGraphLaunch(g->step_exec, s);
        if (e != cudaSuccess) return set_error(RESR_E_CUDA, "cudaGraphLaunch: %s", cudaGetErrorString(e));
        return RESR_OK;
    }
    auto eager = [&]() -> int {
        RESR_TRY(resr_generator_forward_train(g, x, y, n, h, w, workspace, workspace_bytes, stream));
        return resr_generator_backward_l1(g, hr, grads_flat, loss_out, n, h, w, workspace, workspace_bytes, stream);
    };
    // first call with these arguments: run once eagerly (allocations, function attributes, transposed packs), then
    // capture the identical launch sequence (~2400 kernels) into a graph that later calls replay
    RESR_TRY(eager());
    if (g->step_graph_failed || getenv("RESR_NO_GRAPH")) return RESR_OK;
    if (cudaStreamSynchronize(s) != cudaSuccess) return set_error(RESR_E_CUDA, "train step failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (g->step_exec) { cudaGraphExecDestroy(g->step_exec); g->step_exec = nullptr; }
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); g->step_graph_failed = true; return RESR_OK; }
    const int rc = eager();
    const cudaError_t ec = cudaStreamEndCapture(s, &graph);
    if (rc != RESR_OK || ec != cudaSuccess || !graph) {
        cudaGetLastError();
        if (graph) cudaGraphDestroy(graph);
        g->step_graph_failed = true;  // keep running eagerly (the eager result above is already valid)
        return RESR_OK;
    }
    const cudaError_t ei = cudaGraphInstantiate(&g->step_exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ei != cudaSuccess) { cudaGetLastError(); g->step_exec = nullptr; g->step_graph_failed = true; return RESR_OK; }
    memcpy(g->step_key, key, sizeof(key));
    g->step_shape[0] = n; g->step_shape[1] = h; g->step_shape[2] = w;
    g->step_precision = g->precision;
    return RESR_OK;
}

int resr_generator_step_is_graph(resr_generator_t* g) { return g && g->step_exec ? 1 : 0; }

int resr_generator_grad_buckets(size_t* offsets, int max_entries) {
    if (!offsets || max_entries < 5) return set_error(RESR_E_INVALID, "need room for 5 offsets");
    const Table& T = table();
    // layer index of the first convolution of RRDB i: 1 + 15 * i (conv1 is layer 0, 15 convolutions per RRDB)
    offsets[0] = 0;
    offsets[1] = T.c[1 + 15 * kBucketRRDB[2]].p_off;
    offsets[2] = T.c[1 + 15 * kBucketRRDB[1]].p_off;
    offsets[3] = T.c[1 + 15 * kBucketRRDB[0]].p_off;
    offsets[4] = T.n_params;
    return 4;
}

int resr_generator_wait_grad_bucket(resr_generator_t* g, int bucket, void* stream) {
    if (!g || bucket < 0 || bucket > 3) return set_error(RESR_E_INVALID, "bad bucket");
    if (bucket == 0) return RESR_OK;                       // the front of the vector (conv1 ... trunk.4) completes with the step itself
    cudaEvent_t ev = g->ev_bucket[3 - bucket];             // bucket 3 (the end of the vector) is closed by the first event
    if (!ev) return set_error(RESR_E_INVALID, "no training step has recorded bucket %d yet", bucket);
    const cudaError_t e = cudaStreamWaitEvent(static_cast<cudaStream_t>(stream), ev, 0);
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "cudaStreamWaitEvent: %s", cudaGetErrorString(e));
    return RESR_OK;
}

int resr_conv3x3_wgrad(const void* x16, int x_cstride, int fmt_x, const void* dy16_bf16, int n, int h, int w, int cin, int cout,
                       float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream) {
    if (!x16 || !dy16_bf16 || !dw || !workspace) return set_error(RESR_E_INVALID, "null argument");
    if (w % 8 != 0 || cout > 64 || cin > x_cstride) return set_error(RESR_E_INVALID, "unsupported wgrad shape");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t P = static_cast<size_t>(n) * h * w;
    const int xr = (cin + 31) / 32 * 32, yr = (cout + 31) / 32 * 32;
    const size_t need = up1k(P * xr * 2) + up1k(3 * P * yr * 2) + wgrad_partial_bytes(160);
    if (workspace_bytes < need) return set_error(RESR_E_NOMEM, "wgrad workspace too small (need %zu)", need);
    uint16_t* xt = static_cast<uint16_t*>(workspace);
    uint16_t* dyt = reinterpret_cast<uint16_t*>(static_cast<uint8_t*>(workspace) + up1k(P * xr * 2));
    float* partial = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(dyt) + up1k(3 * P * yr * 2));
    nhwc16_to_cf_kernel<false><<<dim3(static_cast<unsigned>((P + 255) / 256), xr / 32), 256, 0, s>>>(static_cast<const uint16_t*>(x16), x_cstride, 0, cin, xr, P, w, fmt_x, xt, nullptr);
    if (db) cudaMemsetAsync(db, 0, cout * sizeof(float), s);
    nhwc16_to_cf_kernel<true><<<dim3(static_cast<unsigned>((P + 255) / 256), yr / 32), 256, 0, s>>>(static_cast<const uint16_t*>(dy16_bf16), 64, 0, cout, yr, P, w, 1, dyt, db);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int rc = wgrad_launch(xt, xr, dyt, yr, n, h, w, cin, cout, partial, dw, nullptr, sms, s);
    if (rc != 0) return set_error(RESR_E_CUDA, "wgrad failed (%d)", rc);
    return RESR_OK;
}

size_t resr_conv3x3_wgrad_nhwc_workspace_bytes(void) { return wgrad_mn_workspace_bytes(160) + 1024; }

int resr_conv3x3_wgrad_nhwc(const void* x_bf16, int x_cstride, const void* dy_bf16, int dy_cstride, int n, int h, int w, int cin, int cout,
                            float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream) {
    if (!x_bf16 || !dy_bf16 || !dw || !workspace) return set_error(RESR_E_INVALID, "null argument");
    if (n <= 0 || h <= 0 || w <= 0 || cin <= 0 || cout <= 0 || cin > 256 || cout > 192 || cin > x_cstride || cout > dy_cstride ||
        (x_cstride & 7) || (dy_cstride & 7))
        return set_error(RESR_E_INVALID, "unsupported wgrad shape (cin <= 256, cout <= 192, channel strides multiples of 8)");
    if (workspace_bytes < resr_conv3x3_wgrad_nhwc_workspace_bytes()) return set_error(RESR_E_NOMEM, "wgrad workspace too small");
    if ((reinterpret_cast<uintptr_t>(workspace) & 15) != 0) return set_error(RESR_E_INVALID, "workspace must be 16-byte aligned");
    int units[4][3], nu = 0;
    for (int ci0 = 0; ci0 < cin; ci0 += 128)
        for (int co0 = 0; co0 < cout;) {
            const int nn = cout - co0 > 64 ? 128 : 64;
            units[nu][0] = ci0; units[nu][1] = co0; units[nu][2] = nn; ++nu;
            co0 += nn;
        }
    WgradMnTable tb;
    for (int cs = 0; cs < 6; ++cs) { tb.dw[cs] = dw; tb.db[cs] = db; tb.cin[cs] = cin; tb.cout[cs] = cout; tb.co_base[cs] = cs * 32; }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms > 160) sms = 160;
    int dyc = (cout + 7) / 8 * 8;
    if (dyc > dy_cstride) dyc = dy_cstride;
    const int rc = wgrad_mn_launch(static_cast<const uint16_t*>(x_bf16), x_cstride, cin, static_cast<const uint16_t*>(dy_bf16), dy_cstride, dyc,
                                   n, h, w, units, nu, tb, db != nullptr, static_cast<float*>(workspace), sms, static_cast<cudaStream_t>(stream));
    if (rc != 0) return set_error(RESR_E_CUDA, "wgrad (nhwc) failed (%d)", rc);
    return RESR_OK;
}

size_t resr_conv3x3_wgrad_workspace_bytes(int n, int h, int w, int cin, int cout) {
    const size_t P = static_cast<size_t>(n) * h * w;
    const int xr = (cin + 31) / 32 * 32, yr = (cout + 31) / 32 * 32;
    return up1k(P * xr * 2) + up1k(3 * P * yr * 2) + wgrad_partial_bytes(160);
}

}  // extern "C"
