// Hot path 2: second-order degradation ops as CUDA kernels for sm_100a (fp32 NCHW images, as the reference holds
// them). Reference: /root/reference/imgproc.py (filter2d_torch :1089, USMSharp :1514, noise :829-1086, DiffJPEG
// :1124-1494, random_crop :1894) and the sequencing in train_realesrnet.py:267-377. See DESIGN.md §5.
#include <curand_kernel.h>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "../../include/resr.h"
#include "device_state.h"
#include "errors.h"
#include "ptx.cuh"

namespace resr {

// Every kernel of this file is launched with programmatic stream serialization (PDL) and starts with griddepcontrol.wait:
// inside the degradation chain (a CUDA graph of ~15 dependent launches of 3 - 50 us each) the next kernel's blocks are
// scheduled while the previous kernel drains, instead of after a full launch round trip per edge.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    static const bool no_pdl = getenv("RESR_NO_PDL") != nullptr;   // A/B switch (profiles/r02_degrade_pdl_ab.txt)
    cfg.attrs = at; cfg.numAttrs = no_pdl ? 0 : 1;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

#define RESR_LAUNCH_CHECK(what)                                                                   \
    do {                                                                                          \
        const cudaError_t e__ = cudaGetLastError();                                               \
        if (e__ != cudaSuccess) return set_error(RESR_E_CUDA, what ": %s", cudaGetErrorString(e__)); \
    } while (0)

__device__ __forceinline__ int reflect_idx(int i, int n) {  // ATen reflection_pad2d rule (imgproc.py:1104)
    i = i < 0 ? -i : i;
    return i >= n ? 2 * (n - 1) - i : i;
}

// a / b and a % b in 32-bit arithmetic whenever the dividend fits: a 64-bit division is a ~100-instruction subroutine, and
// the elementwise kernels below decode one linear index per element
__device__ __forceinline__ size_t div_u(size_t a, unsigned b) {
    return a <= 0xffffffffull ? static_cast<size_t>(static_cast<unsigned>(a) / b) : a / b;
}
__device__ __forceinline__ unsigned mod_u(size_t a, unsigned b) {
    return a <= 0xffffffffull ? static_cast<unsigned>(a) % b : static_cast<unsigned>(a % b);
}

// ===================================================================================== filter2d (a8)
// One block = 64 x (8 * R) output tile of one (sample, channel) plane; 256 threads = 32 columns x 8 row groups, each
// thread owns R consecutive rows of 2 columns (x and x+32). The reflect-padded halo tile and the taps live in shared
// memory. The kernels of the degradation model are 7..21 supports zero-padded to 21 (dataset.py:102-103): the block
// finds the centred square support KS of its sample and runs the KS-specialised body, whose (row, output) loops are fully
// unrolled with the current tap column in registers: 2*R*KS FMAs per (2*(KS+R-1) + KS) shared loads.
// R is chosen per launch so that small images still fill the GPU: 8 rows per thread at 256^2 (768 blocks at cfg2),
// 4 at 128^2, 2 at 64^2 (the 64 x 64 tile of round 1 left 100 of the 148 SMs idle there).
static constexpr int kF2dTileW = 64;

// The two columns of a thread (x, x + 32) ride in ONE packed fp32x2 FMA (Blackwell FFMA2, `__ffma2_rn`: two IEEE fmas per
// instruction, the tap broadcast to both halves by the operand selector): the same arithmetic bit for bit in half the issue
// slots. ncu had this kernel issue-bound (issue slots 78 % busy, FMA pipe 48 %, 60 % of the instructions FMAs).
template <int KS, int R, int tpitch>
__device__ __forceinline__ void filter2d_body(const float* __restrict__ tile, const float* __restrict__ taps, int k,
                                              int off, int tx, int ty0, float2 (&acc)[R]) {
    // taps: full k x k array; the KS x KS centred window starts at (off, off). tile row 0 / col 0 correspond to output
    // (0,0) shifted by -(k/2); the window adds `off` again.
    for (int kx = 0; kx < KS; ++kx) {
        float w[KS];
#pragma unroll
        for (int ky = 0; ky < KS; ++ky) w[ky] = taps[(off + ky) * k + off + kx];
        const float* col = tile + (ty0 + off) * tpitch + tx + off + kx;
#pragma unroll
        for (int rr = 0; rr < KS + R - 1; ++rr) {
            const float2 v = make_float2(col[rr * tpitch], col[rr * tpitch + 32]);
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const int ky = rr - j;
                if (ky >= 0 && ky < KS) acc[j] = __ffma2_rn(v, make_float2(w[ky], w[ky]), acc[j]);
            }
        }
    }
}

// PITCH: row pitch of the shared-memory tile, a compile-time constant so that the (fully unrolled) window loads carry
// immediate offsets instead of one address computation each: 85 for k <= 21 (the degradation model), 127 up to k = 63.
template <int R, int PITCH>
__global__ void __launch_bounds__(R == 16 ? 128 : 256) filter2d_kernel(const float* __restrict__ in, const float* __restrict__ kern,
                                                       float* __restrict__ out, int B, int C, int H, int W, int k,
                                                       int kern_batched) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    constexpr int NW = R == 16 ? 4 : 8;   // warps per block
    constexpr int TH = NW * R;            // tile height
    extern __shared__ float sm[];
    const int r = k / 2;
    const int tw = kF2dTileW + k - 1, th = TH + k - 1;
    constexpr int tpitch = PITCH;
    float* tile = sm;                  // [th][PITCH]
    float* taps = sm + th * tpitch;    // [k][k]
    __shared__ int s_ext;              // max |offset from centre| of a non-zero tap
    const int plane = blockIdx.z;      // b * C + c
    const int b = plane / C;
    const int x0 = blockIdx.x * kF2dTileW, y0 = blockIdx.y * TH;
    const float* src = in + static_cast<size_t>(plane) * H * W;
    const float* kp = kern + (kern_batched ? static_cast<size_t>(b) * k * k : 0);
    if (threadIdx.x == 0) s_ext = 0;
    __syncthreads();
    int ext_mine = 0;                  // per-thread, then per-warp maximum: ONE shared atomic per warp (a dense 21 x 21 sinc
    for (int i = threadIdx.x; i < k * k; i += blockDim.x) {   // kernel used to serialise 441 of them per block)
        const float v = kp[i];
        taps[i] = v;
        if (v != 0.f) ext_mine = max(ext_mine, max(abs(i / k - r), abs(i % k - r)));
    }
    ext_mine = __reduce_max_sync(0xffffffffu, ext_mine);
    if ((threadIdx.x & 31) == 0 && ext_mine > 0) atomicMax(&s_ext, ext_mine);
    __syncthreads();
    const int ext = s_ext;
    const int off = r - ext;           // first row/col of the centred support inside the k x k array
    {   // only the halo the trimmed support needs is fetched: tile rows [off, th - off) / columns [off, tw - off). One tile
        // row per warp pass, coalesced along x; the reflected columns of this lane are computed once. Positions the tile
        // overhang would touch beyond the image are clamped: their outputs are never stored.
        const int lane = threadIdx.x & 31;
        int cxk[4];          // tw <= 64 + 62
#pragma unroll
        for (int q = 0; q < 4; ++q) cxk[q] = min(max(reflect_idx(x0 + off + lane + 32 * q - r, W), 0), W - 1);
        const int span = tw - 2 * off;
        for (int ty = off + (threadIdx.x >> 5); ty < th - off; ty += 2 * NW) {  // two rows (8 loads per lane) in flight
            float v[2][4];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int cy = min(max(reflect_idx(y0 + min(ty + u * NW, th - off - 1) - r, H), 0), H - 1);
                const float* srow = src + static_cast<size_t>(cy) * W;
#pragma unroll
                for (int q = 0; q < 4; ++q) v[u][q] = srow[cxk[q]];
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                if (ty + u * NW < th - off) {
                    float* trow = tile + (ty + u * NW) * tpitch + off;
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (lane + 32 * q < span) trow[lane + 32 * q] = v[u][q];
                }
            }
        }
    }
    __syncthreads();
    const int tx = threadIdx.x & 31;
    const int ty0 = (threadIdx.x >> 5) * R;   // NW warps x R rows
    float2 acc[R];   // .x: column tx, .y: column tx + 32
#pragma unroll
    for (int j = 0; j < R; ++j) acc[j] = make_float2(0.f, 0.f);
    switch (2 * ext + 1) {
        case 1: filter2d_body<1, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 3: filter2d_body<3, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 5: filter2d_body<5, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 7: filter2d_body<7, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 9: filter2d_body<9, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 11: filter2d_body<11, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 13: filter2d_body<13, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 15: filter2d_body<15, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 17: filter2d_body<17, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 19: filter2d_body<19, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        case 21: filter2d_body<21, R, PITCH>(tile, taps, k, off, tx, ty0, acc); break;
        default: {  // generic odd support (k <= 63): rolled loops
            const int ks = 2 * ext + 1;
            for (int kx = 0; kx < ks; ++kx)
                for (int rr = 0; rr < ks + R - 1; ++rr) {
                    const float v0 = tile[(ty0 + off + rr) * tpitch + tx + off + kx];
                    const float v1 = tile[(ty0 + off + rr) * tpitch + tx + 32 + off + kx];
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        const int ky = rr - j;
                        if (ky >= 0 && ky < ks) {
                            const float wv = taps[(off + ky) * k + off + kx];
                            acc[j].x = fmaf(v0, wv, acc[j].x);
                            acc[j].y = fmaf(v1, wv, acc[j].y);
                        }
                    }
                }
        }
    }
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const int gx = x0 + tx + 32 * c;
        if (gx < W) {
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const int gy = y0 + ty0 + j;
                if (gy < H) out[static_cast<size_t>(plane) * H * W + static_cast<size_t>(gy) * W + gx] = c ? acc[j].y : acc[j].x;
            }
        }
    }
}

template <int R>
static void filter2d_launch(const float* in, const float* kern, float* out, int B, int C, int H, int W, int k, int kb,
                            cudaStream_t s) {
    constexpr int NW = R == 16 ? 4 : 8;
    constexpr int TH = NW * R;
    const int th = TH + k - 1;
    dim3 grid((W + kF2dTileW - 1) / kF2dTileW, (H + TH - 1) / TH, B * C);
    if (k <= 21) {
        const size_t smem = (static_cast<size_t>(th) * 85 + static_cast<size_t>(k) * k) * sizeof(float);
        static PerDevice<size_t> attr_set;  // function attributes are per device
        if (smem > 48 * 1024 && smem > attr_set.cur()) {
            cudaFuncSetAttribute(filter2d_kernel<R, 85>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            attr_set.cur() = smem;
        }
        launch_pdl(filter2d_kernel<R, 85>, grid, 32 * NW, smem, s, in, kern, out, B, C, H, W, k, kb);
    } else {
        const size_t smem = (static_cast<size_t>(th) * 127 + static_cast<size_t>(k) * k) * sizeof(float);
        static PerDevice<size_t> attr_set;
        if (smem > 48 * 1024 && smem > attr_set.cur()) {
            cudaFuncSetAttribute(filter2d_kernel<R, 127>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            attr_set.cur() = smem;
        }
        launch_pdl(filter2d_kernel<R, 127>, grid, 32 * NW, smem, s, in, kern, out, B, C, H, W, k, kb);
    }
}

static int filter2d_impl(const float* in, const float* kern, float* out, int B, int C, int H, int W, int k, int kb,
                         cudaStream_t s) {
    if (k % 2 != 1) return set_error(RESR_E_INVALID, "Wrong kernel size.");  // imgproc.py:1106 ValueError
    if (k > 63) return set_error(RESR_E_INVALID, "kernel size %d > 63 unsupported", k);
    if (k / 2 >= H || k / 2 >= W) return set_error(RESR_E_INVALID, "reflect padding %d needs a larger image (%dx%d)", k / 2, H, W);
    // rows per thread: 16 (64 x 64 tile, 128 threads: 32*KS FMAs per 3*KS+30 shared loads, the stencil is shared-memory
    // bandwidth bound below ~4 FMAs per load) when that still gives ~4 blocks per SM, else the largest of 8 / 4 / 2 that
    // gives ~2 blocks per SM
    const long long cols = (W + kF2dTileW - 1) / kF2dTileW, planes = static_cast<long long>(B) * C;
    auto blocks = [&](int R) { return cols * ((H + 8 * R - 1) / (8 * R)) * planes; };
    static const int env_r16 = getenv("RESR_F2D_R16") ? atoi(getenv("RESR_F2D_R16")) : 0;  // measured: no faster than 8
    if (env_r16 && cols * ((H + 63) / 64) * planes >= 592) filter2d_launch<16>(in, kern, out, B, C, H, W, k, kb, s);
    else if (blocks(8) >= 296) filter2d_launch<8>(in, kern, out, B, C, H, W, k, kb, s);
    else if (blocks(4) >= 296) filter2d_launch<4>(in, kern, out, B, C, H, W, k, kb, s);
    else filter2d_launch<2>(in, kern, out, B, C, H, W, k, kb, s);
    RESR_LAUNCH_CHECK("filter2d");
    return RESR_OK;
}

// ===================================================================================== USM sharpen (a7)
// The 51 x 51 kernel is an exact outer product (imgproc.py:1522-1523), so both blurs run as a horizontal and a
// vertical 51-tap pass. Taps: cv2.getGaussianKernel(51, 0) restated on the host in double, stored as fp32.
static constexpr int kUsmMaxTaps = 129;
__constant__ float c_usm_taps[kUsmMaxTaps];

// out = conv_x(in) with reflect padding; one block = one row segment of 256 outputs.
__global__ void __launch_bounds__(256) usm_hpass_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W,
                                                        int k) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    extern __shared__ float row[];
    const int r = k / 2;
    const size_t line = static_cast<size_t>(blockIdx.z) * H + blockIdx.y;
    const int x0 = blockIdx.x * 256;
    const float* src = in + line * W;
    for (int i = threadIdx.x; i < 256 + k - 1; i += 256) {
        const int gx = reflect_idx(x0 + i - r, W);
        row[i] = src[min(max(gx, 0), W - 1)];
    }
    __syncthreads();
    const int x = x0 + threadIdx.x;
    if (x < W) {
        float acc = 0.f;
        for (int t = 0; t < k; ++t) acc = fmaf(row[threadIdx.x + t], c_usm_taps[t], acc);
        out[line * W + x] = acc;
    }
}

// Vertical pass over a 32-wide x 64-tall output tile, then the fused pointwise tail.
//   stage 0: blur = conv_y(tmp); res = x - blur; mask = |res| * 255 > threshold     -> res_out, mask_out
//   stage 1: soft = conv_y(tmp); out = soft * clip(x + weight * res, 0, 1) + (1 - soft) * x
__global__ void __launch_bounds__(256) usm_vpass_kernel(const float* __restrict__ tmp, const float* __restrict__ x,
                                                        float* __restrict__ res, float* __restrict__ mask_or_out, int H,
                                                        int W, int k, int stage, float weight, float threshold,
                                                        float* __restrict__ soft_out) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    extern __shared__ float tile[];  // [64 + k - 1][32]
    const int r = k / 2;
    const int plane = blockIdx.z;
    const int x0 = blockIdx.x * 32, y0 = blockIdx.y * 64;
    const size_t pbase = static_cast<size_t>(plane) * H * W;
    const int tx = threadIdx.x & 31, tyb = threadIdx.x >> 5;  // 8 row groups
    const int gx = min(x0 + tx, W - 1);
    for (int i = tyb; i < 64 + k - 1; i += 8) {
        const int gy = reflect_idx(y0 + i - r, H);
        tile[i * 32 + tx] = tmp[pbase + static_cast<size_t>(min(max(gy, 0), H - 1)) * W + gx];
    }
    __syncthreads();
    if (x0 + tx >= W) return;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
        const int ly = tyb * 8 + j;
        const int gy = y0 + ly;
        if (gy >= H) break;
        float acc = 0.f;
        for (int t = 0; t < k; ++t) acc = fmaf(tile[(ly + t) * 32 + tx], c_usm_taps[t], acc);
        const size_t o = pbase + static_cast<size_t>(gy) * W + x0 + tx;
        const float xv = x[o];
        if (stage == 0) {
            const float rv = xv - acc;                                     // imgproc.py:1528
            res[o] = rv;
            mask_or_out[o] = (fabsf(rv) * 255.f > threshold) ? 1.f : 0.f;  // imgproc.py:1530-1531
        } else {
            const float rv = res[o];
            float sh = __fadd_rn(xv, __fmul_rn(weight, rv));                // imgproc.py:1533 (separate mul, add)
            sh = fminf(fmaxf(sh, 0.f), 1.f);                               // imgproc.py:1534
            mask_or_out[o] = __fadd_rn(__fmul_rn(acc, sh), __fmul_rn(1.f - acc, xv));  // imgproc.py:1535
            if (soft_out) soft_out[o] = acc;   // kept for the backward pass (resr_usm_sharp_backward)
        }
    }
}

// The 51-tap case the training loops use (USMSharp(50, 0)): each blur is a horizontal pass into a scratch image (it
// stays in the 126 MB L2) and a vertical pass with the pointwise tail fused. Both passes are plain 1-D stencils with NO
// recomputation. A thread slides a register window over 8 consecutive outputs ALONG the filter direction for TWO
// independent lines at once (two rows in the horizontal pass, two columns in the vertical one): the two lines share every
// tap, so each step is one packed fp32x2 FMA (FFMA2, tap broadcast by the operand selector) -- 408 packed FMAs + 116
// conflict-free shared loads per 16 outputs, taps in uniform registers. The lane index runs ACROSS the filter direction
// (horizontal pass: lane = row, odd row pitch; vertical pass: lane = column). Global loads are issued in batches ahead
// of their use (ncu showed the first version of these kernels waiting on the long scoreboard for most of its cycles).
static constexpr int kUsmK = 51, kUsmR = kUsmK / 2, kUsmO = 8;   // outputs per thread and line
static constexpr int kUsmHCols = 64, kUsmHRows = 64, kUsmHPitch = kUsmHCols + kUsmK - 1 + 1;  // 115: odd
static constexpr int kUsmVCols = 64, kUsmVRows = 64, kUsmVIn = kUsmVRows + kUsmK - 1;         // 114 input rows

__device__ __forceinline__ void usm_window8x2(const float* __restrict__ p0, const float* __restrict__ p1, int stride,
                                              float2 (&acc)[kUsmO]) {
#pragma unroll
    for (int j = 0; j < kUsmO; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
    for (int t = 0; t < kUsmK + kUsmO - 1; ++t) {
        const float2 v = make_float2(p0[t * stride], p1[t * stride]);
#pragma unroll
        for (int j = 0; j < kUsmO; ++j) {
            const int tap = t - j;
            if (tap >= 0 && tap < kUsmK) acc[j] = __ffma2_rn(v, make_float2(c_usm_taps[tap], c_usm_taps[tap]), acc[j]);
        }
    }
}

// tmp = conv_x(src), reflect padding. Block = 64 rows x 64 columns of outputs, 256 threads: lane = rows (l, l + 32),
// warp = 8 columns.
__global__ void __launch_bounds__(256) usm_h51_kernel(const float* __restrict__ src, float* __restrict__ tmp, int H, int W) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    __shared__ float A[kUsmHRows * kUsmHPitch];
    const int plane = blockIdx.z;
    const int x0 = blockIdx.x * kUsmHCols, y0 = blockIdx.y * kUsmHRows;
    const size_t pbase = static_cast<size_t>(plane) * H * W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    {   // tile rows: warp w takes rows w, w+8, ...; 4 rows (16 loads per lane) in flight, coalesced along x
        int gxk[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) gxk[k] = min(max(reflect_idx(x0 + lane + 32 * k - kUsmR, W), 0), W - 1);
        const bool last_ok = lane + 96 < kUsmHCols + kUsmK - 1;
#pragma unroll
        for (int pass = 0; pass < 2; ++pass) {
            float v[4][4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int ty = warp + 8 * (pass * 4 + u);
                const float* srow = src + pbase + static_cast<size_t>(min(y0 + ty, H - 1)) * W;
#pragma unroll
                for (int k = 0; k < 4; ++k) v[u][k] = srow[gxk[k]];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int ty = warp + 8 * (pass * 4 + u);
#pragma unroll
                for (int k = 0; k < 3; ++k) A[ty * kUsmHPitch + lane + 32 * k] = v[u][k];
                if (last_ok) A[ty * kUsmHPitch + lane + 96] = v[u][3];
            }
        }
    }
    __syncthreads();
    const int c0 = warp * kUsmO;
    float2 acc[kUsmO];
    usm_window8x2(A + lane * kUsmHPitch + c0, A + (lane + 32) * kUsmHPitch + c0, 1, acc);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int gy = y0 + lane + 32 * half;
        if (gy >= H) continue;
        float o8[kUsmO];
#pragma unroll
        for (int j = 0; j < kUsmO; ++j) o8[j] = half ? acc[j].y : acc[j].x;
        float* o = tmp + pbase + static_cast<size_t>(gy) * W + x0 + c0;
        if (x0 + c0 + kUsmO <= W && (W & 3) == 0) {
            reinterpret_cast<float4*>(o)[0] = make_float4(o8[0], o8[1], o8[2], o8[3]);
            reinterpret_cast<float4*>(o)[1] = make_float4(o8[4], o8[5], o8[6], o8[7]);
        } else {
#pragma unroll
            for (int j = 0; j < kUsmO; ++j)
                if (x0 + c0 + j < W) o[j] = o8[j];
        }
    }
}

// conv_y(tmp) + the pointwise tail. Block = 64 x 64 outputs, 256 threads: thread = columns (c, c + 32), 8 consecutive rows.
//   stage 0: blur = conv_y(tmp); res = x - blur; mask = |res| * 255 > threshold     -> res, mask_or_out
//   stage 1: soft = conv_y(tmp); out = soft * clip(x + weight * res, 0, 1) + (1 - soft) * x
__global__ void __launch_bounds__(256) usm_v51_kernel(const float* __restrict__ tmp, const float* __restrict__ x,
                                                      float* __restrict__ res, float* __restrict__ mask_or_out, int H, int W,
                                                      int stage, float weight, float threshold, float* __restrict__ soft_out) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    __shared__ float Bm[kUsmVIn * kUsmVCols];
    const int plane = blockIdx.z;
    const int x0 = blockIdx.x * kUsmVCols, y0 = blockIdx.y * kUsmVRows;
    const size_t pbase = static_cast<size_t>(plane) * H * W;
    {   // 114 rows x 64 columns, coalesced; this thread's rows are g, g+4, ...: 8 loads in flight per batch
        const int cx = threadIdx.x & 63;
        const int gxc = min(x0 + cx, W - 1);
        const int g = threadIdx.x >> 6;
#pragma unroll
        for (int base = 0; base < kUsmVIn; base += 32) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int ty = min(base + g + 4 * u, kUsmVIn - 1);
                const int gy = min(max(reflect_idx(y0 + ty - kUsmR, H), 0), H - 1);
                v[u] = tmp[pbase + static_cast<size_t>(gy) * W + gxc];
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int ty = base + g + 4 * u;
                if (ty < kUsmVIn) Bm[ty * kUsmVCols + cx] = v[u];
            }
        }
    }
    const int cx = threadIdx.x & 31;
    const int r0 = (threadIdx.x >> 5) * kUsmO;
    // the tail's operands, requested before the window so that their latency hides behind the FMAs
    float2 xv[kUsmO], rv[kUsmO];
#pragma unroll
    for (int j = 0; j < kUsmO; ++j) {
        const size_t o = pbase + static_cast<size_t>(min(y0 + r0 + j, H - 1)) * W;
        const int ga = min(x0 + cx, W - 1), gb = min(x0 + cx + 32, W - 1);
        xv[j] = make_float2(x[o + ga], x[o + gb]);
        rv[j] = stage == 0 ? make_float2(0.f, 0.f) : make_float2(res[o + ga], res[o + gb]);
    }
    __syncthreads();
    float2 acc[kUsmO];
    usm_window8x2(Bm + r0 * kUsmVCols + cx, Bm + r0 * kUsmVCols + cx + 32, kUsmVCols, acc);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int gx = x0 + cx + 32 * half;
        if (gx >= W) continue;
#pragma unroll
        for (int j = 0; j < kUsmO; ++j) {
            const int gy = y0 + r0 + j;
            if (gy >= H) break;
            const size_t o = pbase + static_cast<size_t>(gy) * W + gx;
            const float a = half ? acc[j].y : acc[j].x, xx = half ? xv[j].y : xv[j].x;
            if (stage == 0) {
                const float r = xx - a;                                               // imgproc.py:1528
                res[o] = r;
                mask_or_out[o] = (fabsf(r) * 255.f > threshold) ? 1.f : 0.f;          // imgproc.py:1530-1531
            } else {
                const float rr = half ? rv[j].y : rv[j].x;
                float sh = __fadd_rn(xx, __fmul_rn(weight, rr));                      // imgproc.py:1533
                sh = fminf(fmaxf(sh, 0.f), 1.f);                                      // imgproc.py:1534
                mask_or_out[o] = __fadd_rn(__fmul_rn(a, sh), __fmul_rn(1.f - a, xx));  // imgproc.py:1535
                if (soft_out) soft_out[o] = a;   // kept for the backward pass (resr_usm_sharp_backward)
            }
        }
    }
}

// One blur (horizontal + vertical 51-tap pass + the pointwise tail) in ONE kernel: a block owns a 32-column strip of a plane
// over its FULL height, so the horizontal-pass results it needs for the vertical pass are exactly the strip's own rows --
// no halo recomputation, no scratch image, two launches per USM instead of four. The strip's horizontal results live in
// shared memory ([H + 50][33] floats with the 25 reflected rows on either side); the per-output FMA order is that of
// usm_h51_kernel / usm_v51_kernel (same usm_window8x2), so the results are bit-identical. 128 threads: horizontal pass
// in chunks of 64 rows (lane = rows l, l + 32; warp = 8 columns), vertical pass in chunks of 64 rows (lane = column,
// warp = 8 rows of each of the two 32-row halves).
static constexpr int kUsmFCols = 32, kUsmFPitchT = 33, kUsmFPitchA = kUsmFCols + kUsmK - 1 + 1;   // 83: odd
__global__ void __launch_bounds__(128) usm_fused51_kernel(const float* __restrict__ src, const float* __restrict__ x,
                                                          float* __restrict__ res, float* __restrict__ mask_or_out, int H, int W,
                                                          int stage, float weight, float threshold, float* __restrict__ soft_out) {
    grid_dep_wait();
    grid_dep_launch();
    extern __shared__ float usm_sm[];
    float* T = usm_sm;                                   // [H + 2 * kUsmR][33]: row i <-> image row i - 25
    float* A = usm_sm + (H + 2 * kUsmR) * kUsmFPitchT;   // [64][83] staging of the horizontal pass
    const int plane = blockIdx.y, x0 = blockIdx.x * kUsmFCols;
    const size_t pbase = static_cast<size_t>(plane) * H * W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int gxk[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) gxk[k] = min(max(reflect_idx(x0 + lane + 32 * k - kUsmR, W), 0), W - 1);
    const bool last_ok = lane + 64 < kUsmFCols + kUsmK - 1;
    // Horizontal pass in chunks of 64 rows. The global loads of chunk i + 1 are issued (into registers) before the FMAs of
    // chunk i, so their latency hides behind the arithmetic: warp w holds rows w, w + 4, ... of the chunk, 3 columns per lane.
    float v[16][3];
    auto load_chunk = [&](int row0) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const float* srow = src + pbase + static_cast<size_t>(min(row0 + warp + 4 * u, H - 1)) * W;
#pragma unroll
            for (int k = 0; k < 3; ++k) v[u][k] = srow[gxk[k]];
        }
    };
    load_chunk(0);
    for (int row0 = 0; row0 < H; row0 += 64) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            const int ty = warp + 4 * u;
            A[ty * kUsmFPitchA + lane] = v[u][0];
            A[ty * kUsmFPitchA + lane + 32] = v[u][1];
            if (last_ok) A[ty * kUsmFPitchA + lane + 64] = v[u][2];
        }
        __syncthreads();
        if (row0 + 64 < H) load_chunk(row0 + 64);
        const int c0 = warp * kUsmO;
        float2 acc[kUsmO];
        usm_window8x2(A + lane * kUsmFPitchA + c0, A + (lane + 32) * kUsmFPitchA + c0, 1, acc);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int gy = row0 + lane + 32 * half;
            if (gy < H) {
                float* t = T + (gy + kUsmR) * kUsmFPitchT + c0;
#pragma unroll
                for (int j = 0; j < kUsmO; ++j) t[j] = half ? acc[j].y : acc[j].x;
            }
        }
        __syncthreads();
    }
    // reflected halo rows: image row -k = row k, row H - 1 + k = row H - 1 - k  (k = 1 .. 25)
    for (int i = threadIdx.x; i < 2 * kUsmR * kUsmFCols; i += blockDim.x) {
        const int k = i / (2 * kUsmFCols) + 1, side = (i / kUsmFCols) & 1, c = i % kUsmFCols;
        if (side == 0) T[(kUsmR - k) * kUsmFPitchT + c] = T[(kUsmR + k) * kUsmFPitchT + c];
        else T[(kUsmR + H - 1 + k) * kUsmFPitchT + c] = T[(kUsmR + H - 1 - k) * kUsmFPitchT + c];
    }
    __syncthreads();
    const int gx = x0 + lane;
    // Vertical pass in chunks of 64 rows; the tail's operands (x, res) of chunk i + 1 are requested before chunk i's FMAs.
    float2 xv[kUsmO], rv[kUsmO], xn[kUsmO], rn[kUsmO];
    auto load_tail = [&](int row0, float2 (&xo)[kUsmO], float2 (&ro)[kUsmO]) {
        const int r0 = row0 + warp * kUsmO, r1 = r0 + 32;
#pragma unroll
        for (int j = 0; j < kUsmO; ++j) {
            const size_t oa = pbase + static_cast<size_t>(min(r0 + j, H - 1)) * W + min(gx, W - 1);
            const size_t ob = pbase + static_cast<size_t>(min(r1 + j, H - 1)) * W + min(gx, W - 1);
            xo[j] = make_float2(x[oa], x[ob]);
            ro[j] = stage == 0 ? make_float2(0.f, 0.f) : make_float2(res[oa], res[ob]);
        }
    };
    load_tail(0, xn, rn);
    for (int row0 = 0; row0 < H; row0 += 64) {
        const int r0 = row0 + warp * kUsmO, r1 = r0 + 32;      // two lines: the same column, rows r0.. and r0 + 32..
#pragma unroll
        for (int j = 0; j < kUsmO; ++j) { xv[j] = xn[j]; rv[j] = rn[j]; }
        if (row0 + 64 < H) load_tail(row0 + 64, xn, rn);
        float2 acc[kUsmO];
        // T row index of image row r is r + 25, and the window of output row r starts at image row r - 25: T row r
        usm_window8x2(T + min(r0, H - 1) * kUsmFPitchT + lane, T + min(r1, H - 1) * kUsmFPitchT + lane, kUsmFPitchT, acc);
        if (gx >= W) continue;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
            for (int j = 0; j < kUsmO; ++j) {
                const int gy = (half ? r1 : r0) + j;
                if (gy >= H) break;
                const size_t o = pbase + static_cast<size_t>(gy) * W + gx;
                const float a = half ? acc[j].y : acc[j].x, xx = half ? xv[j].y : xv[j].x;
                if (stage == 0) {
                    const float r = xx - a;                                               // imgproc.py:1528
                    res[o] = r;
                    mask_or_out[o] = (fabsf(r) * 255.f > threshold) ? 1.f : 0.f;          // imgproc.py:1530-1531
                } else {
                    const float rr = half ? rv[j].y : rv[j].x;
                    float sh = __fadd_rn(xx, __fmul_rn(weight, rr));                      // imgproc.py:1533
                    sh = fminf(fmaxf(sh, 0.f), 1.f);                                      // imgproc.py:1534
                    mask_or_out[o] = __fadd_rn(__fmul_rn(a, sh), __fmul_rn(1.f - a, xx));  // imgproc.py:1535
                    if (soft_out) soft_out[o] = a;
                }
            }
        }
    }
}

static int usm_taps_count(int radius) { return radius % 2 == 0 ? radius + 1 : radius; }  // imgproc.py:1518-1519

// Argument checks of the USM entry points, made before anything touches the device
static int usm_check_args(int B, int C, int H, int W, int radius) {
    const int k = usm_taps_count(radius);
    if (B <= 0 || C <= 0) return set_error(RESR_E_INVALID, "USM batch %d / channels %d must be positive", B, C);
    if (k < 1 || k > kUsmMaxTaps) return set_error(RESR_E_INVALID, "USM radius %d out of range", radius);
    if (k / 2 >= H || k / 2 >= W) return set_error(RESR_E_INVALID, "USM reflect padding %d needs a larger image (%dx%d)", k / 2, H, W);
    return RESR_OK;
}

static int usm_set_taps(int radius, int sigma, int* k_out) {
    radius = usm_taps_count(radius);
    double sg = sigma;
    if (sg <= 0) sg = 0.3 * ((radius - 1) * 0.5 - 1) + 0.8;  // cv2.getGaussianKernel
    double taps[kUsmMaxTaps], sum = 0;
    for (int i = 0; i < radius; ++i) {
        const double d = i - (radius - 1) * 0.5;
        taps[i] = std::exp(-(d * d) / (2.0 * sg * sg));
        sum += taps[i];
    }
    float tf[kUsmMaxTaps];
    for (int i = 0; i < radius; ++i) tf[i] = static_cast<float>(taps[i] / sum);
    // the constant bank is per device: remember (radius, sigma) + 1 per device (0 = nothing uploaded yet)
    static PerDevice<long long> cached;
    const long long key = (static_cast<long long>(radius) << 32) + sigma + 1;
    if (cached.cur() != key) {
        if (cudaMemcpyToSymbol(c_usm_taps, tf, radius * sizeof(float)) != cudaSuccess)
            return set_error(RESR_E_CUDA, "cudaMemcpyToSymbol failed");
        cached.cur() = key;
    }
    *k_out = radius;
    return RESR_OK;
}

static int usm_impl(const float* x, float* out, float* ws, int B, int C, int H, int W, int radius, int sigma, float weight,
                    float threshold, cudaStream_t s, float* soft_out = nullptr) {
    int k = 0;
    int rc = usm_check_args(B, C, H, W, radius);
    if (rc == RESR_OK) rc = usm_set_taps(radius, sigma, &k);
    if (rc != RESR_OK) return rc;
    const size_t E = static_cast<size_t>(B) * C * H * W;
    float* tmp = ws;
    float* res = ws + E;
    float* mask = ws + 2 * E;
    const dim3 gh((W + 255) / 256, H, B * C), gv((W + 31) / 32, (H + 63) / 64, B * C);
    const size_t sh = (256 + k - 1) * sizeof(float), sv = static_cast<size_t>(64 + k - 1) * 32 * sizeof(float);
    static const int env_fused = getenv("RESR_USM_FUSED") ? atoi(getenv("RESR_USM_FUSED")) : 1;
    const size_t fsm = (static_cast<size_t>(H + 2 * kUsmR) * kUsmFPitchT + 64 * kUsmFPitchA) * sizeof(float);
    if (k == kUsmK && env_fused && fsm <= 100 * 1024) {   // strip height bounded by shared memory (H <= ~570)
        static PerDevice<size_t> attr_set;
        if (fsm > 48 * 1024 && fsm > attr_set.cur()) {
            cudaFuncSetAttribute(usm_fused51_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fsm));
            attr_set.cur() = fsm;
        }
        const dim3 gf((W + kUsmFCols - 1) / kUsmFCols, B * C);
        launch_pdl(usm_fused51_kernel, gf, 128, fsm, s, x, x, res, mask, H, W, 0, weight, threshold, nullptr);
        launch_pdl(usm_fused51_kernel, gf, 128, fsm, s, static_cast<const float*>(mask), x, res, out, H, W, 1, weight, threshold, soft_out);
    } else if (k == kUsmK) {
        const dim3 g51h((W + kUsmHCols - 1) / kUsmHCols, (H + kUsmHRows - 1) / kUsmHRows, B * C);
        const dim3 g51v((W + kUsmVCols - 1) / kUsmVCols, (H + kUsmVRows - 1) / kUsmVRows, B * C);
        launch_pdl(usm_h51_kernel, g51h, 256, 0, s, x, tmp, H, W);
        launch_pdl(usm_v51_kernel, g51v, 256, 0, s, tmp, x, res, mask, H, W, 0, weight, threshold, nullptr);
        launch_pdl(usm_h51_kernel, g51h, 256, 0, s, mask, tmp, H, W);
        launch_pdl(usm_v51_kernel, g51v, 256, 0, s, tmp, x, res, out, H, W, 1, weight, threshold, soft_out);
    } else {
        launch_pdl(usm_hpass_kernel, gh, 256, sh, s, x, tmp, H, W, k);
        launch_pdl(usm_vpass_kernel, gv, 256, sv, s, tmp, x, res, mask, H, W, k, 0, weight, threshold, nullptr);
        launch_pdl(usm_hpass_kernel, gh, 256, sh, s, mask, tmp, H, W, k);
        launch_pdl(usm_vpass_kernel, gv, 256, sv, s, tmp, x, res, out, H, W, k, 1, weight, threshold, soft_out);
    }
    RESR_LAUNCH_CHECK("usm");
    return RESR_OK;
}

// ---- backward of USMSharp (train_realesrgan.py:476-478 sharpens SR inside the pixel / content losses, so the loss
// gradient has to pass through imgproc.py:1526-1535). The 0/1 mask is a comparison, so the soft mask s is a constant:
//     out = s * clip(x + w * (x - K x), 0, 1) + (1 - s) * x
//     g_sh = g * s * [0 <= x + w * r <= 1]                (torch.clip passes the gradient on the closed interval)
//     dL/dx = g * (1 - s) + (1 + w) * g_sh - w * K^T g_sh
// K^T is the adjoint of the REFLECT-padded separable blur: position j also collects what the padded positions -j (for
// 1 <= j <= R) and 2 (L - 1) - j (for L - 1 - R <= j <= L - 2) received in the forward pass.
__global__ void __launch_bounds__(256) usm_gsh_kernel(const float* __restrict__ g, const float* __restrict__ x, const float* __restrict__ res,
                                                      const float* __restrict__ soft, float* __restrict__ gsh, size_t total, float weight) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const float v = __fadd_rn(x[i], __fmul_rn(weight, res[i]));
        gsh[i] = (v >= 0.f && v <= 1.f) ? g[i] * soft[i] : 0.f;
    }
}

// out[j] = sum over the padded positions p that reflect onto j of  sum_i taps[p - i + R] * in[i]   along x (dir 0) or y (dir 1).
// dir 1 also applies the pointwise tail of the backward when g is given: out = g * (1 - soft) + (1 + w) * gsh - w * K^T gsh.
__global__ void __launch_bounds__(256) usm_adjoint_kernel(const float* __restrict__ in, float* __restrict__ out, int planes, int H, int W,
                                                          int k, int dir, const float* __restrict__ g, const float* __restrict__ soft,
                                                          const float* __restrict__ gsh, float weight) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const int R = k / 2;
    const size_t total = static_cast<size_t>(planes) * H * W;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total; idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int x = static_cast<int>(idx % W), y = static_cast<int>((idx / W) % H);
        const size_t pbase = idx - static_cast<size_t>(y) * W - x;
        const int L = dir ? H : W, j = dir ? y : x;
        const size_t stride = dir ? W : 1;
        const float* line = in + pbase + (dir ? static_cast<size_t>(x) : static_cast<size_t>(y) * W);
        float acc = 0.f;
        auto gather = [&](int p) {   // G(p): what padded position p received
            const int i0 = max(0, p - R), i1 = min(L - 1, p + R);
            for (int i = i0; i <= i1; ++i) acc = fmaf(c_usm_taps[p - i + R], line[i * stride], acc);
        };
        gather(j);
        if (j >= 1 && j <= R) gather(-j);
        if (j >= L - 1 - R && j <= L - 2) gather(2 * (L - 1) - j);
        if (dir && g) acc = g[idx] * (1.f - soft[idx]) + (1.f + weight) * gsh[idx] - weight * acc;
        out[idx] = acc;
    }
}

// ===================================================================================== resize (a9)
// One thread per output element; ATen index rules in fp32 (see oracle/degrade.py resize()).
__device__ __forceinline__ float cubic1(float x) { const float A = -0.75f; return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cubic2(float x) { const float A = -0.75f; return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }

__global__ void __launch_bounds__(256) resize_kernel(const float* __restrict__ in, float* __restrict__ out, int planes, int Hi,
                                                     int Wi, int Ho, int Wo, int mode, float sy, float sx) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const size_t total = static_cast<size_t>(planes) * Ho * Wo;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t rowi = div_u(idx, Wo);
        const int ox = static_cast<int>(mod_u(idx, Wo));
        const int oy = static_cast<int>(mod_u(rowi, Ho));
        const size_t p = div_u(rowi, Ho);
        const float* src = in + p * Hi * Wi;
        float v;
        if (mode == 0) {  // area == adaptive_avg_pool2d
            const int ys = (oy * Hi) / Ho, ye = ((oy + 1) * Hi + Ho - 1) / Ho;
            const int xs = (ox * Wi) / Wo, xe = ((ox + 1) * Wi + Wo - 1) / Wo;
            float acc = 0.f;
            for (int y = ys; y < ye; ++y)
                for (int x = xs; x < xe; ++x) acc += src[static_cast<size_t>(y) * Wi + x];
            v = acc / static_cast<float>((ye - ys) * (xe - xs));
        } else if (mode == 1) {  // bilinear, align_corners=False
            const float fy = fmaxf(fmaf(sy, oy + 0.5f, -0.5f), 0.f), fx = fmaxf(fmaf(sx, ox + 0.5f, -0.5f), 0.f);
            const int y0 = static_cast<int>(fy), x0 = static_cast<int>(fx);
            const int y1 = y0 + (y0 < Hi - 1), x1 = x0 + (x0 < Wi - 1);
            const float ly1 = fy - y0, lx1 = fx - x0, ly0 = 1.f - ly1, lx0 = 1.f - lx1;
            const float top = lx0 * src[static_cast<size_t>(y0) * Wi + x0] + lx1 * src[static_cast<size_t>(y0) * Wi + x1];
            const float bot = lx0 * src[static_cast<size_t>(y1) * Wi + x0] + lx1 * src[static_cast<size_t>(y1) * Wi + x1];
            v = ly0 * top + ly1 * bot;
        } else {  // bicubic A=-0.75, indices clamped
            const float fy = fmaf(sy, oy + 0.5f, -0.5f), fx = fmaf(sx, ox + 0.5f, -0.5f);
            const float fly = floorf(fy), flx = floorf(fx);
            const int iy = static_cast<int>(fly), ix = static_cast<int>(flx);
            const float ty = fy - fly, tx = fx - flx;
            const float wy[4] = {cubic2(ty + 1.f), cubic1(ty), cubic1(1.f - ty), cubic2(2.f - ty)};
            const float wx[4] = {cubic2(tx + 1.f), cubic1(tx), cubic1(1.f - tx), cubic2(2.f - tx)};
            v = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int yy = min(max(iy - 1 + i, 0), Hi - 1);
                float rowacc = 0.f;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int xx = min(max(ix - 1 + j, 0), Wi - 1);
                    rowacc += src[static_cast<size_t>(yy) * Wi + xx] * wx[j];
                }
                v += rowacc * wy[i];
            }
        }
        out[idx] = v;
    }
}

static int grid1d(size_t total, int block = 256) {
    size_t g = (total + block - 1) / block;
    if (g > 148 * 32) g = 148 * 32;
    return static_cast<int>(g < 1 ? 1 : g);
}

static int resize_impl(const float* in, float* out, int planes, int Hi, int Wi, int Ho, int Wo, int mode, double scale_h,
                       double scale_w, cudaStream_t s) {
    if (mode < 0 || mode > 2 || Ho <= 0 || Wo <= 0) return set_error(RESR_E_INVALID, "bad resize arguments");
    // ATen area_pixel_compute_scale: 1/scale_factor when the caller passed scale_factor, else in/out, as float
    const float sy = scale_h > 0 ? static_cast<float>(1.0 / scale_h) : static_cast<float>(Hi) / static_cast<float>(Ho);
    const float sx = scale_w > 0 ? static_cast<float>(1.0 / scale_w) : static_cast<float>(Wi) / static_cast<float>(Wo);
    const size_t total = static_cast<size_t>(planes) * Ho * Wo;
    launch_pdl(resize_kernel, grid1d(total), 256, 0, s, in, out, planes, Hi, Wi, Ho, Wo, mode, sy, sx);
    RESR_LAUNCH_CHECK("resize");
    return RESR_OK;
}

// ===================================================================================== noise (a10, a11)
__device__ __forceinline__ float round_u8(float x) {  // clamp(round(x*255), 0, 255) / 255, half-to-even
    return __fdiv_rn(fminf(fmaxf(rintf(__fmul_rn(x, 255.f)), 0.f), 255.f), 255.f);
}
__device__ __forceinline__ float gray_of(float r, float g, float b) {  // torchvision rgb_to_grayscale
    return __fadd_rn(__fadd_rn(__fmul_rn(0.2989f, r), __fmul_rn(0.587f, g)), __fmul_rn(0.114f, b));
}

// clip / rounds tail shared by both noise ops (imgproc.py:1048-1055, 1080-1085)
__device__ __forceinline__ float noise_post(float v, int clip, int rounds) {
    if (clip && rounds) return __fdiv_rn(fminf(fmaxf(rintf(__fmul_rn(v, 255.f)), 0.f), 255.f), 255.f);
    if (clip) return fminf(fmaxf(v, 0.f), 1.f);
    if (rounds) return __fdiv_rn(rintf(__fmul_rn(v, 255.f)), 255.f);
    return v;
}

__global__ void __launch_bounds__(256) gaussian_noise_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                             const float* __restrict__ sigma, const float* __restrict__ gray,
                                                             const float* __restrict__ ncolor,
                                                             const float* __restrict__ ngray, int B, int C, int HW, int clip,
                                                             int rounds) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const size_t total = static_cast<size_t>(B) * C * HW;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int b = static_cast<int>(div_u(idx, static_cast<unsigned>(C) * HW));
        const int p = static_cast<int>(mod_u(idx, HW));
        const float sg = sigma[b];
        float n = __fdiv_rn(__fmul_rn(ncolor[idx], sg), 255.f);  // imgproc.py:858
        if (ngray) {                                             // imgproc.py:853-861
            const float g = gray[b];
            const float ng = __fdiv_rn(__fmul_rn(ngray[p], sg), 255.f);
            n = __fadd_rn(__fmul_rn(n, 1.f - g), __fmul_rn(ng, g));
        }
        out[idx] = noise_post(__fadd_rn(x[idx], n), clip, rounds);
    }
}

// Same arithmetic with the normal deviates drawn in the kernel (production mode of the plan-driven pipeline: no host-drawn
// noise tensors): Philox4x32-10, subsequence = element index for the colour field, = pixel index (shared by all samples
// and channels, imgproc.py:853-856: ONE H x W field) for the gray field with a different key. state[0] is the call counter
// (advanced by the last block to finish, so every block of this launch reads the same value), state[1] the block ticket.
__global__ void __launch_bounds__(256) gaussian_noise_sampled_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                                     const float* __restrict__ sigma, const float* __restrict__ gray,
                                                                     unsigned long long seed, unsigned long long* __restrict__ state,
                                                                     int with_gray, int B, int C, int HW, int clip, int rounds) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const size_t total = static_cast<size_t>(B) * C * HW;
    const unsigned long long call = state[0];
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int b = static_cast<int>(div_u(idx, static_cast<unsigned>(C) * HW));
        const int p = static_cast<int>(mod_u(idx, HW));
        const float sg = sigma[b];
        curandStatePhilox4_32_10_t st;
        curand_init(seed, idx, call * 8ull, &st);
        float n = __fdiv_rn(__fmul_rn(curand_normal(&st), sg), 255.f);  // imgproc.py:858
        if (with_gray) {                                                 // imgproc.py:853-861
            const float g = gray[b];
            curand_init(seed ^ 0x9E3779B97F4A7C15ull, static_cast<unsigned long long>(p), call * 8ull, &st);
            const float ng = __fdiv_rn(__fmul_rn(curand_normal(&st), sg), 255.f);
            n = __fadd_rn(__fmul_rn(n, 1.f - g), __fmul_rn(ng, g));
        }
        out[idx] = noise_post(__fadd_rn(x[idx], n), clip, rounds);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&state[1], 1ull) == gridDim.x - 1) {
            state[1] = 0;
            state[0] = call + 1;
        }
    }
}

// Presence bitmap of the 256 u8 levels per sample, colour image (all channels) and luma: replaces the per-sample
// torch.unique host syncs of imgproc.py:892, 903. bitmaps: [B][2][8] uint32 (0 = colour, 1 = gray), pre-zeroed.
__global__ void __launch_bounds__(256) u8_presence_kernel(const float* __restrict__ x, unsigned* __restrict__ bitmaps, int C,
                                                          int HW, int want_gray, unsigned long long* __restrict__ call_counter) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    if (call_counter && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *call_counter += 1;  // sampled mode
    __shared__ unsigned sbits[16];
    if (threadIdx.x < 16) sbits[threadIdx.x] = 0;
    __syncthreads();
    const int b = blockIdx.y;
    const float* src = x + static_cast<size_t>(b) * C * HW;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += gridDim.x * blockDim.x) {
        float ch[3];
        for (int c = 0; c < C; ++c) {
            ch[c < 3 ? c : 2] = src[static_cast<size_t>(c) * HW + p];
            const int lv = static_cast<int>(fminf(fmaxf(rintf(__fmul_rn(src[static_cast<size_t>(c) * HW + p], 255.f)), 0.f), 255.f));
            atomicOr(&sbits[lv >> 5], 1u << (lv & 31));
        }
        if (want_gray && C == 3) {
            const int lv = static_cast<int>(fminf(fmaxf(rintf(__fmul_rn(gray_of(ch[0], ch[1], ch[2]), 255.f)), 0.f), 255.f));
            atomicOr(&sbits[8 + (lv >> 5)], 1u << (lv & 31));
        }
    }
    __syncthreads();
    if (threadIdx.x < 16 && sbits[threadIdx.x]) atomicOr(&bitmaps[b * 16 + threadIdx.x], sbits[threadIdx.x]);
}

__global__ void unique_counts_kernel(const unsigned* __restrict__ bitmaps, int* __restrict__ counts, float* __restrict__ vals,
                                     int B) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // b*2 + which
    if (i >= 2 * B) return;
    int n = 0;
    for (int w = 0; w < 8; ++w) n += __popc(bitmaps[i * 8 + w]);
    counts[i] = n;
    // 2 ** ceil(log2(n)) (imgproc.py:893, 904): smallest power of two >= n
    int v = 1;
    while (v < n) v <<= 1;
    vals[i] = static_cast<float>(v);
}

__global__ void __launch_bounds__(256) poisson_noise_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                            const float* __restrict__ scale, const float* __restrict__ gray,
                                                            const float* __restrict__ scolor,
                                                            const float* __restrict__ sgray, const float* __restrict__ vals,
                                                            int B, int HW, int clip, int rounds) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const size_t total = static_cast<size_t>(B) * HW;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int b = static_cast<int>(div_u(idx, HW));
        const int p = static_cast<int>(mod_u(idx, HW));
        const size_t base = static_cast<size_t>(b) * 3 * HW + p;
        const float r = x[base], g = x[base + HW], bl = x[base + 2 * static_cast<size_t>(HW)];
        const float vc = vals[2 * b], sc = scale[b];
        float ng = 0.f, gm = 0.f;
        if (sgray) {  // imgproc.py:886-897
            gm = gray[b];
            const float qg = round_u8(gray_of(r, g, bl));
            ng = __fsub_rn(__fdiv_rn(sgray[idx], vals[2 * b + 1]), qg);
        }
        const float in3[3] = {r, g, bl};
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const size_t o = base + static_cast<size_t>(c) * HW;
            const float q = round_u8(in3[c]);                                   // imgproc.py:901
            float n = __fsub_rn(__fdiv_rn(scolor[o], vc), q);                   // imgproc.py:906-907
            if (sgray) n = __fadd_rn(__fmul_rn(n, 1.f - gm), __fmul_rn(ng, gm));  // imgproc.py:910
            n = __fmul_rn(n, sc);                                               // imgproc.py:914
            out[o] = noise_post(__fadd_rn(in3[c], n), clip, rounds);
        }
    }
}

// Same arithmetic with the Poisson draws made in the kernel (production mode of the plan-driven pipeline: no rate tensors,
// no library sampler launches): Philox4x32-10 counter RNG, one subsequence per pixel, `*counter` advances once per call
// (bumped by the presence kernel that runs before), exact rejection / multiplication samplers on top of it (poisson_draw;
// cuRAND's header-only Philox generator supplies the uniforms). vals = 2 ** ceil(log2(#unique)) come straight from the 256-bit presence bitmaps.
__device__ __forceinline__ float vals_of(const unsigned* __restrict__ bm8) {
    int n = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) n += __popc(bm8[w]);
    int v = 1;
    while (v < n) v <<= 1;
    return static_cast<float>(v);
}

// Poisson(lam) from a Philox stream. lam >= 10: PTRS, Hoermann's transformed rejection with squeeze (the algorithm NumPy and
// torch's CPU sampler use; ~1.1 iterations, two uniforms each). lam < 10:
// multiplication method (lam + 1 uniforms on average). Both are exact samplers.
__device__ __forceinline__ float poisson_draw(curandStatePhilox4_32_10_t* st, float lam) {
    if (lam <= 0.f) return 0.f;
    if (lam < 10.f) {
        const float enlam = __expf(-lam);
        float prod = curand_uniform(st);
        int k = 0;
        while (prod > enlam) {
            prod *= curand_uniform(st);
            ++k;
        }
        return static_cast<float>(k);
    }
    const float slam = sqrtf(lam), loglam = logf(lam);
    const float b = 0.931f + 2.53f * slam;
    const float a = -0.059f + 0.02483f * b;
    const float invalpha = 1.1239f + 1.1328f / (b - 3.4f);
    const float vr = 0.9277f - 3.6224f / (b - 2.f);
    while (true) {
        const float U = curand_uniform(st) - 0.5f;
        const float V = curand_uniform(st);
        const float us = 0.5f - fabsf(U);
        const float k = floorf((2.f * a / us + b) * U + lam + 0.43f);
        if (us >= 0.07f && V <= vr) return k;
        if (k < 0.f || (us < 0.013f && V > us)) continue;
        // exact test, reached by ~10 % of the proposals; fp32 logs / lgammaf put an absolute error of ~1e-4 on a log
        // acceptance ratio, i.e. a relative bias of the acceptance probability far below the sampling noise
        const float lhs = logf(V * invalpha / (a / (us * us) + b));
        const float rhs = -lam + k * loglam - lgammaf(k + 1.f);
        if (lhs <= rhs) return k;
    }
}

__global__ void __launch_bounds__(256) poisson_noise_sampled_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                                    const float* __restrict__ scale, const float* __restrict__ gray,
                                                                    const unsigned* __restrict__ bitmaps,
                                                                    const unsigned long long* __restrict__ counter,
                                                                    unsigned long long seed, int with_gray, int B, int HW, int clip,
                                                                    int rounds) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    // four threads per pixel: lanes 0..2 of a quad draw the colour channels, lane 3 the luma sample (the sampler's loop
    // count grows with the rate, so the draws are spread over threads instead of being made one after the other)
    const size_t total = static_cast<size_t>(B) * HW;
    const unsigned long long call = *counter;
    const size_t tid = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    const size_t idx = tid >> 2;
    const int k = static_cast<int>(tid & 3);
    const bool live = idx < total;
    const size_t pi = live ? idx : 0;
    const int b = static_cast<int>(div_u(pi, HW));
    const int p = static_cast<int>(mod_u(pi, HW));
    const size_t base = static_cast<size_t>(b) * 3 * HW + p;
    const float r = x[base], g = x[base + HW], bl = x[base + 2 * static_cast<size_t>(HW)];
    const float vc = vals_of(bitmaps + b * 16);
    const float vg = with_gray ? vals_of(bitmaps + b * 16 + 8) : 1.f;
    const float qg = round_u8(gray_of(r, g, bl));
    const float mine = k == 0 ? r : (k == 1 ? g : bl);
    const float q = k < 3 ? round_u8(mine) : qg;                                 // imgproc.py:888-889, 901
    const float v = k < 3 ? vc : vg;
    float draw = 0.f;
    if (live && (k < 3 || with_gray)) {
        curandStatePhilox4_32_10_t st;
        curand_init(seed, tid, call * 64ull, &st);
        draw = poisson_draw(&st, __fmul_rn(q, v));                               // imgproc.py:895, 906
    }
    float n = __fsub_rn(__fdiv_rn(draw, v), q);                                  // imgproc.py:896-897, 906-907
    const float ng = __shfl_sync(0xffffffffu, n, (threadIdx.x & 31) | 3);       // the quad's luma noise
    if (live && k < 3) {
        if (with_gray) {
            const float gm = gray[b];
            n = __fadd_rn(__fmul_rn(n, 1.f - gm), __fmul_rn(ng, gm));           // imgproc.py:910
        }
        n = __fmul_rn(n, scale[b]);                                             // imgproc.py:914
        out[base + static_cast<size_t>(k) * HW] = noise_post(__fadd_rn(mine, n), clip, rounds);
    }
}

// Rates handed to the Poisson sampler: rate = q * vals (imgproc.py:895, 906). Used to replay host-fed draws.
__global__ void __launch_bounds__(256) poisson_rates_kernel(const float* __restrict__ x, const float* __restrict__ vals,
                                                            float* __restrict__ rate_color, float* __restrict__ rate_gray,
                                                            int B, int HW) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const size_t total = static_cast<size_t>(B) * HW;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int b = static_cast<int>(div_u(idx, HW));
        const int p = static_cast<int>(mod_u(idx, HW));
        const size_t base = static_cast<size_t>(b) * 3 * HW + p;
        const float r = x[base], g = x[base + HW], bl = x[base + 2 * static_cast<size_t>(HW)];
        const float vc = vals[2 * b];
        rate_color[base] = __fmul_rn(round_u8(r), vc);
        rate_color[base + HW] = __fmul_rn(round_u8(g), vc);
        rate_color[base + 2 * static_cast<size_t>(HW)] = __fmul_rn(round_u8(bl), vc);
        if (rate_gray) rate_gray[idx] = __fmul_rn(round_u8(gray_of(r, g, bl)), vals[2 * b + 1]);
    }
}

// ===================================================================================== JPEG (a12)
// One WARP per 16 x 16 MCU (4 Y blocks + Cb + Cr), eight MCUs in flight per block, no block-level synchronisation. The
// reference's 64-term contraction with its cos-product table (imgproc.py:1238-1249, 1358-1368) is evaluated in its
// separable form, D[u,v] = sum_x C[x][u] * (sum_y p[x][y] * C[y][v]) with C[x][u] = cos((2x+1) u pi / 16): the same sum
// in a different fp32 order (the reference's own order is whatever its BLAS picks), 16 instead of 64 FMAs per
// coefficient, and the 8 x 8 cos matrix lives in 48 registers per lane instead of two 16 KB shared-memory tables that
// every block had to reload. Quantisation (table * factor, round-half-even) is the reference arithmetic, op for op.
__device__ float g_cos8[64];          // [x][u] = (float) cos((2x+1) u pi / 16)
__device__ float g_qtab[2][64];       // [0] transposed Annex-K luma table (imgproc.py:40-45), [1] chroma table (:46-49), [u][v]

static constexpr int kJpegWarps = 8;

__global__ void __launch_bounds__(32 * kJpegWarps) jpeg_kernel(const float* __restrict__ x, float* __restrict__ out,
                                                               const float* __restrict__ quality, float* __restrict__ factor_out,
                                                               int B, int H, int W, int clamp_in, int vec_ok,
                                                               float* __restrict__ qy, float* __restrict__ qcb,
                                                               float* __restrict__ qcr) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    __shared__ __align__(16) float s_pix[kJpegWarps][6][64];   // samples -> dequantised coefficients -> reconstruction
    __shared__ __align__(16) float s_tmp[kJpegWarps][6][64];   // row-transformed intermediate
    __shared__ __align__(16) float s_chr[kJpegWarps][2][256];  // full-resolution Cb, Cr of the MCU
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float (*pix)[64] = s_pix[warp];
    float (*tmp)[64] = s_tmp[warp];
    float (*chr)[256] = s_chr[warp];
    // this lane's two transform outputs per 8 x 8 block: row a = lane / 4, columns b0 = 2 * (lane % 4), b0 + 1
    const int a = lane >> 2, b0 = (lane & 3) * 2;
    float c_col[8][2];   // C[i][b0 + j]   (forward row pass: sum over y = i)
    float c_row[2][8];   // C[b0 + j][i]   (inverse row pass: sum over v = i)
    float c_a_col[8];    // C[i][a]        (forward column pass: sum over x = i)
    float c_a_row[8];    // C[a][i]        (inverse column pass: sum over u = i)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        c_col[i][0] = g_cos8[i * 8 + b0];
        c_col[i][1] = g_cos8[i * 8 + b0 + 1];
        c_row[0][i] = g_cos8[b0 * 8 + i];
        c_row[1][i] = g_cos8[(b0 + 1) * 8 + i];
        c_a_col[i] = g_cos8[i * 8 + a];
        c_a_row[i] = g_cos8[a * 8 + i];
    }
    // quantisation constants of this lane's two coefficients (u = a, v = b0 + j)
    float tab_y[2], tab_c[2], alpha[2], scale[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int u = a, v = b0 + j;
        tab_y[j] = g_qtab[0][u * 8 + v];
        tab_c[j] = g_qtab[1][u * 8 + v];
        alpha[j] = (u == 0 ? 0.70710678118654752f : 1.f) * (v == 0 ? 0.70710678118654752f : 1.f);
        scale[j] = (u == 0 && v == 0) ? 0.125f : ((u == 0 || v == 0) ? static_cast<float>(0.25 * 0.70710678118654752) : 0.25f);
    }
    const int Hp = (H + 15) / 16 * 16, Wp = (W + 15) / 16 * 16;
    const int mw = Wp / 16, mh = Hp / 16;
    const int nmcu = B * mh * mw;
    const size_t HW = static_cast<size_t>(H) * W;
    const int py = lane >> 1, px0 = (lane & 1) * 8;   // this lane's 8 consecutive pixels of the MCU
    for (int m = blockIdx.x * kJpegWarps + warp; m < nmcu; m += gridDim.x * kJpegWarps) {
        const int b = m / (mh * mw);
        const int my = (m / mw) % mh, mx = m % mw;
        // quality -> factor in fp32 tensor arithmetic (imgproc.py:1124-1141 applied per element at :1478-1479)
        const float q = quality[b];
        const float factor = __fdiv_rn(q < 50.f ? __fdiv_rn(5000.f, q) : __fsub_rn(200.f, __fmul_rn(q, 2.f)), 100.f);
        if (factor_out && my == 0 && mx == 0 && lane == 0) factor_out[b] = factor;
        const int gy = my * 16 + py, gx0 = mx * 16 + px0;
        const size_t o0 = static_cast<size_t>(b) * 3 * HW + static_cast<size_t>(gy) * W + gx0;
        float rgb[3][8];
        if (gy < H && gx0 + 8 <= W && vec_ok) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float4 v0 = *reinterpret_cast<const float4*>(x + o0 + c * HW);
                const float4 v1 = *reinterpret_cast<const float4*>(x + o0 + c * HW + 4);
                rgb[c][0] = v0.x; rgb[c][1] = v0.y; rgb[c][2] = v0.z; rgb[c][3] = v0.w;
                rgb[c][4] = v1.x; rgb[c][5] = v1.y; rgb[c][6] = v1.z; rgb[c][7] = v1.w;
            }
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int i = 0; i < 8; ++i) rgb[c][i] = (gy < H && gx0 + i < W) ? x[o0 + c * HW + i] : 0.f;  // zero padding (imgproc.py:1489)
        }
        {
            const int blk = (py >> 3) * 2 + (lane & 1);
            float yv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float r = rgb[0][i], g = rgb[1][i], bl = rgb[2][i];
                if (clamp_in) { r = fminf(fmaxf(r, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); bl = fminf(fmaxf(bl, 0.f), 1.f); }
                r = __fmul_rn(r, 255.f); g = __fmul_rn(g, 255.f); bl = __fmul_rn(bl, 255.f);  // imgproc.py:1318
                // imgproc.py:1195-1208 (matrix rows as float32 constants)
                yv[i] = (0.299f * r + 0.587f * g + 0.114f * bl) - 128.f;
                chr[0][py * 16 + px0 + i] = -0.168736f * r + -0.331264f * g + 0.5f * bl + 128.f;
                chr[1][py * 16 + px0 + i] = 0.5f * r + -0.418688f * g + -0.081312f * bl + 128.f;
            }
            float4* dst = reinterpret_cast<float4*>(&pix[blk][(py & 7) * 8]);
            dst[0] = make_float4(yv[0], yv[1], yv[2], yv[3]);
            dst[1] = make_float4(yv[4], yv[5], yv[6], yv[7]);
        }
        __syncwarp();
        {   // 2x2 mean (imgproc.py:1216-1219): 2 planes x 64 samples, 4 per lane
            const int c = lane >> 4;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int i = (lane & 15) * 4 + t, cy = i >> 3, cx = i & 7;
                const float* src = chr[c];
                const float sum = (src[(2 * cy) * 16 + 2 * cx] + src[(2 * cy) * 16 + 2 * cx + 1]) +
                                  (src[(2 * cy + 1) * 16 + 2 * cx] + src[(2 * cy + 1) * 16 + 2 * cx + 1]);
                pix[4 + c][i] = sum * 0.25f - 128.f;
            }
        }
        __syncwarp();
        // ---- forward DCT, row pass: tmp[x][v] = sum_y p[x][y] * C[y][v]   (x = a, v = b0 + j)
#pragma unroll
        for (int blk = 0; blk < 6; ++blk) {
            const float4 p0 = *reinterpret_cast<const float4*>(&pix[blk][a * 8]);
            const float4 p1 = *reinterpret_cast<const float4*>(&pix[blk][a * 8 + 4]);
            const float p[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
            float t0 = 0.f, t1 = 0.f;
#pragma unroll
            for (int y = 0; y < 8; ++y) { t0 = fmaf(p[y], c_col[y][0], t0); t1 = fmaf(p[y], c_col[y][1], t1); }
            *reinterpret_cast<float2*>(&tmp[blk][a * 8 + b0]) = make_float2(t0, t1);
        }
        __syncwarp();
        // ---- column pass + quantise + dequantise: D[u][v] = sum_x C[x][u] * tmp[x][v]   (u = a, v = b0 + j)
#pragma unroll
        for (int blk = 0; blk < 6; ++blk) {
            float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
            for (int xx = 0; xx < 8; ++xx) {
                const float2 t = *reinterpret_cast<const float2*>(&tmp[blk][xx * 8 + b0]);
                acc0 = fmaf(c_a_col[xx], t.x, acc0);
                acc1 = fmaf(c_a_col[xx], t.y, acc1);
            }
            const float accs[2] = {acc0, acc1};
            float cf[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int uv = a * 8 + b0 + j;
                const float d = __fmul_rn(scale[j], accs[j]);                            // imgproc.py:1249
                const float tq = __fmul_rn(blk < 4 ? tab_y[j] : tab_c[j], factor);        // imgproc.py:1270, 1289
                const float qc = rintf(__fdiv_rn(d, tq));                                // imgproc.py:1272-1274
                if (qy) {  // optional dump of the quantised coefficients (tests)
                    if (blk < 4) {
                        const int byi = my * 2 + (blk >> 1), bxi = mx * 2 + (blk & 1);
                        qy[(static_cast<size_t>(b) * (Hp / 8) * (Wp / 8) + static_cast<size_t>(byi) * (Wp / 8) + bxi) * 64 + uv] = qc;
                    } else {
                        float* dst = blk == 4 ? qcb : qcr;
                        dst[(static_cast<size_t>(b) * mh * mw + static_cast<size_t>(my) * mw + mx) * 64 + uv] = qc;
                    }
                }
                cf[j] = __fmul_rn(__fmul_rn(qc, tq), alpha[j]);                           // imgproc.py:1331, 1366
            }
            *reinterpret_cast<float2*>(&pix[blk][a * 8 + b0]) = make_float2(cf[0], cf[1]);  // everyone is past the row pass
        }
        __syncwarp();
        // ---- inverse DCT, row pass: t2[u][y'] = sum_v coef[u][v] * C[y'][v]   (u = a, y' = b0 + j)
#pragma unroll
        for (int blk = 0; blk < 6; ++blk) {
            const float4 p0 = *reinterpret_cast<const float4*>(&pix[blk][a * 8]);
            const float4 p1 = *reinterpret_cast<const float4*>(&pix[blk][a * 8 + 4]);
            const float p[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
            float t0 = 0.f, t1 = 0.f;
#pragma unroll
            for (int v = 0; v < 8; ++v) { t0 = fmaf(p[v], c_row[0][v], t0); t1 = fmaf(p[v], c_row[1][v], t1); }
            *reinterpret_cast<float2*>(&tmp[blk][a * 8 + b0]) = make_float2(t0, t1);
        }
        __syncwarp();
        // ---- column pass: rec[x'][y'] = 0.25 * sum_u C[x'][u] * t2[u][y'] + 128   (x' = a, y' = b0 + j)
#pragma unroll
        for (int blk = 0; blk < 6; ++blk) {
            float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const float2 t = *reinterpret_cast<const float2*>(&tmp[blk][u * 8 + b0]);
                acc0 = fmaf(c_a_row[u], t.x, acc0);
                acc1 = fmaf(c_a_row[u], t.y, acc1);
            }
            *reinterpret_cast<float2*>(&pix[blk][a * 8 + b0]) =
                make_float2(__fadd_rn(__fmul_rn(0.25f, acc0), 128.f), __fadd_rn(__fmul_rn(0.25f, acc1), 128.f));  // imgproc.py:1367-1368
        }
        __syncwarp();
        {   // chroma nearest 2x repeat (imgproc.py:1392-1400), shift (:1412), YCbCr -> RGB (:1405-1419), clamp, / 255
            const int blk = (py >> 3) * 2 + (lane & 1);
            const float4 y0v = *reinterpret_cast<const float4*>(&pix[blk][(py & 7) * 8]);
            const float4 y1v = *reinterpret_cast<const float4*>(&pix[blk][(py & 7) * 8 + 4]);
            const float yy[8] = {y0v.x, y0v.y, y0v.z, y0v.w, y1v.x, y1v.y, y1v.z, y1v.w};
            const float4 cbv = *reinterpret_cast<const float4*>(&pix[4][(py >> 1) * 8 + (px0 >> 1)]);
            const float4 crv = *reinterpret_cast<const float4*>(&pix[5][(py >> 1) * 8 + (px0 >> 1)]);
            const float cb4[4] = {cbv.x, cbv.y, cbv.z, cbv.w}, cr4[4] = {crv.x, crv.y, crv.z, crv.w};
            float o3[3][8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float r0 = yy[i], r1 = cb4[i >> 1] - 128.f, r2 = cr4[i >> 1] - 128.f;
                const float ro = r0 + 1.402f * r2;
                const float go = r0 + -0.344136f * r1 + -0.714136f * r2;
                const float bo = r0 + 1.772f * r1;
                o3[0][i] = __fdiv_rn(fminf(255.f, fmaxf(0.f, ro)), 255.f);  // imgproc.py:1453-1455
                o3[1][i] = __fdiv_rn(fminf(255.f, fmaxf(0.f, go)), 255.f);
                o3[2][i] = __fdiv_rn(fminf(255.f, fmaxf(0.f, bo)), 255.f);
            }
            if (gy < H && gx0 + 8 <= W && vec_ok) {
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    *reinterpret_cast<float4*>(out + o0 + c * HW) = make_float4(o3[c][0], o3[c][1], o3[c][2], o3[c][3]);
                    *reinterpret_cast<float4*>(out + o0 + c * HW + 4) = make_float4(o3[c][4], o3[c][5], o3[c][6], o3[c][7]);
                }
            } else if (gy < H) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if (gx0 + i < W) out[o0 + c * HW + i] = o3[c][i];
            }
        }
        __syncwarp();
    }
}

static int jpeg_init_tables() {
    static PerDevice<bool> done;  // __device__ tables live per device
    if (done.cur()) return RESR_OK;
    const double pi = 3.14159265358979323846;
    float c8[64];
    for (int xx = 0; xx < 8; ++xx)
        for (int u = 0; u < 8; ++u) c8[xx * 8 + u] = static_cast<float>(std::cos((2 * xx + 1) * u * pi / 16));
    static const float ybase[64] = {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57,
                                    69, 56, 14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55,
                                    64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
    static const float cbase[16] = {17, 18, 24, 47, 18, 21, 26, 66, 24, 26, 56, 99, 47, 66, 99, 99};
    float qt[2][64];
    for (int u = 0; u < 8; ++u)
        for (int v = 0; v < 8; ++v) {
            qt[0][u * 8 + v] = ybase[v * 8 + u];  // .T (imgproc.py:45)
            qt[1][u * 8 + v] = (u < 4 && v < 4) ? cbase[v * 4 + u] : 99.f;
        }
    if (cudaMemcpyToSymbol(g_cos8, c8, sizeof(c8)) != cudaSuccess || cudaMemcpyToSymbol(g_qtab, qt, sizeof(qt)) != cudaSuccess)
        return set_error(RESR_E_CUDA, "JPEG table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
    done.cur() = true;
    return RESR_OK;
}

static int jpeg_impl(const float* x, float* out, const float* quality, float* factor_out, int B, int H, int W, int clamp_in,
                     float* qy, float* qcb, float* qcr, cudaStream_t s) {
    const int rc = jpeg_init_tables();
    if (rc != RESR_OK) return rc;
    const int nmcu = B * ((H + 15) / 16) * ((W + 15) / 16);
    int grid = (nmcu + kJpegWarps - 1) / kJpegWarps;
    if (grid > 148 * 8) grid = 148 * 8;   // beyond that, warps loop over MCUs
    // float4 rows need W % 4 == 0 AND 16-byte aligned bases: a contiguous view with a storage offset reaches here as is
    const int vec_ok = (W & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    launch_pdl(jpeg_kernel, grid, 32 * kJpegWarps, 0, s, x, out, quality, factor_out, B, H, W, clamp_in, vec_ok, qy, qcb, qcr);
    RESR_LAUNCH_CHECK("jpeg");
    return RESR_OK;
}

// ===================================================================================== round + crop (a13)
__global__ void __launch_bounds__(256) crop_kernel(const float* __restrict__ in, float* __restrict__ out, int planes, int Hi,
                                                   int Wi, int top, int left, int Ho, int Wo, int round_to_u8) {
    grid_dep_wait();      // programmatic dependent launch: everything the previous kernel wrote is visible from here on
    grid_dep_launch();    // the next kernel of the chain may be scheduled behind this one
    const size_t total = static_cast<size_t>(planes) * Ho * Wo;
    for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
         idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const size_t rowi = div_u(idx, Wo);
        const int ox = static_cast<int>(mod_u(idx, Wo));
        const int oy = static_cast<int>(mod_u(rowi, Ho));
        const size_t p = div_u(rowi, Ho);
        float v = in[(p * Hi + top + oy) * Wi + left + ox];
        if (round_to_u8) v = round_u8(v);  // train_realesrnet.py:374
        out[idx] = v;
    }
}

}  // namespace resr

using namespace resr;

extern "C" {

int resr_filter2d(const float* image, const float* kernel, float* out, int b, int c, int h, int w, int k, int kernel_batch,
                  void* stream) {
    if (!image || !kernel || !out) return set_error(RESR_E_INVALID, "null argument");
    if (b <= 0 || c <= 0) return set_error(RESR_E_INVALID, "filter2d batch %d / channels %d must be positive", b, c);
    if (kernel_batch != 1 && kernel_batch != b) return set_error(RESR_E_INVALID, "kernel batch %d must be 1 or %d", kernel_batch, b);
    return filter2d_impl(image, kernel, out, b, c, h, w, k, kernel_batch != 1, static_cast<cudaStream_t>(stream));
}

size_t resr_usm_workspace_bytes(int b, int c, int h, int w) { return static_cast<size_t>(b) * c * h * w * 4 * 3; }

int resr_usm_sharp(const float* image, float* out, int b, int c, int h, int w, int radius, int sigma, float weight,
                   float threshold, void* workspace, size_t workspace_bytes, void* stream) {
    if (!image || !out || !workspace) return set_error(RESR_E_INVALID, "null argument");
    if (workspace_bytes < resr_usm_workspace_bytes(b, c, h, w)) return set_error(RESR_E_NOMEM, "USM workspace too small");
    return usm_impl(image, out, static_cast<float*>(workspace), b, c, h, w, radius, sigma, weight, threshold,
                    static_cast<cudaStream_t>(stream));
}

size_t resr_usm_backward_workspace_bytes(int b, int c, int h, int w) { return static_cast<size_t>(b) * c * h * w * 4 * 6; }

int resr_usm_sharp_backward(const float* image, const float* grad_out, float* grad_in, int b, int c, int h, int w, int radius, int sigma,
                            float weight, float threshold, void* workspace, size_t workspace_bytes, void* stream) {
    if (!image || !grad_out || !grad_in || !workspace) return set_error(RESR_E_INVALID, "null argument");
    if (workspace_bytes < resr_usm_backward_workspace_bytes(b, c, h, w)) return set_error(RESR_E_NOMEM, "USM backward workspace too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t E = static_cast<size_t>(b) * c * h * w;
    float* ws = static_cast<float*>(workspace);           // [0, 3E): forward scratch (tmp, res, mask)
    float *soft = ws + 3 * E, *gsh = ws + 4 * E, *t = ws + 5 * E;
    // recompute the forward quantities the gradient needs (residual, soft mask); the sharpened image itself lands in `t`
    const int rc = usm_impl(image, t, ws, b, c, h, w, radius, sigma, weight, threshold, s, soft);
    if (rc != RESR_OK) return rc;
    const int k = usm_taps_count(radius);
    launch_pdl(usm_gsh_kernel, grid1d(E), 256, 0, s, grad_out, image, ws + E, soft, gsh, E, weight);
    launch_pdl(usm_adjoint_kernel, grid1d(E), 256, 0, s, gsh, t, b * c, h, w, k, 0, nullptr, nullptr, nullptr, weight);
    launch_pdl(usm_adjoint_kernel, grid1d(E), 256, 0, s, t, grad_in, b * c, h, w, k, 1, grad_out, soft, gsh, weight);
    RESR_LAUNCH_CHECK("usm backward");
    return RESR_OK;
}

int resr_resize(const float* image, float* out, int planes, int h_in, int w_in, int h_out, int w_out, int mode,
                double scale_h, double scale_w, void* stream) {
    if (!image || !out) return set_error(RESR_E_INVALID, "null argument");
    if (planes <= 0 || h_in <= 0 || w_in <= 0) return set_error(RESR_E_INVALID, "bad resize input %d x %d x %d", planes, h_in, w_in);
    return resize_impl(image, out, planes, h_in, w_in, h_out, w_out, mode, scale_h, scale_w, static_cast<cudaStream_t>(stream));
}

int resr_gaussian_noise_apply(const float* image, float* out, const float* sigma, const float* gray,
                              const float* noise_color, const float* noise_gray, int b, int c, int h, int w, int clip,
                              int rounds, void* stream) {
    if (!image || !out || !sigma || !noise_color) return set_error(RESR_E_INVALID, "null argument");
    if (noise_gray && !gray) return set_error(RESR_E_INVALID, "noise_gray needs gray flags");
    const size_t total = static_cast<size_t>(b) * c * h * w;
    launch_pdl(gaussian_noise_kernel, grid1d(total), 256, 0, static_cast<cudaStream_t>(stream), image, out, sigma, gray, noise_color,
                                                                                       noise_gray, b, c, h * w, clip, rounds);
    RESR_LAUNCH_CHECK("gaussian_noise");
    return RESR_OK;
}

int resr_gaussian_noise_sampled(const float* image, float* out, const float* sigma, const float* gray, int b, int c, int h, int w,
                                int clip, int rounds, unsigned long long seed, unsigned long long* call_state, void* stream) {
    if (!image || !out || !sigma || !call_state) return set_error(RESR_E_INVALID, "null argument");
    const size_t total = static_cast<size_t>(b) * c * h * w;
    launch_pdl(gaussian_noise_sampled_kernel, grid1d(total), 256, 0, static_cast<cudaStream_t>(stream), image, out, sigma, gray, seed, call_state,
                                                                                               gray != nullptr, b, c, h * w, clip, rounds);
    RESR_LAUNCH_CHECK("gaussian_noise_sampled");
    return RESR_OK;
}

size_t resr_poisson_workspace_bytes(int b) { return static_cast<size_t>(b) * (16 * 4 + 2 * 4 + 2 * 4); }

static int poisson_prepare(const float* image, int b, int c, int h, int w, int want_gray, void* workspace, size_t wsb,
                           cudaStream_t s, unsigned** bm, int** counts, float** vals, bool reuse = false) {
    if (c != 3) return set_error(RESR_E_INVALID, "Poisson noise expects RGB images");
    if (wsb < resr_poisson_workspace_bytes(b)) return set_error(RESR_E_NOMEM, "Poisson workspace too small");
    *bm = static_cast<unsigned*>(workspace);
    *counts = reinterpret_cast<int*>(*bm + static_cast<size_t>(b) * 16);
    *vals = reinterpret_cast<float*>(*counts + 2 * b);
    if (reuse) return RESR_OK;  // counts / vals of this image are already in the workspace (resr_poisson_rates)
    cudaMemsetAsync(*bm, 0, static_cast<size_t>(b) * 16 * 4, s);
    const int HW = h * w;
    int gx = (HW + 255) / 256;
    if (gx > 64) gx = 64;
    launch_pdl(u8_presence_kernel, dim3(gx, b), 256, 0, s, image, *bm, c, HW, want_gray, nullptr);
    launch_pdl(unique_counts_kernel, (2 * b + 127) / 128, 128, 0, s, *bm, *counts, *vals, b);
    RESR_LAUNCH_CHECK("poisson_prepare");
    return RESR_OK;
}

int resr_unique_count_u8(const float* image, int* counts_color, int* counts_gray, int b, int c, int h, int w, void* workspace,
                         size_t workspace_bytes, void* stream) {
    if (!image || !counts_color || !workspace) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned* bm; int* counts; float* vals;
    const int rc = poisson_prepare(image, b, c, h, w, counts_gray != nullptr, workspace, workspace_bytes, s, &bm, &counts, &vals);
    if (rc != RESR_OK) return rc;
    cudaMemcpy2DAsync(counts_color, 4, counts, 8, 4, b, cudaMemcpyDeviceToDevice, s);
    if (counts_gray) cudaMemcpy2DAsync(counts_gray, 4, counts + 1, 8, 4, b, cudaMemcpyDeviceToDevice, s);
    RESR_LAUNCH_CHECK("unique_count");
    return RESR_OK;
}

int resr_poisson_rates(const float* image, float* rate_color, float* rate_gray, int b, int c, int h, int w, void* workspace,
                       size_t workspace_bytes, void* stream) {
    if (!image || !rate_color || !workspace) return set_error(RESR_E_INVALID, "null argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned* bm; int* counts; float* vals;
    const int rc = poisson_prepare(image, b, c, h, w, rate_gray != nullptr, workspace, workspace_bytes, s, &bm, &counts, &vals);
    if (rc != RESR_OK) return rc;
    launch_pdl(poisson_rates_kernel, grid1d(static_cast<size_t>(b) * h * w), 256, 0, s, image, vals, rate_color, rate_gray, b, h * w);
    RESR_LAUNCH_CHECK("poisson_rates");
    return RESR_OK;
}

int resr_poisson_noise_apply(const float* image, float* out, const float* scale, const float* gray, const float* samples_color,
                             const float* samples_gray, int b, int c, int h, int w, int clip, int rounds, void* workspace,
                             size_t workspace_bytes, int reuse_counts, void* stream) {
    if (!image || !out || !scale || !samples_color || !workspace) return set_error(RESR_E_INVALID, "null argument");
    if (samples_gray && !gray) return set_error(RESR_E_INVALID, "samples_gray needs gray flags");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned* bm; int* counts; float* vals;
    const int rc = poisson_prepare(image, b, c, h, w, samples_gray != nullptr, workspace, workspace_bytes, s, &bm, &counts, &vals,
                                   reuse_counts != 0);
    if (rc != RESR_OK) return rc;
    launch_pdl(poisson_noise_kernel, grid1d(static_cast<size_t>(b) * h * w), 256, 0, s, image, out, scale, gray, samples_color,
                                                                              samples_gray, vals, b, h * w, clip, rounds);
    RESR_LAUNCH_CHECK("poisson_noise");
    return RESR_OK;
}

int resr_poisson_noise_sampled(const float* image, float* out, const float* scale, const float* gray, int b, int c, int h, int w,
                               int clip, int rounds, unsigned long long seed, unsigned long long* call_counter, void* workspace,
                               size_t workspace_bytes, void* stream) {
    if (!image || !out || !scale || !workspace || !call_counter) return set_error(RESR_E_INVALID, "null argument");
    if (c != 3) return set_error(RESR_E_INVALID, "Poisson noise expects RGB images");
    if (workspace_bytes < resr_poisson_workspace_bytes(b)) return set_error(RESR_E_NOMEM, "Poisson workspace too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    unsigned* bm = static_cast<unsigned*>(workspace);
    unsigned long long* counter = call_counter;  // advances on every call / CUDA-graph replay: fresh Philox offsets
    cudaMemsetAsync(bm, 0, static_cast<size_t>(b) * 16 * 4, s);
    const int HW = h * w;
    int gx = (HW + 255) / 256;
    if (gx > 64) gx = 64;
    launch_pdl(u8_presence_kernel, dim3(gx, b), 256, 0, s, image, bm, c, HW, gray != nullptr, counter);
    launch_pdl(poisson_noise_sampled_kernel, static_cast<unsigned>((static_cast<size_t>(b) * HW * 4 + 255) / 256), 256, 0, s, image, out, scale, gray, bm, counter, seed,
                                                                                  gray != nullptr, b, HW, clip, rounds);
    RESR_LAUNCH_CHECK("poisson_noise_sampled");
    return RESR_OK;
}

int resr_jpeg(const float* image, float* out, const float* quality, float* factor_out, int b, int h, int w, int clamp_input,
              float* q_y, float* q_cb, float* q_cr, void* stream) {
    if (!image || !out || !quality) return set_error(RESR_E_INVALID, "null argument");
    if ((q_y != nullptr) != (q_cb != nullptr) || (q_y != nullptr) != (q_cr != nullptr))
        return set_error(RESR_E_INVALID, "pass all three coefficient dumps or none");
    if (b <= 0 || h <= 0 || w <= 0) return set_error(RESR_E_INVALID, "bad JPEG image %d x 3 x %d x %d", b, h, w);
    return jpeg_impl(image, out, quality, factor_out, b, h, w, clamp_input, q_y, q_cb, q_cr, static_cast<cudaStream_t>(stream));
}

int resr_crop(const float* image, float* out, int planes, int h_in, int w_in, int top, int left, int h_out, int w_out,
              int round_to_u8, void* stream) {
    if (!image || !out) return set_error(RESR_E_INVALID, "null argument");
    if (planes <= 0 || h_out <= 0 || w_out <= 0) return set_error(RESR_E_INVALID, "bad crop size %d x %d x %d", planes, h_out, w_out);
    if (top < 0 || left < 0 || top + h_out > h_in || left + w_out > w_in) return set_error(RESR_E_INVALID, "crop window out of range");
    const size_t total = static_cast<size_t>(planes) * h_out * w_out;
    if (!round_to_u8 && h_out == h_in && w_out == w_in) {  // the window is the whole image (cfg2: HR is already 256^2)
        if (cudaMemcpyAsync(out, image, total * sizeof(float), cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)) != cudaSuccess)
            return set_error(RESR_E_CUDA, "crop copy failed");
        return RESR_OK;
    }
    launch_pdl(crop_kernel, grid1d(total), 256, 0, static_cast<cudaStream_t>(stream), image, out, planes, h_in, w_in, top, left, h_out,
                                                                            w_out, round_to_u8);
    RESR_LAUNCH_CHECK("crop");
    return RESR_OK;
}

// ------------------------------------------------------------------------------------------------ whole block in one call
// train_realesrnet.py:267-377 from a POD plan (every host decision of the block + device pointers to its per-sample
// parameters and, optionally, host-fed random draws). Same kernels and same order as the op-level entry points above.
static size_t degrade_max_elems(const resr_degrade_plan* p) {
    auto out_hw = [](int h, int w, const resr_resize_spec& r, int* oh, int* ow) {
        if (r.scale > 0) { *oh = static_cast<int>(floor(static_cast<double>(h) * r.scale)); *ow = static_cast<int>(floor(static_cast<double>(w) * r.scale)); }
        else { *oh = r.out_h; *ow = r.out_w; }
    };
    int h = p->hr_h, w = p->hr_w, h1, w1, h2, w2, h3, w3;
    out_hw(h, w, p->resize1, &h1, &w1);
    out_hw(h1, w1, p->resize2, &h2, &w2);
    out_hw(h2, w2, p->resize3, &h3, &w3);
    size_t m = static_cast<size_t>(h) * w;
    if (static_cast<size_t>(h1) * w1 > m) m = static_cast<size_t>(h1) * w1;
    if (static_cast<size_t>(h2) * w2 > m) m = static_cast<size_t>(h2) * w2;
    if (static_cast<size_t>(h3) * w3 > m) m = static_cast<size_t>(h3) * w3;
    return m * 3 * static_cast<size_t>(p->batch);
}
static size_t up256(size_t v) { return (v + 255) / 256 * 256; }

size_t resr_degrade_workspace_bytes(const resr_degrade_plan* p) {
    if (!p || p->batch <= 0 || p->hr_h <= 0 || p->hr_w <= 0) return 0;
    const size_t img = up256(degrade_max_elems(p) * 4);
    return 2 * img + up256(resr_usm_workspace_bytes(p->batch, 3, p->hr_h, p->hr_w)) + up256(resr_poisson_workspace_bytes(p->batch)) +
           up256(static_cast<size_t>(p->batch) * 4);
}

int resr_degrade_batch(const resr_degrade_plan* p, const float* hr, const float* kernel1, const float* kernel2,
                       const float* sinc_kernel, float* lr_out, float* hr_out, void* workspace, size_t workspace_bytes,
                       void* stream) {
    if (!p || !hr || !lr_out || !hr_out || !workspace || !sinc_kernel) return set_error(RESR_E_INVALID, "null argument");
    if ((p->blur1 && !kernel1) || (p->blur2 && !kernel2) || !p->jpeg1_quality || !p->jpeg2_quality)
        return set_error(RESR_E_INVALID, "plan needs kernels / jpeg qualities");
    if (workspace_bytes < resr_degrade_workspace_bytes(p)) return set_error(RESR_E_NOMEM, "degradation workspace too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int B = p->batch, k = p->kernel_size > 0 ? p->kernel_size : 21;
    uint8_t* base = static_cast<uint8_t*>(workspace);
    const size_t img = up256(degrade_max_elems(p) * 4);
    float* bufs[2] = {reinterpret_cast<float*>(base), reinterpret_cast<float*>(base + img)};
    float* usm_ws = reinterpret_cast<float*>(base + 2 * img);
    void* pws = base + 2 * img + up256(resr_usm_workspace_bytes(B, 3, p->hr_h, p->hr_w));
    float* qtmp = reinterpret_cast<float*>(static_cast<uint8_t*>(pws) + up256(resr_poisson_workspace_bytes(B)));
    int cur = 0, h = p->hr_h, w = p->hr_w;
#define RESR_STEP(expr) do { const int rc__ = (expr); if (rc__ != RESR_OK) return rc__; } while (0)
    auto resize = [&](const resr_resize_spec& r) -> int {
        int oh, ow;
        if (r.scale > 0) { oh = static_cast<int>(floor(static_cast<double>(h) * r.scale)); ow = static_cast<int>(floor(static_cast<double>(w) * r.scale)); }
        else { oh = r.out_h; ow = r.out_w; }
        if (oh == h && ow == w && (r.scale <= 0 || r.scale == 1.0)) return RESR_OK;  // bit-exact identity (SURVEY a12b)
        const int rc = resize_impl(bufs[cur], bufs[cur ^ 1], B * 3, h, w, oh, ow, r.mode, r.scale > 0 ? r.scale : 0.0,
                                   r.scale > 0 ? r.scale : 0.0, s);
        cur ^= 1; h = oh; w = ow;
        return rc;
    };
    auto blur = [&](const float* kern, int kb) -> int {
        const int rc = filter2d_impl(bufs[cur], kern, bufs[cur ^ 1], B, 3, h, w, k, kb, s);
        cur ^= 1;
        return rc;
    };
    auto jpeg = [&](const float* quality) -> int {
        const int rc = jpeg_impl(bufs[cur], bufs[cur ^ 1], quality, qtmp, B, h, w, 1, nullptr, nullptr, nullptr, s);
        cur ^= 1;
        return rc;
    };
    auto noise = [&](const resr_noise_spec& n, int which) -> int {
        if (!n.param) return set_error(RESR_E_INVALID, "noise spec without parameters");
        const float* gray = n.gray_any ? n.gray : nullptr;
        int rc;
        if (n.type == 0) {
            if (n.draws_color) rc = resr_gaussian_noise_apply(bufs[cur], bufs[cur ^ 1], n.param, n.gray, n.draws_color,
                                                              n.gray_any ? n.draws_gray : nullptr, B, 3, h, w, 1, 0, stream);
            else if (!p->rng_state) return set_error(RESR_E_INVALID, "in-kernel noise needs plan->rng_state");
            else rc = resr_gaussian_noise_sampled(bufs[cur], bufs[cur ^ 1], n.param, gray, B, 3, h, w, 1, 0, n.seed,
                                                  p->rng_state + 4 * which, stream);
        } else {
            if (n.draws_color) rc = resr_poisson_noise_apply(bufs[cur], bufs[cur ^ 1], n.param, n.gray, n.draws_color,
                                                             n.gray_any ? n.draws_gray : nullptr, B, 3, h, w, 1, 0, pws,
                                                             resr_poisson_workspace_bytes(B), 0, stream);
            else if (!p->rng_state) return set_error(RESR_E_INVALID, "in-kernel noise needs plan->rng_state");
            else rc = resr_poisson_noise_sampled(bufs[cur], bufs[cur ^ 1], n.param, gray, B, 3, h, w, 1, 0, n.seed,
                                                 p->rng_state + 4 * which + 2, pws, resr_poisson_workspace_bytes(B), stream);
        }
        cur ^= 1;
        return rc;
    };
    RESR_STEP(usm_impl(hr, bufs[cur], usm_ws, B, 3, h, w, p->usm_radius > 0 ? p->usm_radius : 50, p->usm_sigma,
                       p->usm_weight, p->usm_threshold, s));                                        // train:268
    if (p->blur1) RESR_STEP(blur(kernel1, 1));                                                       // train:275-276
    RESR_STEP(resize(p->resize1));                                                                   // train:279-288
    RESR_STEP(noise(p->noise1, 0));                                                                  // train:291-304
    RESR_STEP(jpeg(p->jpeg1_quality));                                                               // train:307-309
    if (p->blur2) RESR_STEP(blur(kernel2, 1));                                                       // train:313-314
    RESR_STEP(resize(p->resize2));                                                                   // train:317-329
    RESR_STEP(noise(p->noise2, 1));                                                                  // train:332-345
    if (p->final_order == 0) {                                                                       // train:347-358
        RESR_STEP(resize(p->resize3));
        RESR_STEP(blur(sinc_kernel, p->sinc_batched));
        RESR_STEP(jpeg(p->jpeg2_quality));
    } else {                                                                                         // train:360-371
        RESR_STEP(jpeg(p->jpeg2_quality));
        RESR_STEP(resize(p->resize3));
        RESR_STEP(blur(sinc_kernel, p->sinc_batched));
    }
#undef RESR_STEP
    const int up = p->upscale > 0 ? p->upscale : 4, ls = p->image_size / up;                         // train:374-377
    int rc = resr_crop(bufs[cur], lr_out, B * 3, h, w, p->crop_top / up, p->crop_left / up, ls, ls, 1, stream);
    if (rc != RESR_OK) return rc;
    return resr_crop(hr, hr_out, B * 3, p->hr_h, p->hr_w, p->crop_top, p->crop_left, p->image_size, p->image_size, 0, stream);
}

}  // extern "C"
