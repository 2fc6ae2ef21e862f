// What the two tcgen05 convolution kernels (conv3x3_tc.cu: one CTA, conv3x3_pair.cu: CTA pairs) share: the
// shared-memory layout constants, operand descriptors, the bias-armed accumulator init, the whole epilogue after the
// accumulator row has been drained into registers, and the host launch.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstring>

#include "conv3x3.cuh"
#include "device_state.h"
#include "ptx.cuh"

namespace resr {

static constexpr int kStageBytes = 17408;  // 136 rows x 128 B (mode 0 uses BW + 2 rows, mode 1 uses 128)
static constexpr int kMaxStages = 12;
static constexpr int kMiscBytes = 1024;
static constexpr int kSmemMax = 232448;    // 227 KB opt-in limit per CTA
static constexpr int kTileFBytes = 16384;  // 128 px x 32 fp32

struct RowRange {   // 32-bit on purpose: 64-bit divisions are ~100-instruction subroutines and every role decodes its strips
    int g0, g1;     // (the launcher refuses problems with rows_total * grid >= 2^31)
};

// K-major, 128B-swizzled operand descriptor: constant high word (SBO = 1024 B, version 1, SWIZZLE_128B) + low word.
static constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t desc_of(uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; }

// One staging buffer of an epilogue group: [fp32 tile][16-bit tile of `subw` channels]. A group holds epi_bufs of them.
__host__ __device__ inline int epi_buf_bytes(const ConvArgs& a, int subw) {
    const int f = a.has_outf ? kTileFBytes : 0;
    const int h = a.has_out16 ? 128 * subw * 2 : 0;
    return f + (h + 1023) / 1024 * 1024;
}
__host__ __device__ inline int epi_group_bytes(const ConvArgs& a, int subw) {
    return (a.epi_bufs == 2 ? 2 : 1) * epi_buf_bytes(a, subw);
}

template <int W>
__device__ __forceinline__ void tmem_ld_w(uint32_t taddr, float* v) {
    if (W == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
}
// Re-arm an accumulator with the layer's BIAS instead of zero: the MMAs then accumulate on top of it and the epilogue
// needs no bias add (32 FADDs + their shared loads per pass for 8 vector loads; the epilogue warps are issue-bound:
// 41.0 -> 39.8 ms per cfg3 forward, same-box A/B in profiles/r02_epilogue_ab.txt).
template <int W>
__device__ __forceinline__ void tmem_init_bias(uint32_t taddr, const float* __restrict__ bias_w) {
    float b[W];
#pragma unroll
    for (int i = 0; i < W / 4; ++i) {
        const float4 q = reinterpret_cast<const float4*>(bias_w)[i];
        b[4 * i] = q.x; b[4 * i + 1] = q.y; b[4 * i + 2] = q.z; b[4 * i + 3] = q.w;
    }
    if (W == 32) tmem_st32(taddr, b); else tmem_st16(taddr, b);
}

// eight 16-bit values (fp16 or bf16) of a uint4 -> fp32
__device__ __forceinline__ void unpack16x8(const uint4 q, int fmt, float (&f)[8]) {
    const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (fmt == 1) {
            f[2 * i] = __uint_as_float(w4[i] << 16);
            f[2 * i + 1] = __uint_as_float(w4[i] & 0xFFFF0000u);
        } else {
            const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&w4[i]));
            f[2 * i] = h.x;
            f[2 * i + 1] = h.y;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------ epilogue
//
// One epilogue pass handles W channels (32, or 16 for the RGB output convolution) of one output pixel per thread. `ls`
// is the pass's logical W-channel slice: it selects the channel offsets and the per-slice output flags.

// Cout slice `ls` takes part in an output / input whose per-slice opt-out bit mask is `off_mask`.
__device__ __forceinline__ bool slice_on(int has, unsigned off_mask, int ls) { return has && !((off_mask >> ls) & 1u); }

// The epilogue thread's pixel in the output row being drained.
struct EpiPixel {
    int n, x, y;     // image, column, row
    int n0, x0;      // origin of the tile (TMA store coordinates)
    bool valid;      // a real pixel (lanes past W or N carry padding)
    bool inside;     // packed canvas: the pixel belongs to an image (always true without a canvas)
    size_t pix;      // NHWC pixel index (pixel 0 of row y for an invalid lane, so its loads stay in bounds)
};

template <bool MASKED>
__device__ __forceinline__ EpiPixel epi_pixel(const ConvArgs& a, int n0, int x0, int n, int x, int y, bool emit) {
    EpiPixel p;
    p.n = n; p.x = x; p.y = y; p.n0 = n0; p.x0 = x0;
    p.valid = (n < a.N) && (x < a.W);
    p.pix = (static_cast<size_t>(p.valid ? n : 0) * a.H + y) * a.W + (p.valid ? x : 0);
    p.inside = true;   // canvas pixel of an image (vmask), read before the accumulator wait like the residual
    if (MASKED && emit) {
        const int lx = (p.valid ? x : 0) >> a.vmask_shift, ly = y >> a.vmask_shift;
        p.inside = (__ldg(a.vmask + static_cast<size_t>(ly) * a.vmask_words + (lx >> 5)) >> (lx & 31)) & 1u;
    }
    return p;
}

// The residual of this pass: fp32, or (res16) W 16-bit values in the first W / 8 entries. Issued before the wait for the
// accumulator, so that the latency hides behind the row's MMAs.
template <int W>
__device__ __forceinline__ void epi_load_res1(const ConvArgs& a, size_t pix, int ls, float4 (&resv)[W / 4]) {
    if (a.res16) {
        const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.res1) + pix * a.res1_cstride +
                                                         a.res_choff + ls * W);
#pragma unroll
        for (int i = 0; i < W / 8; ++i) {
            const uint4 q4 = rp[i];
            resv[i] = make_float4(__uint_as_float(q4.x), __uint_as_float(q4.y), __uint_as_float(q4.z), __uint_as_float(q4.w));
        }
    } else {
        const float4* rp = reinterpret_cast<const float4*>(static_cast<const float*>(a.res1) + pix * a.res1_cstride +
                                                           a.res_choff + ls * W);
#pragma unroll
        for (int i = 0; i < W / 4; ++i) resv[i] = rp[i];
    }
}

// An epilogue warp group (4 warps, 128 threads: one pixel of the tile each) and its staging buffers.
struct EpiGroup {
    uint8_t* tiles;   // the group's staging buffer(s)
    int buf_bytes;    // bytes of one buffer
    bool two_bufs;    // alternate two buffers: a pass never waits for the TMA store of the pass before
    uint32_t pass;    // staged passes so far (selects the buffer)
    int gi;           // group index: named barrier 1 + gi
    int m;            // this thread's pixel of the tile (== TMEM lane)
    bool lead_warp;   // the group's first warp issues its TMA traffic
};

// Everything after the drain: residuals, RRDB / ADD2, LeakyReLU, canvas mask, pre-clamp NCHW copy, clamp, staging
// (fp32 tile, LeakyReLU' mask, out16 scale, 16-bit pack), TMA stores, NCHW and u8 stores. `val` holds the accumulator
// (bias included); `resv` what epi_load_res1 fetched, if this slice reads res1.
template <int W, bool MASKED>
__device__ __forceinline__ void epi_pass(const ConvArgs& a, const CUtensorMap* tmapO16, const CUtensorMap* tmapOF,
                                         EpiGroup& grp, const EpiPixel& p, int ls, float (&val)[W], float4 (&resv)[W / 4]) {
    const bool use_res1 = slice_on(a.has_res1, a.slice_nores_mask, ls);
    const bool use_outf = slice_on(a.has_outf, a.slice_noutf_mask, ls);
    const bool use_o16 = slice_on(a.has_out16, a.slice_no16_mask, ls);
    const bool staged = use_o16 || use_outf;
    const int m = grp.m;

    if (use_res1 && a.res16) {  // widen the 16-bit residual in place (consumed below as fp32)
        float wide[W];
#pragma unroll
        for (int i = 0; i < W / 8; ++i) {
            float f8[8];
            unpack16x8(make_uint4(__float_as_uint(resv[i].x), __float_as_uint(resv[i].y), __float_as_uint(resv[i].z),
                                  __float_as_uint(resv[i].w)), a.res16_fmt, f8);
#pragma unroll
            for (int e = 0; e < 8; ++e) wide[8 * i + e] = f8[e];
        }
#pragma unroll
        for (int i = 0; i < W / 4; ++i) resv[i] = make_float4(wide[4 * i], wide[4 * i + 1], wide[4 * i + 2], wide[4 * i + 3]);
    }
    if (use_res1) {
#pragma unroll
        for (int i = 0; i < W / 4; ++i) {
            const float4 r4 = resv[i];
            if (a.ep_mode == EP_SKIP || a.ep_mode == EP_ADD2) {
                val[4 * i + 0] = __fadd_rn(r4.x, val[4 * i + 0]);
                val[4 * i + 1] = __fadd_rn(r4.y, val[4 * i + 1]);
                val[4 * i + 2] = __fadd_rn(r4.z, val[4 * i + 2]);
                val[4 * i + 3] = __fadd_rn(r4.w, val[4 * i + 3]);
            } else {   // v * 0.2 + r: separately rounded product and sum (reference order), two lanes per instruction
                const float2 p01 = __fmul2_rn(make_float2(val[4 * i + 0], val[4 * i + 1]), make_float2(0.2f, 0.2f));
                const float2 p23 = __fmul2_rn(make_float2(val[4 * i + 2], val[4 * i + 3]), make_float2(0.2f, 0.2f));
                const float2 s01 = __fadd2_rn(p01, make_float2(r4.x, r4.y));
                const float2 s23 = __fadd2_rn(p23, make_float2(r4.z, r4.w));
                val[4 * i + 0] = s01.x; val[4 * i + 1] = s01.y; val[4 * i + 2] = s23.x; val[4 * i + 3] = s23.y;
            }
        }
    }
    uint8_t* const tileR = grp.tiles + ((grp.two_bufs && (grp.pass & 1u)) ? grp.buf_bytes : 0);  // fp32 output tile
    uint8_t* const tile16 = tileR + (a.has_outf ? kTileFBytes : 0);                                 // 16-bit output tile
    if (staged) {
        // the staging buffer is free once the TMA stores that last used it have read it: the previous pass's (one
        // buffer) or the pass before that (two buffers: the wait is normally already satisfied)
        if (grp.lead_warp) { if (grp.two_bufs) tma_store_wait_read1(); else tma_store_wait_read(); }
        named_bar_sync(1 + grp.gi, 128);
        ++grp.pass;
    }
    if (a.ep_mode == EP_RRDB) {
        if (a.res16) {
            // plain (coherent) loads: in the inference trunk res2 is the RRDB input held in the very buffer this launch
            // overwrites -- each element is read by the thread that later stores its replacement
            const uint4* r2 = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.res2) + p.pix * a.res2_cstride +
                                                             a.res_choff + ls * W);
#pragma unroll
            for (int i = 0; i < W / 8; ++i) {
                float f8[8];
                unpack16x8(r2[i], a.res16_fmt, f8);
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                    const float2 pp = __fmul2_rn(make_float2(val[8 * i + e], val[8 * i + e + 1]), make_float2(0.2f, 0.2f));
                    const float2 ss = __fadd2_rn(pp, make_float2(f8[e], f8[e + 1]));
                    val[8 * i + e] = ss.x; val[8 * i + e + 1] = ss.y;
                }
            }
        } else {
            const float4* r2 = reinterpret_cast<const float4*>(static_cast<const float*>(a.res2) + p.pix * a.res2_cstride +
                                                               a.res_choff + ls * W);
#pragma unroll
            for (int i = 0; i < W / 4; ++i) {
                const float4 r4 = __ldg(r2 + i);
                val[4 * i + 0] = __fadd_rn(__fmul_rn(val[4 * i + 0], 0.2f), r4.x);
                val[4 * i + 1] = __fadd_rn(__fmul_rn(val[4 * i + 1], 0.2f), r4.y);
                val[4 * i + 2] = __fadd_rn(__fmul_rn(val[4 * i + 2], 0.2f), r4.z);
                val[4 * i + 3] = __fadd_rn(__fmul_rn(val[4 * i + 3], 0.2f), r4.w);
            }
        }
    }
    if (a.ep_mode == EP_ADD2 && a.res2) {
        const float4* r2 = reinterpret_cast<const float4*>(static_cast<const float*>(a.res2) + p.pix * a.res2_cstride + a.res_choff + ls * W);
#pragma unroll
        for (int i = 0; i < W / 4; ++i) {
            const float4 r4 = __ldg(r2 + i);
            val[4 * i + 0] = fmaf(a.res2_scale, r4.x, val[4 * i + 0]);
            val[4 * i + 1] = fmaf(a.res2_scale, r4.y, val[4 * i + 1]);
            val[4 * i + 2] = fmaf(a.res2_scale, r4.z, val[4 * i + 2]);
            val[4 * i + 3] = fmaf(a.res2_scale, r4.w, val[4 * i + 3]);
        }
    }
    if (a.lrelu) {   // max(v, 0.2 v) == (v > 0 ? v : 0.2 v) for every finite v; the product is one packed FMUL2 per pair
#pragma unroll
        for (int i = 0; i < W / 2; ++i) {
            const float2 t = __fmul2_rn(make_float2(val[2 * i], val[2 * i + 1]), make_float2(0.2f, 0.2f));
            val[2 * i] = fmaxf(val[2 * i], t.x);
            val[2 * i + 1] = fmaxf(val[2 * i + 1], t.y);
        }
    }
    if (MASKED && !p.inside) {   // gutter / canvas margin: 0 in every output, as the zero padding around an image
#pragma unroll
        for (int i = 0; i < W; ++i) val[i] = 0.f;
    }
    if (a.out_nchw_raw && p.valid) {
        const size_t plane = static_cast<size_t>(a.H) * a.W;
        float* o = a.out_nchw_raw + static_cast<size_t>(p.n) * a.out_nchw_c * plane + static_cast<size_t>(p.y) * a.W + p.x;
#pragma unroll
        for (int c = 0; c < W; ++c) {
            const int cc = ls * W + c;
            if (cc < a.out_nchw_c) o[static_cast<size_t>(cc) * plane] = val[c];
        }
    }
    if (a.clamp01) {
#pragma unroll
        for (int i = 0; i < W; ++i) val[i] = fminf(fmaxf(val[i], 0.f), 1.f);
    }
    if (use_outf) {  // fp32 master (W == 32 only)
#pragma unroll
        for (int i = 0; i < W / 4; ++i)
            *reinterpret_cast<float4*>(tileR + m * 128 + ((i ^ (m & 7)) << 4)) =
                make_float4(val[4 * i], val[4 * i + 1], val[4 * i + 2], val[4 * i + 3]);
    }
    if (use_o16 && a.mask16) {  // LeakyReLU backward: slope 1 where the saved activation is > 0, else 0.2
        const uint4* mk = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.mask16) + p.pix * a.mask16_cstride +
                                                         a.mask16_choff + ls * W);
#pragma unroll
        for (int i = 0; i < W / 8; ++i) {
            const uint4 q4 = __ldg(mk + i);
            const uint32_t w4[4] = {q4.x, q4.y, q4.z, q4.w};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const uint32_t h16 = (w4[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu;
                const bool pos = ((h16 & 0x8000u) == 0) && ((h16 & 0x7FFFu) != 0);
                if (!pos) val[8 * i + e] = __fmul_rn(val[8 * i + e], 0.2f);
            }
        }
    }
    if (use_o16 && a.out16_scale != 0.f) {
#pragma unroll
        for (int i = 0; i < W; ++i) val[i] = __fmul_rn(val[i], a.out16_scale);
    }
    if (use_o16) {
        uint32_t pk[W / 2];
#pragma unroll
        for (int i = 0; i < W / 2; ++i) {
            if (a.out16_fmt == 1) {
                __nv_bfloat162 hh = __floats2bfloat162_rn(val[2 * i], val[2 * i + 1]);
                pk[i] = *reinterpret_cast<uint32_t*>(&hh);
            } else {
                pk[i] = pack_f16x2_sat(val[2 * i], val[2 * i + 1]);  // saturate, never inf
            }
        }
        // (Storing the pixel's channels straight from registers instead -- no staging tile, no proxy fence, no block
        // barrier -- was tried and is slower: 45.5 vs 43.0 ms per cfg3 forward, profiles/r02_direct_store_ab.txt.)
        uint4* dst = reinterpret_cast<uint4*>(tile16 + m * (W * 2));
#pragma unroll
        for (int i = 0; i < W / 8; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
    }
    if (staged) {
        fence_proxy_async_smem();
        named_bar_sync(1 + grp.gi, 128);
        if (grp.lead_warp) {
            if (elect_one()) {
                if (use_outf) tma_store_4d(tmapOF, tileR, a.outf_choff + ls * W, p.x0, p.y, p.n0);
                if (use_o16) {
                    const int c0 = a.out16_choff + (a.out16_slice_fixed ? 0 : ls * W);
                    if (!a.out16_up2) {
                        tma_store_4d(tmapO16, tile16, c0, p.x0, p.y, p.n0);
                    } else {
#pragma unroll
                        for (int s = 0; s < 4; ++s) tma_store_5d(tmapO16, tile16, c0, s & 1, p.x0, 2 * p.y + (s >> 1), p.n0);
                    }
                }
                tma_store_commit();
            }
            __syncwarp();
        }
    }
    if (a.out_nchw && p.valid) {
        const size_t plane = static_cast<size_t>(a.H) * a.W;
        float* o = a.out_nchw + static_cast<size_t>(p.n) * a.out_nchw_c * plane + static_cast<size_t>(p.y) * a.W + p.x;
#pragma unroll
        for (int c = 0; c < W; ++c) {
            const int cc = ls * W + c;
            if (cc < a.out_nchw_c) o[static_cast<size_t>(cc) * plane] = val[c];
        }
    }
    if (a.out_u8 && p.valid) {   // clamp01 has been applied: v * 255 lies in [0, 255], the cast truncates
        unsigned char* o = a.out_u8 + ((static_cast<size_t>(p.n) * a.H + p.y) * a.W + p.x) * a.out_nchw_c;
#pragma unroll
        for (int c = 0; c < W; ++c) {
            const int cc = ls * W + c;
            if (cc < a.out_nchw_c) o[cc] = static_cast<unsigned char>(fminf(fmaxf(__fmul_rn(val[c], 255.f), 0.f), 255.f));
        }
    }
}

// ----------------------------------------------------------------------------------------------------------- host side

// Shared-memory bytes of the weights a CTA keeps resident: `nout` accumulator columns per output row, split over the
// `cluster` CTAs that share one MMA.
inline int conv3x3_weight_bytes(const ConvArgs& a, int nout, int cluster) { return a.nchunks * 3 * (3 * nout / cluster) * 128; }

// The single-CTA kernel's launch (conv3x3_tc.cu); conv3x3_run calls it with normalised arguments.
cudaError_t conv3x3_tc_launch(const ConvMaps& maps, const ConvArgs& args, int nout, int nslices, int num_sms, cudaStream_t stream);

// Launches one persistent convolution grid: clusters of `cluster` CTAs over `units` (column group, row) work units,
// `nslices` Cout slices on blockIdx.y, the full 227 KB of shared memory (exactly one CTA -- one 512-column TMEM
// allocation -- per SM), and programmatic stream serialisation so that the next launch's prologue overlaps this one's tail.
template <auto Kernel>
static cudaError_t conv3x3_launch_grid(const ConvMaps& maps, const ConvArgs& args, int nout, int cluster, long long units,
                                       int nslices, int num_sms, cudaStream_t stream) {
    const int subw = nout == 64 ? 32 : nout;
    const int smem = 1024 + conv3x3_weight_bytes(args, nout, cluster) + args.nstages * kStageBytes +
                     args.nepi * epi_group_bytes(args, subw) + kMiscBytes;
    if (args.nstages < 2 || args.nepi < 1 || args.nepi > 3 || smem > kSmemMax) return cudaErrorInvalidConfiguration;
    const long long nclusters = conv3x3_clusters(units, cluster, nslices, num_sms);
    if (units * (nclusters + 1) >= (1ll << 31)) return cudaErrorInvalidValue;   // the kernel's strip arithmetic is 32-bit

    static PerDevice<bool> attr;  // function attributes are per device
    if (!attr.cur()) {
        const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
        if (e != cudaSuccess) return e;
        attr.cur() = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(static_cast<unsigned>(cluster * nclusters), static_cast<unsigned>(nslices), 1);
    cfg.blockDim = dim3(128 + 128 * args.nepi, 1, 1);
    cfg.dynamicSmemBytes = kSmemMax;
    cfg.stream = stream;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    at[1].id = cudaLaunchAttributeClusterDimension;
    at[1].val.clusterDim.x = cluster;
    at[1].val.clusterDim.y = 1;
    at[1].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = cluster > 1 ? 2 : 1;
    return cudaLaunchKernelEx(&cfg, Kernel, maps.a, maps.o16, maps.of, args);
}

}  // namespace resr
