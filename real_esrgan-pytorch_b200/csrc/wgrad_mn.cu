// Weight gradient of 3x3 convolutions on the tensor cores, operands read STRAIGHT from the NHWC buffers the forward and
// the data-gradient convolutions leave behind (no channels-first copies, no pre-shifted copies):
//     dW[co][ci][dy][dx] = sum_{n,y,x} dY[n,y,x,co] * X[n, y+dy-1, x+dx-1, ci]          (autograd of model.py:75-79)
// The contraction runs over pixels, and in an NHWC tensor the pixel index is the SLOW dimension of both operands: a TMA box
// of 64 channels x R pixels lands in shared memory as R rows of 128 bytes (128B swizzle), which is exactly the canonical
// MN-MAJOR operand layout of tcgen05.mma (cute/arch/mma_sm100_desc.hpp: ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units;
// LBO = distance between 64-channel chunks, SBO = 1024 B between groups of eight pixel rows). Both operands are MN-major
// (instruction-descriptor bits 15 / 16). A one-pixel shift along x is a 128-byte shift of the descriptor start address
// (the swizzle is a function of the absolute shared-memory address, the same property the forward kernel uses for its
// dx shifts), a shift along y is a TMA coordinate; borders are zero-filled by TMA.
//
// One pipeline stage = 64 pixels of one image row of dY (x0 .. x0+63) and the 66 pixels x0-1 .. x0+64 of row y+dy-1 of X:
//     A  = X tile   [128 ci x 66 px]   (two 64-channel chunks; channels past the tensor's end are zero-filled)   M = 128
//     B  = dY tile  [n co x 64 px]     (n = 64 or 128)
//     D[dx] (TMEM, 128 x n fp32) += A(rows dx .. dx+63) * B       for dx = 0, 1, 2  -> 3 accumulators, 3n <= 384 columns
// A CTA owns one unit (ci block, co chunk), ONE dy, and a contiguous range of pixel stages (split-K); its three
// accumulators go to a partial buffer and wgrad_mn_reduce_kernel sums the splits into the OIHW gradients of the layers
// that own the channel slices (a dense block's five layers share X and sit side by side in dYcat', train.cu).
// Requires X and dY in ONE 16-bit format, bf16 (train.cu converts the fp16 recipe's saved activations first).
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "conv3x3.cuh"
#include "device_state.h"
#include "ptx.cuh"
#include "wgrad.cuh"

namespace resr {

static constexpr int kMnXChunk = 72 * 128;                       // 66 rows loaded, rounded up to whole 8-row groups
static constexpr int kMnYChunk = 64 * 128;
static constexpr int kMnSlabBytes = 2 * kMnXChunk + 2 * kMnYChunk;  // 34,816: one 64-pixel slab (X tile + dY tile)
static constexpr int kMnSub = 2;                                 // slabs per pipeline stage (one barrier round trip per 24 MMAs)
static constexpr int kMnStageBytes = kMnSub * kMnSlabBytes;      // 69,632
static constexpr int kMnStages = 3;
static constexpr int kMnTileFloats = 3 * 128 * 128;              // one CTA's partial tile [dx][ci][co (16-byte groups XOR-swizzled by ci & 7)]

// MN-major, 128B-swizzled operand: start address | LBO (bits 16..29) in the low word; SBO = 1024 B, version 1, SWIZZLE_128B.
static constexpr uint32_t kMnDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t mn_desc(uint32_t addr16, uint32_t lbo16) {
    return (static_cast<uint64_t>(kMnDescHi) << 32) | (lbo16 << 16) | (addr16 & 0x3FFFu);
}
__device__ __forceinline__ void bulk_store_1d(void* gdst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(reinterpret_cast<uint64_t>(gdst)),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}

__global__ void __launch_bounds__(256, 1)
wgrad_mn_kernel(const __grid_constant__ CUtensorMap tmapX, const __grid_constant__ CUtensorMap tmapDY, const WgradMnArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* misc = smem + kMnStages * kMnStageBytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(misc);
    uint64_t* empty = full + kMnStages;
    uint64_t* done = empty + kMnStages;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(done + 1);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    int kind = 0;
    while (kind + 1 < a.nkinds && static_cast<int>(blockIdx.x) >= a.kind[kind + 1].cta0) ++kind;
    const WgradMnKind kd = a.kind[kind];
    const uint32_t split = blockIdx.x - kd.cta0;
    // 32-bit index arithmetic throughout (the launcher checks kslabs * nsplit < 2^32): 64-bit divisions are subroutine
    // calls of ~1 us each on one warp
    const uint32_t k0 = a.kslabs * split / static_cast<uint32_t>(kd.nsplit);
    const uint32_t k1 = a.kslabs * (split + 1) / static_cast<uint32_t>(kd.nsplit);
    const int nyc = kd.n >> 6;  // 64-channel chunks of dY
    // bias gradient = column sums of dY: the CTAs of the (ci block 0, dy = 1) kinds see every dY tile exactly once, their
    // four epilogue warps (idle during the main loop) sum the tiles out of shared memory
    const bool bias_cta = a.bias_partial != nullptr && kd.dy == 1 && kd.ci0 == 0;

    if (threadIdx.x == 0) {
        prefetch_tmap(&tmapX);
        prefetch_tmap(&tmapDY);
        for (int i = 0; i < kMnStages; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, bias_cta ? 5 : 1); }
        mbar_init(done, 1);
        fence_mbar_init();
    }
    if (warp == 2) { tmem_alloc(tmem_ptr, 512); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = *tmem_ptr;
    const uint32_t segs = a.segs_per_row;

    if (warp == 0) {
        int stage = 0; uint32_t phase = 0;
        // (xs, y, n) of the first slab, then incremented
        uint32_t xs = k0 % segs, y = (k0 / segs) % static_cast<uint32_t>(a.H), n = k0 / (segs * static_cast<uint32_t>(a.H));
        for (uint32_t k = k0; k < k1; k += kMnSub) {
            const int cnt = k1 - k < kMnSub ? static_cast<int>(k1 - k) : kMnSub;
            mbar_wait(empty + stage, phase ^ 1);
            if (elect_one()) {
                uint8_t* st = smem + stage * kMnStageBytes;
                mbar_expect_tx(full + stage, cnt * (2 * 66 * 128 + nyc * kMnYChunk));
                uint32_t xs2 = xs, y2 = y, n2 = n;
                for (int sub = 0; sub < cnt; ++sub, st += kMnSlabBytes) {
                    const int px = static_cast<int>(xs2) * 64, yy = static_cast<int>(y2), nn = static_cast<int>(n2);
                    tma_load_4d(st, &tmapX, full + stage, kd.ci0, px - 1, yy + kd.dy - 1, nn);
                    tma_load_4d(st + kMnXChunk, &tmapX, full + stage, kd.ci0 + 64, px - 1, yy + kd.dy - 1, nn);
                    for (int j = 0; j < nyc; ++j)
                        tma_load_4d(st + 2 * kMnXChunk + j * kMnYChunk, &tmapDY, full + stage, kd.co0 + 64 * j, px, yy, nn);
                    if (++xs2 == segs) { xs2 = 0; if (++y2 == static_cast<uint32_t>(a.H)) { y2 = 0; ++n2; } }
                }
            }
            __syncwarp();
            if (++stage == kMnStages) { stage = 0; phase ^= 1; }
            for (int sub = 0; sub < kMnSub; ++sub)
                if (++xs == segs) { xs = 0; if (++y == static_cast<uint32_t>(a.H)) { y = 0; ++n; } }
        }
    } else if (warp == 1) {
        const uint32_t idesc = make_idesc_f16(1, 128, kd.n) | (1u << 15) | (1u << 16);   // A and B MN-major
        const uint32_t s16 = (smem_u32(smem) & 0x3FFFFu) >> 4;
        int stage = 0; uint32_t phase = 0;
        uint32_t acc = 0;
        for (uint32_t k = k0; k < k1; k += kMnSub) {
            const int cnt = k1 - k < kMnSub ? static_cast<int>(k1 - k) : kMnSub;
            mbar_wait(full + stage, phase);
            tc_fence_after();
            if (elect_one()) {
                for (int sub = 0; sub < cnt; ++sub) {
                    const uint32_t xa = s16 + ((stage * kMnStageBytes + sub * kMnSlabBytes) >> 4);
                    const uint32_t ya = xa + ((2 * kMnXChunk) >> 4);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t bd = mn_desc(ya + ks * (2048 >> 4), kMnYChunk >> 4);
#pragma unroll
                        for (int dx = 0; dx < 3; ++dx)
                            umma_f16(tbase + dx * kd.n, mn_desc(xa + ks * (2048 >> 4) + dx * (128 >> 4), kMnXChunk >> 4), bd, idesc,
                                     (acc | sub | ks) ? 1u : 0u);
                    }
                }
                umma_commit(empty + stage);
            }
            __syncwarp();
            acc = 1;
            if (++stage == kMnStages) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) umma_commit(done);
        __syncwarp();
    } else if (warp >= 4) {
        const int q = warp & 3;
        const int m = q * 32 + lane;  // ci row within the unit
        if (bias_cta) {
            const int t = threadIdx.x - 128, half = kd.n >> 1;     // thread -> (channel pair, row group)
            const int cp = t % half, rg = t / half, rows = (64 * half) >> 7;   // 256 / n row groups of 64 / (256 / n) rows
            const uint32_t coff = 2 * kMnXChunk + (cp >> 5) * kMnYChunk + (cp & 3) * 4;
            const int c16 = (cp & 31) >> 2;
            float s0 = 0.f, s1 = 0.f;
            int stage = 0; uint32_t phase = 0;
            for (uint32_t k = k0; k < k1; k += kMnSub) {
                const int cnt = k1 - k < kMnSub ? static_cast<int>(k1 - k) : kMnSub;
                mbar_wait(full + stage, phase);
                for (int sub = 0; sub < cnt; ++sub) {
                    const uint8_t* yt = smem + stage * kMnStageBytes + sub * kMnSlabBytes + coff;
#pragma unroll 8
                    for (int r = rg * rows; r < (rg + 1) * rows; ++r) {
                        const uint32_t v = *reinterpret_cast<const uint32_t*>(yt + r * 128 + ((c16 ^ (r & 7)) << 4));
                        s0 += __uint_as_float(v << 16);
                        s1 += __uint_as_float(v & 0xFFFF0000u);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty + stage);
                if (++stage == kMnStages) { stage = 0; phase ^= 1; }
            }
            float* bp = a.bias_partial + static_cast<size_t>(blockIdx.x) * 256 + rg * kd.n + 2 * cp;
            bp[0] = s0; bp[1] = s1;
        }
        mbar_wait(done, 0);
        tc_fence_after();
        named_bar_sync(1, 128);   // every warp has left the bias loop: the stage buffers may be overwritten
        // Accumulators -> shared memory (the pipeline buffers are free now) -> ONE 64 KB bulk store per dx. Row m of a tile
        // is 512 B; its 16-byte groups are XOR-swizzled by (m & 7) so that a quarter-warp's float4 stores hit distinct
        // banks; the global partial tile keeps that layout and the reduction kernel un-swizzles.
        const bool any = k1 > k0;
#pragma unroll 1
        for (int dx = 0; dx < 3; ++dx) {
            float4* row = reinterpret_cast<float4*>(smem + dx * 65536 + m * 512);
#pragma unroll 1
            for (int c = 0; c < kd.n; c += 32) {
                float v[32];
                tmem_ld32(tbase + (static_cast<uint32_t>(q * 32) << 16) + dx * kd.n + c, v);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    row[((c >> 2) + i) ^ (m & 7)] = any ? make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (threadIdx.x == 128) {
            float* dst = a.partial + static_cast<size_t>(blockIdx.x) * kMnTileFloats;
            for (int dx = 0; dx < 3; ++dx) bulk_store_1d(dst + dx * 16384, smem + dx * 65536, 65536);
            tma_store_commit();
            tma_store_wait_read();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tbase, 512);
}

// dW of the layer owning each 32-channel slice of dY: sum over the splits of a kind. One thread per partial element
// (kind, dx, ci, co): the split-strided reads are coalesced along co, the OIHW write happens once. The first `nbias`
// threads also finish the bias gradients from the per-block column sums.
__global__ void __launch_bounds__(256) wgrad_mn_reduce_kernel(const WgradMnArgs a, const WgradMnTable tb, int nbias) {
    const size_t total = static_cast<size_t>(a.nkinds) * kMnTileFloats;
    for (size_t e = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; e < total; e += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const int col = e & 127;
        const int m = (e >> 7) & 127;
        const int dx = static_cast<int>((e >> 14) % 3);
        const int kind = static_cast<int>(e / kMnTileFloats);
        const WgradMnKind kd = a.kind[kind];
        if (col >= kd.n) continue;
        const int ci = kd.ci0 + m, cc = kd.co0 + col, cs = cc >> 5;
        const int co = tb.co_base[cs] + (cc & 31);
        if (ci >= tb.cin[cs] || co >= tb.cout[cs]) continue;
        // (dx, m) tile row, 16-byte group XOR-swizzled by m & 7 (the epilogue's shared-memory layout, kept in global memory)
        const float* p = a.partial + static_cast<size_t>(kd.cta0) * kMnTileFloats + (static_cast<size_t>(dx) * 128 + m) * 128 +
                         ((((col >> 2) ^ (m & 7)) << 2) | (col & 3));
        // fixed summation order (bit-reproducible), four independent loads in flight per thread
        float s = 0.f;
        int sp = 0;
        for (; sp + 4 <= kd.nsplit; sp += 4) {
            const float v0 = p[static_cast<size_t>(sp) * kMnTileFloats], v1 = p[static_cast<size_t>(sp + 1) * kMnTileFloats];
            const float v2 = p[static_cast<size_t>(sp + 2) * kMnTileFloats], v3 = p[static_cast<size_t>(sp + 3) * kMnTileFloats];
            s += v0; s += v1; s += v2; s += v3;
        }
        for (; sp < kd.nsplit; ++sp) s += p[static_cast<size_t>(sp) * kMnTileFloats];
        tb.dw[cs][((static_cast<size_t>(co) * tb.cin[cs] + ci) * 3 + kd.dy) * 3 + dx] = s;
    }
    const size_t gt = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (gt < static_cast<size_t>(nbias) && a.bias_partial) {
        const int cc = static_cast<int>(gt), cs = cc >> 5;
        const int co = tb.co_base[cs] + (cc & 31);
        if (co < tb.cout[cs]) {
            float s = 0.f;
            for (int kind = 0; kind < a.nkinds; ++kind) {
                const WgradMnKind kd = a.kind[kind];
                if (kd.dy != 1 || kd.ci0 != 0 || cc < kd.co0 || cc >= kd.co0 + kd.n) continue;
                const int nrg = 256 / kd.n;
                for (int sp = 0; sp < kd.nsplit; ++sp)
                    for (int rg = 0; rg < nrg; ++rg) s += a.bias_partial[static_cast<size_t>(kd.cta0 + sp) * 256 + rg * kd.n + (cc - kd.co0)];
            }
            tb.db[cs][co] = s;
        }
    }
}

// NHWC 16-bit tensor [N][H][W][cstride], channels [0, C) visible (the rest of a 64-channel box is zero-filled);
// box = 64 channels x `rows` pixels of one image row.
static int make_nhwc_map(CUtensorMap* out, const void* base, int C, int cstride, int N, int H, int W, int rows) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return -1;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(N)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(cstride) * 2, static_cast<cuuint64_t>(W) * cstride * 2,
                                   static_cast<cuuint64_t>(H) * W * cstride * 2};
    const cuuint32_t box[4] = {64, static_cast<cuuint32_t>(rows), 1, 1};
    const cuuint32_t es[4] = {1, 1, 1, 1};
    const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

size_t wgrad_mn_workspace_bytes(int num_sms) {
    return static_cast<size_t>(num_sms + 16) * (kMnTileFloats + 256) * sizeof(float);
}

static int wgrad_mn_set_smem_attr(int smem) {
    static PerDevice<bool> attr;
    if (!attr.cur()) {
        if (cudaFuncSetAttribute(wgrad_mn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -3;
        attr.cur() = true;
    }
    return 0;
}

// units: (ci0, co0, n) triples; every unit is expanded into its three dy kinds. CTAs are dealt to the kinds in proportion
// to their per-slab MMA cost, every kind gets at least one.
int wgrad_mn_launch(const uint16_t* x, int x_cstride, int x_channels, const uint16_t* dy, int dy_cstride, int dy_channels,
                    int N, int H, int W, const int (*units)[3], int nunits, const WgradMnTable& tb, bool with_bias,
                    float* workspace, int num_sms, cudaStream_t s) {
    if (nunits < 1 || nunits * 3 > kMnMaxKinds) return -2;
    if ((x_cstride & 7) || (dy_cstride & 7) || (dy_channels & 7) || dy_channels > 192) return -2;
    WgradMnArgs a;
    memset(&a, 0, sizeof(a));
    a.N = N; a.H = H; a.W = W;
    a.segs_per_row = (W + 63) / 64;
    const long long kslabs = static_cast<long long>(N) * H * a.segs_per_row;
    if (kslabs * (num_sms + 16) >= (1ll << 32)) return -2;   // the kernel's index arithmetic is 32-bit
    a.kslabs = static_cast<uint32_t>(kslabs);
    a.partial = workspace;
    a.nkinds = nunits * 3;
    int weight[kMnMaxKinds], share[kMnMaxKinds];
    long long wsum = 0;
    for (int u = 0; u < nunits; ++u)
        for (int d = 0; d < 3; ++d) {
            WgradMnKind& k = a.kind[u * 3 + d];
            k.ci0 = units[u][0]; k.co0 = units[u][1]; k.n = units[u][2]; k.dy = d;
            if (k.n != 64 && k.n != 128) return -2;
            // cost of a slab = 12 MMAs: 64 cycles each at N = 128, 48 at N = 64 (shared-memory operand bound, tools/mma_mn_bench.cu)
            weight[u * 3 + d] = k.n == 128 ? 4 : 3;
            wsum += weight[u * 3 + d];
        }
    long long cap = kslabs / 4;
    if (cap < 1) cap = 1;
    int used = 0;
    for (int i = 0; i < a.nkinds; ++i) {
        long long v = static_cast<long long>(num_sms) * weight[i] / wsum;
        if (v < 1) v = 1;
        if (v > cap) v = cap;
        share[i] = static_cast<int>(v);
        used += share[i];
    }
    // hand the SMs left over by the rounding to the heaviest kinds first
    for (int pass = 0; pass < 2 && used < num_sms; ++pass)
        for (int i = 0; i < a.nkinds && used < num_sms; ++i)
            if (weight[i] >= (pass == 0 ? 4 : 0) && share[i] < cap) { ++share[i]; ++used; }
    int cta = 0;
    for (int i = 0; i < a.nkinds; ++i) { a.kind[i].cta0 = cta; a.kind[i].nsplit = share[i]; cta += share[i]; }
    if (cta > num_sms + 16) return -2;
    CUtensorMap mx, my;
    int rc = make_nhwc_map(&mx, x, x_channels, x_cstride, N, H, W, 66);
    rc |= make_nhwc_map(&my, dy, dy_channels, dy_cstride, N, H, W, 64);
    if (rc != 0) return rc;
    const int smem = 1024 + kMnStages * kMnStageBytes + 256;
    if (wgrad_mn_set_smem_attr(smem) != 0) return -3;
    a.bias_partial = with_bias ? workspace + static_cast<size_t>(num_sms + 16) * kMnTileFloats : nullptr;
    wgrad_mn_kernel<<<cta, 256, smem, s>>>(mx, my, a);
    const size_t total = static_cast<size_t>(a.nkinds) * kMnTileFloats;
    wgrad_mn_reduce_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(a, tb, with_bias ? dy_channels : 0);
    return cudaGetLastError() == cudaSuccess ? 0 : -4;
}

}  // namespace resr
