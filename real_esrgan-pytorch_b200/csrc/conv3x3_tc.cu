// 3x3 / stride 1 / zero-pad 1 convolution on the 5th-gen tensor cores (tcgen05 + TMEM), NHWC 16-bit activations.
//
// Replaces nn.Conv2d(…, (3,3), (1,1), (1,1)) + torch.cat + LeakyReLU + residual arithmetic of the reference
// generator (/root/reference/model.py:75-98, 123-132, 255-272). Design ("row-rolling implicit GEMM"):
//
//   * One M tile = 128 output columns of ONE image row (or BW columns x BN images when W < 128): TMEM lane = pixel.
//   * The three vertical taps are folded into the MMA N dimension: for input row r the tensor core computes
//         D'_r[x, (dy, co)] = sum_{dx, ci} in[r, x + dx - 1, ci] * w[co, ci, dy, dx]            (N = 3 * Cout_slice)
//     so every activation row is read from shared memory once per dx instead of once per tap.
//   * out[y] = D'_{y-1}[dy=0] + D'_y[dy=1] + D'_{y+1}[dy=2] is summed BY THE TENSOR CORE: output-row accumulators live
//     in a ring of 16 TMEM slots laid out in descending row order, so the (dy=0, dy=1, dy=2) column blocks of one MMA
//     land exactly on the accumulators of rows (r+1, r, r-1). Every MMA accumulates; the epilogue zeroes a slot after
//     draining it. (At the ring seam the N = 3*NOUT MMA is split into an N = NOUT and an N = 2*NOUT MMA.)
//   * Horizontal taps: mode 0 loads BW+2 pixels once (TMA zero-fills x = -1 and x = W) and shifts the UMMA
//     shared-memory descriptor by dx * 128 B; mode 1 issues one TMA load per dx (used when the lanes span images).
//   * Weights of the CTA's Cout slice stay resident in shared memory for the whole launch (bulk copies).
//   * CTAs are persistent over a contiguous range of (column group, row) work; grid = #SMs / #slices.
//   * Epilogue: one or two groups of 4 warps take alternate output rows: TMEM -> registers -> bias / LeakyReLU /
//     residual -> shared-memory staging tile -> TMA store (coalesced NHWC writes, also the 2x nearest-upsampled
//     variant); the fp32 residual tile arrives by TMA load while the row's MMAs are still running.
//
// Warp roles: warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer, warp 2 = TMEM allocator,
// warps 4-7 (and 8-11) = epilogue groups.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>

#include "conv3x3.cuh"
#include "device_state.h"
#include "ptx.cuh"

// Kernel perturbation flags for bottleneck experiments (tools/power_probe.py); compiled out of the product build.
#ifdef RESR_EXPERIMENTS
#define DBGF(x) ((a.dbg_flags & (x)) != 0)
#else
#define DBGF(x) false
#endif

namespace resr {

static constexpr int kStageBytes = 17408;  // 136 rows x 128 B (mode 0 uses 130 rows, mode 1 uses 128)
static constexpr int kMaxStages = 12;
static constexpr int kSlots = 16;          // TMEM accumulator ring
static constexpr int kMiscBytes = 1024;
static constexpr int kSmemMax = 232448;    // 227 KB opt-in limit per CTA
static constexpr int kTileFBytes = 16384;  // 128 px x 32 fp32

struct RowRange {   // 32-bit on purpose: 64-bit divisions are ~100-instruction subroutines and every role decodes its strips
    int g0, g1;     // (the launcher refuses problems with rows_total * grid >= 2^31)
};

__device__ __forceinline__ RowRange cta_rows(const ConvArgs& a) {
    RowRange r;
    const unsigned rows = static_cast<unsigned>(a.rows_total);
    r.g0 = static_cast<int>(rows * blockIdx.x / gridDim.x);
    r.g1 = static_cast<int>(rows * (blockIdx.x + 1) / gridDim.x);
    return r;
}

__device__ __forceinline__ unsigned long long gtimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define RESR_DBG(slot) do { if (a.dbg && blockIdx.x == 0 && blockIdx.y == 0 && (threadIdx.x & 31) == 0) a.dbg[slot] = gtimer(); } while (0)

__device__ __forceinline__ uint32_t slot_of(uint32_t v) { return (16u - (v & 15u)) & 15u; }

__host__ __device__ inline int epi_group_bytes(const ConvArgs& a, int nout) {
    const int f = a.has_outf ? kTileFBytes : 0;  // fp32 output tile (TMA store)
    const int h = a.has_out16 ? 128 * nout * 2 : 0;
    return f + (h + 1023) / 1024 * 1024;
}


// K-major, 128B-swizzled operand descriptor: constant high word (SBO = 1024 B, version 1, SWIZZLE_128B) + low word.
static constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t desc_of(uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; }

// All MMAs of one pipeline stage, straight-line. SPLIT: 0 = one N=3*NOUT MMA at d0; 1 / 2 = ring seam (slot 14 / 15),
// the (dy=0,1 | dy=2) resp. (dy=0 | dy=1,2) column blocks go to d0 and to the start of the ring. NDX: horizontal taps
// served by this stage (3 in mode 0: descriptor shifted by dx pixels; 1 in mode 1).
template <int NOUT, int SPLIT, int KS, int I0, int I1>
__device__ __forceinline__ void issue_range(uint32_t d0, uint32_t ring0, uint32_t a_lo, uint32_t b_lo, uint32_t idesc3,
                                            uint32_t idesc2, uint32_t idesc1) {
    constexpr uint32_t WT = (3 * NOUT * 128) >> 4;   // one (chunk, dx) weight tile, in 16-byte units
    constexpr uint32_t ROWS = (NOUT * 128) >> 4;     // NOUT weight rows
#pragma unroll
    for (int i = I0; i < I1; ++i) {                  // i = dx * KS + ks; KS = K16 steps that carry real channels
        const int dx = i / KS, ks = i % KS;
        const uint64_t ad = desc_of(a_lo + dx * 8 + ks * 2);
        const uint32_t bl = b_lo + dx * WT + ks * 2;
        if (SPLIT == 0) {
            umma_f16(d0, ad, desc_of(bl), idesc3, 1);
        } else if (SPLIT == 1) {
            umma_f16(d0, ad, desc_of(bl), idesc2, 1);
            umma_f16(ring0, ad, desc_of(bl + 2 * ROWS), idesc1, 1);
        } else {
            umma_f16(d0, ad, desc_of(bl), idesc1, 1);
            umma_f16(ring0, ad, desc_of(bl + ROWS), idesc2, 1);
        }
    }
}
// MMAs [I0, I1) of a stage, dispatching on the ring-seam case (uniform per output row).
template <int NOUT, int KS, int I0, int I1>
__device__ __forceinline__ void issue_part(uint32_t s0, uint32_t d0, uint32_t ring0, uint32_t a_lo, uint32_t b_lo,
                                           uint32_t idesc3, uint32_t idesc2, uint32_t idesc1) {
    if (s0 <= 13) issue_range<NOUT, 0, KS, I0, I1>(d0, ring0, a_lo, b_lo, idesc3, idesc2, idesc1);
    else if (s0 == 14) issue_range<NOUT, 1, KS, I0, I1>(d0, ring0, a_lo, b_lo, idesc3, idesc2, idesc1);
    else issue_range<NOUT, 2, KS, I0, I1>(d0, ring0, a_lo, b_lo, idesc3, idesc2, idesc1);
}


// First (HALF = 0) or second (HALF = 1) half of the MMAs of one pipeline step whose chunk carries `ks` K16 steps of real
// channels (4 for a full 64-channel chunk; fewer for the zero-padded tail chunk of Cin = 96 / 160 / 3).
template <int NOUT, int NDX, int HALF>
__device__ __forceinline__ void issue_half(int ks, uint32_t s0, uint32_t d0, uint32_t ring0, uint32_t a_lo, uint32_t b_lo,
                                           uint32_t idesc3, uint32_t idesc2, uint32_t idesc1) {
#define RESR_HALF(KS)                                                                                              \
    if (HALF == 0) issue_part<NOUT, KS, 0, (NDX * KS) / 2>(s0, d0, ring0, a_lo, b_lo, idesc3, idesc2, idesc1);       \
    else issue_part<NOUT, KS, (NDX * KS) / 2, NDX * KS>(s0, d0, ring0, a_lo, b_lo, idesc3, idesc2, idesc1)
    if (ks == 2) { RESR_HALF(2); }
    else if (ks == 1) { RESR_HALF(1); }
    else { RESR_HALF(4); }
#undef RESR_HALF
}

// Re-arm an accumulator slot with the layer's BIAS instead of zero (see conv3x3_pair.cu tmem_init_bias): the MMAs
// accumulate on top of it and the epilogue needs no bias add.
template <int W>
__device__ __forceinline__ void tmem_init_bias_w(uint32_t taddr, const float* __restrict__ bias_w) {
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

// The MMA-issuing warp. The tensor core is fed by ONE instruction stream with a shallow queue, so every non-MMA
// instruction of this warp is tensor-pipe idle time (tools/mma_bench3.cu): the loop keeps 32-bit incremental
// bookkeeping, probes the NEXT step's barriers (non-blocking test_wait) between the two halves of the current step's
// MMAs, and spaces the two tcgen05.commit of a row (stage release of the previous step, accumulator completion) at
// least six MMAs apart (back-to-back commits cost ~190 cycles each, spaced ones ~90).
template <int NOUT, int MODE>
__device__ __forceinline__ void mma_role(const ConvArgs& a, const RowRange rr, const uint32_t tbase, const uint32_t wsm_addr,
                                         const uint32_t stg_addr, const uint32_t full_a, const uint32_t empty_a,
                                         const uint32_t accfull_a, const uint32_t slotfree_a) {
    constexpr uint32_t WT = (3 * NOUT * 128) >> 4;
    const uint32_t idesc3 = make_idesc_f16(a.fmt_in, 128, 3 * NOUT);
    const uint32_t idesc2 = make_idesc_f16(a.fmt_in, 128, 2 * NOUT);
    const uint32_t idesc1 = make_idesc_f16(a.fmt_in, 128, NOUT);
    const uint32_t w_lo = (wsm_addr & 0x3FFFFu) >> 4;
    const uint32_t s_lo = (stg_addr & 0x3FFFFu) >> 4;
    const int nsteps = MODE == 0 ? a.nchunks : a.nchunks * 3;
    const uint32_t b_step = (MODE == 0 ? 3 : 1) * WT;
    const int nstages = a.nstages;
    const int H = a.H;
    const bool dbg_quarter = DBGF(4), dbg_nomma = DBGF(16);
    int stage = 0;
    uint32_t phase = 0;
    uint32_t a_lo = s_lo;
    int pending_empty = -1;          // stage whose release commit has not been issued yet
    bool full_ready = false, slot_ready = false;
    uint32_t vnew = 1;               // virtual index of the NEWEST accumulator the next row touches (out row r+1)
    uint32_t acq = 0;                // accumulators acquired so far (virtual indices < acq)
    for (int g = rr.g0; g < rr.g1;) {
        const int ya = g % H;
        const int yb = min(H, ya + (rr.g1 - g));
        const int ra = max(ya - 1, 0), rb = min(yb, H - 1);
        vnew += 1;                   // a strip touches rows ra-1 .. rb+1: first row's newest accumulator is v0 + 2
        for (int r = ra; r <= rb; ++r, ++vnew) {
            // accumulators of rows r-1, r, r+1 (virtual vnew-2 .. vnew) must be zeroed & free
            if (slot_ready && acq == vnew) {
                ++acq;
            } else {
                while (static_cast<int>(vnew - acq) >= 0) {
                    mbar_wait_a(slotfree_a + (((0u - acq) & 15u) << 3), (acq >> 4) & 1u);
                    ++acq;
                }
            }
            slot_ready = false;
            tc_fence_after();
            const uint32_t s0 = (0u - vnew) & 15u;
            const uint32_t d0 = tbase + s0 * NOUT;
            uint32_t b_lo = w_lo;
            for (int st = 0; st < nsteps; ++st, b_lo += b_step) {
                if (!full_ready) mbar_wait_a(full_a + (stage << 3), phase);
                tc_fence_after();
                const bool last = (st == nsteps - 1);
                const int ks = dbg_quarter ? 1 : ((st >= nsteps - (MODE == 0 ? 1 : 3)) ? a.tail_ksteps : 4);  // steps of the last K chunk
                if (elect_one()) {
                    if (!dbg_nomma) issue_half<NOUT, MODE == 0 ? 3 : 1, 0>(ks, s0, d0, tbase, a_lo, b_lo, idesc3, idesc2, idesc1);
                    if (pending_empty >= 0) umma_commit_a(empty_a + (pending_empty << 3));
                }
                __syncwarp();
                pending_empty = stage;
                // advance the ring, then probe the next step's barriers behind the MMAs just queued
                const uint32_t a_cur = a_lo;
                if (++stage == nstages) { stage = 0; phase ^= 1u; a_lo = s_lo; } else { a_lo += kStageBytes >> 4; }
                full_ready = mbar_test_wait_a(full_a + (stage << 3), phase);
                if (last && r < rb) slot_ready = mbar_test_wait_a(slotfree_a + (((0u - (vnew + 1)) & 15u) << 3), ((vnew + 1) >> 4) & 1u);
                if (elect_one()) {
                    if (!dbg_nomma) issue_half<NOUT, MODE == 0 ? 3 : 1, 1>(ks, s0, d0, tbase, a_cur, b_lo, idesc3, idesc2, idesc1);
                    if (last) {
                        umma_commit_a(accfull_a + (((s0 + 2) & 15u) << 3));      // row r-1 has its last contribution
                        if (r == rb) {                                            // strip end: rows rb, rb+1 get no more
                            umma_commit_a(accfull_a + (((s0 + 1) & 15u) << 3));
                            umma_commit_a(accfull_a + (s0 << 3));
                        }
                    }
                }
                __syncwarp();
            }
        }
        vnew += 1;                   // strip used rb-ra+3 virtual indices
        g += yb - ya;
    }
    if (pending_empty >= 0) {
        if (elect_one()) umma_commit_a(empty_a + (pending_empty << 3));
        __syncwarp();
    }
}

// MASKED: the packed-canvas variant (ConvArgs::vmask set); the other instantiation carries no mask code at all
template <int NOUT, bool MASKED>
__global__ void __launch_bounds__(512, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapO16,
                  const __grid_constant__ CUtensorMap tmapOF,
                  const ConvArgs a) {
    constexpr int NT = 3 * NOUT;     // MMA N: (dy, co)
    constexpr int WTILE = NT * 128;  // bytes of one (chunk, dx) weight tile: NT rows x 64 ch x 2 B
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

    // warp-uniform role index (shuffle => provably uniform: TMA / MMA operands then live in uniform registers)
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int slice = blockIdx.y;
    if (threadIdx.x == 0) RESR_DBG(0);  // kernel entry
    const uint32_t wbytes = static_cast<uint32_t>(a.nchunks) * 3u * WTILE;
    const int epi_bytes = epi_group_bytes(a, NOUT);

    uint8_t* wsm = smem;
    uint8_t* stg = smem + wbytes;
    uint8_t* epi = stg + a.nstages * kStageBytes;
    uint8_t* misc = epi + a.nepi * epi_bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(misc);
    uint64_t* empty = full + kMaxStages;
    uint64_t* acc_full = empty + kMaxStages;
    uint64_t* slot_free = acc_full + kSlots;
    uint64_t* wbar = slot_free + kSlots;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(wbar + 1);
    float* bias_s = reinterpret_cast<float*>(misc + 512);

    if (threadIdx.x == 0) {
        prefetch_tmap(&tmapA);
        if (a.has_out16) prefetch_tmap(&tmapO16);
        if (a.has_outf) prefetch_tmap(&tmapOF);
        for (int i = 0; i < a.nstages; ++i) {
            mbar_init(full + i, 1);
            mbar_init(empty + i, 1);
        }
        for (int i = 0; i < kSlots; ++i) {
            mbar_init(acc_full + i, 1);
            mbar_init(slot_free + i, 128);
        }
        mbar_init(wbar, 1);
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr, 512);
        tmem_relinquish();
    }
    if (threadIdx.x >= 128 && threadIdx.x < 128 + NOUT) bias_s[threadIdx.x - 128] = a.bias[slice * NOUT + threadIdx.x - 128];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = *tmem_ptr;
    if (threadIdx.x == 0) RESR_DBG(1);  // setup done (barriers, TMEM)
    // Programmatic dependent launch: the next kernel in the stream may take over SMs as soon as CTAs of this grid
    // retire (it parks in griddepcontrol.wait until this whole grid has completed and flushed).
    grid_dep_launch();

    const RowRange rr = cta_rows(a);
    const int H = a.H;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (whole warp, one elected lane issues)
        // weights do not depend on the previous kernel: fetch them before the grid dependency resolves
        if (elect_one()) {
            mbar_expect_tx(wbar, wbytes);
            const uint8_t* wsrc = a.wpack + static_cast<size_t>(slice) * wbytes;
            for (int c = 0; c < a.nchunks; ++c) bulk_load_1d(wsm + c * 3 * WTILE, wsrc + static_cast<size_t>(c) * 3 * WTILE, 3 * WTILE, wbar);
        }
        __syncwarp();
        grid_dep_wait();
        RESR_DBG(2);  // previous grid complete
        int stage = 0;
        uint32_t phase = 0;
        const int ndx = a.mode == 0 ? 1 : 3;
        const uint32_t tx_bytes = a.mode == 0 ? (a.BW + 2) * 128 : 128 * 128;
        for (int g = rr.g0; g < rr.g1;) {
            const int cg = g / H;
            const int ya = g % H;
            const int yb = min(H, ya + (rr.g1 - g));
            const int n0 = (cg / a.nxs) * a.BN;
            const int x0 = (cg % a.nxs) * a.BW;
            const int ra = max(ya - 1, 0), rb = min(yb, H - 1);
            for (int r = ra; r <= rb; ++r) {
                for (int c = 0; c < a.nchunks; ++c) {
                    for (int dx = 0; dx < ndx; ++dx) {
                        mbar_wait(empty + stage, phase ^ 1);
                        if (elect_one()) {
                            if (DBGF(32)) {
                                mbar_arrive(full + stage);
                            } else {
                                mbar_expect_tx(full + stage, tx_bytes);
                                tma_load_4d(stg + stage * kStageBytes, &tmapA, full + stage, c * 64,
                                            a.mode == 0 ? x0 - 1 : x0 + dx - 1, DBGF(2) ? 0 : r, DBGF(2) ? 0 : n0);
                            }
                        }
                        __syncwarp();
                        if (++stage == a.nstages) { stage = 0; phase ^= 1; }
                    }
                }
            }
            g += yb - ya;
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (whole warp, one elected lane issues)
        mbar_wait(wbar, 0);
        RESR_DBG(3);  // weights resident
        tc_fence_after();
        if (a.mode == 0) mma_role<NOUT, 0>(a, rr, tbase, smem_u32(wsm), smem_u32(stg), smem_u32(full), smem_u32(empty), smem_u32(acc_full), smem_u32(slot_free));
        else mma_role<NOUT, 1>(a, rr, tbase, smem_u32(wsm), smem_u32(stg), smem_u32(full), smem_u32(empty), smem_u32(acc_full), smem_u32(slot_free));
        RESR_DBG(5);  // all MMAs issued
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue groups
        const int gi = (warp - 4) >> 2;
        const int q = warp & 3;        // TMEM lane quadrant this warp may access
        const int m = q * 32 + lane;   // M row == TMEM lane == pixel of the tile
        const bool lead_warp = ((warp - 4) & 3) == 0;  // first warp of the group issues its TMA traffic
        // per-slice output selection (backward: only the top slice produces the masked 16-bit dY, the others
        // accumulate into the fp32 gradient buffer)
        const bool use_res1 = a.has_res1 && !((a.slice_nores_mask >> slice) & 1u);
        const bool use_outf = a.has_outf && !((a.slice_noutf_mask >> slice) & 1u);
        const bool use_o16 = a.has_out16 && !((a.slice_no16_mask >> slice) & 1u);
        const bool staged = use_o16 || use_outf;
        uint8_t* tileR = epi + gi * epi_bytes;                       // fp32 output tile (TMA store)
        uint8_t* tile16 = tileR + (a.has_outf ? kTileFBytes : 0);  // 16-bit output tile (TMA store)
        const uint32_t lane_base = tbase + (static_cast<uint32_t>(q * 32) << 16);
        const int img_in_tile = m / a.BW;
        const int x_in_tile = m % a.BW;
        {   // zero this group's share of the accumulator ring, then hand the slots to the MMA issuer
            const int s_lo = gi * kSlots / a.nepi, s_hi = (gi + 1) * kSlots / a.nepi;
            for (int s = s_lo; s < s_hi; ++s) tmem_init_bias_w<NOUT>(lane_base + s * NOUT, bias_s);
            tmem_st_wait();
            tc_fence_before();
            for (int s = s_lo; s < s_hi; ++s) mbar_arrive(slot_free + s);
        }
        grid_dep_wait();  // residual reads / output writes below touch buffers of the previous kernel
        uint32_t v0 = 0;
        for (int g = rr.g0; g < rr.g1;) {
            const int cg = g / H;
            const int ya = g % H;
            const int yb = min(H, ya + (rr.g1 - g));
            const int n0 = (cg / a.nxs) * a.BN;
            const int x0 = (cg % a.nxs) * a.BW;
            const int n = n0 + img_in_tile;
            const int x = x0 + x_in_tile;
            const bool valid = (n < a.N) && (x < a.W);
            const int ra = max(ya - 1, 0), rb = min(yb, H - 1);
            const int n_acc = rb - ra + 3;
            for (int j = 0; j < n_acc; ++j) {
                const uint32_t v = v0 + j;
                if (static_cast<int>(v % static_cast<uint32_t>(a.nepi)) != gi) continue;
                const int y = ra - 1 + j;
                const bool emit = (y >= ya) && (y < yb) && !DBGF(8);
                const uint32_t slot = slot_of(v);
                float4 resv[NOUT / 4];   // fp32 residual, or (res16) NOUT 16-bit values in the first NOUT / 8 entries
                if (emit && use_res1) {
                    // this row's residual: contiguous bytes per thread, requested before the wait for the accumulator so
                    // the latency hides behind the row's MMAs
                    const size_t pix = (static_cast<size_t>(valid ? n : 0) * a.H + y) * a.W + (valid ? x : 0);
                    if (a.res16) {
                        const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.res1) + pix * a.res1_cstride +
                                                                         a.res_choff + slice * NOUT);
#pragma unroll
                        for (int i = 0; i < NOUT / 8; ++i) {
                            const uint4 q4 = rp[i];
                            resv[i] = make_float4(__uint_as_float(q4.x), __uint_as_float(q4.y), __uint_as_float(q4.z), __uint_as_float(q4.w));
                        }
                    } else {
                        const float4* rp = reinterpret_cast<const float4*>(static_cast<const float*>(a.res1) + pix * a.res1_cstride +
                                                                           a.res_choff + slice * NOUT);
#pragma unroll
                        for (int i = 0; i < NOUT / 4; ++i) resv[i] = rp[i];
                    }
                }
                bool inside = true;   // canvas pixel of an image (vmask), read before the accumulator wait like the residual
                if (MASKED && emit) {
                    const int lx = (valid ? x : 0) >> a.vmask_shift, ly = y >> a.vmask_shift;
                    inside = (__ldg(a.vmask + static_cast<size_t>(ly) * a.vmask_words + (lx >> 5)) >> (lx & 31)) & 1u;
                }
                mbar_wait(acc_full + slot, static_cast<uint32_t>(v >> 4) & 1);
                tc_fence_after();
                float val[NOUT];
                if (NOUT == 32) tmem_ld32(lane_base + slot * NOUT, val); else tmem_ld16(lane_base + slot * NOUT, val);
                tmem_ld_wait();
                tmem_init_bias_w<NOUT>(lane_base + slot * NOUT, bias_s);
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(slot_free + slot);
                if (!emit) continue;

                // (no bias add here: the accumulator was armed with the bias)
                if (use_res1 && a.res16) {  // widen the 16-bit residual in place (consumed below as fp32)
                    float wide[NOUT];
#pragma unroll
                    for (int i = 0; i < NOUT / 8; ++i) {
                        float f8[8];
                        unpack16x8(make_uint4(__float_as_uint(resv[i].x), __float_as_uint(resv[i].y), __float_as_uint(resv[i].z),
                                              __float_as_uint(resv[i].w)), a.res16_fmt, f8);
#pragma unroll
                        for (int e = 0; e < 8; ++e) wide[8 * i + e] = f8[e];
                    }
#pragma unroll
                    for (int i = 0; i < NOUT / 4; ++i) resv[i] = make_float4(wide[4 * i], wide[4 * i + 1], wide[4 * i + 2], wide[4 * i + 3]);
                }
                if (use_res1) {
#pragma unroll
                    for (int i = 0; i < NOUT / 4; ++i) {
                        const float4 r4 = resv[i];
                        if (a.ep_mode == EP_SKIP || a.ep_mode == EP_ADD2) {
                            val[4 * i + 0] = __fadd_rn(r4.x, val[4 * i + 0]);
                            val[4 * i + 1] = __fadd_rn(r4.y, val[4 * i + 1]);
                            val[4 * i + 2] = __fadd_rn(r4.z, val[4 * i + 2]);
                            val[4 * i + 3] = __fadd_rn(r4.w, val[4 * i + 3]);
                        } else {
                            val[4 * i + 0] = __fadd_rn(__fmul_rn(val[4 * i + 0], 0.2f), r4.x);
                            val[4 * i + 1] = __fadd_rn(__fmul_rn(val[4 * i + 1], 0.2f), r4.y);
                            val[4 * i + 2] = __fadd_rn(__fmul_rn(val[4 * i + 2], 0.2f), r4.z);
                            val[4 * i + 3] = __fadd_rn(__fmul_rn(val[4 * i + 3], 0.2f), r4.w);
                        }
                    }
                }
                if (staged) {  // the output tiles are free once the previous row's TMA stores have read them
                    if (lead_warp) tma_store_wait_read();
                    named_bar_sync(1 + gi, 128);
                }
                if (a.ep_mode == EP_RRDB) {
                    const size_t pix = (static_cast<size_t>(valid ? n : 0) * a.H + y) * a.W + (valid ? x : 0);
                    if (a.res16) {
                        // plain (coherent) loads: in the inference trunk res2 is the RRDB input held in the very buffer
                        // this launch overwrites -- each element is read by the thread that later stores its replacement
                        const uint4* r2 = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.res2) + pix * a.res2_cstride +
                                                                         a.res_choff + slice * NOUT);
#pragma unroll
                        for (int i = 0; i < NOUT / 8; ++i) {
                            float f8[8];
                            unpack16x8(r2[i], a.res16_fmt, f8);
#pragma unroll
                            for (int e = 0; e < 8; ++e) val[8 * i + e] = __fadd_rn(__fmul_rn(val[8 * i + e], 0.2f), f8[e]);
                        }
                    } else {
                        const float4* r2 = reinterpret_cast<const float4*>(static_cast<const float*>(a.res2) + pix * a.res2_cstride +
                                                                           a.res_choff + slice * NOUT);
#pragma unroll
                        for (int i = 0; i < NOUT / 4; ++i) {
                            const float4 r4 = __ldg(r2 + i);
                            val[4 * i + 0] = __fadd_rn(__fmul_rn(val[4 * i + 0], 0.2f), r4.x);
                            val[4 * i + 1] = __fadd_rn(__fmul_rn(val[4 * i + 1], 0.2f), r4.y);
                            val[4 * i + 2] = __fadd_rn(__fmul_rn(val[4 * i + 2], 0.2f), r4.z);
                            val[4 * i + 3] = __fadd_rn(__fmul_rn(val[4 * i + 3], 0.2f), r4.w);
                        }
                    }
                }
                if (a.ep_mode == EP_ADD2 && a.res2) {
                    const size_t pix = (static_cast<size_t>(valid ? n : 0) * a.H + y) * a.W + (valid ? x : 0);
                    const float4* r2 = reinterpret_cast<const float4*>(static_cast<const float*>(a.res2) + pix * a.res2_cstride + a.res_choff + slice * NOUT);
#pragma unroll
                    for (int i = 0; i < NOUT / 4; ++i) {
                        const float4 r4 = __ldg(r2 + i);
                        val[4 * i + 0] = fmaf(a.res2_scale, r4.x, val[4 * i + 0]);
                        val[4 * i + 1] = fmaf(a.res2_scale, r4.y, val[4 * i + 1]);
                        val[4 * i + 2] = fmaf(a.res2_scale, r4.z, val[4 * i + 2]);
                        val[4 * i + 3] = fmaf(a.res2_scale, r4.w, val[4 * i + 3]);
                    }
                }
                if (a.lrelu) {   // max(v, 0.2 v) == (v > 0 ? v : 0.2 v); the product is one packed FMUL2 per pair
#pragma unroll
                    for (int i = 0; i < NOUT / 2; ++i) {
                        const float2 t = __fmul2_rn(make_float2(val[2 * i], val[2 * i + 1]), make_float2(0.2f, 0.2f));
                        val[2 * i] = fmaxf(val[2 * i], t.x);
                        val[2 * i + 1] = fmaxf(val[2 * i + 1], t.y);
                    }
                }
                if (MASKED && !inside) {   // gutter / canvas margin: 0 in every output, as the zero padding around an image
#pragma unroll
                    for (int i = 0; i < NOUT; ++i) val[i] = 0.f;
                }
                if (a.out_nchw_raw && valid) {
                    const size_t plane = static_cast<size_t>(a.H) * a.W;
                    float* o = a.out_nchw_raw + static_cast<size_t>(n) * a.out_nchw_c * plane + static_cast<size_t>(y) * a.W + x;
#pragma unroll
                    for (int c = 0; c < NOUT; ++c) {
                        const int cc = slice * NOUT + c;
                        if (cc < a.out_nchw_c) o[static_cast<size_t>(cc) * plane] = val[c];
                    }
                }
                if (a.clamp01) {
#pragma unroll
                    for (int i = 0; i < NOUT; ++i) val[i] = fminf(fmaxf(val[i], 0.f), 1.f);
                }
                if (use_outf) {  // fp32 master
#pragma unroll
                    for (int i = 0; i < NOUT / 4; ++i)
                        *reinterpret_cast<float4*>(tileR + m * 128 + ((i ^ (m & 7)) << 4)) =
                            make_float4(val[4 * i], val[4 * i + 1], val[4 * i + 2], val[4 * i + 3]);
                }
                if (use_o16 && a.mask16) {  // LeakyReLU backward: slope 1 where the saved activation is > 0, else 0.2
                    const size_t pix = (static_cast<size_t>(valid ? n : 0) * a.H + y) * a.W + (valid ? x : 0);
                    const uint4* mk = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.mask16) + pix * a.mask16_cstride +
                                                                     a.mask16_choff + slice * NOUT);
#pragma unroll
                    for (int i = 0; i < NOUT / 8; ++i) {
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
                    for (int i = 0; i < NOUT; ++i) val[i] = __fmul_rn(val[i], a.out16_scale);
                }
                if (use_o16) {
                    uint32_t pk[NOUT / 2];
#pragma unroll
                    for (int i = 0; i < NOUT / 2; ++i) {
                        if (a.out16_fmt == 1) {
                            __nv_bfloat162 h = __floats2bfloat162_rn(val[2 * i], val[2 * i + 1]);
                            pk[i] = *reinterpret_cast<uint32_t*>(&h);
                        } else {

                            pk[i] = pack_f16x2_sat(val[2 * i], val[2 * i + 1]);  // saturate, never inf
                        }
                    }
                    // rotate the 16-byte chunk order per lane so that a quarter-warp does not hammer two bank groups
                    uint4* dst = reinterpret_cast<uint4*>(tile16 + m * (NOUT * 2));
#pragma unroll
                    for (int i = 0; i < NOUT / 8; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
                }
                if (staged) {
                    fence_proxy_async_smem();
                    named_bar_sync(1 + gi, 128);
                    if (lead_warp) {
                      if (elect_one()) {
                        if (use_outf && !DBGF(1) && !DBGF(64)) tma_store_4d(&tmapOF, tileR, a.outf_choff + slice * NOUT, x0, y, n0);
                        if (use_o16 && !DBGF(1) && !(DBGF(128) && a.has_res1)) {
                            const int c0 = a.out16_choff + (a.out16_slice_fixed ? 0 : slice * NOUT);
                            if (!a.out16_up2) {
                                tma_store_4d(&tmapO16, tile16, c0, x0, y, n0);
                            } else {
#pragma unroll
                                for (int s = 0; s < 4; ++s) tma_store_5d(&tmapO16, tile16, c0, s & 1, x0, 2 * y + (s >> 1), n0);
                            }
                        }
                        tma_store_commit();
                      }
                      __syncwarp();
                    }
                }
                if (a.out_nchw && valid) {
                    const size_t plane = static_cast<size_t>(a.H) * a.W;
                    float* o = a.out_nchw + static_cast<size_t>(n) * a.out_nchw_c * plane + static_cast<size_t>(y) * a.W + x;
#pragma unroll
                    for (int c = 0; c < NOUT; ++c) {
                        const int cc = slice * NOUT + c;
                        if (cc < a.out_nchw_c) o[static_cast<size_t>(cc) * plane] = val[c];
                    }
                }
                if (a.out_u8 && valid) {   // clamp01 has been applied: v * 255 lies in [0, 255], the cast truncates
                    unsigned char* o = a.out_u8 + ((static_cast<size_t>(n) * a.H + y) * a.W + x) * a.out_nchw_c;
#pragma unroll
                    for (int c = 0; c < NOUT; ++c) {
                        const int cc = slice * NOUT + c;
                        if (cc < a.out_nchw_c) o[cc] = static_cast<unsigned char>(fminf(fmaxf(__fmul_rn(val[c], 255.f), 0.f), 255.f));
                    }
                }
            }
            v0 += n_acc;
            g += yb - ya;
        }
        if (lead_warp) tma_store_wait_all();
        if (gi == 0 && lead_warp) RESR_DBG(6);  // epilogue group 0 drained
    }

    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) RESR_DBG(7);  // CTA done
    if (warp == 2) tmem_dealloc(tbase, 512);
}

// --------------------------------------------------------------------------------------------- host side

bool conv3x3_plan_smem(ConvArgs* a, int cout_slice) {
    const int wbytes = a->nchunks * 3 * (3 * cout_slice) * 128;
    // The per-row epilogue latency (TMEM drain, staging, TMA store; ~1.6k cycles, more with an fp32 output tile) is hidden
    // by running several epilogue groups on consecutive rows. Three groups whenever they fit beside at least four
    // stages (8 KB of shared memory each without an fp32 tile); two with the 24 KB fp32 variant.
    int nepi = a->has_outf ? 2 : 3;
    const char* env = getenv("RESR_CONV_NEPI");
    if (env) nepi = atoi(env);
    if (nepi < 1) nepi = 1;
    if (nepi > 3) nepi = 3;
    for (;; --nepi) {
        a->nepi = nepi;
        const int fixed = 1024 + wbytes + nepi * epi_group_bytes(*a, cout_slice) + kMiscBytes;
        int ns = (kSmemMax - fixed) / kStageBytes;
        if (ns > kMaxStages) ns = kMaxStages;
        if (ns >= 4 || nepi == 1) {
            a->nstages = ns;
            return ns >= 2;
        }
    }
}

void conv3x3_pick_tile(int W, int* BW, int* BN) {
    if (W == 64 || W == 32 || W == 16 || W == 8) {
        *BW = W;
        *BN = 128 / W;
    } else {
        *BW = 128;
        *BN = 1;
    }
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

int conv3x3_make_tmap_act(CUtensorMap* out, const void* base, int N, int H, int W, int C, int mode, int BW, int BN,
                          int cvalid) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return -1;
    // Channels at and beyond `cvalid` are out of bounds for the map: the 64-channel box of the tail chunk is zero-filled
    // there instead of fetching the neighbouring (zero-weight) channels of the concat buffer from DRAM.
    int cdim = cvalid > 0 ? (cvalid + 7) / 8 * 8 : C;
    if (cdim > C) cdim = C;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(cdim), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                                static_cast<cuuint64_t>(N)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(W) * C * 2,
                                   static_cast<cuuint64_t>(H) * W * C * 2};
    cuuint32_t box[4] = {64, static_cast<cuuint32_t>(mode == 0 ? BW + 2 : BW), 1, static_cast<cuuint32_t>(mode == 0 ? 1 : BN)};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    // L2 promotion: 128 B fetches suit full 64-channel chunks (128 B per pixel); a layer whose last chunk holds only 32
    // channels (Cin = 96 / 160) would drag the other half of every 128-byte line in from DRAM (ncu: 278 MB read for the
    // 201 MB a 96-channel layer needs), so those maps promote to 64 B. RESR_TMAP_PROMO = 0 / 1 / 2 / 3 forces none / 64 / 128 / 256.
    static const int env_promo = getenv("RESR_TMAP_PROMO") ? atoi(getenv("RESR_TMAP_PROMO")) : -1;
    CUtensorMapL2promotion promo = (cdim % 64 != 0) ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    if (env_promo == 0) promo = CU_TENSOR_MAP_L2_PROMOTION_NONE;
    else if (env_promo == 1) promo = CU_TENSOR_MAP_L2_PROMOTION_L2_64B;
    else if (env_promo == 2) promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    else if (env_promo == 3) promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
    const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

int conv3x3_make_tmap_out16(CUtensorMap* out, const void* base, int N, int H, int W, int C, int nout, int BW, int BN,
                            int up2) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return -1;
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r;
    if (!up2) {
        const cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                                    static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[3] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(W) * C * 2,
                                       static_cast<cuuint64_t>(H) * W * C * 2};
        const cuuint32_t box[4] = {static_cast<cuuint32_t>(nout), static_cast<cuuint32_t>(BW), 1, static_cast<cuuint32_t>(BN)};
        r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        // destination [N, 2H, 2W, C] viewed as (c, b, x, Y' = 2y + a, n): pixel (Y', 2x + b)
        const cuuint64_t dims[5] = {static_cast<cuuint64_t>(C), 2, static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(2 * H),
                                    static_cast<cuuint64_t>(N)};
        const cuuint64_t strides[4] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(C) * 4,
                                       static_cast<cuuint64_t>(2 * W) * C * 2, static_cast<cuuint64_t>(2 * H) * 2 * W * C * 2};
        const cuuint32_t box[5] = {static_cast<cuuint32_t>(nout), 1, static_cast<cuuint32_t>(BW), 1, static_cast<cuuint32_t>(BN)};
        r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

int conv3x3_make_tmap_f32(CUtensorMap* out, const void* base, int N, int H, int W, int C, int BW, int BN) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return -1;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                                static_cast<cuuint64_t>(N)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(C) * 4, static_cast<cuuint64_t>(W) * C * 4,
                                   static_cast<cuuint64_t>(H) * W * C * 4};
    const cuuint32_t box[4] = {32, static_cast<cuuint32_t>(BW), 1, static_cast<cuuint32_t>(BN)};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

template <int NOUT, bool MASKED>
static cudaError_t launch_t(const ConvMaps& maps, const ConvArgs& args, dim3 grid, int threads, cudaStream_t stream) {
    static PerDevice<bool> attr;  // function attributes are per device
    if (!attr.cur()) {
        const cudaError_t e = cudaFuncSetAttribute(conv3x3_tc_kernel<NOUT, MASKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
        if (e != cudaSuccess) return e;
        attr.cur() = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = kSmemMax;  // always the full 227 KB: exactly one CTA (one 512-column TMEM allocation) per SM
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, conv3x3_tc_kernel<NOUT, MASKED>, maps.a, maps.o16, maps.of, args);
}

cudaError_t conv3x3_launch(const ConvMaps& maps, const ConvArgs& args, int cout_slice, int nslices, int num_sms,
                           cudaStream_t stream) {
    const int wbytes = args.nchunks * 3 * (3 * cout_slice) * 128;
    const int smem = 1024 + wbytes + args.nstages * kStageBytes + args.nepi * epi_group_bytes(args, cout_slice) + kMiscBytes;
    if (args.nstages < 2 || args.nepi < 1 || args.nepi > 3 || smem > kSmemMax) return cudaErrorInvalidConfiguration;
    long long gx = num_sms / nslices;
    const long long min_rows = 4;  // do not shred tiny problems into 1-row strips (2 halo rows each)
    const long long cap = (args.rows_total + min_rows - 1) / min_rows;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    if (args.rows_total * (gx + 1) >= (1ll << 31)) return cudaErrorInvalidValue;   // the kernel's strip arithmetic is 32-bit
    const dim3 grid(static_cast<unsigned>(gx), static_cast<unsigned>(nslices), 1);
    const int threads = 128 + 128 * args.nepi;
    static const int env_flags = getenv("RESR_CONV_DBGFLAGS") ? atoi(getenv("RESR_CONV_DBGFLAGS")) : 0;  // experiments only
    if (env_flags && !(args.dbg_flags & 0x40000000)) {
        ConvArgs fixed = args;
        fixed.dbg_flags |= env_flags | 0x40000000;
        return conv3x3_launch(maps, fixed, cout_slice, nslices, num_sms, stream);
    }
    if (args.tail_ksteps != 1 && args.tail_ksteps != 2 && args.tail_ksteps != 4) {
        ConvArgs fixed = args;
        fixed.tail_ksteps = 4;
        return conv3x3_launch(maps, fixed, cout_slice, nslices, num_sms, stream);
    }
    if (args.vmask) {
        if (cout_slice == 32) return launch_t<32, true>(maps, args, grid, threads, stream);
        if (cout_slice == 16) return launch_t<16, true>(maps, args, grid, threads, stream);
        return cudaErrorInvalidValue;
    }
    if (cout_slice == 32) return launch_t<32, false>(maps, args, grid, threads, stream);
    if (cout_slice == 16) return launch_t<16, false>(maps, args, grid, threads, stream);
    return cudaErrorInvalidValue;
}

}  // namespace resr
