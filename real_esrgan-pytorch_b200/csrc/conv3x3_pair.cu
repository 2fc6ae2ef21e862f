// 3x3 / stride 1 / zero-pad 1 convolution on CTA PAIRS: tcgen05.mma.cta_group::2 (M = 256) + TMEM + TMA.
//
// Same "row-rolling implicit GEMM" as conv3x3_tc.cu (read its header first), re-shaped so that two SMs share one MMA
// stream (reference: /root/reference/model.py:75-98, 123-132, 255-272):
//
//   * A cluster of two CTAs works on TWO column groups (two images at cfg3, two 128-pixel column strips of one image
//     at cfg5) over the SAME row range. Each CTA loads its own activation rows (its 128 TMEM lanes = its pixels) and
//     holds only HALF of the weight rows: one cta_group::2 MMA multiplies both CTAs' 128 x K activation tiles with the
//     N = 3 * NOUT weight rows gathered from the two shared memories (rows [0, N/2) from rank 0, [N/2, N) from rank 1;
//     profiles/r02_mma_pair_check.txt). Per FLOP a CTA reads half as many weight rows from shared memory as the
//     single-CTA kernel: an N = 96 stream runs at the full tensor rate instead of 86 % and at 1719 instead of 1526
//     TFLOP/s under the board's power cap (profiles/r02_mma_pair_power.txt), and the 192 -> 64 convolution of a dense
//     block becomes ONE N = 192 MMA per K step (NOUT = 64) instead of two N = 96 streams on separate SMs.
//   * Only rank 0 issues MMAs. Completion (tcgen05.commit) is multicast to the barriers at the same offsets in both
//     CTAs; rank 1's TMA loads signal rank 0's stage barrier (cp.async.bulk.tensor ... cta_group::2); the epilogue
//     warps of both CTAs drain their own TMEM and release accumulator slots on rank 0's barriers (remote arrive).
//   * The accumulator ring has no seam: it has S ring positions plus two overflow slots, so the three (dy) column
//     blocks of an MMA that starts at ring position S-2 / S-1 simply run on into the overflow slots instead of being
//     split into two MMAs (a split would need weight rows the issuing half does not hold). The rows whose ring
//     position is 0 or 1 therefore have their sum in two slots; the epilogue adds them.
//   * The weight packs are the ones conv3x3_tc.cu uses ([slice32][chunk][dx][(dy, co) x 64 ch], 128B-swizzled): each
//     CTA bulk-copies the row blocks that make up its half.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>

#include "conv3x3.cuh"
#include "device_state.h"
#include "ptx.cuh"

namespace resr {

// Wait-time profile (development builds with -DRESR_PROFILE_WAITS): cycles each role spends blocked, summed over CTAs.
//   [0] MMA warp total  [1] .. waiting for activation stages  [2] .. waiting for free accumulator slots  [3] steps
//   [4] producer total  [5] .. waiting for empty stages
//   [6] epilogue (group 0, warp 0) total  [7] .. waiting for accumulators  [8] .. waiting for its staging tile
__device__ unsigned long long g_wait_prof[16];
#ifdef RESR_PROFILE_WAITS
#define PROF_DECL(name) long long name = 0
#define PROF_T0(t) const long long t = clock64()
#define PROF_ADD(acc, t) acc += clock64() - t
#define PROF_FLUSH(idx, v) do { if ((threadIdx.x & 31) == 0) atomicAdd(&g_wait_prof[idx], static_cast<unsigned long long>(v)); } while (0)
#else
#define PROF_DECL(name)
#define PROF_T0(t)
#define PROF_ADD(acc, t)
#define PROF_FLUSH(idx, v)
#endif

namespace {

constexpr int kStageBytes = 17408;  // 136 rows x 128 B (mode 0 uses BW + 2 rows, mode 1 uses 128)
constexpr int kMaxStages = 12;
constexpr int kMiscBytes = 1024;
constexpr int kSmemMax = 232448;    // 227 KB opt-in limit per CTA
constexpr int kTileFBytes = 16384;  // 128 px x 32 fp32

struct RowRange {   // 32-bit on purpose: 64-bit divisions are ~100-instruction subroutines and every role decodes its strips
    int g0, g1;     // (the launcher refuses problems with rows_total * grid >= 2^31)
};

// K-major, 128B-swizzled operand descriptor: constant high word (SBO = 1024 B, version 1, SWIZZLE_128B) + low word.
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint64_t desc_of(uint32_t lo) { return (static_cast<uint64_t>(kDescHi) << 32) | lo; }

// one staging buffer of an epilogue group: [fp32 tile][16-bit tile]
__host__ __device__ inline int epi_buf_bytes_pair(const ConvArgs& a, int subw) {
    const int f = a.has_outf ? kTileFBytes : 0;
    const int h = a.has_out16 ? 128 * subw * 2 : 0;
    return f + (h + 1023) / 1024 * 1024;
}
__host__ __device__ inline int epi_group_bytes_pair(const ConvArgs& a, int subw) {
    return (a.epi_bufs == 2 ? 2 : 1) * epi_buf_bytes_pair(a, subw);
}

template <int S>
__device__ __forceinline__ uint32_t ring_slot(uint32_t v) { return (S - v % S) % S; }
template <int S>
__device__ __forceinline__ uint32_t ring_parity(uint32_t v) { return (v / S) & 1u; }

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

// MMAs [I0, I1) of one pipeline stage (i = dx * KS + ks), straight-line. One N = 3 * NOUT instruction per K16 step.
template <int NOUT, int KS, int I0, int I1>
__device__ __forceinline__ void issue_range(uint32_t d0, uint32_t a_lo, uint32_t b_lo, uint32_t idesc) {
    constexpr uint32_t WT = (3 * NOUT / 2 * 128) >> 4;  // one (chunk, dx) HALF weight tile, in 16-byte units
#pragma unroll
    for (int i = I0; i < I1; ++i) {
        const int dx = i / KS, ks = i % KS;
        umma2_f16(d0, desc_of(a_lo + dx * 8 + ks * 2), desc_of(b_lo + dx * WT + ks * 2), idesc, 1);
    }
}

template <int NOUT, int NDX, int HALF>
__device__ __forceinline__ void issue_half(int ks, uint32_t d0, uint32_t a_lo, uint32_t b_lo, uint32_t idesc) {
#define RESR_HALF(KS)                                                                       \
    if (HALF == 0) issue_range<NOUT, KS, 0, (NDX * KS) / 2>(d0, a_lo, b_lo, idesc);          \
    else issue_range<NOUT, KS, (NDX * KS) / 2, NDX * KS>(d0, a_lo, b_lo, idesc)
    if (ks == 2) { RESR_HALF(2); }
    else if (ks == 1) { RESR_HALF(1); }
    else { RESR_HALF(4); }
#undef RESR_HALF
}

// The MMA-issuing warp of the pair's leader CTA (see conv3x3_tc.cu mma_role for the scheduling rationale).
template <int NOUT, int MODE, int S>
__device__ __forceinline__ void mma_role(const ConvArgs& a, const RowRange rr, const uint32_t tbase, const uint32_t wsm_addr,
                                         const uint32_t stg_addr, const uint32_t full_a, const uint32_t empty_a,
                                         const uint32_t accfull_a, const uint32_t slotfree_a) {
    constexpr uint32_t WT = (3 * NOUT / 2 * 128) >> 4;
    const uint32_t idesc = make_idesc_f16(a.fmt_in, 256, 3 * NOUT);
    const uint32_t w_lo = (wsm_addr & 0x3FFFFu) >> 4;
    const uint32_t s_lo = (stg_addr & 0x3FFFFu) >> 4;
    const int nsteps = MODE == 0 ? a.nchunks : a.nchunks * 3;
    const uint32_t b_step = (MODE == 0 ? 3 : 1) * WT;
    const int nstages = a.nstages;
    const int H = a.H;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t a_lo = s_lo;
    int pending_empty = -1;          // stage whose release commit has not been issued yet
    bool full_ready = false, slot_ready = false;
    uint32_t vnew = 1;               // virtual index of the NEWEST accumulator the next row touches (out row r+1)
    uint32_t acq = 0;                // accumulators acquired so far (virtual indices < acq)
    PROF_DECL(p_full); PROF_DECL(p_slot); PROF_DECL(p_steps);
    PROF_T0(p_t0);
    for (int g = rr.g0; g < rr.g1;) {
        const int ya = g % H;
        const int yb = min(H, ya + (rr.g1 - g));
        const int ra = max(ya - 1, 0), rb = min(yb, H - 1);
        vnew += 1;                   // a strip touches rows ra-1 .. rb+1: first row's newest accumulator is v0 + 2
        for (int r = ra; r <= rb; ++r, ++vnew) {
            // accumulators of rows r-1, r, r+1 (virtual vnew-2 .. vnew) must be zeroed & free in BOTH CTAs
            if (slot_ready && acq == vnew) {
                ++acq;
            } else {
                PROF_T0(p_t);
                while (static_cast<int>(vnew - acq) >= 0) {
                    mbar_wait_a(slotfree_a + (ring_slot<S>(acq) << 3), ring_parity<S>(acq));
                    ++acq;
                }
                PROF_ADD(p_slot, p_t);
            }
            slot_ready = false;
            tc_fence_after();
            const uint32_t s0 = ring_slot<S>(vnew), s1 = ring_slot<S>(vnew - 1), s2 = ring_slot<S>(vnew - 2);
            const uint32_t d0 = tbase + s0 * NOUT;   // the three dy blocks land on s0, s0+1, s0+2 (possibly overflow slots)
            uint32_t b_lo = w_lo;
            for (int st = 0; st < nsteps; ++st, b_lo += b_step) {
                if (!full_ready) { PROF_T0(p_t); mbar_wait_a(full_a + (stage << 3), phase); PROF_ADD(p_full, p_t); }
                tc_fence_after();
#ifdef RESR_PROFILE_WAITS
                ++p_steps;
#endif
                const bool last = (st == nsteps - 1);
                const int ks = (st >= nsteps - (MODE == 0 ? 1 : 3)) ? a.tail_ksteps : 4;  // steps of the last K chunk
                if (elect_one()) {
                    issue_half<NOUT, MODE == 0 ? 3 : 1, 0>(ks, d0, a_lo, b_lo, idesc);
                    if (pending_empty >= 0) umma2_commit_mc(empty_a + (pending_empty << 3), 3);
                }
                __syncwarp();
                pending_empty = stage;
                const uint32_t a_cur = a_lo;
                if (++stage == nstages) { stage = 0; phase ^= 1u; a_lo = s_lo; } else { a_lo += kStageBytes >> 4; }
                full_ready = mbar_test_wait_a(full_a + (stage << 3), phase);
                if (last && r < rb) slot_ready = mbar_test_wait_a(slotfree_a + (ring_slot<S>(vnew + 1) << 3), ring_parity<S>(vnew + 1));
                if (elect_one()) {
                    issue_half<NOUT, MODE == 0 ? 3 : 1, 1>(ks, d0, a_cur, b_lo, idesc);
                    if (last) {
                        umma2_commit_mc(accfull_a + (s2 << 3), 3);          // row r-1 has its last contribution
                        if (r == rb) {                                       // strip end: rows rb, rb+1 get no more
                            umma2_commit_mc(accfull_a + (s1 << 3), 3);
                            umma2_commit_mc(accfull_a + (s0 << 3), 3);
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
        if (elect_one()) umma2_commit_mc(empty_a + (pending_empty << 3), 3);
        __syncwarp();
    }
#ifdef RESR_PROFILE_WAITS
    PROF_FLUSH(0, clock64() - p_t0); PROF_FLUSH(1, p_full); PROF_FLUSH(2, p_slot); PROF_FLUSH(3, p_steps);
#endif
}

template <int W>
__device__ __forceinline__ void tmem_ld_w(uint32_t taddr, float* v) {
    if (W == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
}
template <int W>
__device__ __forceinline__ void tmem_zero_w(uint32_t taddr) {
    if (W == 32) tmem_st_zero32(taddr); else tmem_st_zero16(taddr);
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

}  // namespace

// MASKED: the packed-canvas variant (ConvArgs::vmask set); the other instantiation carries no mask code at all
template <int NOUT, bool MASKED>
__global__ void __launch_bounds__(512, 1)
conv3x3_pair_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapO16,
                    const __grid_constant__ CUtensorMap tmapOF, const ConvArgs a) {
    constexpr int NT = 3 * NOUT;            // MMA N: (dy, co)
    constexpr int NH = NT / 2;              // weight rows held by each CTA of the pair
    constexpr int WHALF = NH * 128;         // bytes of one (chunk, dx) half tile
    constexpr int NSUB = NOUT == 64 ? 2 : 1;  // epilogue passes per output row
    constexpr int SUBW = NOUT / NSUB;       // channels per pass (32, or 16 for the RGB output convolution)
    constexpr int SLOTS = NOUT == 64 ? 8 : 16;
    constexpr int S = SLOTS - 2;            // ring positions; physical slots S and S+1 take the overflow of positions 0 and 1
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int slice = blockIdx.y;
    const uint32_t rank = cluster_ctarank();
    const uint32_t wbytes = static_cast<uint32_t>(a.nchunks) * 3u * WHALF;
    const int epi_bytes = epi_group_bytes_pair(a, SUBW);

    uint8_t* wsm = smem;
    uint8_t* stg = smem + wbytes;
    uint8_t* epi = stg + a.nstages * kStageBytes;
    uint8_t* misc = epi + a.nepi * epi_bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(misc);
    uint64_t* empty = full + kMaxStages;
    uint64_t* acc_full = empty + kMaxStages;
    uint64_t* slot_free = acc_full + 16;
    uint64_t* wbar = slot_free + 16;
    uint64_t* wpair = wbar + 1;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(wpair + 1);
    float* bias_s = reinterpret_cast<float*>(misc + 512);

    if (threadIdx.x == 0) {
        prefetch_tmap(&tmapA);
        if (a.has_out16) prefetch_tmap(&tmapO16);
        if (a.has_outf) prefetch_tmap(&tmapOF);
        for (int i = 0; i < a.nstages; ++i) {
            mbar_init(full + i, 1);       // rank 0 arrives and expects BOTH CTAs' bytes; rank 1's loads only complete_tx
            mbar_init(empty + i, 1);      // multicast tcgen05.commit
        }
        for (int i = 0; i < S; ++i) {
            mbar_init(acc_full + i, 1);   // multicast tcgen05.commit
            mbar_init(slot_free + i, 8);  // 4 epilogue warps of the draining group in each CTA
        }
        mbar_init(wbar, 1);
        mbar_init(wpair, 2);
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc2(tmem_ptr, 512);
        tmem_relinquish2();
    }
    if (threadIdx.x >= 128 && threadIdx.x < 128 + NOUT) bias_s[threadIdx.x - 128] = a.bias[slice * NOUT + threadIdx.x - 128];
    tc_fence_before();
    __syncthreads();      // CTA-level ordering of the prologue's shared-memory writes (TMEM base, bias, barrier words) ...
    cluster_sync_all();   // ... and both CTAs' barriers are initialised before anyone signals across the pair
    tc_fence_after();
    const uint32_t tbase = *tmem_ptr;
    grid_dep_launch();

    // the pair's work: a contiguous range of (pair column group, row); this CTA takes column group 2 * cg2 + rank
    RowRange rr;
    {
        const unsigned npairs = gridDim.x >> 1, pidx = blockIdx.x >> 1, rows = static_cast<unsigned>(a.rows_total_pair);
        rr.g0 = static_cast<int>(rows * pidx / npairs);
        rr.g1 = static_cast<int>(rows * (pidx + 1) / npairs);
    }
    const int H = a.H;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (one elected lane issues)
        if (elect_one()) {
            mbar_expect_tx(wbar, wbytes);
            // this CTA's half of every (chunk, dx) tile, gathered from the [slice32][chunk][dx][(dy, co32) x 64] pack in blocks of
            // G rows (a block never straddles a dy boundary); in reverse mode the dy blocks are taken in flipped order
            constexpr int G = NOUT == 64 ? 32 : NOUT / 2;          // rows per gathered block
            constexpr int BPD = NOUT / G;                           // blocks per dy: 2
            constexpr int NB = 3 * BPD / 2;                         // blocks per CTA: 3
            for (int c = 0; c < a.nchunks; ++c) {
                for (int dx = 0; dx < 3; ++dx) {
                    uint8_t* dst = wsm + (c * 3 + dx) * WHALF;
#pragma unroll
                    for (int j = 0; j < NB; ++j) {
                        const int blk = static_cast<int>(rank) * NB + j;   // position in the (dy', part) order of the MMA's N rows
                        const int dyv = blk / BPD, part = blk % BPD;
                        const int dy = a.reverse ? 2 - dyv : dyv;
                        const uint8_t* src;
                        if (NOUT == 64)   // part = 32-channel pack slice
                            src = a.wpack + ((static_cast<size_t>(slice * 2 + part) * a.nchunks + c) * 3 + dx) * (96 * 128) +
                                  static_cast<size_t>(dy) * 32 * 128;
                        else              // part = half of the slice's channels
                            src = a.wpack + ((static_cast<size_t>(slice) * a.nchunks + c) * 3 + dx) * (NT * 128) +
                                  static_cast<size_t>(dy * NOUT + part * G) * 128;
                        bulk_load_1d(dst + j * G * 128, src, G * 128, wbar);
                    }
                }
            }
        }
        __syncwarp();
        grid_dep_wait();
        int stage = 0;
        uint32_t phase = 0;
        const int ndx = a.mode == 0 ? 1 : 3;
        const uint32_t tx_bytes = a.mode == 0 ? (a.BW + 2) * 128 : 128 * 128;
        const uint32_t full0 = map_to_cta(smem_u32(full), 0);  // the leader's stage barriers
        PROF_DECL(p_empty);
        PROF_T0(p_t0);
        const int ncg2 = (a.ncg + 1) >> 1;
        for (int g = rr.g0; g < rr.g1;) {
            const int cg2 = g / H;
            const int cg = 2 * (a.reverse ? ncg2 - 1 - cg2 : cg2) + static_cast<int>(rank);  // may be == ncg (odd count): all out of bounds
            const int ya = g % H;
            const int yb = min(H, ya + (rr.g1 - g));
            const int n0 = (cg / a.nxs) * a.BN;
            const int x0 = (cg % a.nxs) * a.BW;
            const int ra = max(ya - 1, 0), rb = min(yb, H - 1);
            for (int r = ra; r <= rb; ++r) {
                for (int c = 0; c < a.nchunks; ++c) {
                    for (int dx = 0; dx < ndx; ++dx) {
                        { PROF_T0(p_t); mbar_wait(empty + stage, phase ^ 1); PROF_ADD(p_empty, p_t); }
                        if (elect_one()) {
                            // rank 1 does not arrive: its bytes are counted by the leader's expect_tx (the transaction count
                            // may go negative for a moment; the phase cannot complete before the leader's own arrive, and
                            // rank 1 re-uses a stage only after the commit that follows the leader's wait on this phase)
                            if (rank == 0) mbar_expect_tx(full + stage, 2 * tx_bytes);
                            tma_load_4d_pair(stg + stage * kStageBytes, &tmapA, full0 + (stage << 3), c * 64,
                                             a.mode == 0 ? x0 - 1 : x0 + dx - 1, a.reverse ? H - 1 - r : r, n0);
                        }
                        __syncwarp();
                        if (++stage == a.nstages) { stage = 0; phase ^= 1; }
                    }
                }
            }
            g += yb - ya;
        }
#ifdef RESR_PROFILE_WAITS
        PROF_FLUSH(4, clock64() - p_t0); PROF_FLUSH(5, p_empty);
#endif
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        mbar_wait(wbar, 0);   // this CTA's half of the weights is resident
        if (elect_one()) mbar_arrive_cluster(map_to_cta(smem_u32(wpair), 0));
        __syncwarp();
        if (rank == 0) {
            mbar_wait(wpair, 0);  // ... and the peer's half
            tc_fence_after();
            if (a.mode == 0) mma_role<NOUT, 0, S>(a, rr, tbase, smem_u32(wsm), smem_u32(stg), smem_u32(full), smem_u32(empty), smem_u32(acc_full), smem_u32(slot_free));
            else mma_role<NOUT, 1, S>(a, rr, tbase, smem_u32(wsm), smem_u32(stg), smem_u32(full), smem_u32(empty), smem_u32(acc_full), smem_u32(slot_free));
        }
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue groups (both CTAs, own TMEM)
        const int gi = (warp - 4) >> 2;
        const int q = warp & 3;        // TMEM lane quadrant this warp may access
        const int m = q * 32 + lane;   // M row == TMEM lane == pixel of this CTA's tile
        const bool lead_warp = ((warp - 4) & 3) == 0;
        uint8_t* const tile_base = epi + gi * epi_bytes;
        const int buf_bytes = epi_buf_bytes_pair(a, SUBW);
        const bool two_bufs = a.epi_bufs == 2;
        uint32_t pass = 0;   // staged passes of this group so far (selects the staging buffer)
        const uint32_t lane_base = tbase + (static_cast<uint32_t>(q * 32) << 16);
        const uint32_t free0 = map_to_cta(smem_u32(slot_free), 0);  // the leader's slot barriers
        const int img_in_tile = m / a.BW;
        const int x_in_tile = m % a.BW;
        {   // zero this group's share of the accumulator ring (+ the overflow slots of positions 0 / 1), then hand it over
            const int s_lo = gi * S / a.nepi, s_hi = (gi + 1) * S / a.nepi;
            for (int s = s_lo; s < s_hi; ++s) {
#pragma unroll
                for (int c = 0; c < NOUT; c += SUBW) {
                    tmem_init_bias<SUBW>(lane_base + s * NOUT + c, bias_s + c);
                    if (s < 2) tmem_zero_w<SUBW>(lane_base + (S + s) * NOUT + c);   // overflow twin: plain zero
                }
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0)
                for (int s = s_lo; s < s_hi; ++s) mbar_arrive_cluster(free0 + (s << 3));
        }
        grid_dep_wait();  // residual reads / output writes below touch buffers of the previous kernel
        PROF_DECL(p_acc); PROF_DECL(p_tile); PROF_DECL(p_drain); PROF_DECL(p_math); PROF_DECL(p_store); PROF_DECL(p_rows);
        PROF_T0(p_t0);
        uint32_t v0 = 0;
        const int ncg2 = (a.ncg + 1) >> 1;
        for (int g = rr.g0; g < rr.g1;) {
            const int cg2 = g / H;
            const int cg = 2 * (a.reverse ? ncg2 - 1 - cg2 : cg2) + static_cast<int>(rank);
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
                if (static_cast<int>(v % a.nepi) != gi) continue;
                const int yv = ra - 1 + j;                       // row in traversal order
                const bool emit = (yv >= ya) && (yv < yb);
                const int y = a.reverse ? H - 1 - yv : yv;       // image row
                const uint32_t slot = ring_slot<S>(v);
                const uint32_t col = slot * NOUT;
                const uint32_t col2 = (S + slot) * NOUT;  // overflow twin (ring positions 0 and 1 only)
                const bool dual = slot < 2;
                const size_t pix = (static_cast<size_t>(valid ? n : 0) * a.H + y) * a.W + (valid ? x : 0);
                bool inside = true;   // canvas pixel of an image (vmask), read before the accumulator wait like the residual
                if (MASKED && emit) {
                    const int lx = (valid ? x : 0) >> a.vmask_shift, ly = y >> a.vmask_shift;
                    inside = (__ldg(a.vmask + static_cast<size_t>(ly) * a.vmask_words + (lx >> 5)) >> (lx & 31)) & 1u;
                }
                bool waited = false;
#pragma unroll 1
                for (int h = 0; h < NSUB; ++h) {
                    const int ls = slice * NSUB + h;   // logical 32-channel slice (channel offsets, per-slice flags)
                    const bool use_res1 = a.has_res1 && !((a.slice_nores_mask >> ls) & 1u);
                    const bool use_outf = a.has_outf && !((a.slice_noutf_mask >> ls) & 1u);
                    const bool use_o16 = a.has_out16 && !((a.slice_no16_mask >> ls) & 1u);
                    const bool staged = use_o16 || use_outf;
                    float4 resv[SUBW / 4];   // fp32 residual, or (res16) SUBW 16-bit values in the first SUBW / 8 entries
                    if (emit && use_res1) {
                        // requested before the wait for the accumulator: the latency hides behind the row's MMAs
                        if (a.res16) {
                            const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.res1) + pix * a.res1_cstride +
                                                                             a.res_choff + ls * SUBW);
#pragma unroll
                            for (int i = 0; i < SUBW / 8; ++i) {
                                const uint4 q4 = rp[i];
                                resv[i] = make_float4(__uint_as_float(q4.x), __uint_as_float(q4.y), __uint_as_float(q4.z), __uint_as_float(q4.w));
                            }
                        } else {
                            const float4* rp = reinterpret_cast<const float4*>(static_cast<const float*>(a.res1) + pix * a.res1_cstride +
                                                                               a.res_choff + ls * SUBW);
#pragma unroll
                            for (int i = 0; i < SUBW / 4; ++i) resv[i] = rp[i];
                        }
                    }
                    if (!waited) {
                        PROF_T0(p_t);
                        mbar_wait(acc_full + slot, ring_parity<S>(v));
                        PROF_ADD(p_acc, p_t);
                        tc_fence_after();
                        waited = true;
                    }
                    float val[SUBW];
                    PROF_T0(p_td);
                    tmem_ld_w<SUBW>(lane_base + col + h * SUBW, val);
                    if (dual) {
                        float val2[SUBW];
                        tmem_ld_w<SUBW>(lane_base + col2 + h * SUBW, val2);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < SUBW; ++i) val[i] = __fadd_rn(val[i], val2[i]);
                        tmem_zero_w<SUBW>(lane_base + col2 + h * SUBW);
                    } else {
                        tmem_ld_wait();
                    }
                    tmem_init_bias<SUBW>(lane_base + col + h * SUBW, bias_s + h * SUBW);
                    if (h == NSUB - 1) {   // the whole slot is drained and zeroed: give it back to the MMA issuer
                        tmem_st_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(free0 + (slot << 3));
                    }
                    PROF_ADD(p_drain, p_td);
                    if (!emit) continue;
                    PROF_T0(p_tm);
#ifdef RESR_PROFILE_WAITS
                    ++p_rows;
#endif

                    // (no bias add here: the accumulator was armed with the bias, tmem_init_bias)
                    if (use_res1 && a.res16) {  // widen the 16-bit residual in place (consumed below as fp32)
                        float wide[SUBW];
#pragma unroll
                        for (int i = 0; i < SUBW / 8; ++i) {
                            float f8[8];
                            unpack16x8(make_uint4(__float_as_uint(resv[i].x), __float_as_uint(resv[i].y), __float_as_uint(resv[i].z),
                                                  __float_as_uint(resv[i].w)), a.res16_fmt, f8);
#pragma unroll
                            for (int e = 0; e < 8; ++e) wide[8 * i + e] = f8[e];
                        }
#pragma unroll
                        for (int i = 0; i < SUBW / 4; ++i) resv[i] = make_float4(wide[4 * i], wide[4 * i + 1], wide[4 * i + 2], wide[4 * i + 3]);
                    }
                    if (use_res1) {
#pragma unroll
                        for (int i = 0; i < SUBW / 4; ++i) {
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
                    PROF_ADD(p_math, p_tm);
                    uint8_t* const tileR = tile_base + ((two_bufs && (pass & 1u)) ? buf_bytes : 0);  // fp32 output tile
                    uint8_t* const tile16 = tileR + (a.has_outf ? kTileFBytes : 0);                  // 16-bit output tile
                    if (staged) {
                        // the staging buffer is free once the TMA stores that last used it have read it: the previous pass's
                        // (one buffer) or the pass before that (two buffers: the wait is normally already satisfied)
                        PROF_T0(p_t);
                        if (lead_warp) { if (two_bufs) tma_store_wait_read1(); else tma_store_wait_read(); }
                        named_bar_sync(1 + gi, 128);
                        PROF_ADD(p_tile, p_t);
                        ++pass;
                    }
                    PROF_T0(p_ts);
                    if (a.ep_mode == EP_RRDB) {
                        if (a.res16) {
                            // plain (coherent) loads: in the inference trunk res2 is the RRDB input held in the very buffer
                            // this launch overwrites -- each element is read by the thread that later stores its replacement
                            const uint4* r2 = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.res2) + pix * a.res2_cstride +
                                                                             a.res_choff + ls * SUBW);
#pragma unroll
                            for (int i = 0; i < SUBW / 8; ++i) {
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
                            const float4* r2 = reinterpret_cast<const float4*>(static_cast<const float*>(a.res2) + pix * a.res2_cstride +
                                                                               a.res_choff + ls * SUBW);
#pragma unroll
                            for (int i = 0; i < SUBW / 4; ++i) {
                                const float4 r4 = __ldg(r2 + i);
                                val[4 * i + 0] = __fadd_rn(__fmul_rn(val[4 * i + 0], 0.2f), r4.x);
                                val[4 * i + 1] = __fadd_rn(__fmul_rn(val[4 * i + 1], 0.2f), r4.y);
                                val[4 * i + 2] = __fadd_rn(__fmul_rn(val[4 * i + 2], 0.2f), r4.z);
                                val[4 * i + 3] = __fadd_rn(__fmul_rn(val[4 * i + 3], 0.2f), r4.w);
                            }
                        }
                    }
                    if (a.ep_mode == EP_ADD2 && a.res2) {
                        const float4* r2 = reinterpret_cast<const float4*>(static_cast<const float*>(a.res2) + pix * a.res2_cstride + a.res_choff + ls * SUBW);
#pragma unroll
                        for (int i = 0; i < SUBW / 4; ++i) {
                            const float4 r4 = __ldg(r2 + i);
                            val[4 * i + 0] = fmaf(a.res2_scale, r4.x, val[4 * i + 0]);
                            val[4 * i + 1] = fmaf(a.res2_scale, r4.y, val[4 * i + 1]);
                            val[4 * i + 2] = fmaf(a.res2_scale, r4.z, val[4 * i + 2]);
                            val[4 * i + 3] = fmaf(a.res2_scale, r4.w, val[4 * i + 3]);
                        }
                    }
                    if (a.lrelu) {   // max(v, 0.2 v) == (v > 0 ? v : 0.2 v) for every finite v; the product is one packed FMUL2 per pair
#pragma unroll
                        for (int i = 0; i < SUBW / 2; ++i) {
                            const float2 t = __fmul2_rn(make_float2(val[2 * i], val[2 * i + 1]), make_float2(0.2f, 0.2f));
                            val[2 * i] = fmaxf(val[2 * i], t.x);
                            val[2 * i + 1] = fmaxf(val[2 * i + 1], t.y);
                        }
                    }
                    if (MASKED && !inside) {   // gutter / canvas margin: 0 in every output, as the zero padding around an image
#pragma unroll
                        for (int i = 0; i < SUBW; ++i) val[i] = 0.f;
                    }
                    if (a.out_nchw_raw && valid) {
                        const size_t plane = static_cast<size_t>(a.H) * a.W;
                        float* o = a.out_nchw_raw + static_cast<size_t>(n) * a.out_nchw_c * plane + static_cast<size_t>(y) * a.W + x;
#pragma unroll
                        for (int c = 0; c < SUBW; ++c) {
                            const int cc = ls * SUBW + c;
                            if (cc < a.out_nchw_c) o[static_cast<size_t>(cc) * plane] = val[c];
                        }
                    }
                    if (a.clamp01) {
#pragma unroll
                        for (int i = 0; i < SUBW; ++i) val[i] = fminf(fmaxf(val[i], 0.f), 1.f);
                    }
                    if (use_outf) {  // fp32 master (SUBW == 32 only)
#pragma unroll
                        for (int i = 0; i < SUBW / 4; ++i)
                            *reinterpret_cast<float4*>(tileR + m * 128 + ((i ^ (m & 7)) << 4)) =
                                make_float4(val[4 * i], val[4 * i + 1], val[4 * i + 2], val[4 * i + 3]);
                    }
                    if (use_o16 && a.mask16) {  // LeakyReLU backward: slope 1 where the saved activation is > 0, else 0.2
                        const uint4* mk = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.mask16) + pix * a.mask16_cstride +
                                                                         a.mask16_choff + ls * SUBW);
#pragma unroll
                        for (int i = 0; i < SUBW / 8; ++i) {
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
                        for (int i = 0; i < SUBW; ++i) val[i] = __fmul_rn(val[i], a.out16_scale);
                    }
                    if (use_o16) {
                        uint32_t pk[SUBW / 2];
#pragma unroll
                        for (int i = 0; i < SUBW / 2; ++i) {
                            if (a.out16_fmt == 1) {
                                __nv_bfloat162 hh = __floats2bfloat162_rn(val[2 * i], val[2 * i + 1]);
                                pk[i] = *reinterpret_cast<uint32_t*>(&hh);
                            } else {
                                pk[i] = pack_f16x2_sat(val[2 * i], val[2 * i + 1]);  // saturate, never inf
                            }
                        }
                        // (Storing the pixel's channels straight from registers instead -- no staging tile, no proxy fence, no
                        // block barrier -- was tried and is slower: 45.5 vs 43.0 ms per cfg3 forward, profiles/r02_direct_store_ab.txt.)
                        uint4* dst = reinterpret_cast<uint4*>(tile16 + m * (SUBW * 2));
#pragma unroll
                        for (int i = 0; i < SUBW / 8; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
                    }
                    if (staged) {
                        fence_proxy_async_smem();
                        named_bar_sync(1 + gi, 128);
                        if (lead_warp) {
                            if (elect_one()) {
                                if (use_outf) tma_store_4d(&tmapOF, tileR, a.outf_choff + ls * SUBW, x0, y, n0);
                                if (use_o16) {
                                    const int c0 = a.out16_choff + (a.out16_slice_fixed ? 0 : ls * SUBW);
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
                    PROF_ADD(p_store, p_ts);
                    if (a.out_nchw && valid) {
                        const size_t plane = static_cast<size_t>(a.H) * a.W;
                        float* o = a.out_nchw + static_cast<size_t>(n) * a.out_nchw_c * plane + static_cast<size_t>(y) * a.W + x;
#pragma unroll
                        for (int c = 0; c < SUBW; ++c) {
                            const int cc = ls * SUBW + c;
                            if (cc < a.out_nchw_c) o[static_cast<size_t>(cc) * plane] = val[c];
                        }
                    }
                    if (a.out_u8 && valid) {   // clamp01 has been applied: v * 255 lies in [0, 255], the cast truncates
                        unsigned char* o = a.out_u8 + ((static_cast<size_t>(n) * a.H + y) * a.W + x) * a.out_nchw_c;
#pragma unroll
                        for (int c = 0; c < SUBW; ++c) {
                            const int cc = ls * SUBW + c;
                            if (cc < a.out_nchw_c) o[cc] = static_cast<unsigned char>(fminf(fmaxf(__fmul_rn(val[c], 255.f), 0.f), 255.f));
                        }
                    }
                }
            }
            v0 += n_acc;
            g += yb - ya;
        }
        if (lead_warp) tma_store_wait_all();
#ifdef RESR_PROFILE_WAITS
        if (warp == 4) {
            PROF_FLUSH(6, clock64() - p_t0); PROF_FLUSH(7, p_acc); PROF_FLUSH(8, p_tile);
            PROF_FLUSH(9, p_drain); PROF_FLUSH(10, p_math); PROF_FLUSH(11, p_store); PROF_FLUSH(12, p_rows);
        }
#endif
    }

    // no CTA of the pair may exit while its peer can still signal its barriers / read its shared memory
    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc2(tbase, 512);
}

// --------------------------------------------------------------------------------------------- host side

bool conv3x3_pair_plan_smem(ConvArgs* a, int nout) {
    const int subw = nout == 64 ? 32 : nout;
    const int wbytes = a->nchunks * 3 * (3 * nout / 2) * 128;
    int nepi = a->has_outf ? 2 : 3;
    const char* env = getenv("RESR_CONV_NEPI");
    if (env) nepi = atoi(env);
    if (nepi < 1) nepi = 1;
    if (nepi > 3) nepi = 3;
    static const int env_bufs = getenv("RESR_CONV_EPI_BUFS") ? atoi(getenv("RESR_CONV_EPI_BUFS")) : 2;
    for (;; --nepi) {
        a->nepi = nepi;
        for (int bufs = env_bufs == 2 ? 2 : 1; bufs >= 1; --bufs) {
            a->epi_bufs = bufs;
            const int fixed = 1024 + wbytes + nepi * epi_group_bytes_pair(*a, subw) + kMiscBytes;
            int ns = (kSmemMax - fixed) / kStageBytes;
            if (ns > kMaxStages) ns = kMaxStages;
            // two staging tiles per group only where they do not eat into the activation ring (>= 6 stages left)
            if ((bufs == 2 && ns >= 6) || (bufs == 1 && (ns >= 4 || nepi == 1))) {
                a->nstages = ns;
                return ns >= 2;
            }
        }
    }
}

template <int NOUT, bool MASKED>
static cudaError_t launch_pair_t(const ConvMaps& maps, const ConvArgs& args, dim3 grid, int threads, cudaStream_t stream) {
    static PerDevice<bool> attr;  // function attributes are per device
    if (!attr.cur()) {
        cudaError_t e = cudaFuncSetAttribute(conv3x3_pair_kernel<NOUT, MASKED>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemMax);
        if (e != cudaSuccess) return e;
        attr.cur() = true;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = kSmemMax;  // the full 227 KB: exactly one CTA (one 512-column TMEM allocation) per SM
    cfg.stream = stream;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    at[1].id = cudaLaunchAttributeClusterDimension;
    at[1].val.clusterDim.x = 2;
    at[1].val.clusterDim.y = 1;
    at[1].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 2;
    return cudaLaunchKernelEx(&cfg, conv3x3_pair_kernel<NOUT, MASKED>, maps.a, maps.o16, maps.of, args);
}

// `nout`: accumulator columns per output row and pair (64, 32, 16); `nslices` pair-slices cover Cout (blockIdx.y).
cudaError_t conv3x3_pair_launch(const ConvMaps& maps, const ConvArgs& args_in, int nout, int nslices, int num_sms,
                                cudaStream_t stream) {
    ConvArgs args = args_in;
    const int subw = nout == 64 ? 32 : nout;
    const int wbytes = args.nchunks * 3 * (3 * nout / 2) * 128;
    const int smem = 1024 + wbytes + args.nstages * kStageBytes + args.nepi * epi_group_bytes_pair(args, subw) + kMiscBytes;
    if (args.nstages < 2 || args.nepi < 1 || args.nepi > 3 || smem > kSmemMax) return cudaErrorInvalidConfiguration;
    if (args.has_outf && subw != 32) return cudaErrorInvalidConfiguration;
    const long long ncg2 = (args.ncg + 1) / 2;
    args.rows_total_pair = ncg2 * args.H;
    long long npairs = (num_sms / 2) / nslices;
    const long long min_rows = 4;  // do not shred tiny problems into 1-row strips (2 halo rows each)
    const long long cap = (args.rows_total_pair + min_rows - 1) / min_rows;
    if (npairs > cap) npairs = cap;
    if (npairs < 1) npairs = 1;
    if (args.rows_total_pair * (npairs + 1) >= (1ll << 31)) return cudaErrorInvalidValue;   // the kernel's strip arithmetic is 32-bit
    if (args.tail_ksteps != 1 && args.tail_ksteps != 2 && args.tail_ksteps != 4) args.tail_ksteps = 4;
    const dim3 grid(static_cast<unsigned>(2 * npairs), static_cast<unsigned>(nslices), 1);
    const int threads = 128 + 128 * args.nepi;
    if (args.vmask) {
        if (nout == 64) return launch_pair_t<64, true>(maps, args, grid, threads, stream);
        if (nout == 32) return launch_pair_t<32, true>(maps, args, grid, threads, stream);
        if (nout == 16) return launch_pair_t<16, true>(maps, args, grid, threads, stream);
        return cudaErrorInvalidValue;
    }
    if (nout == 64) return launch_pair_t<64, false>(maps, args, grid, threads, stream);
    if (nout == 32) return launch_pair_t<32, false>(maps, args, grid, threads, stream);
    if (nout == 16) return launch_pair_t<16, false>(maps, args, grid, threads, stream);
    return cudaErrorInvalidValue;
}

int conv3x3_wait_profile(unsigned long long* out16, int reset) {
    if (out16 && cudaMemcpyFromSymbol(out16, g_wait_prof, sizeof(unsigned long long) * 16) != cudaSuccess) return -1;
    if (reset) {
        unsigned long long z[16] = {0};
        if (cudaMemcpyToSymbol(g_wait_prof, z, sizeof(z)) != cudaSuccess) return -1;
    }
    return 0;
}

// 0: never pair, 1: pair when the problem is large enough (default), 2: pair whenever two column groups exist
static int g_pair_policy = -1;
int conv3x3_set_pair_policy(int policy) {
    if (g_pair_policy < 0) g_pair_policy = getenv("RESR_CONV_PAIR") ? atoi(getenv("RESR_CONV_PAIR")) : 1;
    const int prev = g_pair_policy;
    if (policy >= 0 && policy <= 2) g_pair_policy = policy;
    return prev;
}

bool conv3x3_choose(ConvArgs* a, int pack_nout, int pack_nslices, ConvLaunchCfg* cfg) {
    const int env_pair = conv3x3_set_pair_policy(-1);
    static const int env_n64 = getenv("RESR_CONV_PAIR_N64") ? atoi(getenv("RESR_CONV_PAIR_N64")) : 1;
    cfg->pair = 0;
    cfg->nout = pack_nout;
    cfg->nslices = pack_nslices;
    // Pairs pay off once every pair has a real strip of rows: below ~6 rows per pair (cfg4's 16x3x64x64 training batch:
    // 256 pair-rows over 74 pairs) the launch is dominated by its prologue and the two halo rows per strip, and the
    // single-CTA kernel is as fast or faster (measured 25.6 vs 26.4 ms per training step). RESR_CONV_PAIR=2 forces pairs.
    const long long pair_rows = static_cast<long long>((a->ncg + 1) / 2) * a->H;
    const bool big_enough = pair_rows >= 6 * 74 || env_pair == 2;
    if (env_pair && a->ncg >= 2 && big_enough) {
        ConvArgs t = *a;
        int nout = pack_nout, nslices = pack_nslices;
        if (env_n64 && pack_nout == 32 && pack_nslices % 2 == 0) { nout = 64; nslices = pack_nslices / 2; }
        if (conv3x3_pair_plan_smem(&t, nout)) {
            *a = t;
            cfg->pair = 1; cfg->nout = nout; cfg->nslices = nslices;
            return true;
        }
    }
    return conv3x3_plan_smem(a, pack_nout);
}

cudaError_t conv3x3_run(const ConvMaps& maps, const ConvArgs& args, const ConvLaunchCfg& cfg, int num_sms, cudaStream_t stream) {
    if (cfg.pair) return conv3x3_pair_launch(maps, args, cfg.nout, cfg.nslices, num_sms, stream);
    return conv3x3_launch(maps, args, cfg.nout, cfg.nslices, num_sms, stream);
}

}  // namespace resr
