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
#include <cstdlib>

#include "conv3x3_common.cuh"

namespace resr {

namespace {

template <int S>
__device__ __forceinline__ uint32_t ring_slot(uint32_t v) { return (S - v % S) % S; }
template <int S>
__device__ __forceinline__ uint32_t ring_parity(uint32_t v) { return (v / S) & 1u; }

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
                while (static_cast<int>(vnew - acq) >= 0) {
                    mbar_wait_a(slotfree_a + (ring_slot<S>(acq) << 3), ring_parity<S>(acq));
                    ++acq;
                }
            }
            slot_ready = false;
            tc_fence_after();
            const uint32_t s0 = ring_slot<S>(vnew), s1 = ring_slot<S>(vnew - 1), s2 = ring_slot<S>(vnew - 2);
            const uint32_t d0 = tbase + s0 * NOUT;   // the three dy blocks land on s0, s0+1, s0+2 (possibly overflow slots)
            uint32_t b_lo = w_lo;
            for (int st = 0; st < nsteps; ++st, b_lo += b_step) {
                if (!full_ready) mbar_wait_a(full_a + (stage << 3), phase);
                tc_fence_after();
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
}

template <int W>
__device__ __forceinline__ void tmem_zero_w(uint32_t taddr) {
    if (W == 32) tmem_st_zero32(taddr); else tmem_st_zero16(taddr);
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
    const int epi_bytes = epi_group_bytes(a, SUBW);

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
                        mbar_wait(empty + stage, phase ^ 1);
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
        EpiGroup grp{epi + gi * epi_bytes, epi_buf_bytes(a, SUBW), a.epi_bufs == 2, 0, gi, m, lead_warp};
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
        uint32_t v0 = 0;
        const int ncg2 = (a.ncg + 1) >> 1;
        for (int g = rr.g0; g < rr.g1;) {
            const int cg2 = g / H;
            const int cg = 2 * (a.reverse ? ncg2 - 1 - cg2 : cg2) + static_cast<int>(rank);
            const int ya = g % H;
            const int yb = min(H, ya + (rr.g1 - g));
            const int n0 = (cg / a.nxs) * a.BN;
            const int x0 = (cg % a.nxs) * a.BW;
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
                const EpiPixel px = epi_pixel<MASKED>(a, n0, x0, n0 + img_in_tile, x0 + x_in_tile, y, emit);
                bool waited = false;
#pragma unroll 1
                for (int h = 0; h < NSUB; ++h) {
                    const int ls = slice * NSUB + h;   // logical 32-channel slice (channel offsets, per-slice flags)
                    float4 resv[SUBW / 4];
                    if (emit && slice_on(a.has_res1, a.slice_nores_mask, ls)) epi_load_res1<SUBW>(a, px.pix, ls, resv);
                    if (!waited) {
                        mbar_wait(acc_full + slot, ring_parity<S>(v));
                        tc_fence_after();
                        waited = true;
                    }
                    float val[SUBW];
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
                    if (emit) epi_pass<SUBW, MASKED>(a, &tmapO16, &tmapOF, grp, px, ls, val, resv);
                }
            }
            v0 += n_acc;
            g += yb - ya;
        }
        if (lead_warp) tma_store_wait_all();
    }

    // no CTA of the pair may exit while its peer can still signal its barriers / read its shared memory
    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) tmem_dealloc2(tbase, 512);
}

// --------------------------------------------------------------------------------------------- host side

// Fills nepi / epi_bufs / nstages from the shared-memory budget of a CTA that keeps `wbytes` of weights resident and
// stages `subw` channels per epilogue pass; `max_bufs` (1 or 2) staging buffers per epilogue group at most. Returns
// false if the configuration does not fit.
static bool plan_smem(ConvArgs* a, int wbytes, int subw, int max_bufs) {
    // The per-row epilogue latency (TMEM drain, staging, TMA store; ~1.6k cycles, more with an fp32 output tile) is hidden
    // by running several epilogue groups on consecutive rows. Three groups whenever they fit beside at least four
    // stages (8 KB of shared memory each without an fp32 tile); two with the 24 KB fp32 variant.
    for (int nepi = a->has_outf ? 2 : 3;; --nepi) {
        a->nepi = nepi;
        for (int bufs = max_bufs; bufs >= 1; --bufs) {
            a->epi_bufs = bufs;
            const int fixed = 1024 + wbytes + nepi * epi_group_bytes(*a, subw) + kMiscBytes;
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

// 0: never pair, 1: pair when the problem is large enough (default), 2: pair whenever two column groups exist
// Read by every plan, possibly from several host threads at once: an atomic, initialised once from the environment.
static std::atomic<int>& pair_policy() {
    static std::atomic<int> p{getenv("RESR_CONV_PAIR") ? atoi(getenv("RESR_CONV_PAIR")) : 1};
    return p;
}
int conv3x3_set_pair_policy(int policy) {
    std::atomic<int>& p = pair_policy();
    return policy >= 0 && policy <= 2 ? p.exchange(policy) : p.load();
}

bool conv3x3_choose(ConvArgs* a, int pack_nout, int pack_nslices, ConvLaunchCfg* cfg) {
    const int policy = conv3x3_set_pair_policy(-1);
    cfg->pair = 0;
    cfg->nout = pack_nout;
    cfg->nslices = pack_nslices;
    // Pairs pay off once every pair has a real strip of rows: below ~6 rows per pair (cfg4's 16x3x64x64 training batch:
    // 256 pair-rows over 74 pairs) the launch is dominated by its prologue and the two halo rows per strip, and the
    // single-CTA kernel is as fast or faster (measured 25.6 vs 26.4 ms per training step). RESR_CONV_PAIR=2 forces pairs.
    const long long pair_rows = static_cast<long long>((a->ncg + 1) / 2) * a->H;
    const bool big_enough = pair_rows >= 6 * 74 || policy == 2;
    if (policy && a->ncg >= 2 && big_enough) {
        ConvArgs t = *a;
        int nout = pack_nout, nslices = pack_nslices;
        // two 32-channel pack slices per pair: the 192 -> 64 convolution of a dense block is ONE N = 192 MMA per K step
        if (pack_nout == 32 && pack_nslices % 2 == 0) { nout = 64; nslices = pack_nslices / 2; }
        if (plan_smem(&t, conv3x3_weight_bytes(t, nout, 2), nout == 64 ? 32 : nout, 2)) {
            *a = t;
            cfg->pair = 1; cfg->nout = nout; cfg->nslices = nslices;
            return true;
        }
    }
    return plan_smem(a, conv3x3_weight_bytes(*a, pack_nout, 1), pack_nout, 1);   // the single-CTA kernel stages in one buffer
}

cudaError_t conv3x3_run(const ConvMaps& maps, const ConvArgs& args_in, const ConvLaunchCfg& cfg, int num_sms, cudaStream_t stream) {
    ConvArgs args = args_in;
    if (args.tail_ksteps != 1 && args.tail_ksteps != 2 && args.tail_ksteps != 4) args.tail_ksteps = 4;
    if (!cfg.pair) return conv3x3_tc_launch(maps, args, cfg.nout, cfg.nslices, num_sms, stream);
    // `nout`: accumulator columns per output row and pair (64, 32, 16); `nslices` pair-slices cover Cout (blockIdx.y)
    const int nout = cfg.nout, nslices = cfg.nslices;
    if (args.has_outf && nout == 16) return cudaErrorInvalidConfiguration;   // the fp32 tile holds 32 channels
    args.rows_total_pair = static_cast<long long>((args.ncg + 1) / 2) * args.H;
    const long long units = args.rows_total_pair;
    if (args.vmask) {
        if (nout == 64) return conv3x3_launch_grid<conv3x3_pair_kernel<64, true>>(maps, args, 64, 2, units, nslices, num_sms, stream);
        if (nout == 32) return conv3x3_launch_grid<conv3x3_pair_kernel<32, true>>(maps, args, 32, 2, units, nslices, num_sms, stream);
        if (nout == 16) return conv3x3_launch_grid<conv3x3_pair_kernel<16, true>>(maps, args, 16, 2, units, nslices, num_sms, stream);
        return cudaErrorInvalidValue;
    }
    if (nout == 64) return conv3x3_launch_grid<conv3x3_pair_kernel<64, false>>(maps, args, 64, 2, units, nslices, num_sms, stream);
    if (nout == 32) return conv3x3_launch_grid<conv3x3_pair_kernel<32, false>>(maps, args, 32, 2, units, nslices, num_sms, stream);
    if (nout == 16) return conv3x3_launch_grid<conv3x3_pair_kernel<16, false>>(maps, args, 16, 2, units, nslices, num_sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace resr
