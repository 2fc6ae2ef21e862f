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
//   * Epilogue (conv3x3_common.cuh, shared with the CTA-pair kernel): one to three groups of 4 warps take alternate
//     output rows: TMEM -> registers -> residual / LeakyReLU -> shared-memory staging tile -> TMA store (coalesced NHWC
//     writes, also the 2x nearest-upsampled variant). Each thread reads its pixel's residual channels straight into
//     registers, issued before the wait for the accumulator so that the latency hides behind the row's MMAs.
//
// Warp roles: warp 0 lane 0 = TMA producer, warp 1 lane 0 = MMA issuer, warp 2 = TMEM allocator,
// warps 4-7 (8-11, 12-15) = epilogue groups.
#include "conv3x3_common.cuh"

namespace resr {

static constexpr int kSlots = 16;          // TMEM accumulator ring

__device__ __forceinline__ RowRange cta_rows(const ConvArgs& a) {
    RowRange r;
    const unsigned rows = static_cast<unsigned>(a.rows_total);
    r.g0 = static_cast<int>(rows * blockIdx.x / gridDim.x);
    r.g1 = static_cast<int>(rows * (blockIdx.x + 1) / gridDim.x);
    return r;
}

__device__ __forceinline__ uint32_t slot_of(uint32_t v) { return (16u - (v & 15u)) & 15u; }

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
                const int ks = (st >= nsteps - (MODE == 0 ? 1 : 3)) ? a.tail_ksteps : 4;  // steps of the last K chunk
                if (elect_one()) {
                    issue_half<NOUT, MODE == 0 ? 3 : 1, 0>(ks, s0, d0, tbase, a_lo, b_lo, idesc3, idesc2, idesc1);
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
                    issue_half<NOUT, MODE == 0 ? 3 : 1, 1>(ks, s0, d0, tbase, a_cur, b_lo, idesc3, idesc2, idesc1);
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
                            mbar_expect_tx(full + stage, tx_bytes);
                            tma_load_4d(stg + stage * kStageBytes, &tmapA, full + stage, c * 64, a.mode == 0 ? x0 - 1 : x0 + dx - 1, r, n0);
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
        tc_fence_after();
        if (a.mode == 0) mma_role<NOUT, 0>(a, rr, tbase, smem_u32(wsm), smem_u32(stg), smem_u32(full), smem_u32(empty), smem_u32(acc_full), smem_u32(slot_free));
        else mma_role<NOUT, 1>(a, rr, tbase, smem_u32(wsm), smem_u32(stg), smem_u32(full), smem_u32(empty), smem_u32(acc_full), smem_u32(slot_free));
    } else if (warp >= 4) {
        // ------------------------------------------------------------------ epilogue groups
        const int gi = (warp - 4) >> 2;
        const int q = warp & 3;        // TMEM lane quadrant this warp may access
        const int m = q * 32 + lane;   // M row == TMEM lane == pixel of the tile
        const bool lead_warp = ((warp - 4) & 3) == 0;  // first warp of the group issues its TMA traffic
        // per-slice residual selection (backward: slices whose input gradient is not accumulated skip res1)
        const bool use_res1 = slice_on(a.has_res1, a.slice_nores_mask, slice);
        EpiGroup grp{epi + gi * epi_bytes, 0, false, 0, gi, m, lead_warp};   // one staging buffer per group
        const uint32_t lane_base = tbase + (static_cast<uint32_t>(q * 32) << 16);
        const int img_in_tile = m / a.BW;
        const int x_in_tile = m % a.BW;
        {   // zero this group's share of the accumulator ring, then hand the slots to the MMA issuer
            const int s_lo = gi * kSlots / a.nepi, s_hi = (gi + 1) * kSlots / a.nepi;
            for (int s = s_lo; s < s_hi; ++s) tmem_init_bias<NOUT>(lane_base + s * NOUT, bias_s);
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
            const int ra = max(ya - 1, 0), rb = min(yb, H - 1);
            const int n_acc = rb - ra + 3;
            for (int j = 0; j < n_acc; ++j) {
                const uint32_t v = v0 + j;
                if (static_cast<int>(v % static_cast<uint32_t>(a.nepi)) != gi) continue;
                const int y = ra - 1 + j;
                const bool emit = (y >= ya) && (y < yb);
                const uint32_t slot = slot_of(v);
                const EpiPixel px = epi_pixel<MASKED>(a, n0, x0, n0 + img_in_tile, x0 + x_in_tile, y, emit);
                float4 resv[NOUT / 4];
                if (emit && use_res1) epi_load_res1<NOUT>(a, px.pix, slice, resv);
                mbar_wait(acc_full + slot, static_cast<uint32_t>(v >> 4) & 1);
                tc_fence_after();
                float val[NOUT];
                tmem_ld_w<NOUT>(lane_base + slot * NOUT, val);
                tmem_ld_wait();
                tmem_init_bias<NOUT>(lane_base + slot * NOUT, bias_s);
                tmem_st_wait();
                tc_fence_before();
                mbar_arrive(slot_free + slot);
                if (emit) epi_pass<NOUT, MASKED>(a, &tmapO16, &tmapOF, grp, px, slice, val, resv);
            }
            v0 += n_acc;
            g += yb - ya;
        }
        if (lead_warp) tma_store_wait_all();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tbase, 512);
}

// --------------------------------------------------------------------------------------------- host side

void conv3x3_init_geometry(ConvArgs* a, int N, int H, int W, int cin, int mode) {
    a->N = N; a->H = H; a->W = W;
    if (W == 64 || W == 32 || W == 16 || W == 8) {   // BN images of W columns share one 128-lane tile
        a->BW = W;
        a->BN = 128 / W;
    } else {
        a->BW = 128;
        a->BN = 1;
    }
    a->mode = a->BN != 1 ? 1 : (mode >= 0 ? mode : 0);   // lanes that span images need one load per dx
    a->nxs = (W + a->BW - 1) / a->BW;
    a->ncg = ((N + a->BN - 1) / a->BN) * a->nxs;
    a->rows_total = static_cast<long long>(a->ncg) * H;
    // K16 steps of the last 64-channel chunk that hold real input channels; the zero-weight rest is not issued
    const int r = cin % 64;
    a->tail_ksteps = r == 0 || r > 32 ? 4 : (r > 16 ? 2 : 1);
}

PFN_encodeTiled get_encode_fn() {
    // looked up once per process; the initialisation of a function-local static is thread-safe (several host threads
    // plan forwards at once)
    static const PFN_encodeTiled fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            return reinterpret_cast<PFN_encodeTiled>(p);
        return static_cast<PFN_encodeTiled>(nullptr);
    }();
    return fn;
}

int conv3x3_make_tmap_act(CUtensorMap* out, const void* base, int N, int H, int W, int C, int mode, int BW, int BN,
                          int cvalid) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return -1;
    // Channels at and beyond `cvalid` are out of bounds for the map: the 64-channel box of the tail chunk is zero-filled
    // there instead of fetching the neighbouring (zero-weight) channels of the concat buffer from DRAM. The map ends at
    // exactly `cvalid` (TMA extents need no alignment, only the strides do): a zero weight times a NaN or Inf in a
    // channel past `cvalid` would still be NaN. A caller that owns zeroed padding channels may pass cvalid rounded up
    // to 8: a 16-byte row per pixel loads faster than a 6-byte one (the 3-channel first convolution).
    int cdim = cvalid > 0 ? cvalid : C;
    if (cdim > C) cdim = C;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(cdim), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                                static_cast<cuuint64_t>(N)};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(W) * C * 2,
                                   static_cast<cuuint64_t>(H) * W * C * 2};
    cuuint32_t box[4] = {64, static_cast<cuuint32_t>(mode == 0 ? BW + 2 : BW), 1, static_cast<cuuint32_t>(mode == 0 ? 1 : BN)};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    // L2 promotion: 128 B fetches suit full 64-channel chunks (128 B per pixel); a layer whose last chunk holds only 32
    // channels (Cin = 96 / 160) would drag the other half of every 128-byte line in from DRAM (ncu: 278 MB read for the
    // 201 MB a 96-channel layer needs), so those maps promote to 64 B.
    const CUtensorMapL2promotion promo = (cdim % 64 != 0) ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B : CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
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

cudaError_t conv3x3_tc_launch(const ConvMaps& maps, const ConvArgs& args, int nout, int nslices, int num_sms,
                              cudaStream_t stream) {
    const long long units = args.rows_total;
    if (args.vmask) {
        if (nout == 32) return conv3x3_launch_grid<conv3x3_tc_kernel<32, true>>(maps, args, 32, 1, units, nslices, num_sms, stream);
        if (nout == 16) return conv3x3_launch_grid<conv3x3_tc_kernel<16, true>>(maps, args, 16, 1, units, nslices, num_sms, stream);
        return cudaErrorInvalidValue;
    }
    if (nout == 32) return conv3x3_launch_grid<conv3x3_tc_kernel<32, false>>(maps, args, 32, 1, units, nslices, num_sms, stream);
    if (nout == 16) return conv3x3_launch_grid<conv3x3_tc_kernel<16, false>>(maps, args, 16, 1, units, nslices, num_sms, stream);
    return cudaErrorInvalidValue;
}

}  // namespace resr
