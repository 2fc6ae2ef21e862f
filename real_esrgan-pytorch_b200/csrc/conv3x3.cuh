// Internal interface of the tcgen05 3x3 convolution ("row-rolling implicit GEMM", see DESIGN.md §3).
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace resr {

// Epilogue arithmetic selector (what the reference does after each nn.Conv2d).
enum EpMode : int {
    EP_PLAIN = 0,  // v = acc + b                       (model.py:90-93 conv1..4, :258, :264-269)
    EP_RDB = 1,    // v = (acc + b) * 0.2 + res1         (model.py:94-96)
    EP_RRDB = 2,   // v = ((acc + b) * 0.2 + res1) * 0.2 + res2   (model.py:94-96 then :129-130)
    EP_SKIP = 3,   // v = res1 + (acc + b)               (model.py:261-262)
    EP_ADD2 = 4,   // v = (acc + b) [+ res1] + res2_scale * res2   (backward: gradient accumulation)
};

struct ConvArgs {
    // geometry of this convolution (input resolution == output resolution, stride 1, zero pad 1)
    int N, H, W;
    int BW, BN;     // one 128-lane M tile = BW consecutive x  *  BN consecutive images
    int nxs;        // x segments per image row = ceil(W / BW)
    int ncg;        // column groups = ceil(N / BN) * nxs
    int nchunks;    // input channels / 64 (zero-padded weights cover the remainder)
    int tail_ksteps;  // K16 steps of the LAST chunk that carry real channels (1..4); the zero-weight rest is not issued
    int mode;       // 0: one TMA load of BW+2 px per (row, chunk), dx taken by shifting the smem descriptor
                    // 1: three TMA loads per (row, chunk), one per dx (any BW x BN split)
    int nstages;    // activation ring depth
    int nepi;       // epilogue warp groups (1 .. 3), rows alternate between them
    int reverse;    // pair kernel: traverse the work back to front (rows bottom-up, column groups last to first, dy taps
                    // flipped when the weights are gathered). Consecutive layers alternate direction, so a launch starts
                    // on the data its predecessor touched last -- what is still in the 126 MB L2.
    int epi_bufs;   // staging tiles per epilogue group (2 = a pass never waits for the previous pass's TMA store; the
                    // single-CTA kernel uses 1)
    int fmt_in;     // MMA operand format: 0 fp16, 1 bf16
    long long rows_total;  // ncg * H
    long long rows_total_pair;  // ceil(ncg / 2) * H: work units of the CTA-pair kernel (filled by its launcher)
    const uint8_t* wpack;  // [slice][chunk][dx][(dy,co) x 64ch] 16-bit, 128B-swizzled, ready for a bulk copy
    const float* bias;     // [nslices * NOUT]
    // epilogue
    int ep_mode, lrelu, clamp01;
    int has_out16;         // 16-bit NHWC output through tmapO16 (TMA store from a staging tile)
    int out16_fmt;         // 0 fp16, 1 bf16
    int out16_choff;       // first destination channel of slice 0
    int out16_up2;         // 1: destination is [N,2H,2W,*]; every pixel is written to its 2x2 nearest-upsampled sites
    int has_outf;          // fp32 NHWC output: each epilogue thread stores its pixel's 128 contiguous bytes directly
    int outf_choff;
    float* outf;           // base of the fp32 NHWC output, outf_cstride channels per pixel
    int outf_cstride;
    int has_res1;          // fp32 NHWC residual: each epilogue thread loads its pixel's channels straight into registers
    int res_choff;         //   before it waits for the accumulator (no shared-memory tile, no dependency on the TMA queue)
    const void* res1;
    int res1_cstride;
    int res16;             // 0: res1 / res2 are fp32; 1: both are 16-bit NHWC tensors in format res16_fmt (the residual
    int res16_fmt;         //    stream of the inference trunk IS the fp16 conv input: no fp32 master is kept)
    const void* res2;      // second residual (EP_RRDB / EP_ADD2): plain global loads
    int res2_cstride;
    float* out_nchw;       // NCHW fp32 output with out_nchw_c channels (or null)
    int out_nchw_c;
    unsigned char* out_u8; // NHWC u8 image output with out_nchw_c channels (or null): tensor_to_image fused into the last conv
                           // (imgproc.py:1594: mul(255).clamp(0, 255) then astype(uint8) = truncation)
    // ---- backward (data-gradient) extensions; all zero in the forward pass
    unsigned slice_nores_mask;  // bit s: Cout slice s does not read res1
    unsigned slice_noutf_mask;  // bit s: slice s does not write the fp32 output
    unsigned slice_no16_mask;   // bit s: slice s does not write the 16-bit output
    int out16_slice_fixed;      // 1: every writing slice stores at out16_choff (instead of out16_choff + slice * cout_slice)
    const void* mask16;         // LeakyReLU' mask source: NHWC 16-bit activations; v *= (act > 0 ? 1 : 0.2) before out16
    int mask16_cstride, mask16_choff;
    float res2_scale;           // EP_ADD2
    float out16_scale;          // != 0: the 16-bit output stores out16_scale * v (the fp32 output keeps v): the next dense block's dY5
    float* out_nchw_raw;        // pre-clamp copy of the NCHW output (training: clamp backward needs it)
    // ---- packed canvas of several images (N == 1; generator.cu resr_generator_forward_many): null = every pixel is valid
    const uint32_t* vmask;      // bitmap of the valid LR pixels, row-major, vmask_words 32-bit words per LR row (non-null
                                // selects the kernels' MASKED instantiation; the unmasked one is the code without canvas)
    int vmask_words;
    int vmask_shift;            // this layer's resolution: pixel (x, y) is valid iff LR bit (x >> shift, y >> shift) is set;
                                // every output of an invalid pixel is written as 0, so a zero gutter between images stays zero
};

// Fills the launch geometry of an N x H x W convolution: N / H / W, the lane split BW x BN, mode (-1: automatic, i.e. 0
// when a tile is one image row; lanes that span images always take mode 1), nxs, ncg, rows_total, and tail_ksteps from
// the real input channels `cin` (0: every 64-channel chunk is full).
void conv3x3_init_geometry(ConvArgs* args, int N, int H, int W, int cin, int mode);

struct ConvMaps {
    CUtensorMap a;    // activations (load)
    CUtensorMap o16;  // 16-bit output (store), 4-D or 5-D (up2)
    CUtensorMap of;   // fp32 output (store)
};

// Kernel choice for one convolution whose weights are packed in `pack_nout`-channel slices (`pack_nslices` of them).
struct ConvLaunchCfg {
    int pair;     // 1: CTA-pair kernel, 0: single-CTA kernel
    int nout;     // channels per launch slice
    int nslices;  // blockIdx.y extent
};
// Picks the kernel: the CTA-pair kernel (conv3x3_pair.cu: tcgen05 cta_group::2, M = 256, same weight packs) whenever
// there are at least two column groups to pair up and enough rows, the single-CTA kernel (conv3x3_tc.cu) otherwise;
// RESR_CONV_PAIR=0 forces the single-CTA kernel. Fills args->nstages / nepi / epi_bufs. Returns false if the
// configuration does not fit in shared memory.
int conv3x3_set_pair_policy(int policy);  // returns the previous policy; -1 only queries
bool conv3x3_choose(ConvArgs* args, int pack_nout, int pack_nslices, ConvLaunchCfg* cfg);

// Clusters of `cluster` CTAs per Cout slice of the persistent grid over `units` work units: as many as the SMs hold,
// but at least 4 rows of work each (tiny problems are not shredded into 1-row strips with 2 halo rows each).
inline long long conv3x3_clusters(long long units, int cluster, int nslices, int num_sms) {
    long long nclusters = (num_sms / cluster) / nslices;
    const long long min_rows = 4;
    const long long cap = (units + min_rows - 1) / min_rows;
    if (nclusters > cap) nclusters = cap;
    return nclusters < 1 ? 1 : nclusters;
}
cudaError_t conv3x3_run(const ConvMaps& maps, const ConvArgs& args, const ConvLaunchCfg& cfg, int num_sms, cudaStream_t stream);

// Tensor maps. base: NHWC tensor [N,H,W,C].
int conv3x3_make_tmap_act(CUtensorMap* out, const void* base, int N, int H, int W, int C, int mode, int BW, int BN,
                          int cvalid = 0);  // cvalid: channels the convolution reads (0 = all C)
int conv3x3_make_tmap_out16(CUtensorMap* out, const void* base, int N, int H, int W, int C, int nout, int BW, int BN,
                            int up2);  // N,H,W = geometry of the CONVOLUTION (destination is 2H x 2W when up2)
int conv3x3_make_tmap_f32(CUtensorMap* out, const void* base, int N, int H, int W, int C, int BW, int BN);

}  // namespace resr
