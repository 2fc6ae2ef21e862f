// Internal interface of the tensor-core weight-gradient kernel (wgrad_mn.cu): operands straight from the NHWC buffers,
// one 16-bit format (bf16) for X and dY.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace resr {

static constexpr int kMnMaxKinds = 12;
struct WgradMnKind { int ci0, co0, n, dy, cta0, nsplit; };   // unit (128 input channels from ci0) x (n = 64 / 128 dY channels from co0), one dy
struct WgradMnArgs {
    int N, H, W;
    int segs_per_row;         // ceil(W / 64)
    uint32_t kslabs;          // N * H * segs_per_row (one slab = 64 pixels of one row)
    float* partial;           // [cta][3 dx][128 ci][128 co] fp32
    float* bias_partial;      // [cta][256 / n row groups][n] column sums of dY from the (ci0 = 0, dy = 1) CTAs, or null
    int nkinds;
    WgradMnKind kind[kMnMaxKinds];
};
// dY channel slice cs (32 channels) belongs to the layer with gradient dw[cs] (OIHW, cin[cs] x cout[cs]); the slice's first
// channel is output channel co_base[cs] of that layer; db[cs] is the layer's bias gradient (indexed by output channel).
struct WgradMnTable {
    float* dw[6];
    float* db[6];
    int cin[6], cout[6], co_base[6];
};
size_t wgrad_mn_workspace_bytes(int num_sms);
// x: NHWC bf16 [N][H][W][x_cstride] (channels >= x_channels are never read); dy: NHWC bf16 [N][H][W][dy_cstride], channels
// [0, dy_channels). units: (ci0, co0, n) triples with n = 64 or 128. workspace: wgrad_mn_workspace_bytes(num_sms).
int wgrad_mn_launch(const uint16_t* x, int x_cstride, int x_channels, const uint16_t* dy, int dy_cstride, int dy_channels,
                    int N, int H, int W, const int (*units)[3], int nunits, const WgradMnTable& tb, bool with_bias,
                    float* workspace, int num_sms, cudaStream_t s);

}  // namespace resr
