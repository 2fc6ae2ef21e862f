// Shared between generator.cu (inference) and train.cu (training forward / backward): layer table, plan, handle.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "conv3x3.cuh"

namespace resr {

// ------------------------------------------------------------------------------------------- layer table
struct ConvSpec {
    int cin, cout;
    int nout;      // channels per CTA slice (32, or 16 for the 3-channel output conv)
    int nslices;
    int nchunks;   // ceil(cin / 64)
    int fmt;       // operand format: 0 fp16, 1 bf16
    size_t p_off;  // offset of weight in the flat fp32 parameter vector (bias follows the weight)
    size_t w_off;  // byte offset of the packed weights
    size_t b_off;  // float offset of the padded bias
    size_t wt_off; // byte offset of the packed TRANSPOSED weights (data-gradient convolution: Cin' = cout, Cout' = cin)
    int t_nslices; // ceil(cin / 32)
    int t_nchunks; // ceil(cout / 64)
};

static const int kNumConvs = 351;
static const int kNumRRDB = 23;

struct Table {
    ConvSpec c[kNumConvs];
    size_t n_params, pack_bytes, bias_floats, packt_bytes;
    Table() {
        int i = 0;
        auto add = [&](int cin, int cout, int fmt) {
            ConvSpec& s = c[i++];
            s.cin = cin;
            s.cout = cout;
            s.nout = cout >= 32 ? 32 : 16;
            s.nslices = (cout + s.nout - 1) / s.nout;
            s.nchunks = (cin + 63) / 64;
            s.fmt = fmt;
        };
        // Forward operands are fp16 everywhere (same tensor rate as bf16, 3 more mantissa bits; stored activations
        // saturate at +-65504 -- the reference trains under fp16 autocast, train_realesrnet.py:97). Gradients stay bf16.
        add(3, 64, 0);  // conv1
        for (int r = 0; r < kNumRRDB * 3; ++r) {
            for (int k = 0; k < 4; ++k) add(64 + 32 * k, 32, 0);
            add(192, 64, 0);
        }
        add(64, 64, 0);  // conv2 reads the fp16 trunk output
        add(64, 64, 0);  // upsampling1.0   (tail runs with fp16 operands, SURVEY.md §7.3-1)
        add(64, 64, 0);  // upsampling2.0
        add(64, 64, 0);  // conv3.0
        add(64, 3, 0);   // conv4
        size_t p = 0, w = 0, b = 0, wt = 0;
        for (int k = 0; k < kNumConvs; ++k) {
            c[k].p_off = p;
            p += static_cast<size_t>(c[k].cout) * c[k].cin * 9 + c[k].cout;
            c[k].w_off = w;
            w += static_cast<size_t>(c[k].nslices) * c[k].nchunks * 3 * (3 * c[k].nout) * 128;
            c[k].b_off = b;
            b += static_cast<size_t>(c[k].nslices) * c[k].nout;
            c[k].t_nslices = (c[k].cin + 31) / 32;
            c[k].t_nchunks = (c[k].cout + 63) / 64;
            c[k].wt_off = wt;
            wt += static_cast<size_t>(c[k].t_nslices) * c[k].t_nchunks * 3 * 96 * 128;
        }
        n_params = p;
        pack_bytes = w;
        bias_floats = b;
        packt_bytes = wt;
    }
};
inline const Table& table() {
    static Table t;
    return t;
}


// ------------------------------------------------------------------------------------------- generator object
struct Step {
    int conv;   // index into the layer table
    ConvMaps maps;
    ConvArgs a;
    ConvLaunchCfg cfg;  // which kernel runs it (CTA pair or single CTA) and its slicing
};

struct Plan {
    int N = 0, H = 0, W = 0;
    void* ws = nullptr;
    std::vector<Step> steps;
    uint16_t* xin = nullptr;
    int pair_policy = -1;  // conv3x3_set_pair_policy value the steps were planned under
    bool valid = false;
};

}  // namespace resr

struct resr_generator {
    // training-step CUDA graph (train.cu): one cached instantiation per argument set
    cudaGraphExec_t step_exec = nullptr;
    const void* step_key[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int step_shape[3] = {0, 0, 0};
    int step_precision = -1;      // recipe the graph was captured under: its kernels and pack formats are that recipe's
    bool step_graph_failed = false;
    // pipelined host path (generator.cu): copy streams, per-slot events, call counter
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_fwd[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    unsigned long long host_calls = 0;
    int host_shape[3] = {0, 0, 0};   // shape / workspace of the previous pipelined host call (staging-slot layout)
    const void* host_ws = nullptr;
    // second stream of the backward pass: the weight-gradient chain of a layer runs beside the data-gradient chain
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_dy = nullptr, ev_join = nullptr;
    cudaEvent_t ev_dyc[3] = {nullptr, nullptr, nullptr};  // the weight gradient has read this dYcat buffer (side stream)
    bool ev_dyc_valid[3] = {false, false, false};
    // gradient buckets (data-parallel training): bucket i of the flat gradient vector is complete when ev_bucket[i] fires
    // (recorded on the weight-gradient stream inside the backward, as an EXTERNAL event when the step is being captured)
    cudaEvent_t ev_bucket[4] = {nullptr, nullptr, nullptr, nullptr};
    uint8_t* wpack_t = nullptr;   // transposed packs for the backward data-gradient convolutions (lazily allocated)
    uint8_t* wpack_t2 = nullptr;  // mirrored dense-block data-gradient packs (train.cu), laid out like the forward packs
    float* zero_bias = nullptr;
    bool packed_t = false;
    const float* flat_params = nullptr;  // last parameter vector handed to load_params (device memory, caller-owned)
    uint8_t* wpack = nullptr;
    void* pack_jobs = nullptr;    // device tables of the batched weight-pack kernel (forward / transposed)
    void* pack_jobs_t = nullptr;
    float* bias = nullptr;
    bool loaded = false;
    int num_sms = 148;
    int precision = 0;            // inference recipe: 0 = fp16 operands / fp16 residual stream, 1 = bf16 operands + fp32 residual masters
    resr::Plan plan;
    std::vector<resr::Plan> canvas_plans;  // packed-canvas plans of resr_generator_forward_many, oldest first (a few shapes)
};


namespace resr {
int grid_for(size_t total, int block);

// One convolution of the training path (train.cu) or of the VGG19 content loss (vgg.cu), launched with tensor maps encoded
// per call: what goes in, which weights, which epilogue, what comes out.
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
    const void* mask16 = nullptr; int mask16_c = 64, mask16_choff = 0, mask16_relu = 0;
    int ep_mode = EP_PLAIN, lrelu = 0, clamp01 = 0, relu = 0;
    float out16_scale = 0.f;
    float* out_nchw = nullptr; float* out_nchw_raw = nullptr; int out_nchw_c = 3;
};
int launch_conv_io(int num_sms, const Geo& q, int N, const ConvIO& io, cudaStream_t s);
// OIHW fp32 -> packed 16-bit tiles (generator.cu). transposed=1 packs the data-gradient convolution
// W'[ci][co][dy][dx] = W[co][ci][2-dy][2-dx] (cin/cout are the FORWARD channel counts; bias ignored).
// (re)builds the transposed packs if the handle has them allocated or `force` is set (train.cu)
void ensure_transposed_packs(resr_generator* g, cudaStream_t s, bool force);
int launch_pack_all(resr_generator* g, const float* flat, int transposed, cudaStream_t s);
int launch_pack_rdb_bwd(resr_generator* g, const float* flat, uint8_t* wpack_t2, cudaStream_t s);
void launch_pack_conv(const float* w, const float* bias, uint16_t* wp, float* bp, int cin, int cout, int nout, int nslices,
                      int nchunks, int fmt, int transposed, cudaStream_t s);
}  // namespace resr
