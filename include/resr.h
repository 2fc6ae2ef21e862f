/*
 * resr.h — C ABI of libresr.so: the sm_100a (B200) implementation of the two hot paths of
 * Lornatang/Real_ESRGAN-PyTorch.
 *
 * The reference has no FFI layer: its boundary is the Python module API (SURVEY.md §8b). Each entry point below
 * names the reference call site it replaces (file:line under /root/reference). The reference-side binding a
 * maintainer would add is a ctypes stub; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - the caller owns all memory; the library never frees caller memory and never allocates across the ABI
 *     (handles own their packed weights and cached tensor maps only);
 *   - every function returns 0 on success, non-zero on failure; resr_last_error() gives the message
 *     (thread-local). There is no CPU fallback: without a CUDA device every compute call fails with RESR_E_CUDA.
 *   - image tensors are fp32 NCHW contiguous in [0,1] exactly as the reference scripts hold them.
 */
#ifndef RESR_H_
#define RESR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RESR_OK 0
#define RESR_E_INVALID 1  /* bad argument (the reference would raise ValueError / a shape error) */
#define RESR_E_CUDA 2     /* CUDA runtime / launch failure */
#define RESR_E_NOMEM 3    /* workspace too small */

int resr_version(void);
const char* resr_last_error(void);

/* ------------------------------------------------------------------------------------------------------------
 * Hot path 1 — RRDBNet x4 generator. Replaces model.Generator(3, 3, 4).forward (model.py:206-275),
 * ResidualResidualDenseBlock.forward (model.py:123-132) and ResidualDenseBlock.forward (model.py:87-98).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct resr_generator resr_generator_t;

/* model.py:207-252. Only (in=3, out=3, upscale=4) — the configuration the north star names — is implemented;
 * anything else returns RESR_E_INVALID. */
int resr_generator_create(resr_generator_t** out, int in_channels, int out_channels, int upscale_factor);
void resr_generator_destroy(resr_generator_t* g);

/* Number of fp32 parameters (16,697,987) and of parameter tensors (702) in state_dict order:
 * conv1.{weight,bias}, trunk.{0..22}.rdb{1,2,3}.conv{1..5}.{weight,bias}, conv2.*, upsampling1.0.*,
 * upsampling2.0.*, conv3.0.*, conv4.*  (model.py:223-252). */
size_t resr_generator_num_params(void);
int resr_generator_num_tensors(void);
/* Element offset of tensor `index` (0..701) inside the flat parameter vector, and its element count. */
int resr_generator_tensor_span(int index, size_t* offset, size_t* count);

/* Repack OIHW fp32 weights (flat vector in state_dict order, device memory) into the tap-major 16-bit swizzled
 * tiles the tensor-core kernel streams. Replaces load_state_dict (inference.py:32-33). */
int resr_generator_load_params(resr_generator_t* g, const float* flat_params, void* stream);

size_t resr_generator_workspace_bytes(int n, int h, int w);
/* Inference precision recipe of a handle (north_star names bf16; fp16 is the default because it is more accurate at the
 * same tensor rate): 0 = fp16 MMA operands, the trunk's residual stream is the fp16 conv input itself; 1 = bf16 MMA
 * operands and stored activations with fp32 masters of the residual stream (model.py:94-96, 129-130 evaluated in fp32).
 * After a change the caller must call resr_generator_load_params again (the weight packs carry the operand format).
 * resr_generator_workspace_bytes_for: workspace of THIS handle's recipe (the bf16 recipe adds four fp32 master buffers). */
int resr_generator_set_precision(resr_generator_t* g, int precision);
size_t resr_generator_workspace_bytes_for(const resr_generator_t* g, int n, int h, int w);

/* y[n,3,4h,4w] = clamp(G(x[n,3,h,w]), 0, 1). x, y fp32 NCHW contiguous. model.py:255-275. */
int resr_generator_forward(resr_generator_t* g, const float* x, float* y, int n, int h, int w, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Same, but x_host / y_host are (pinned) HOST buffers: H2D, forward, D2H on `stream`, then a stream synchronise.
 * This is the call inference.py:46-56 turns into. */
/* I/O edges fused into the first / last kernels (SURVEY.md §8 f4): x_u8 is an NHWC u8 RGB batch [n,h,w,3] as decoded by
 * cv2.imread + cvtColor (inference.py:40-46: image / 255 -> image_to_tensor, imgproc.py:1540-1567), y_u8 the NHWC u8 result
 * [n,4h,4w,3] that tensor_to_image (imgproc.py:1570-1596: mul(255).clamp(0,255), uint8 truncation) would produce from the
 * fp32 output. 16x fewer bytes than the fp32 tensors on the way in, 4x fewer on the way out. _host: pinned host buffers,
 * H2D + forward + D2H + synchronise inside the call (staging at the end of the workspace: + n*3*h*w*17 bytes + 2 KB). */
int resr_generator_forward_u8(resr_generator_t* g, const unsigned char* x_u8, unsigned char* y_u8, int n, int h, int w,
                              void* workspace, size_t workspace_bytes, void* stream);
int resr_generator_forward_u8_host(resr_generator_t* g, const unsigned char* x_u8_host, unsigned char* y_u8_host, int n, int h, int w,
                                   void* workspace, size_t workspace_bytes, void* stream);
/* imgproc.tensor_to_image(tensor, range_norm, half) (imgproc.py:1570-1596) on the device: NCHW fp32 [1,c,h,w] -> HWC u8. */
int resr_tensor_to_image_u8(const float* x, unsigned char* out_hwc, int c, int h, int w, int range_norm, int half, void* stream);

int resr_generator_forward_host(resr_generator_t* g, const float* x_host, float* y_host, int n, int h, int w,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Pipelined serving variant of forward_host: returns as soon as the work is queued. Two staging slots rotate, the
 * H2D copy of call k+1 and the D2H copy of call k-1 run on the handle's own copy streams while call k computes on
 * `stream`. y_host of a call is complete after resr_generator_host_sync (or after the second following call returned
 * from its internal wait). The workspace must hold resr_generator_workspace_bytes + 2 x (1 KB-aligned input + output).
 * Use ONE stream and ONE workspace per handle for all async calls. */
int resr_generator_forward_host_async(resr_generator_t* g, const float* x_host, float* y_host, int n, int h, int w,
                                      void* workspace, size_t workspace_bytes, void* stream);
/* Waits for every queued async call of this handle (copies included). */
int resr_generator_host_sync(resr_generator_t* g);

/* A list of differently sized images as ONE packed forward. The reference's image loops (test.py, validate() in
 * train_realesrnet.py / train_realesrgan.py, inference.py over a directory) pass images one at a time; each then pays the
 * full chain of launches at a size that leaves most SMs idle. Here the images are packed into one N = 1 canvas with a
 * zero LR pixel between neighbours, and every convolution writes 0 outside the images, so each result is that image's
 * own forward (DESIGN.md §3.2, packed canvas).
 *
 * resr_canvas_pack: the deterministic shelf packer (host only, no device). hs / ws: count image sizes (1..16384 per side);
 * max_width: widest canvas row of images, <= 0 for a near-square canvas. Returns each image's LR offset (x0, y0) and the
 * canvas size, rounded up to a multiple of 16 rows and 128 columns. Rectangles plus a one-pixel gutter do not overlap.
 * resr_generator_forward_many(_workspace_bytes): xs[i] is image i, fp32 NCHW [1,3,hs[i],ws[i]]; ys[i] receives
 * clamp(G(xs[i]), 0, 1), fp32 NCHW [1,3,4hs[i],4ws[i]]. _u8: NHWC u8 [hs[i],ws[i],3] in, [4hs[i],4ws[i],3] out, with the
 * conversions of resr_generator_forward_u8. The pointer and size ARRAYS are host memory, the images device memory;
 * count is 1..65535. Plans are cached per canvas size beside the single-shape plan of resr_generator_forward. */
int resr_canvas_pack(const int* hs, const int* ws, int count, int max_width, int* x0, int* y0, int* canvas_h, int* canvas_w);
size_t resr_generator_forward_many_workspace_bytes(const resr_generator_t* g, const int* hs, const int* ws, int count);
int resr_generator_forward_many(resr_generator_t* g, const float* const* xs, float* const* ys, const int* hs, const int* ws, int count,
                                void* workspace, size_t workspace_bytes, void* stream);
int resr_generator_forward_many_u8(resr_generator_t* g, const unsigned char* const* xs, unsigned char* const* ys, const int* hs,
                                   const int* ws, int count, void* workspace, size_t workspace_bytes, void* stream);

/* Number of kernels of this library that one resr_generator_forward launches (for bench accounting). */
int resr_generator_launches_per_forward(void);
/* Kernel policy of the 3x3 convolutions: 0 = single-CTA kernel only, 1 = CTA-pair kernel (tcgen05 cta_group::2) when
 * every pair gets a real strip of rows (default; env RESR_CONV_PAIR sets the initial value), 2 = CTA pairs whenever two
 * column groups exist (tests use it to push small / awkward shapes through the pair kernel). Returns the previous policy;
 * a value outside 0..2 only queries. Takes effect for plans built afterwards (new shapes / workspaces). */
int resr_set_conv_pair_policy(int policy);

/* One 3x3 convolution through the same tensor-core kernel (test / building block).
 * in16: NHWC 16-bit activations [n,h,w,c_total]; exactly the first `cin` channels are read (the tensor map ends there:
 * whatever the channels [cin, c_total) hold, NaN included, does not reach the output). c_total is a multiple of 8 and
 * at least cin rounded up to 64. weight: OIHW fp32 [cout,cin,3,3]; bias: fp32 [cout] or NULL.
 * Outputs and residuals are addressed per 32-channel Cout slice: an NHWC output (out16 / outf) needs cout % 32 == 0 and
 * choff + cout <= cstride; cout < 32 (the RGB convolution) writes out_nchw / out_nchw_raw / out_u8 only. 16-bit NHWC
 * strides and offsets are multiples of 8 channels, fp32 ones multiples of 4 (16-byte vector accesses).
 * Every argument is checked on the host before any device work; a bad one returns RESR_E_INVALID. */
typedef struct resr_conv_desc {
    const void* in16;
    int n, h, w, c_total, cin, cout;
    int fmt_in;  /* 0 fp16, 1 bf16 */
    int mode;    /* -1 auto, 0 shifted-descriptor loads, 1 three loads per row */
    const float* weight;
    const float* bias;
    int ep_mode; /* 0 plain, 1 rdb: 0.2*v+res1, 2 rrdb: 0.2*(0.2*v+res1)+res2, 3 skip: res1+v,
                    4 add2: v [+ res1] + res2_scale*res2 (fp32 res2) */
    int lrelu, clamp01;
    void* out16;
    int out16_fmt, out16_cstride, out16_choff, out16_up2;
    float* outf;
    int outf_cstride, outf_choff;
    const void* res1;        /* fp32 NHWC, or 16-bit NHWC when res16 != 0 */
    const void* res2;
    int res_cstride, res_choff;
    int res16, res16_fmt;    /* res16 = 1: res1 / res2 are 16-bit tensors of format res16_fmt (0 fp16, 1 bf16) */
    float* out_nchw;
    int out_nchw_c;          /* channels of out_nchw / out_nchw_raw / out_u8: must equal cout */
    /* ---- what the generator's and the training step's launches set as well (zero: off) */
    int reverse;             /* CTA-pair kernel: walk rows and column groups back to front (serpentine layer order) */
    const uint32_t* vmask;   /* packed canvas: bit (x >> vmask_shift, y >> vmask_shift) of a row-major bitmap with */
    int vmask_words;         /* vmask_words 32-bit words per row marks a valid pixel; every output of an invalid pixel */
    int vmask_shift;         /* is written as 0 */
    unsigned char* out_u8;   /* NHWC u8 [n,h,w,out_nchw_c]: (unsigned char)(255 * v) of the clamped value */
    float* out_nchw_raw;     /* NCHW fp32 copy of the value before clamp01 */
    const void* mask16;      /* LeakyReLU' mask: 16-bit NHWC activations (fp16 or bf16); out16 stores v where the */
    int mask16_cstride, mask16_choff;  /* activation is > 0 and 0.2 v elsewhere (-0 and +0 count as not positive) */
    float out16_scale;       /* != 0: out16 stores out16_scale * v (outf keeps v) */
    float res2_scale;        /* ep_mode 4 */
    int res2_cstride;        /* 0: res_cstride */
    unsigned slice_nores_mask, slice_noutf_mask, slice_no16_mask;  /* bit s: 32-channel slice s skips res1 / outf / out16 */
    int out16_slice_fixed;   /* 1: every writing slice stores at out16_choff instead of out16_choff + 32 s */
} resr_conv_desc;
int resr_conv3x3(const resr_conv_desc* d, void* stream);

/* The launch configuration resr_conv3x3 uses for `d` on a device with `num_sms` SMs. Host only: needs no device, reads
 * no pointer of `d` (only whether it is NULL), honours resr_set_conv_pair_policy. resr_conv3x3 plans through this very
 * function, so the report cannot drift from what runs. Returns RESR_E_INVALID (and fills nothing) for every
 * descriptor resr_conv3x3 would reject, including one whose weights and staging do not fit in shared memory. */
typedef struct resr_conv_plan {
    int pair;           /* 1: CTA-pair kernel (tcgen05 cta_group::2), 0: single-CTA kernel */
    int nout;           /* accumulator channels per output row and launch slice: 64 (pairs only), 32 or 16 */
    int nslices;        /* Cout slices of nout channels (grid y) */
    int bw, bn;         /* one 128-lane tile = bw consecutive columns x bn consecutive images */
    int mode;           /* 0: one activation load per (row, chunk); 1: one per (row, chunk, dx) */
    int nxs, ncg;       /* column segments per image row, column groups */
    int tail_ksteps;    /* K16 steps of the last 64-channel chunk (1, 2 or 4) */
    int nepi, epi_bufs; /* epilogue warp groups, staging buffers per group */
    int nstages;        /* activation pipeline stages */
    int masked;         /* the packed-canvas (vmask) instantiation */
    long long units;    /* work units: (column group, row), or (pair of column groups, row) for pairs */
    long long clusters; /* clusters in the grid (one or two CTAs each) per Cout slice */
} resr_conv_plan;
int resr_conv3x3_plan(const resr_conv_desc* d, int num_sms, resr_conv_plan* plan);

/* Layout helpers used by the generator (exposed for tests): NCHW fp32 -> NHWC 16-bit, channels zero-padded. */
int resr_nchw_to_nhwc16(const float* x, void* out16, int n, int c, int h, int w, int c_pad, int fmt, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Hot path 2 — second-order degradation synthesis (train_realesrnet.py:267-377 and the imgproc.py ops it calls).
 * Images: fp32 NCHW contiguous, device memory. Random decisions and random tensors are INPUTS (drawn by the
 * caller: torch RNG on the host side, or recorded from the reference for parity).
 * filter2d, USM, resize, JPEG and crop return RESR_E_INVALID for an empty or negative size (batch, channels, planes,
 * input or output height / width) before they touch the device.
 * ---------------------------------------------------------------------------------------------------------- */

/* imgproc.filter2d_torch (imgproc.py:1089-1121): reflect-pad k/2, cross-correlation; kernel [kernel_batch,k,k] with
 * kernel_batch == b (one kernel per sample, all channels) or 1 (shared). Even k -> RESR_E_INVALID "Wrong kernel size."
 * (the reference raises ValueError, imgproc.py:1106). */
int resr_filter2d(const float* image, const float* kernel, float* out, int b, int c, int h, int w, int k,
                  int kernel_batch, void* stream);

/* imgproc.USMSharp(radius, sigma).forward(image, weight, threshold) (imgproc.py:1514-1537). Workspace: 3 images. */
size_t resr_usm_workspace_bytes(int b, int c, int h, int w);
int resr_usm_sharp(const float* image, float* out, int b, int c, int h, int w, int radius, int sigma, float weight,
                   float threshold, void* workspace, size_t workspace_bytes, void* stream);
/* Backward of USMSharp.forward: d loss / d image from d loss / d out. train_realesrgan.py:476-478 sharpens the generator
 * output inside the pixel and content losses, so the loss gradient passes through imgproc.py:1526-1535 (autograd of the
 * reflect-padded blur, the clip and the blend; the 0/1 mask and hence the soft mask are constants). The forward
 * quantities are recomputed from `image`. */
size_t resr_usm_backward_workspace_bytes(int b, int c, int h, int w);
int resr_usm_sharp_backward(const float* image, const float* grad_out, float* grad_in, int b, int c, int h, int w,
                            int radius, int sigma, float weight, float threshold, void* workspace,
                            size_t workspace_bytes, void* stream);

/* torch.nn.functional.interpolate(image, size= | scale_factor=, mode=) as called at train_realesrnet.py:288, 326,
 * 349, 366. mode: 0 area, 1 bilinear, 2 bicubic (align_corners=False, no antialias). scale_h/scale_w: the
 * scale_factor when the reference call used scale_factor= (coordinate scale is then 1/scale_factor), or 0 when
 * it used size= (coordinate scale in/out). planes = b*c. */
int resr_resize(const float* image, float* out, int planes, int h_in, int w_in, int h_out, int w_out, int mode,
                double scale_h, double scale_w, void* stream);

/* imgproc.random_add_gaussian_noise_torch(clip, rounds) with its draws fed in (imgproc.py:829-863,
 * 1029-1057): sigma[b], gray[b] in {0,1}, noise_color = randn(b,c,h,w), noise_gray = randn(h,w) or NULL when no
 * sample drew gray. */
int resr_gaussian_noise_apply(const float* image, float* out, const float* sigma, const float* gray,
                              const float* noise_color, const float* noise_gray, int b, int c, int h, int w, int clip,
                              int rounds, void* stream);

/* Poisson branch (imgproc.py:866-916, 1060-1086). */
size_t resr_poisson_workspace_bytes(int b);
/* len(torch.unique(...)) of the u8-quantised colour image / luma per sample (imgproc.py:892, 903), no host sync.
 * counts_gray may be NULL. */
int resr_unique_count_u8(const float* image, int* counts_color, int* counts_gray, int b, int c, int h, int w,
                         void* workspace, size_t workspace_bytes, void* stream);
/* The rate tensors the reference hands to torch.poisson: q*vals [b,3,h,w] and (optional) q_gray*vals_gray [b,1,h,w]. */
int resr_poisson_rates(const float* image, float* rate_color, float* rate_gray, int b, int c, int h, int w,
                       void* workspace, size_t workspace_bytes, void* stream);
/* random_add_poisson_noise_torch(clip, rounds) with its draws fed in: scale[b], gray[b],
 * samples_color = poisson(rate_color), samples_gray = poisson(rate_gray) or NULL. reuse_counts=1: the unique counts of
 * this image are already in `workspace` (left there by resr_poisson_rates on the same image), skip recounting. */
int resr_poisson_noise_apply(const float* image, float* out, const float* scale, const float* gray,
                             const float* samples_color, const float* samples_gray, int b, int c, int h, int w, int clip,
                             int rounds, void* workspace, size_t workspace_bytes, int reuse_counts, void* stream);

/* Production variant of resr_gaussian_noise_apply: the normal deviates are drawn inside the kernel (Philox4x32-10; the gray
 * field is ONE H x W field shared by the batch, imgproc.py:853-856). gray == NULL: no sample uses the gray field.
 * `call_state`: two persistent, zero-initialised device u64 owned by the caller ([0] call counter, [1] scratch): every
 * call / CUDA-graph replay draws fresh noise for a fixed seed. */
int resr_gaussian_noise_sampled(const float* image, float* out, const float* sigma, const float* gray, int b, int c, int h, int w,
                                int clip, int rounds, unsigned long long seed, unsigned long long* call_state, void* stream);

/* Production variant of resr_poisson_noise_apply: the Poisson draws are made inside the kernel (Philox4x32-10 counter RNG,
 * one subsequence per draw; exact samplers: Hoermann's PTRS rejection for rate >= 10, multiplication method below), so no
 * rate tensors and no sampler launches are needed: memset + presence bitmap + one fused kernel. gray == NULL: no sample uses
 * the luma branch (imgproc.py:886). `call_counter`: one persistent device u64 owned by the caller; every call (and every
 * replay of a captured CUDA graph) increments it and draws from a fresh Philox offset. */
int resr_poisson_noise_sampled(const float* image, float* out, const float* scale, const float* gray, int b, int c, int h, int w,
                               int clip, int rounds, unsigned long long seed, unsigned long long* call_counter,
                               void* workspace, size_t workspace_bytes, void* stream);

/* imgproc.DiffJPEG(differentiable=False).forward(image, quality[b]) (imgproc.py:1462-1494). quality is NOT modified;
 * the factor the reference writes back in place (imgproc.py:1478-1479) is returned in factor_out[b] (may be NULL).
 * clamp_input=1 fuses the torch.clamp(out, 0, 1) of train_realesrnet.py:308. q_y/q_cb/q_cr (all or none): dump of the
 * quantised coefficients, [b, (hp/8)*(wp/8), 8, 8] and [b, (hp/16)*(wp/16), 8, 8] with hp, wp = h, w rounded up to 16. */
int resr_jpeg(const float* image, float* out, const float* quality, float* factor_out, int b, int h, int w,
              int clamp_input, float* q_y, float* q_cb, float* q_cr, void* stream);

/* Training-image augmentation of the dataset (dataset.py:66-79) for a whole batch: random_rotate by 0 / 90 / 180 / 270 degrees
 * about (w//2, h//2) (imgproc.py:1937-1963, cv2.warpAffine: exact pixel copies, zeros where the canvas has no source),
 * random horizontal / vertical flip (imgproc.py:1966-2001), BGR -> RGB, image_to_tensor (HWC -> CHW) and the / 255 of
 * dataset.py:67. images_bgr_hwc: decoded u8 images [b,h,w,3]; out_rgb_nchw: fp32 [b,3,h,w]; ops[b] (device):
 * bits 0-1 = angle index (0, 90, 180, 270), bit 2 = horizontal flip, bit 3 = vertical flip -- the caller's draws
 * (imgproc.draw_augment_ops keeps the reference's RNG order). Bit-exact against the reference functions. */
int resr_augment_batch_u8(const unsigned char* images_bgr_hwc, float* out_rgb_nchw, const int* ops, int b, int h, int w,
                          void* stream);

/* Paired crop (imgproc.random_crop, imgproc.py:1894-1934) and the u8-grid rounding of train_realesrnet.py:374. */
int resr_crop(const float* image, float* out, int planes, int h_in, int w_in, int top, int left, int h_out, int w_out,
              int round_to_u8, void* stream);

/* Blur-kernel synthesis in float64 on the device (imgproc.py:72-90, 170-327, 576-603). One entry per kernel; the
 * random draws (type, size, sigmas, angle, beta, cutoff) are made by the caller in the reference's RNG order
 * (dataset.py:81-141). type: 0 Gaussian, 1 generalized Gaussian, 2 plateau, 3 sinc (Bessel J1), 4 delta.
 * Every kernel is normalised to sum 1 and written centred, zero-padded to pad x pad (pad = 0: no padding, all
 * sizes must then be equal). out_f64 / out_f32: [count, P, P], either may be NULL. params_host is HOST memory. */
typedef struct resr_kernel_params {
    int type, kernel_size, isotropic, reserved;
    double sigma_x, sigma_y, theta, beta, cutoff;
} resr_kernel_params;
int resr_synthesize_kernels(const resr_kernel_params* params_host, int count, int pad, double* out_f64, float* out_f32,
                            void* stream);
/* The same synthesis from parameters that already live on the device (kmax = largest kernel_size among them, <= pad). */
int resr_synthesize_kernels_device(const resr_kernel_params* params_dev, int count, int kmax, int pad, double* out_f64,
                                   float* out_f32, void* stream);
/* Device-side replacement of the per-sample host loop of dataset.py:81-141: draws, for every sample of a batch, the
 * parameters of kernel1, kernel2 and the final sinc / delta kernel (params_dev: [batch][3]) with the reference's
 * distributions (config.py:20-39) from a Philox counter RNG; *call_state (device u64, may be NULL) advances per call so
 * that a fixed seed yields fresh draws on every call / graph replay. Feed the result to resr_synthesize_kernels_device. */
typedef struct resr_kernel_draw_config {
    int n_sizes, sizes[16];           /* gaussian_kernel_range */
    int sinc_size_split;              /* sizes below it draw cutoff in [pi/3, pi], the others in [pi/5, pi] (dataset.py:85-88: 13) */
    int final_size;                   /* sinc_kernel_size: size of the delta kernel */
    double sinc_prob1, sinc_prob2, sinc_prob3;
    double prob1[6], prob2[6];        /* gaussian_kernel_probability1/2 over (iso, aniso, generalized iso/aniso, plateau iso/aniso) */
    double sigma_range1[2], sigma_range2[2];
    double gen_beta_range1[2], gen_beta_range2[2], plateau_beta_range1[2], plateau_beta_range2[2];
} resr_kernel_draw_config;
int resr_draw_degradation_kernel_params(const resr_kernel_draw_config* cfg, int batch, unsigned long long seed,
                                        unsigned long long* call_state, resr_kernel_params* params_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Hot path 1, training: forward that keeps activations, fused L1 loss, full backward (SURVEY.md row a5).
 * Replaces `sr = model(lr); loss = L1(sr, hr); loss.backward()` (train_realesrnet.py:383-388) for the generator.
 * grads_flat: fp32 [resr_generator_num_params()] in state_dict order (layout of resr_generator_tensor_span); every
 * element is overwritten. The flat parameter vector given to resr_generator_load_params must stay alive (the
 * transposed weight packs of the data-gradient convolutions are built from it on the first backward).
 * Two recipes (resr_generator_set_precision): 0 = fp16 activations + bf16 gradients; 1 = bf16 activations and gradients
 * with an fp32 residual stream. Both take their weight gradients from the NHWC buffers (csrc/wgrad_mn.cu; the fp16
 * recipe's activations pass through a bf16 copy first) and have no shape rule beyond n, h, w >= 1. Bias and weight
 * gradients are summed in a fixed order: identical steps give bit-identical grads_flat.
 * ---------------------------------------------------------------------------------------------------------- */
size_t resr_generator_train_workspace_bytes(int n, int h, int w);
int resr_generator_forward_train(resr_generator_t* g, const float* x, float* y, int n, int h, int w, void* workspace,
                                 size_t workspace_bytes, void* stream);
/* loss = mean |y - hr| (nn.L1Loss, train_realesrnet.py:190-194), written to loss_out (device float, may be NULL),
 * followed by the backward pass of the forward_train call that last used `workspace`. hr: fp32 NCHW [n,3,4h,4w]. */
int resr_generator_backward_l1(resr_generator_t* g, const float* hr, float* grads_flat, float* loss_out, int n, int h,
                               int w, void* workspace, size_t workspace_bytes, void* stream);
/* forward_train + L1 + backward in one call. The first call with a given argument set runs eagerly and captures the
 * launch sequence (~2,400 kernels) into a CUDA graph; later calls with the SAME pointers and shape replay it, so keep
 * x / hr / y / grads_flat / loss_out in persistent buffers. resr_generator_step_is_graph() tells whether a graph is live. */
int resr_generator_train_step_l1(resr_generator_t* g, const float* x, const float* hr, float* y, float* grads_flat,
                                 float* loss_out, int n, int h, int w, void* workspace, size_t workspace_bytes,
                                 void* stream);
int resr_generator_step_is_graph(resr_generator_t* g);
/* Data-parallel training (SURVEY.md §8e; the reference trains on one GPU): the backward finishes gradients from the END of
 * the flat vector towards its front (tail, trunk.22 ... trunk.0, conv1), so the vector is cut into 4 contiguous buckets that
 * complete in the order 3, 2, 1, 0 of their position: bucket k = [offsets[k], offsets[k+1]) (returns the bucket count, 4).
 * resr_generator_wait_grad_bucket makes `stream` wait until bucket k of the most recently enqueued training step is complete
 * (k = 3 finishes first; k = 0 finishes with the step itself: no wait is inserted), so that an all-reduce of that slice can run under the
 * rest of the backward. Works for the eager step and for the CUDA-graph replay (external event-record nodes). */
int resr_generator_grad_buckets(size_t* offsets, int max_entries);
int resr_generator_wait_grad_bucket(resr_generator_t* g, int bucket, void* stream);
/* Backward from an upstream gradient dL/dy (fp32 NCHW [n,3,4h,4w]); the clamp of model.py:270 is applied inside. */
int resr_generator_backward(resr_generator_t* g, const float* dy, float* grads_flat, int n, int h, int w, void* workspace,
                            size_t workspace_bytes, void* stream);

/* Weight / bias gradient of one 3x3 convolution (test / building block) straight from NHWC bf16 operands: both operands
 * are MN-major tcgen05 operands, pixel shifts are descriptor / TMA-coordinate shifts (csrc/wgrad_mn.cu).
 * x_bf16: [n,h,w,x_cstride] (first cin channels, cin <= 256); dy_bf16: [n,h,w,dy_cstride] (first cout channels,
 * cout <= 192; when cout is not a multiple of 8 the channels up to the next multiple of 8 must be zero). dw: OIHW fp32
 * [cout,cin,3,3]; db: [cout] or NULL. No restriction on w. This is the kernel both training recipes use for every layer
 * (autograd of model.py:75-79, 87-98). */
size_t resr_conv3x3_wgrad_nhwc_workspace_bytes(void);
int resr_conv3x3_wgrad_nhwc(const void* x_bf16, int x_cstride, const void* dy_bf16, int dy_cstride, int n, int h, int w,
                            int cin, int cout, float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * NIQE on the device (image_quality_assessment.py:886-998 `_niqe_torch`, class NIQE :1001-1033): the per-block feature
 * extraction. image_rgb: fp32 NCHW [b,3,h,w] in [0,1]; features: float64 [b, nblocks, 36] (18 AGGD features of the MSCN
 * coefficients per block at two scales; block order row-major -- the reference's column-first order only permutes the
 * rows of a matrix whose mean and covariance are taken). crop_border pixels are dropped on every side, then the image
 * is cropped to whole block x block tiles (block must be even: the second scale uses block / 2 on the half-size image).
 * The 36-dimensional Gaussian fit against the pristine statistics (nanmean / nancov / pinv, :879-884) is a 36 x 36
 * problem left to the caller (resr_b200/iqa.py). */
int resr_niqe_num_blocks(int h, int w, int crop_border, int block);
size_t resr_niqe_workspace_bytes(int b, int h, int w, int crop_border, int block);
int resr_niqe_features(const float* image_rgb, double* features, int b, int h, int w, int crop_border, int block,
                       void* workspace, size_t workspace_bytes, void* stream);
/* A list of differently sized images in one call: the reference's test.py / validate() score one image at a time, and
 * benchmark sets differ in size. images[i] is fp32 NCHW [1,3,hs[i],ws[i]] in device memory; the pointer and size ARRAYS are
 * host memory. features: float64 [total_blocks, 36]; image i's blocks are rows [block_offsets[i], block_offsets[i+1]) in
 * the row-major order of resr_niqe_features, and each image's rows are bit-identical to its own resr_niqe_features call.
 * block_offsets (host, count + 1 entries) is filled by the call. crop_border and block apply to every image; an image
 * without a block after cropping, an empty or negative size or a bad block returns RESR_E_INVALID before any device work
 * (the message names the image). resr_niqe_many_workspace_bytes returns 0 for any such argument. */
size_t resr_niqe_many_workspace_bytes(const int* hs, const int* ws, int count, int crop_border, int block);
int resr_niqe_features_many(const float* const* images, const int* hs, const int* ws, int count, int crop_border, int block,
                            double* features, int* block_offsets, void* workspace, size_t workspace_bytes, void* stream);

/* ---- the whole degradation block in one call (train_realesrnet.py:267-377 == train_realesrgan.py:347-457) ---------------
 * A POD plan holds every host decision of one execution of the block; per-sample parameters and host-fed random draws
 * are DEVICE pointers owned by the caller. Stage order, kernels and arithmetic are those of the op-level entry points. */
typedef struct resr_resize_spec {
    int mode;        /* 0 area, 1 bilinear, 2 bicubic (random.choice, train:279, 317, 349) */
    int out_h, out_w;/* used when scale <= 0: F.interpolate(size=...) (coordinate scale in/out) */
    double scale;    /* > 0: F.interpolate(scale_factor=scale): out = floor(in * scale), coordinate scale 1/scale (train:288) */
} resr_resize_spec;
typedef struct resr_noise_spec {
    int type;                 /* 0 Gaussian (imgproc.py:1029-1057), 1 Poisson (imgproc.py:1060-1086) */
    const float* param;       /* [B] sigma (Gaussian) or scale (Poisson) */
    const float* gray;        /* [B] gray flags */
    int gray_any;             /* host-side: any gray flag set (imgproc.py:852, 884) */
    const float* draws_color; /* host-fed draws: normal field / Poisson samples [B,3,h,w]; NULL: drawn inside the kernel */
    const float* draws_gray;  /* normal field [h,w] / Poisson samples [B,1,h,w], read only when gray_any */
    unsigned long long seed;  /* Philox seed of the in-kernel samplers */
} resr_noise_spec;
typedef struct resr_degrade_plan {
    int batch, hr_h, hr_w;
    int usm_radius, usm_sigma;            /* 50, 0 (train:232) */
    float usm_weight, usm_threshold;      /* 0.5, 10 (imgproc.py:1525) */
    int blur1, blur2, final_order;        /* blur flags (train:275, 313); 0: resize-sinc-jpeg, 1: jpeg-resize-sinc (train:347) */
    int kernel_size, sinc_batched;        /* 21; 1 when sinc_kernel is [B,k,k], 0 when [1,k,k] */
    resr_resize_spec resize1, resize2, resize3;
    resr_noise_spec noise1, noise2;
    const float* jpeg1_quality;           /* [B] (train:307, 356/361); not modified (the factor goes to the workspace) */
    const float* jpeg2_quality;
    int crop_top, crop_left, image_size, upscale;   /* HR crop window (imgproc.py:1894-1934), LR offsets = HR offsets / upscale */
    unsigned long long* rng_state;        /* 8 persistent zero-initialised device u64 (in-kernel samplers), or NULL */
} resr_degrade_plan;
size_t resr_degrade_workspace_bytes(const resr_degrade_plan* plan);
/* hr: [B,3,hr_h,hr_w]; kernel1 / kernel2: [B,k,k]; sinc_kernel: [B or 1,k,k]; lr_out: [B,3,image_size/upscale,..] on
 * the u8 grid; hr_out: [B,3,image_size,image_size] (the unsharpened target, train:377). */
int resr_degrade_batch(const resr_degrade_plan* plan, const float* hr, const float* kernel1, const float* kernel2,
                       const float* sinc_kernel, float* lr_out, float* hr_out, void* workspace, size_t workspace_bytes,
                       void* stream);

/* ---- optimizer side of the training step (SURVEY.md §8 row f1) ------------------------------------------------------
 * One fused elementwise pass over flat fp32 vectors of n elements (resr_generator_num_params for the whole generator):
 *   torch.optim.Adam(lr, betas=(beta1, beta2), eps) step number `step` (1-based; no weight decay, no amsgrad), arithmetic
 *   order of torch's single-tensor implementation (train_realesrnet.py:197-200, 390), on grads * grad_scale
 *   (grad_scale = 1 / loss_scale replaces GradScaler's unscale_, train_realesrnet.py:388-391), then
 *   EMA.update(): shadow = (1 - ema_decay) * param + ema_decay * shadow (model.py:42-49); ema_shadow may be NULL.
 * All pointers are device pointers; params / exp_avg / exp_avg_sq / ema_shadow are updated in place. */
int resr_adam_ema_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* ema_shadow, size_t n,
                       float lr, float beta1, float beta2, float eps, long long step, float ema_decay, float grad_scale,
                       void* stream);

/* ---- VGG19 content loss of the RealESRGAN generator step (ContentLoss, model.py:278-335; train_realesrgan.py:473-487) -----
 * losses[k] = mean |F_k(Normalize(sr)) - F_k(Normalize(gt))| for each requested node k, F_k = vgg19().features up to
 * features.<node> as create_feature_extractor returns it: the conv output, rewritten by the in-place ReLU that follows it
 * unless it is the deepest requested node. Weights are frozen; the backward gives d/d sr only.
 *
 * resr_vgg_create takes the node list as features indices (host; any of 0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28,
 * 30, 32, 34, no repeats; losses come out in this order) and Normalize's mean / std (host, 3 floats each). It allocates
 * nothing on the device. resr_vgg_load_params packs the 16 convolutions from one flat fp32 device vector of
 * resr_vgg_num_params() (20,024,384) values: features.{0,2,...,34}.weight then .bias, torchvision order; it needs an sm_100a
 * device (RESR_E_CUDA otherwise) and binds the handle to the current device. Convolutions past the deepest node never run.
 *
 * resr_vgg_forward: sr, gt [n,3,h,w] fp32 NCHW; losses: device fp32 [count]. SR and GT run as one 2n batch; the workspace
 * (resr_vgg_workspace_bytes, 1024-byte aligned) keeps the activations the backward needs. The sums are fp64 in a fixed
 * order: two identical calls give identical bits. h and w must leave at least one pixel at the deepest node (2x2 / stride 2
 * floor pooling); resr_vgg_workspace_bytes returns 0 for a shape that does not.
 * resr_vgg_backward: grad_losses (device fp32 [count], read on the device: no host sync) -> grad_sr fp32 NCHW [n,3,h,w].
 * It needs the workspace and shape of the handle's last forward; anything else is RESR_E_INVALID.
 * Every argument is checked on the host before any device work; a bad one returns RESR_E_INVALID. */
typedef struct resr_vgg resr_vgg_t;
size_t resr_vgg_num_params(void);
int resr_vgg_create(resr_vgg_t** out, const int* features_host, int count, const float* mean_host, const float* std_host);
void resr_vgg_destroy(resr_vgg_t* v);
int resr_vgg_load_params(resr_vgg_t* v, const float* flat_params, void* stream);
size_t resr_vgg_workspace_bytes(const resr_vgg_t* v, int n, int h, int w);
int resr_vgg_forward(resr_vgg_t* v, const float* sr, const float* gt, float* losses, int n, int h, int w, void* workspace,
                     size_t workspace_bytes, void* stream);
int resr_vgg_backward(resr_vgg_t* v, const float* grad_losses, float* grad_sr, int n, int h, int w, void* workspace,
                      size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RESR_H_ */
