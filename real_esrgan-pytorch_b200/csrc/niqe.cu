// NIQE feature extraction on the device (SURVEY.md §8 f4; reference /root/reference/image_quality_assessment.py:886-998
// `_niqe_torch` and the helpers it calls, imgproc.py:1815-1840 for the Y channel). Everything after the Y channel is
// float64, as in the reference. Stages for each of the two scales (block = 96, then 48 on the half-size image):
//   Y * 255 rounded (fp32 arithmetic like the reference, then float64)
//   MSCN coefficients: 7 x 7 Gaussian (sigma 7/6, replicate padding) local mean / deviation, (y - mu) / (sigma + 1)
//   per block and per map (the block itself + its products with four circularly shifted copies, torch.roll): six sums
//   AGGD fit per (block, map): shape parameter by table search over 0.2 : 0.001 : 10, left / right scale, mean -> 18 features
//   MATLAB-style antialiased bicubic x0.5 (ten taps, one weight set, symmetric padding) for the second scale
// The 36-dimensional Gaussian fit over the blocks (nanmean, covariance, pseudo-inverse: a 36 x 36 problem) is left to the
// caller (resr_b200/iqa.py does it with torch.linalg on the device).
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>

#include "../../include/resr.h"
#include "device_state.h"
#include "errors.h"

namespace resr {

static constexpr int kGamN = 9801;   // torch.arange(0.2, 10.001, 0.001)
__constant__ double c_niqe_win[49];
__constant__ double c_niqe_rw[10];   // resize weights

// One image of a call. Every image is cropped to hh x ww = whole blocks after `crop_border`, so hh and ww are even and
// each image's plane size is a multiple of 4: its arena offset at a level whose rows and / or columns are halved is
// `off >> shift` (shift 0: full size, 1: rows halved, 2: both halved), and the planes of all images stay packed.
struct NiqeImage {
    const float* src;   // fp32 NCHW [1, 3, H, W]
    int H, W, hh, ww;
    size_t off;         // first element of this image's full-size plane in the packed fp64 arenas
    int nbw, row0;      // blocks per row; first block (= feature row) of this image
};

// Image of arena element i at `shift`: the last image whose plane starts at or before i (planes are never empty).
__device__ __forceinline__ int niqe_image_of_pixel(const NiqeImage* __restrict__ t, int count, size_t i, int shift) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((t[mid].off >> shift) <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ int niqe_image_of_block(const NiqeImage* __restrict__ t, int count, int blk) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (t[mid].row0 <= blk) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Y channel of rgb2ycbcr_torch(only_use_y_channel=True) in fp32, * 255, round (half to even), as float64; the crop of
// `crop_border` pixels and the crop to whole blocks are folded into the indexing.
__global__ void __launch_bounds__(256) niqe_y_kernel(const NiqeImage* __restrict__ tab, int count, double* __restrict__ y, size_t total,
                                                     int border) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const NiqeImage& im = tab[niqe_image_of_pixel(tab, count, i, 0)];
        const size_t li = i - im.off, plane = static_cast<size_t>(im.H) * im.W;
        const int xx = static_cast<int>(li % im.ww), yy = static_cast<int>(li / im.ww);
        const float* p = im.src + static_cast<size_t>(yy + border) * im.W + xx + border;
        float v = __fadd_rn(__fadd_rn(__fmul_rn(p[0], 65.481f), __fmul_rn(p[plane], 128.553f)), __fmul_rn(p[2 * plane], 24.966f));
        v = __fdiv_rn(__fadd_rn(v, 16.0f), 255.0f);            // imgproc.py:1830, 1838
        y[i] = static_cast<double>(rintf(__fmul_rn(v, 255.0f)));   // image_quality_assessment.py:984-985
    }
}

// structdis = (y - mu) / (sqrt(|E[y^2] - mu^2| + 1e-8) + 1), 7 x 7 window, replicate padding (image_quality_assessment.py:869-873).
// lvl 0: full-size planes, 1: both sides halved (second scale).
__global__ void __launch_bounds__(256) niqe_mscn_kernel(const NiqeImage* __restrict__ tab, int count, const double* __restrict__ y,
                                                        double* __restrict__ sd, size_t total, int lvl) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const NiqeImage& im = tab[niqe_image_of_pixel(tab, count, i, 2 * lvl)];
        const size_t base = im.off >> (2 * lvl);
        const int h = im.hh >> lvl, w = im.ww >> lvl;
        const int xx = static_cast<int>((i - base) % w), yy = static_cast<int>((i - base) / w);
        const double* img = y + base;
        double mu = 0.0, e2 = 0.0;
        for (int dy = 0; dy < 7; ++dy) {
            const int sy = min(max(yy + dy - 3, 0), h - 1);
            for (int dx = 0; dx < 7; ++dx) {
                const int sx = min(max(xx + dx - 3, 0), w - 1);
                const double v = img[static_cast<size_t>(sy) * w + sx], k = c_niqe_win[dy * 7 + dx];
                mu += k * v;
                e2 += k * (v * v);
            }
        }
        const double sigma = sqrt(fabs(e2 - mu * mu) + 1e-8);
        sd[i] = (img[static_cast<size_t>(yy) * w + xx] - mu) / (sigma + 1.0);
    }
}

// One CUDA block per image block of s x s MSCN coefficients (s = block >> lvl). Map m = 0: the block; m = 1..4:
// block * roll(block, shift_m) with shifts (0,1), (1,0), (1,1), (1,-1) (torch.roll: circular inside the block,
// image_quality_assessment.py:851-853). stats[(block * 5 + m) * 6 + {count<0, count>0, sum v^2 over v<0, sum v^2 over v>0,
// sum |v|, sum v^2}]; `block` counts over all images, in feature-row order.
__global__ void __launch_bounds__(256) niqe_block_stats_kernel(const NiqeImage* __restrict__ tab, int count, const double* __restrict__ sd,
                                                               double* __restrict__ stats, int s, int lvl) {
    __shared__ double red[8][30];
    const int blk = blockIdx.x;                       // (image, block row, block column)
    const NiqeImage& im = tab[niqe_image_of_block(tab, count, blk)];
    const int w = im.ww >> lvl, local = blk - im.row0;
    const int bw_i = local % im.nbw, bh_i = local / im.nbw;
    const double* base = sd + (im.off >> (2 * lvl)) + static_cast<size_t>(bh_i) * s * w + static_cast<size_t>(bw_i) * s;
    double acc[30];
#pragma unroll
    for (int i = 0; i < 30; ++i) acc[i] = 0.0;
    const int sy[5] = {0, 0, 1, 1, 1}, sx[5] = {0, 1, 0, 1, -1};
    for (int p = threadIdx.x; p < s * s; p += blockDim.x) {
        const int i = p / s, j = p % s;
        const double v0 = base[static_cast<size_t>(i) * w + j];
#pragma unroll
        for (int m = 0; m < 5; ++m) {
            double v = v0;
            if (m > 0) {
                const int ii = (i - sy[m] + s) % s, jj = (j - sx[m] + s) % s;
                v = v0 * base[static_cast<size_t>(ii) * w + jj];
            }
            const double v2 = v * v;
            if (v < 0) { acc[m * 6 + 0] += 1.0; acc[m * 6 + 2] += v2; }
            if (v > 0) { acc[m * 6 + 1] += 1.0; acc[m * 6 + 3] += v2; }
            acc[m * 6 + 4] += fabs(v);
            acc[m * 6 + 5] += v2;
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 30; ++i) {
        double v = acc[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 30) {
        double v = 0.0;
        for (int k = 0; k < 8; ++k) v += red[k][threadIdx.x];
        stats[static_cast<size_t>(blk) * 30 + threadIdx.x] = v;
    }
}

// AGGD fit of one (block, map) (image_quality_assessment.py:790-836 with get_sigma=True) and its slot of the 18 features
// (:845-858): one CUDA block; the table search is a parallel arg-min (first minimum wins, like torch.argmin). Blocks
// count over all images of the call, so block `blk` writes feature row `blk` and needs no image table.
__global__ void __launch_bounds__(256) niqe_aggd_kernel(const double* __restrict__ stats, const double* __restrict__ r_gam,
                                                        double* __restrict__ feat, int s, int col0) {
    __shared__ double s_val[256];
    __shared__ int s_idx[256];
    const int bm = blockIdx.x, blk = bm / 5, m = bm % 5;
    const double* st = stats + static_cast<size_t>(bm) * 6;
    const double n = static_cast<double>(s) * s;
    const double left_std = sqrt(st[2] / (st[0] + 1e-8)), right_std = sqrt(st[3] / (st[1] + 1e-8));
    const double gamma_hat = left_std / right_std;
    const double mean_abs = st[4] / n;
    const double rhat = mean_abs * mean_abs / (st[5] / n);
    const double g2 = gamma_hat * gamma_hat;
    const double rhat_norm = (rhat * (g2 * gamma_hat + 1.0) * (gamma_hat + 1.0)) / ((g2 + 1.0) * (g2 + 1.0));
    double best = INFINITY;
    int bi = 0x7fffffff;
    for (int i = threadIdx.x; i < kGamN; i += blockDim.x) {
        const double d = fabs(r_gam[i] - rhat_norm);
        if (d < best) { best = d; bi = i; }   // i increases: the first minimum of this thread's entries is kept
    }
    s_val[threadIdx.x] = best; s_idx[threadIdx.x] = bi;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (static_cast<int>(threadIdx.x) < o) {
            const double v = s_val[threadIdx.x + o];
            const int ix = s_idx[threadIdx.x + o];
            if (v < s_val[threadIdx.x] || (v == s_val[threadIdx.x] && ix < s_idx[threadIdx.x])) { s_val[threadIdx.x] = v; s_idx[threadIdx.x] = ix; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // a NaN distance (a constant block: 0 / 0) loses every comparison: torch.argmin returns the first NaN's index (0)
        const int pos = s_idx[0] == 0x7fffffff ? 0 : s_idx[0];
        const double alpha = 0.2 + 0.001 * pos;
        const double sc = sqrt(exp(lgamma(1.0 / alpha) - lgamma(3.0 / alpha)));
        const double lb = left_std * sc, rb = right_std * sc;
        double* f = feat + static_cast<size_t>(blk) * 36 + col0;
        if (m == 0) {
            f[0] = alpha; f[1] = (lb + rb) / 2.0;
        } else {
            const double mean = (rb - lb) * exp(lgamma(2.0 / alpha) - lgamma(1.0 / alpha));
            double* q = f + 2 + (m - 1) * 4;
            q[0] = alpha; q[1] = mean; q[2] = lb; q[3] = rb;
        }
    }
}

// MATLAB imresize(x / 255, 0.5) * 255 with antialiasing along one axis (image_quality_assessment.py:517-585 for scale 0.5:
// ten taps, pos = 2 i + 0.5, base = 2 i - 4, one weight set, symmetric padding of four: the edge element is used twice).
// axis 0: rows (hh x ww -> hh / 2 x ww), axis 1: columns (hh / 2 x ww -> hh / 2 x ww / 2); `total` counts output elements.
// div_in / scale_out fold the / 255 and * 255 of :877-878 into the passes.
__global__ void __launch_bounds__(256) niqe_resize_half_kernel(const NiqeImage* __restrict__ tab, int count, const double* __restrict__ in,
                                                               double* __restrict__ out, size_t total, int axis, double div_in,
                                                               double scale_out) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const NiqeImage& im = tab[niqe_image_of_pixel(tab, count, i, axis + 1)];
        const size_t off = im.off;
        const int h = im.hh >> axis, w = im.ww;
        const int wo = w >> axis;
        const size_t li = i - (off >> (axis + 1));
        const int xx = static_cast<int>(li % wo), yy = static_cast<int>(li / wo);
        const double* img = in + (off >> axis);
        const int n = axis == 0 ? h : w, o = axis == 0 ? yy : xx;
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            int idx = 2 * o - 4 + k;
            idx = idx < 0 ? -idx - 1 : (idx >= n ? 2 * n - idx - 1 : idx);
            const double v = axis == 0 ? img[static_cast<size_t>(idx) * w + xx] : img[static_cast<size_t>(yy) * w + idx];
            acc += (v / div_in) * c_niqe_rw[k];
        }
        out[i] = acc * scale_out;
    }
}

static int grid_of(size_t total) {
    size_t g = (total + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    return static_cast<int>(g < 1 ? 1 : g);
}

static double cubic_w(double x) {   // image_quality_assessment.py:388-404, a = -0.5
    const double a = -0.5, ax = fabs(x), ax2 = ax * ax, ax3 = ax * ax2;
    if (ax <= 1) return (a + 2) * ax3 - (a + 3) * ax2 + 1;
    if (ax <= 2) return a * ax3 - 5 * a * ax2 + 8 * a * ax - 4 * a;
    return 0.0;
}

struct NiqeTables { bool ready = false; double* r_gam = nullptr; };

static int niqe_tables(double** r_gam_out, cudaStream_t s) {
    static PerDevice<NiqeTables> tabs;
    NiqeTables& t = tabs.cur();
    if (!t.ready) {
        // Gaussian window: fspecial('gaussian', 7, 7/6) in double, kept as float32 by the reference (:215-240)
        double win[49], sum = 0.0, mx = 0.0;
        const double sigma = 7.0 / 6.0;
        for (int i = 0; i < 49; ++i) {
            const double yy = i / 7 - 3.0, xx = i % 7 - 3.0;
            win[i] = exp(-(xx * xx + yy * yy) / (2.0 * sigma * sigma));
            mx = fmax(mx, win[i]);
        }
        for (int i = 0; i < 49; ++i) { if (win[i] < 2.220446049250313e-16 * mx) win[i] = 0.0; sum += win[i]; }
        for (int i = 0; i < 49; ++i) win[i] = static_cast<double>(static_cast<float>(win[i] / sum));
        double rw[10], rs = 0.0;
        for (int k = 0; k < 10; ++k) { rw[k] = cubic_w((4.5 - k) * 0.5); rs += rw[k]; }
        for (int k = 0; k < 10; ++k) rw[k] /= rs;
        double* host = new double[kGamN];
        for (int i = 0; i < kGamN; ++i) {
            const double a = 0.2 + 0.001 * i;
            host[i] = exp(2.0 * lgamma(2.0 / a) - (lgamma(1.0 / a) + lgamma(3.0 / a)));
        }
        cudaError_t e = cudaMemcpyToSymbol(c_niqe_win, win, sizeof(win));
        if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_niqe_rw, rw, sizeof(rw));
        if (e == cudaSuccess) e = cudaMalloc(&t.r_gam, kGamN * sizeof(double));
        if (e == cudaSuccess) e = cudaMemcpyAsync(t.r_gam, host, kGamN * sizeof(double), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        delete[] host;
        if (e != cudaSuccess) return set_error(RESR_E_CUDA, "NIQE tables: %s", cudaGetErrorString(e));
        t.ready = true;
    }
    *r_gam_out = t.r_gam;
    return RESR_OK;
}

// Workspace of one call: the packed fp64 arenas (Y, MSCN, the row-halved resize pass; `pixels` full-size elements each,
// the second scale reuses their first quarter), the 30 block sums per block, then the image table.
struct NiqeLayout {
    size_t pixels = 0, stats = 0, table = 0, total = 0;
    int blocks = 0;
};

// Table and layout of `count` images of sizes hs[i] x ws[i] (src pointers are filled by the caller). Rejects every bad
// argument before any device work; an image without a block after cropping is named by its index.
static int niqe_plan(const int* hs, const int* ws, int count, int crop_border, int block, std::vector<NiqeImage>& tab, NiqeLayout& L) {
    if (!hs || !ws) return set_error(RESR_E_INVALID, "null argument");
    if (count <= 0) return set_error(RESR_E_INVALID, "NIQE: %d images", count);
    if (block <= 0 || (block & 1) || crop_border < 0)
        return set_error(RESR_E_INVALID, "NIQE: block %d must be positive and even, crop_border %d non-negative", block, crop_border);
    tab.assign(count, NiqeImage{});
    size_t off = 0;
    long long row = 0;
    for (int i = 0; i < count; ++i) {
        if (hs[i] <= 0 || ws[i] <= 0) return set_error(RESR_E_INVALID, "NIQE: image %d has size %d x %d", i, hs[i], ws[i]);
        if (resr_niqe_num_blocks(hs[i], ws[i], crop_border, block) == 0)
            return set_error(RESR_E_INVALID, "NIQE: image %d (%d x %d) is smaller than one %d x %d block after cropping %d pixels", i, hs[i],
                             ws[i], block, block, crop_border);
        const int nbh = (hs[i] - 2 * crop_border) / block, nbw = (ws[i] - 2 * crop_border) / block;
        tab[i] = NiqeImage{nullptr, hs[i], ws[i], nbh * block, nbw * block, off, nbw, static_cast<int>(row)};
        off += static_cast<size_t>(nbh * block) * (nbw * block);
        row += static_cast<long long>(nbh) * nbw;
        if (row > 0x7fffffff / 5) return set_error(RESR_E_INVALID, "NIQE: more than %d blocks in one call", 0x7fffffff / 5);
    }
    L.pixels = off;
    L.blocks = static_cast<int>(row);
    L.stats = 3 * off * sizeof(double);
    L.table = (L.stats + static_cast<size_t>(L.blocks) * 30 * sizeof(double) + 255) & ~static_cast<size_t>(255);
    L.total = L.table + static_cast<size_t>(count) * sizeof(NiqeImage) + 1024;   // + the alignment of the workspace to 256 bytes
    return RESR_OK;
}

// Features of every image of `tab` into rows [row0, row0 + blocks) of `features`: five kernels per scale, whatever the
// number of images.
static int niqe_run(const std::vector<NiqeImage>& tab, const NiqeLayout& L, int crop_border, int block, double* features,
                    void* workspace, size_t workspace_bytes, cudaStream_t s) {
    if (workspace_bytes < L.total) return set_error(RESR_E_NOMEM, "NIQE workspace too small (need %zu bytes)", L.total);
    double* r_gam = nullptr;
    const int rc = niqe_tables(&r_gam, s);
    if (rc != RESR_OK) return rc;
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~static_cast<uintptr_t>(255));
    double* y = reinterpret_cast<double*>(base);
    double* sd = y + L.pixels;
    double* tmp = sd + L.pixels;
    double* stats = reinterpret_cast<double*>(base + L.stats);
    NiqeImage* tab_d = reinterpret_cast<NiqeImage*>(base + L.table);
    const int count = static_cast<int>(tab.size());
    // (pageable source: the copy is staged before the call returns, so `tab` may go out of scope)
    if (cudaMemcpyAsync(tab_d, tab.data(), tab.size() * sizeof(NiqeImage), cudaMemcpyHostToDevice, s) != cudaSuccess)
        return set_error(RESR_E_CUDA, "NIQE: table copy failed");
    niqe_y_kernel<<<grid_of(L.pixels), 256, 0, s>>>(tab_d, count, y, L.pixels, crop_border);
    for (int lvl = 0; lvl <= 1; ++lvl) {
        const size_t cur = L.pixels >> (2 * lvl);
        const int bs = block >> lvl;
        niqe_mscn_kernel<<<grid_of(cur), 256, 0, s>>>(tab_d, count, y, sd, cur, lvl);
        niqe_block_stats_kernel<<<L.blocks, 256, 0, s>>>(tab_d, count, sd, stats, bs, lvl);
        niqe_aggd_kernel<<<L.blocks * 5, 256, 0, s>>>(stats, r_gam, features, bs, lvl * 18);
        if (lvl == 0) {   // y = imresize(y / 255, 0.5) * 255: rows first, then columns (:877-878, :517-585)
            niqe_resize_half_kernel<<<grid_of(cur / 2), 256, 0, s>>>(tab_d, count, y, tmp, cur / 2, 0, 255.0, 1.0);
            niqe_resize_half_kernel<<<grid_of(cur / 4), 256, 0, s>>>(tab_d, count, tmp, y, cur / 4, 1, 1.0, 255.0);
        }
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(RESR_E_CUDA, "NIQE launch: %s", cudaGetErrorString(e));
    return RESR_OK;
}

}  // namespace resr

using namespace resr;

extern "C" {

int resr_niqe_num_blocks(int h, int w, int crop_border, int block) {
    if (block <= 0 || (block & 1) || crop_border < 0) return 0;
    const int hh = h - 2 * crop_border, ww = w - 2 * crop_border;
    if (hh < block || ww < block) return 0;
    return (hh / block) * (ww / block);
}

// A batch is a table of b equal images: one implementation for batches and lists.
static int niqe_uniform_plan(int b, int h, int w, int crop_border, int block, std::vector<NiqeImage>& tab, NiqeLayout& L) {
    const std::vector<int> hs(b > 0 ? b : 0, h), ws(b > 0 ? b : 0, w);
    return niqe_plan(hs.data(), ws.data(), b, crop_border, block, tab, L);
}

size_t resr_niqe_workspace_bytes(int b, int h, int w, int crop_border, int block) {
    std::vector<NiqeImage> tab;
    NiqeLayout L;
    return niqe_uniform_plan(b, h, w, crop_border, block, tab, L) == RESR_OK ? L.total : 0;
}

int resr_niqe_features(const float* image_rgb, double* features, int b, int h, int w, int crop_border, int block, void* workspace,
                       size_t workspace_bytes, void* stream) {
    if (!image_rgb || !features || !workspace) return set_error(RESR_E_INVALID, "null argument");
    std::vector<NiqeImage> tab;
    NiqeLayout L;
    const int rc = niqe_uniform_plan(b, h, w, crop_border, block, tab, L);
    if (rc != RESR_OK) return rc;
    for (int i = 0; i < b; ++i) tab[i].src = image_rgb + static_cast<size_t>(i) * 3 * h * w;
    return niqe_run(tab, L, crop_border, block, features, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t resr_niqe_many_workspace_bytes(const int* hs, const int* ws, int count, int crop_border, int block) {
    std::vector<NiqeImage> tab;
    NiqeLayout L;
    return niqe_plan(hs, ws, count, crop_border, block, tab, L) == RESR_OK ? L.total : 0;
}

int resr_niqe_features_many(const float* const* images, const int* hs, const int* ws, int count, int crop_border, int block,
                            double* features, int* block_offsets, void* workspace, size_t workspace_bytes, void* stream) {
    if (!images || !features || !block_offsets || !workspace) return set_error(RESR_E_INVALID, "null argument");
    std::vector<NiqeImage> tab;
    NiqeLayout L;
    const int rc = niqe_plan(hs, ws, count, crop_border, block, tab, L);
    if (rc != RESR_OK) return rc;
    for (int i = 0; i < count; ++i) {
        if (!images[i]) return set_error(RESR_E_INVALID, "NIQE: null image pointer %d", i);
        tab[i].src = images[i];
        block_offsets[i] = tab[i].row0;
    }
    block_offsets[count] = L.blocks;
    return niqe_run(tab, L, crop_border, block, features, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
