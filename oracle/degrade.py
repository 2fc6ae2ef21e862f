"""Oracle for hot path 2: numpy restatement of the reference second-order degradation ops. TEST INFRASTRUCTURE ONLY.

Every function cites the reference lines it follows (/root/reference/imgproc.py, train_realesrnet.py) or, where the
arithmetic lives in a third-party dependency that is not part of /root/reference, the library routine it restates:
  torch 2.11.0 ATen: adaptive_avg_pool2d / upsample_bilinear2d / upsample_bicubic2d (align_corners=False, no antialias),
                     reflection_pad2d, round (half to even)
  torchvision 0.26.0: rgb_to_grayscale
  opencv 4.13.0: getGaussianKernel
Pinned by tests/golden/degrade_*.npz (outputs of the unmodified reference, oracle/make_golden.py).

All images are float32 NCHW numpy arrays. Arithmetic is float32 where the reference's result depends on fp32 rounding
(index math, quantisation factors, u8 rounding); long dot products accumulate in float64 (the reference's own fp32
summation order is library-dependent; the difference is ~1e-7, far inside the 1e-5 contract).
"""
import numpy as np

f32 = np.float32

# --------------------------------------------------------------------------------------------- blur (a8)


def reflect_index(i, n):
    """ATen reflection_pad2d index rule (no edge repeat): -1 -> 1, n -> n-2."""
    i = np.where(i < 0, -i, i)
    return np.where(i >= n, 2 * (n - 1) - i, i)


def filter2d(img, kernel, method="auto"):
    """imgproc.py:1089-1121 filter2d_torch: reflect-pad k//2, cross-correlation (no flip); kernel [B,k,k] is applied
    per sample to all channels, kernel [1,k,k] to every sample. float64 accumulation, one rounding to float32.
    method "direct": tap-by-tap sum (the definition); "fft": the same float64 cross-correlation evaluated with
    scipy.signal.fftconvolve (agrees with "direct" to ~1e-15; tests/test_oracle_cpu.py checks it) so that BASELINE-size
    inputs (16x3x256x256, 51x51 taps) finish in seconds; "auto" picks "fft" for large problems."""
    b, c, h, w = img.shape
    k = kernel.shape[-1]
    if k % 2 != 1:
        raise ValueError("Wrong kernel size.")  # imgproc.py:1106
    r = k // 2
    ys = reflect_index(np.arange(-r, h + r), h)
    xs = reflect_index(np.arange(-r, w + r), w)
    pad = img[:, :, ys][:, :, :, xs].astype(np.float64)
    kern = np.broadcast_to(kernel.astype(np.float64), (b, k, k)) if kernel.shape[0] == 1 else kernel.astype(np.float64)
    if method == "auto":
        method = "fft" if float(b) * c * h * w * k * k > 2e8 else "direct"
    if method == "fft":
        from scipy.signal import fftconvolve
        out = np.empty((b, c, h, w), np.float64)
        for i in range(b):  # correlation == convolution with the flipped kernel
            out[i] = fftconvolve(pad[i], kern[i, ::-1, ::-1][None], mode="valid", axes=(1, 2))
        return out.astype(f32)
    out = np.zeros((b, c, h, w), np.float64)
    for i in range(k):
        for j in range(k):
            if not np.any(kern[:, i, j]):
                continue  # zero-padded border of the 7..21 supports (dataset.py:102-103)
            out += kern[:, i, j][:, None, None, None] * pad[:, :, i:i + h, j:j + w]
    return out.astype(f32)


# --------------------------------------------------------------------------------------------- USM sharpen (a7)


def gaussian_kernel_1d(ksize, sigma=0.0):
    """cv2.getGaussianKernel(ksize, sigma) for ksize > 7 (general formula): sigma<=0 -> 0.3*((ksize-1)*0.5-1)+0.8."""
    if sigma <= 0:
        sigma = 0.3 * ((ksize - 1) * 0.5 - 1) + 0.8
    x = np.arange(ksize, dtype=np.float64) - (ksize - 1) * 0.5
    k = np.exp(-(x * x) / (2.0 * sigma * sigma))
    return k / k.sum()


def usm_kernel_2d(radius=50, sigma=0):
    """imgproc.py:1516-1524: radius made odd, outer product of the 1-D kernel in float64, cast to float32."""
    if radius % 2 == 0:
        radius += 1
    k = gaussian_kernel_1d(radius, sigma)
    return np.outer(k, k).astype(f32)[None]


def usm_sharp(img, weight=0.5, threshold=10, radius=50, sigma=0, return_parts=False):
    """imgproc.py:1526-1537 USMSharp.forward."""
    kern = usm_kernel_2d(radius, sigma)
    blur = filter2d(img, kern)
    residual = img - blur
    mask = (np.abs(residual) * f32(255) > f32(threshold)).astype(f32)
    soft = filter2d(mask, kern)
    out = img + f32(weight) * residual
    out = np.clip(out, 0, 1)
    out = soft * out + (f32(1) - soft) * img
    if return_parts:
        return out.astype(f32), residual.astype(f32), mask, soft
    return out.astype(f32)


# --------------------------------------------------------------------------------------------- resize (a9)

AREA, BILINEAR, BICUBIC = 0, 1, 2
MODE_ID = {"area": AREA, "bilinear": BILINEAR, "bicubic": BICUBIC}


def interp_out_size(in_size, scale_factor):
    """F.interpolate(scale_factor=s): floor(float(in) * s) (torch/nn/functional.py)."""
    return int(np.floor(float(in_size) * scale_factor))


def _src_scale(in_size, out_size, scale_factor):
    """ATen area_pixel_compute_scale, align_corners=False: 1/scale_factor when given, else in/out; as float32."""
    if scale_factor is not None:
        return f32(1.0 / float(scale_factor))
    return f32(in_size) / f32(out_size)


def _src_index(scale, out_size, cubic):
    """ATen area_pixel_compute_source_index in fp32: scale * (dst + 0.5) - 0.5, evaluated with one fused
    multiply-add (SURVEY.md §8a9); clamped at 0 for (bi)linear only."""
    d = np.arange(out_size, dtype=np.float64) + 0.5
    src = (np.float64(scale) * d - 0.5).astype(f32)  # exact product/sum in float64, ONE rounding == fmaf
    if not cubic:
        src = np.maximum(src, f32(0))
    return src


def _resize_area(img, oh, ow):
    """ATen adaptive_avg_pool2d: start = floor(o*in/out), end = ceil((o+1)*in/out), mean over the window."""
    b, c, h, w = img.shape

    def bounds(n_in, n_out):
        o = np.arange(n_out)
        return (o * n_in) // n_out, -((-(o + 1) * n_in) // n_out)

    y0, y1 = bounds(h, oh)
    x0, x1 = bounds(w, ow)
    acc = img.astype(np.float64)
    # integral image for exact window sums
    ii = np.zeros((b, c, h + 1, w + 1), np.float64)
    ii[:, :, 1:, 1:] = acc.cumsum(2).cumsum(3)
    s = (ii[:, :, y1][:, :, :, x1] - ii[:, :, y0][:, :, :, x1] - ii[:, :, y1][:, :, :, x0] + ii[:, :, y0][:, :, :, x0])
    cnt = ((y1 - y0)[:, None] * (x1 - x0)[None, :]).astype(np.float64)
    return (s / cnt).astype(f32)


def _cubic_coeffs(t):
    """ATen get_cubic_upsample_coefficients, A = -0.75, fp32."""
    A = f32(-0.75)
    t = t.astype(f32)

    def cc1(x):
        return ((A + f32(2)) * x - (A + f32(3))) * x * x + f32(1)

    def cc2(x):
        return ((A * x - f32(5) * A) * x + f32(8) * A) * x - f32(4) * A

    return np.stack([cc2(t + f32(1)), cc1(t), cc1(f32(1) - t), cc2(f32(2) - t)], 0).astype(f32)


def resize(img, out_h, out_w, mode, scale_h=None, scale_w=None):
    """F.interpolate(img, size= | scale_factor=, mode=area|bilinear|bicubic) as called at train_realesrnet.py:288,
    326, 349, 366. mode: 0 area, 1 bilinear, 2 bicubic. scale_*: the scale_factor when the call used scale_factor=
    (first resize), None when it used size=."""
    if isinstance(mode, str):
        mode = MODE_ID[mode]
    b, c, h, w = img.shape
    if mode == AREA:
        return _resize_area(img, out_h, out_w)
    sy = _src_index(_src_scale(h, out_h, scale_h), out_h, mode == BICUBIC)
    sx = _src_index(_src_scale(w, out_w, scale_w), out_w, mode == BICUBIC)
    x64 = img.astype(np.float64)
    if mode == BILINEAR:
        y0 = sy.astype(np.int64)
        x0 = sx.astype(np.int64)
        y1 = y0 + (y0 < h - 1)
        x1 = x0 + (x0 < w - 1)
        ly1 = (sy - y0.astype(f32)).astype(f32)
        lx1 = (sx - x0.astype(f32)).astype(f32)
        ly0 = (f32(1) - ly1).astype(np.float64)[None, None, :, None]
        lx0 = (f32(1) - lx1).astype(np.float64)[None, None, None, :]
        ly1 = ly1.astype(np.float64)[None, None, :, None]
        lx1 = lx1.astype(np.float64)[None, None, None, :]
        top = x64[:, :, y0][:, :, :, x0] * lx0 + x64[:, :, y0][:, :, :, x1] * lx1
        bot = x64[:, :, y1][:, :, :, x0] * lx0 + x64[:, :, y1][:, :, :, x1] * lx1
        return (top * ly0 + bot * ly1).astype(f32)
    # bicubic
    fy = np.floor(sy)
    fx = np.floor(sx)
    wy = _cubic_coeffs(sy - fy).astype(np.float64)  # [4, oh]
    wx = _cubic_coeffs(sx - fx).astype(np.float64)  # [4, ow]
    iy = fy.astype(np.int64)
    ix = fx.astype(np.int64)
    out = np.zeros((b, c, out_h, out_w), np.float64)
    for i in range(4):
        yy = np.clip(iy - 1 + i, 0, h - 1)
        rowsel = x64[:, :, yy]
        acc = np.zeros((b, c, out_h, out_w), np.float64)
        for j in range(4):
            xx = np.clip(ix - 1 + j, 0, w - 1)
            acc += rowsel[:, :, :, xx] * wx[j][None, None, None, :]
        out += acc * wy[i][None, None, :, None]
    return out.astype(f32)


# --------------------------------------------------------------------------------------------- noise (a10, a11)


def round_u8(x):
    """clamp(round(x * 255), 0, 255) / 255 in fp32 with round-half-to-even (torch.round); imgproc.py:889, 898."""
    return (np.clip(np.rint(x.astype(f32) * f32(255)), 0, 255) / f32(255)).astype(f32)


def rgb_to_gray(img):
    """torchvision rgb_to_grayscale: 0.2989 r + 0.587 g + 0.114 b, fp32, left to right; imgproc.py:887."""
    r, g, bl = img[:, 0:1], img[:, 1:2], img[:, 2:3]
    return ((f32(0.2989) * r + f32(0.587) * g).astype(f32) + f32(0.114) * bl).astype(f32)


def noise_post(out, clip=True, rounds=False):
    """The clip / rounds tail of both noise ops; imgproc.py:1048-1055, 1080-1085."""
    out = out.astype(f32)
    if clip and rounds:
        return (np.clip(np.rint(out * f32(255)), 0, 255) / f32(255)).astype(f32)
    if clip:
        return np.clip(out, 0, 1).astype(f32)
    if rounds:
        return (np.rint(out * f32(255)) / f32(255)).astype(f32)
    return out


def gaussian_noise_apply(img, sigma, gray, noise_color, noise_gray, clip=True, rounds=False):
    """imgproc.py:829-863 + 1029-1057 with the random tensors fed in:
    sigma[B], gray[B] (0/1), noise_color = randn(B,3,H,W), noise_gray = randn(H,W) (or None when sum(gray) == 0)."""
    b = img.shape[0]
    s = sigma.astype(f32).reshape(b, 1, 1, 1)
    noise = (noise_color.astype(f32) * s / f32(255)).astype(f32)
    if noise_gray is not None:
        g = gray.astype(f32).reshape(b, 1, 1, 1)
        ng = (noise_gray.astype(f32)[None, None] * s / f32(255)).astype(f32)  # ONE field shared by the batch
        noise = (noise * (f32(1) - g) + ng * g).astype(f32)
    return noise_post(img + noise, clip, rounds)


def unique_count_u8(q):
    """len(torch.unique(q_b)) per sample for u8-grid values; imgproc.py:892, 903."""
    lv = np.rint(q * f32(255)).astype(np.int64).reshape(q.shape[0], -1)
    return np.array([np.unique(r).size for r in lv], np.int64)


def poisson_vals(counts):
    """2 ** ceil(log2(n)); imgproc.py:893, 904."""
    return (2.0 ** np.ceil(np.log2(counts.astype(np.float64)))).astype(f32)


def poisson_rates(img, gray_any):
    """The rate tensors the reference hands to torch.poisson (imgproc.py:895, 906), for recording / replay."""
    q = round_u8(img)
    vals = poisson_vals(unique_count_u8(q)).reshape(-1, 1, 1, 1)
    out = {"q": q, "vals": vals, "rate": (q * vals).astype(f32)}
    if gray_any:
        qg = round_u8(rgb_to_gray(img))
        vg = poisson_vals(unique_count_u8(qg)).reshape(-1, 1, 1, 1)
        out.update({"qg": qg, "vals_g": vg, "rate_g": (qg * vg).astype(f32)})
    return out


def poisson_noise_apply(img, scale, gray, samples_color, samples_gray, clip=True, rounds=False):
    """imgproc.py:866-916 + 1060-1086 with the Poisson draws fed in: samples_color = poisson(q * vals) [B,3,H,W],
    samples_gray = poisson(q_gray * vals_gray) [B,1,H,W] or None."""
    b = img.shape[0]
    r = poisson_rates(img, samples_gray is not None)
    noise = (samples_color.astype(f32) / r["vals"] - r["q"]).astype(f32)
    if samples_gray is not None:
        g = gray.astype(f32).reshape(b, 1, 1, 1)
        ng = (samples_gray.astype(f32) / r["vals_g"] - r["qg"]).astype(f32)
        noise = (noise * (f32(1) - g) + ng * g).astype(f32)
    noise = (noise * scale.astype(f32).reshape(b, 1, 1, 1)).astype(f32)
    return noise_post(img + noise, clip, rounds)


# --------------------------------------------------------------------------------------------- JPEG (a12)

Y_TABLE = np.array(
    [[16, 11, 10, 16, 24, 40, 51, 61], [12, 12, 14, 19, 26, 58, 60, 55], [14, 13, 16, 24, 40, 57, 69, 56],
     [14, 17, 22, 29, 51, 87, 80, 62], [18, 22, 37, 56, 68, 109, 103, 77], [24, 35, 55, 64, 81, 104, 113, 92],
     [49, 64, 78, 87, 103, 121, 120, 101], [72, 92, 95, 98, 112, 100, 103, 99]], dtype=f32).T  # imgproc.py:40-45
C_TABLE = np.full((8, 8), 99, dtype=f32)  # imgproc.py:46-49
C_TABLE[:4, :4] = np.array([[17, 18, 24, 47], [18, 21, 26, 66], [24, 26, 56, 99], [47, 66, 99, 99]], dtype=f32).T


def jpeg_quality_to_factor(quality):
    """imgproc.py:1124-1141 applied to fp32 tensor elements (imgproc.py:1478-1479): every op rounded to fp32."""
    q = np.asarray(quality, dtype=f32)
    lo = (f32(5000.0) / q).astype(f32)
    hi = (f32(200.0) - (q * f32(2)).astype(f32)).astype(f32)
    return (np.where(q < 50, lo, hi).astype(f32) / f32(100.0)).astype(f32)


def _dct_basis():
    """imgproc.py:1238-1243 / 1358-1362: cos table in float64 -> float32."""
    t = np.zeros((8, 8, 8, 8), np.float64)
    for x in range(8):
        for y in range(8):
            for u in range(8):
                for v in range(8):
                    t[x, y, u, v] = np.cos((2 * x + 1) * u * np.pi / 16) * np.cos((2 * y + 1) * v * np.pi / 16)
    return t.astype(f32)


_BASIS = _dct_basis()
_ALPHA = np.array([1.0 / np.sqrt(2)] + [1] * 7)
_SCALE = (np.outer(_ALPHA, _ALPHA) * 0.25).astype(f32)  # imgproc.py:1244-1245
_ALPHA2 = np.outer(_ALPHA, _ALPHA).astype(f32)  # imgproc.py:1356-1357


def _blocks(plane):
    """imgproc.py:1222-1234: [B,H,W] -> [B, (H/8)*(W/8), 8, 8], row-major blocks."""
    b, h, w = plane.shape
    return plane.reshape(b, h // 8, 8, w // 8, 8).transpose(0, 1, 3, 2, 4).reshape(b, -1, 8, 8)


def _unblocks(blk, h, w):
    """imgproc.py:1374-1386."""
    b = blk.shape[0]
    return blk.reshape(b, h // 8, w // 8, 8, 8).transpose(0, 1, 3, 2, 4).reshape(b, h, w)


def jpeg(img, quality, return_parts=False):
    """imgproc.py:1462-1494 DiffJPEG(differentiable=False).forward(img, quality[B]). Returns the decoded image
    (and, with return_parts, factor[B] and the quantised coefficients / pre-rounding ratios per component)."""
    b, _, h, w = img.shape
    factor = jpeg_quality_to_factor(quality)  # the reference overwrites `quality` in place with this
    hp, wp = (16 - h % 16) % 16, (16 - w % 16) % 16
    x = np.zeros((b, 3, h + hp, w + wp), f32)
    x[:, :, :h, :w] = img
    H, W = h + hp, w + wp
    x = (x * f32(255)).astype(f32)  # imgproc.py:1318
    M = np.array([[0.299, 0.587, 0.114], [-0.168736, -0.331264, 0.5], [0.5, -0.418688, -0.081312]], dtype=f32)
    px = x.transpose(0, 2, 3, 1).astype(np.float64)
    ycc = (px @ M.T.astype(np.float64)).astype(f32) + np.array([0, 128, 128], f32)  # imgproc.py:1204-1208
    ycc = ycc.astype(f32)
    yy = ycc[..., 0]
    pool = lambda p: p.reshape(b, H // 2, 2, W // 2, 2).astype(np.float64).mean((2, 4)).astype(f32)  # :1216-1219
    comps = {"y": yy, "cb": pool(ycc[..., 1]), "cr": pool(ycc[..., 2])}
    parts = {"factor": factor}
    dec = {}
    for name, plane in comps.items():
        table = (Y_TABLE if name == "y" else C_TABLE)
        tq = (table[None, None] * factor.reshape(b, 1, 1, 1)).astype(f32)  # imgproc.py:1270-1272
        blk = _blocks(plane) - f32(128)  # imgproc.py:1248
        d = (np.tensordot(blk.astype(np.float64), _BASIS.astype(np.float64), axes=2)).astype(f32)
        d = (_SCALE * d).astype(f32)  # imgproc.py:1249
        ratio = (d / tq).astype(f32)
        qc = np.rint(ratio).astype(f32)  # torch.round: half to even (imgproc.py:1274)
        parts[name + "_ratio"], parts[name + "_q"] = ratio, qc
        deq = (qc * tq).astype(f32)  # imgproc.py:1327-1333
        z = (deq * _ALPHA2).astype(f32)  # imgproc.py:1366
        idct_basis = _BASIS.transpose(2, 3, 0, 1)  # tensor[x,y,u,v] of the decoder = cos((2u+1)x..)cos((2v+1)y..)
        rec = (f32(0.25) * np.tensordot(z.astype(np.float64), idct_basis.astype(np.float64), axes=2).astype(f32)
               + f32(128)).astype(f32)  # imgproc.py:1367-1368
        ph, pw = (H, W) if name == "y" else (H // 2, W // 2)
        dec[name] = _unblocks(rec, ph, pw)
    up = lambda p: np.repeat(np.repeat(p, 2, 1), 2, 2)  # imgproc.py:1392-1400
    ycc2 = np.stack([dec["y"], up(dec["cb"]), up(dec["cr"])], -1) + np.array([0, -128, -128], f32)
    M2 = np.array([[1., 0., 1.402], [1, -0.344136, -0.714136], [1, 1.772, 0]], dtype=f32)
    rgb = (ycc2.astype(np.float64) @ M2.T.astype(np.float64)).astype(f32)  # imgproc.py:1417-1419
    rgb = (np.minimum(f32(255), np.maximum(f32(0), rgb)) / f32(255)).astype(f32)  # imgproc.py:1453-1455
    out = rgb.transpose(0, 3, 1, 2)[:, :, :h, :w]
    if return_parts:
        return np.ascontiguousarray(out), parts
    return np.ascontiguousarray(out)


# --------------------------------------------------------------------------------------------- tail (a13)


def round_and_crop(out, hr, hr_top, hr_left, image_size, upscale):
    """train_realesrnet.py:374 + imgproc.py:1894-1934 random_crop with the (single, batch-wide) offset fed in."""
    lr = round_u8(out)
    ls = image_size // upscale
    lt, ll = hr_top // upscale, hr_left // upscale
    return (np.ascontiguousarray(lr[:, :, lt:lt + ls, ll:ll + ls]),
            np.ascontiguousarray(hr[:, :, hr_top:hr_top + image_size, hr_left:hr_left + image_size]))


# --------------------------------------------------------------------------------------------- whole block


def degrade_batch(hr, kernel1, kernel2, sinc_kernel, plan, stages=None, draw_rng=None):
    """train_realesrnet.py:267-377 driven by a recorded plan (dict, see oracle/plan.py). Returns (lr, hr_crop).
    If `stages` is a list, every intermediate image is appended to it. Plans without recorded random tensors (the
    CPU-baseline timing of bench.py) draw them here from `draw_rng` (numpy Generator) at the point the reference calls
    torch.randn / torch.poisson (imgproc.py:854-858, 895, 906)."""
    def rec(name, t):
        if stages is not None:
            stages.append((name, t))
        return t

    def noise(x, p):
        if p["type"] == "gaussian":
            nc, ng = p.get("noise_color"), p.get("noise_gray")
            if nc is None:
                if p["gray"].sum() > 0:
                    ng = draw_rng.standard_normal(x.shape[2:], dtype=f32)
                nc = draw_rng.standard_normal(x.shape, dtype=f32)
            return gaussian_noise_apply(x, p["sigma"], p["gray"], nc, ng)
        sc, sg = p.get("samples_color"), p.get("samples_gray")
        if sc is None:
            with_gray = bool(p["gray"].sum() > 0)
            r = poisson_rates(x, with_gray)
            sg = draw_rng.poisson(r["rate_g"]).astype(f32) if with_gray else None
            sc = draw_rng.poisson(r["rate"]).astype(f32)
        return poisson_noise_apply(x, p["scale"], p["gray"], sc, sg)

    out = rec("usm", usm_sharp(hr, 0.5, 10))
    if plan["blur1"]:
        out = rec("blur1", filter2d(out, kernel1))
    r = plan["resize1"]
    out = rec("resize1", resize(out, r["out_h"], r["out_w"], r["mode"], r["scale"], r["scale"]))
    out = rec("noise1", noise(out, plan["noise1"]))
    out = rec("jpeg1", jpeg(np.clip(out, 0, 1), plan["jpeg1_quality"]))
    if plan["blur2"]:
        out = rec("blur2", filter2d(out, kernel2))
    r = plan["resize2"]
    out = rec("resize2", resize(out, r["out_h"], r["out_w"], r["mode"]))
    out = rec("noise2", noise(out, plan["noise2"]))
    r = plan["resize3"]
    if plan["final_order"] == 0:  # resize -> sinc -> jpeg  (train_realesrnet.py:346-358)
        out = rec("resize3", resize(out, r["out_h"], r["out_w"], r["mode"]))
        out = rec("sinc", filter2d(out, sinc_kernel))
        out = rec("jpeg2", jpeg(np.clip(out, 0, 1), plan["jpeg2_quality"]))
    else:  # jpeg -> resize -> sinc  (train_realesrnet.py:360-371)
        out = rec("jpeg2", jpeg(np.clip(out, 0, 1), plan["jpeg2_quality"]))
        out = rec("resize3", resize(out, r["out_h"], r["out_w"], r["mode"]))
        out = rec("sinc", filter2d(out, sinc_kernel))
    c = plan["crop"]
    return round_and_crop(out, hr, c["hr_top"], c["hr_left"], c["image_size"], c["upscale"])
