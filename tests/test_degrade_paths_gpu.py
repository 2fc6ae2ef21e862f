"""Every dispatch path of the degradation kernels (csrc/degrade.cu) against the float64 numpy oracle (oracle/degrade.py),
at the shapes where the launchers switch kernels, template instantiations or loop forms.

Each case names the path it is meant to reach, and `_*_path` recomputes that name from the launcher's own selection
formulas; the two must agree, and `test_every_path_has_a_case` checks that every path appears in some case, so a change
of a threshold cannot quietly move a path out of coverage. The ops are called through the C ABI into an output buffer
pre-filled with NaN and framed by GUARD sentinel floats on either side: every output element must be written, and
nothing outside the output may be."""
import ctypes
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
TOL = 1e-5
GUARD = 4096            # floats on either side of an output; 16 KiB keeps the output 16-byte aligned
SENTINEL = -12345.5
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
f32 = np.float32


def _L():
    import resr_b200
    return resr_b200._lib


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


class Guarded:
    """A NaN-filled output of `shape` framed by sentinel guards."""

    def __init__(self, shape, offset=0):
        self.n = int(np.prod(shape))
        self.lo = GUARD + offset
        self.buf = torch.full((self.lo + self.n + GUARD,), float("nan"), device="cuda")
        self.buf[:self.lo] = SENTINEL
        self.buf[self.lo + self.n:] = SENTINEL
        self.t = self.buf[self.lo:self.lo + self.n].view(shape)

    def ptr(self):
        return ctypes.c_void_p(self.t.data_ptr())

    def check(self, what):
        torch.cuda.synchronize()
        assert bool(torch.isfinite(self.t).all()), f"{what}: output elements left unwritten"
        assert bool((self.buf[:self.lo] == SENTINEL).all()), f"{what}: store before the output"
        assert bool((self.buf[self.lo + self.n:] == SENTINEL).all()), f"{what}: store past the output"
        return self.t.cpu().numpy()


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _cdiv(a, b):
    return -(-a // b)


# ============================================================================================== filter2d
def _f2d_path(b, c, h, w, k, exts, r16=False):
    """filter2d_impl / filter2d_launch: rows per thread R, shared-tile PITCH, and the support bodies the blocks run."""
    cols, planes = _cdiv(w, 64), b * c
    blocks = lambda r: cols * _cdiv(h, 8 * r) * planes
    if r16 and cols * _cdiv(h, 64) * planes >= 592:
        r = 16
    elif blocks(8) >= 296:
        r = 8
    elif blocks(4) >= 296:
        r = 4
    else:
        r = 2
    bodies = sorted({2 * e + 1 for e in exts})
    names = "+".join(f"KS{s}" if s <= 21 else "KSgen" for s in bodies)
    return f"R{r} P{85 if k <= 21 else 127} {names}"


def _f2d_tags(path, k, exts):
    r, p, ks = path.split(" ")
    tags = {f"filter2d {r}", f"filter2d {p}"} | {f"filter2d {s}" for s in ks.split("+")}
    if any(2 * e + 1 > 21 and e < k // 2 for e in exts):
        tags.add("filter2d KSgen off>0")
    return tags


def _f2d_kernel(rng, k, ext, side):
    """k x k taps whose non-zero support reaches exactly `ext` from the centre; `side` places it one-sidedly."""
    r = k // 2
    w = rng.random((2 * ext + 1, 2 * ext + 1)).astype(f32) + f32(0.05)
    if side == "low":            # offsets <= 0 only (top-left quadrant)
        w[ext + 1:, :] = 0
        w[:, ext + 1:] = 0
    elif side == "high":         # offsets >= 0 only
        w[:ext, :] = 0
        w[:, :ext] = 0
    elif side == "row":          # horizontal support only
        w[:ext, :] = 0
        w[ext + 1:, :] = 0
    elif side == "corner":       # the centre and one far corner tap
        w[:] = 0
        w[ext, ext] = 1
        w[2 * ext, 0] = 0.5
    kern = np.zeros((k, k), f32)
    kern[r - ext:r + ext + 1, r - ext:r + ext + 1] = w
    return (kern / kern.sum(dtype=np.float64)).astype(f32)


# (id, b, c, h, w, k, ext per kernel, side, kernel_batch, path)
F2D_CASES = [(f"ks{2 * e + 1}", 1, 3, 40, 70, 21, [e], "both", 1, f"R2 P85 KS{2 * e + 1}") for e in range(11)] + [
    ("low1", 2, 3, 37, 45, 21, [1], "low", 1, "R2 P85 KS3"),
    ("high4", 2, 3, 37, 45, 21, [4], "high", 1, "R2 P85 KS9"),
    ("low10", 2, 3, 37, 45, 21, [10], "low", 1, "R2 P85 KS21"),
    ("row7", 1, 3, 37, 45, 21, [7], "row", 1, "R2 P85 KS15"),
    ("corner5", 1, 3, 37, 45, 21, [5], "corner", 1, "R2 P85 KS11"),
    ("mixed-batch", 4, 3, 30, 50, 21, [0, 3, 10, 6], "both", 4, "R2 P85 KS1+KS7+KS13+KS21"),
    ("mixed-batch-sides", 3, 2, 29, 66, 21, [2, 9, 5], "high", 3, "R2 P85 KS5+KS11+KS19"),
    ("k23", 1, 3, 40, 70, 23, [11], "both", 1, "R2 P127 KSgen"),
    ("k31", 1, 3, 40, 70, 31, [15], "both", 1, "R2 P127 KSgen"),
    ("k31-trim12", 2, 3, 40, 70, 31, [12], "both", 1, "R2 P127 KSgen"),
    ("k31-trim12-low", 1, 3, 40, 70, 31, [12], "low", 1, "R2 P127 KSgen"),
    ("k31-ks11", 1, 3, 40, 70, 31, [5], "both", 1, "R2 P127 KS11"),
    ("k63", 1, 2, 40, 70, 63, [31], "both", 1, "R2 P127 KSgen"),
    ("k63-trim15", 1, 2, 40, 70, 63, [15], "high", 1, "R2 P127 KSgen"),
    ("k63-ks1", 1, 2, 40, 70, 63, [0], "both", 1, "R2 P127 KS1"),
    ("r4", 13, 3, 128, 128, 21, [6], "both", 1, "R4 P85 KS13"),
    ("r4-h33", 50, 3, 33, 64, 21, [10], "both", 1, "R4 P85 KS21"),
    ("r8", 7, 3, 256, 256, 21, [4], "both", 1, "R8 P85 KS9"),
    ("r8-h65", 25, 3, 65, 100, 21, [2], "low", 1, "R8 P85 KS5"),
    ("r8-k31-trim13", 7, 3, 256, 256, 31, [13], "both", 1, "R8 P127 KSgen"),
    ("r2-h17", 1, 3, 17, 63, 21, [8], "both", 1, "R2 P85 KS17"),
    ("min-k3", 1, 3, 2, 2, 3, [1], "both", 1, "R2 P85 KS3"),
    ("min-k21", 2, 3, 11, 11, 21, [10], "both", 1, "R2 P85 KS21"),
    ("min-k31", 1, 1, 16, 16, 31, [15], "both", 1, "R2 P127 KSgen"),
    ("min-k63", 1, 1, 32, 32, 63, [31], "both", 1, "R2 P127 KSgen"),
    ("w63", 1, 3, 20, 63, 21, [10], "both", 1, "R2 P85 KS21"),
    ("w64", 1, 3, 20, 64, 21, [7], "both", 1, "R2 P85 KS15"),
    ("w65", 2, 3, 19, 65, 21, [10], "high", 1, "R2 P85 KS21"),
    ("w129", 1, 3, 24, 129, 21, [3], "both", 1, "R2 P85 KS7"),
]

# run in a child process with RESR_F2D_R16=1 (the knob is read once per process)
F2D_R16_CASES = [
    ("r16", 50, 3, 128, 128, 21, [10], "both", 1, "R16 P85 KS21"),
    ("r16-ks7", 50, 3, 128, 128, 21, [3], "low", 1, "R16 P85 KS7"),
    ("r16-k31-trim13", 50, 3, 128, 128, 31, [13], "both", 1, "R16 P127 KSgen"),
]


def _f2d_inputs(case):
    name, b, c, h, w, k, exts, side, kb, _ = case
    rng = _rng(name)
    x = rng.random((b, c, h, w), dtype=f32)
    kern = np.stack([_f2d_kernel(rng, k, e, side) for e in exts])
    return x, kern


def _f2d_run(case):
    name, b, c, h, w, k, exts, side, kb, _ = case
    x, kern = _f2d_inputs(case)
    L = _L()
    xd, kd = _t(x), _t(kern)
    out = Guarded((b, c, h, w))
    L.check(L.lib().resr_filter2d(_p(xd), _p(kd), out.ptr(), b, c, h, w, k, kb, L.stream_ptr()))
    return out.check(name)


def _f2d_compare(case, y):
    name, b, c, h, w, k, exts, side, kb, _ = case
    from oracle import degrade as od
    x, kern = _f2d_inputs(case)
    ref = od.filter2d(x, kern)
    d = float(np.abs(y.astype(np.float64) - ref).max())
    assert d <= TOL, (name, d)
    if all(e == 0 for e in exts):   # a centre-tap-only kernel (tap 1.0) returns the input bit for bit
        assert np.array_equal(y, x), name


@pytest.mark.parametrize("case", F2D_CASES, ids=[c[0] for c in F2D_CASES])
def test_filter2d_paths(case):
    name, b, c, h, w, k, exts, side, kb, path = case
    assert _f2d_path(b, c, h, w, k, exts) == path
    _f2d_compare(case, _f2d_run(case))


def _child_run(kind, out_path):
    """Body of the child processes that run the paths behind a once-per-process environment knob."""
    res = {}
    if kind == "f2d_r16":
        for case in F2D_R16_CASES:
            res[case[0]] = _f2d_run(case)
    elif kind == "usm_split":
        x = _usm_input(USM_EQ_SHAPE)
        res["usm"] = _usm_run(x, 50, 0)
    np.savez(out_path, **res)


def _child(kind, env, tmp_path):
    out = str(tmp_path / f"{kind}.npz")
    code = f"import sys; sys.path[:0] = [{ROOT!r}, {HERE!r}]; import test_degrade_paths_gpu as t; t._child_run({kind!r}, {out!r})"
    subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), cwd=ROOT, check=True, timeout=900)
    return np.load(out)


def test_filter2d_r16_in_child_process(tmp_path):
    res = _child("f2d_r16", {"RESR_F2D_R16": "1"}, tmp_path)
    for case in F2D_R16_CASES:
        name, b, c, h, w, k, exts, side, kb, path = case
        assert _f2d_path(b, c, h, w, k, exts, r16=True) == path
        _f2d_compare(case, res[name])


# ============================================================================================== USM forward
def _usm_path(h, radius, fused_env=True):
    """usm_impl: the fused 51-tap kernel while its [H + 50][33] + [64][83] fp32 strip fits 100 KiB (H <= 564), the split
    51-tap kernels above that, the generic passes for any other tap count."""
    k = radius + 1 if radius % 2 == 0 else radius
    if k != 51:
        return "generic"
    return "fused" if fused_env and ((h + 50) * 33 + 64 * 83) * 4 <= 100 * 1024 else "split"


# (b, c, h, w, radius, sigma, path)
USM_CASES = [
    (1, 3, 26, 26, 50, 0, "fused"), (1, 3, 26, 100, 50, 0, "fused"), (1, 2, 564, 33, 50, 0, "fused"),
    (1, 1, 564, 65, 50, 0, "fused"), (1, 3, 80, 90, 50, 3, "fused"),
    (1, 2, 565, 64, 50, 0, "split"), (1, 3, 565, 26, 50, 0, "split"), (1, 1, 700, 100, 50, 0, "split"),
    (2, 1, 700, 33, 50, 0, "split"), (1, 1, 600, 65, 50, 0, "split"),
    (1, 3, 60, 50, 20, 0, "generic"), (2, 3, 40, 64, 7, 0, "generic"), (1, 2, 45, 300, 20, 0, "generic"),
    (1, 3, 26, 27, 7, 0, "generic"),
]
USM_EQ_SHAPE = (1, 3, 300, 200)
WEIGHT, THRESH = 0.5, 10.0


def _usm_input(shape):
    return _rng(f"usm{shape}").random(shape, dtype=f32)


def _usm_run(x, radius, sigma):
    L = _L()
    b, c, h, w = x.shape
    out = Guarded(x.shape)
    need = L.lib().resr_usm_workspace_bytes(b, c, h, w)
    ws, xd = torch.empty(need, dtype=torch.uint8, device="cuda"), _t(x)
    L.check(L.lib().resr_usm_sharp(_p(xd), out.ptr(), b, c, h, w, radius, sigma, WEIGHT, THRESH, _p(ws), need,
                                   L.stream_ptr()))
    return out.check(f"usm {x.shape} r{radius}")


@pytest.mark.parametrize("case", USM_CASES, ids=[f"{c[6]}-{c[0]}x{c[1]}x{c[2]}x{c[3]}-r{c[4]}-s{c[5]}" for c in USM_CASES])
def test_usm_forward_paths(case):
    """Tolerance rule: a pixel whose |residual| * 255 sits within fp32 noise (255 * 4e-6) of the threshold may take
    either mask value. A flipped mask pixel p moves the soft mask at q by K[q - p], and the output at q by that times
    |clip(x + w r, 0, 1) - x|[q]; the bound allows exactly that on top of 1e-5."""
    from oracle import degrade as od
    b, c, h, w, radius, sigma, path = case
    assert _usm_path(h, radius) == path
    x = _usm_input((b, c, h, w))
    y = _usm_run(x, radius, sigma)
    ref, res, mask, soft = od.usm_sharp(x, WEIGHT, THRESH, radius, sigma, return_parts=True)
    amb = (np.abs(np.abs(res.astype(np.float64)) * 255 - THRESH) <= 255 * 4e-6).astype(f32)
    spread = od.filter2d(amb, od.usm_kernel_2d(radius, sigma)).astype(np.float64)
    lever = np.abs(np.clip(x + f32(WEIGHT) * res, 0, 1).astype(np.float64) - x)
    bound = TOL + spread * lever
    d = np.abs(y.astype(np.float64) - ref)
    print(f"usm {case}: {int(amb.sum())} ambiguous mask pixels, max diff {d.max():.2e}")
    assert (d <= bound).all(), (case, float((d - bound).max()))


def test_usm_split_is_bit_identical_to_fused(tmp_path):
    """DESIGN §4: the split 51-tap kernels (RESR_USM_FUSED=0, read once per process) and the fused kernel evaluate every
    output with the same FMA order."""
    assert _usm_path(USM_EQ_SHAPE[2], 50) == "fused" and _usm_path(USM_EQ_SHAPE[2], 50, fused_env=False) == "split"
    fused = _usm_run(_usm_input(USM_EQ_SHAPE), 50, 0)
    split = _child("usm_split", {"RESR_USM_FUSED": "0"}, tmp_path)["usm"]
    assert torch.equal(torch.from_numpy(fused), torch.from_numpy(split))


# ============================================================================================== USM backward
# (b, c, h, w, radius, path)
USM_BWD_CASES = [(1, 1, 600, 40, 50, "split"), (1, 3, 60, 50, 7, "generic"), (1, 2, 48, 40, 20, "generic")]


def _usm_ref64(x, kernel2d, weight, threshold):
    import torch.nn.functional as F
    b, c, h, w = x.shape
    K = kernel2d.shape[-1]
    R = K // 2
    k = kernel2d.to(x).view(1, 1, K, K)

    def blur(t):
        return F.conv2d(F.pad(t.reshape(b * c, 1, h, w), (R, R, R, R), mode="reflect"), k).view(b, c, h, w)

    residual = x - blur(x)
    soft = blur((torch.abs(residual) * 255 > threshold).to(x.dtype))
    return soft * torch.clip(x + weight * residual, 0, 1) + (1 - soft) * x, residual


@pytest.mark.parametrize("case", USM_BWD_CASES, ids=[f"{c[5]}-{c[2]}x{c[3]}-r{c[4]}" for c in USM_BWD_CASES])
def test_usm_backward_paths(case):
    from oracle import degrade as od
    b, c, h, w, radius, path = case
    assert _usm_path(h, radius) == path
    k64 = torch.from_numpy(od.usm_kernel_2d(radius, 0)[0]).double()
    for seed in range(20):
        # a draw without a pixel inside fp32 noise of the mask threshold or of the clip bounds: there fp32 and fp64 may
        # take different branches, and the gradient differs by design
        gen = torch.Generator().manual_seed(seed)
        x, g = torch.rand(b, c, h, w, generator=gen), torch.randn(b, c, h, w, generator=gen)
        xr = x.double().requires_grad_(True)
        ref, res = _usm_ref64(xr, k64, WEIGHT, THRESH)
        v = (xr + WEIGHT * res).detach()
        if (res.detach().abs() * 255 - THRESH).abs().min().item() > 5e-5 and min(v.abs().min().item(), (v - 1).abs().min().item()) > 2e-6:
            break
    else:
        raise AssertionError("no draw with a safe margin")
    (ref * g.double()).sum().backward()
    L = _L()
    out = Guarded((b, c, h, w))
    need = L.lib().resr_usm_backward_workspace_bytes(b, c, h, w)
    ws, xd, gd = torch.empty(need, dtype=torch.uint8, device="cuda"), x.cuda(), g.cuda()
    L.check(L.lib().resr_usm_sharp_backward(_p(xd), _p(gd), out.ptr(), b, c, h, w, radius, 0, WEIGHT, THRESH, _p(ws),
                                            need, L.stream_ptr()))
    gi = out.check(f"usm backward {case}")
    err = float(np.abs(gi - xr.grad.numpy()).max())
    scale = float(xr.grad.abs().max())
    print(f"usm backward {case}: seed {seed}, max err {err:.2e} (gradient scale {scale:.2e})")
    assert err <= 1e-5 * max(1.0, scale)


# ============================================================================================== resize
RESIZE_CAP = 148 * 32 * 256    # grid1d: beyond this many outputs every thread loops
MODES = ("area", "bilinear", "bicubic")


def _resize_path(mode, planes, ho, wo):
    return f"{mode} {'stride' if planes * ho * wo > RESIZE_CAP else 'grid'}"


def _out_size(n, s):
    return int(np.floor(float(n) * s))


# (id, b, c, hi, wi, ho, wo, scale (sh, sw) or None)
RESIZE_GEOMS = [
    ("1x1-7x5", 1, 3, 1, 1, 7, 5, None),
    ("7x5-1x1", 1, 3, 7, 5, 1, 1, None),
    ("1xN-Mx1", 2, 3, 1, 37, 23, 1, None),
    ("Nx1-1xM", 1, 2, 29, 1, 1, 41, None),
    ("mixed-40x90-70x31", 1, 3, 40, 90, 70, 31, None),
    ("area-256-17", 1, 2, 256, 256, 17, 17, None),
    ("window-6000", 1, 1, 1, 6000, 3, 1, None),
    ("above-cap", 1, 3, 400, 500, 700, 600, None),
] + [(f"sf{s:.4g}", 2, 3, 48, 56, _out_size(48, s), _out_size(56, s), (s, s)) for s in (0.15, 1 / 3, 0.5, 0.7, 1.37, 1.5)] + [
    ("sf0.7x1.37", 1, 3, 45, 61, _out_size(45, 0.7), _out_size(61, 1.37), (0.7, 1.37)),
    ("sf1.5-odd", 1, 3, 7, 9, _out_size(7, 1.5), _out_size(9, 1.5), (1.5, 1.5)),
]
RESIZE_CASES = [(g, m) for g in RESIZE_GEOMS for m in MODES]


def _area_window(n_in, n_out):
    o = np.arange(n_out)
    return int((-(-(o + 1) * n_in // n_out) - (o * n_in) // n_out).max())


@pytest.mark.parametrize("geom, mode", RESIZE_CASES, ids=[f"{g[0]}-{m}" for g, m in RESIZE_CASES])
def test_resize_paths(geom, mode):
    from oracle import degrade as od
    name, b, c, hi, wi, ho, wo, sf = geom
    assert _resize_path(mode, b * c, ho, wo) == (f"{mode} stride" if name == "above-cap" else f"{mode} grid")
    x = _rng(name).random((b, c, hi, wi), dtype=f32)
    sh, sw = sf if sf is not None else (0.0, 0.0)
    L = _L()
    xd = _t(x)
    out = Guarded((b, c, ho, wo))
    L.check(L.lib().resr_resize(_p(xd), out.ptr(), b * c, hi, wi, ho, wo, od.MODE_ID[mode], float(sh), float(sw), L.stream_ptr()))
    y = out.check(f"resize {name} {mode}")
    ref = od.resize(x, ho, wo, mode, sf[0] if sf else None, sf[1] if sf else None)
    tol = TOL
    if mode == "area":
        # the kernel sums an area window sequentially in fp32: beyond a 64 x 64 window the rounding of that sum
        # (at most n * 2^-24 of the mean for n terms) outgrows 1e-5
        n = _area_window(hi, ho) * _area_window(wi, wo)
        if n > 64 * 64:
            tol = n * 2.0 ** -24
    d = float(np.abs(y.astype(np.float64) - ref).max())
    assert d <= tol, (name, mode, d, tol)


# ============================================================================================== JPEG
JPEG_MCU_CAP = 148 * 8 * 8    # 148 * 8 blocks of 8 warps: beyond this many MCUs warps loop


def _jpeg_path(b, h, w, aligned=True):
    vec = "vec" if w % 4 == 0 and aligned else "scalar"
    loop = b * _cdiv(h, 16) * _cdiv(w, 16) > JPEG_MCU_CAP
    return f"jpeg {vec}" + (" loop" if loop else "")


JPEG_SIDES = (1, 7, 8, 9, 15, 16, 17, 33, 50)
JPEG_QUALITIES = np.array([1, 30, 49.99, 50, 50.01, 95, 99], f32)


def _jpeg_run(x, q, clamp=0, x_off=0, out_off=0):
    """resr_jpeg with every output (image and the three coefficient dumps) guarded; x_off / out_off shift the image and
    output base pointers by that many floats."""
    L = _L()
    b, _, h, w = x.shape
    hp, wp = _cdiv(h, 16) * 16, _cdiv(w, 16) * 16
    src = torch.zeros(x.size + x_off, device="cuda")
    src[x_off:] = _t(x).reshape(-1)
    out = Guarded(x.shape, out_off)
    factor = Guarded((b,))
    qy, qcb, qcr = Guarded((b, hp * wp // 64, 8, 8)), Guarded((b, hp * wp // 256, 8, 8)), Guarded((b, hp * wp // 256, 8, 8))
    qd = _t(q)
    L.check(L.lib().resr_jpeg(ctypes.c_void_p(src.data_ptr() + 4 * x_off), out.ptr(), _p(qd), factor.ptr(), b, h, w, clamp,
                              qy.ptr(), qcb.ptr(), qcr.ptr(), L.stream_ptr()))
    tag = f"jpeg {x.shape}"
    return out.check(tag), factor.check(tag), tuple(g.check(tag) for g in (qy, qcb, qcr))


def _jpeg_verify(x, q, y, factor, coefs):
    """factor bit-exact; a coefficient may differ from the oracle only at a rounding tie, by one step; every 16 x 16 MCU
    whose coefficients all match agrees with the oracle to 1e-5 (an MCU's output depends on its own coefficients only)."""
    from oracle import degrade as od
    ref, parts = od.jpeg(x, q, return_parts=True)
    assert np.array_equal(factor, parts["factor"]), "quantisation factor must be bit-exact"
    b, _, h, w = x.shape
    mh, mw = _cdiv(h, 16), _cdiv(w, 16)
    flipped = np.zeros((b, mh, mw), bool)
    flips = 0
    for name, qn in zip(("y", "cb", "cr"), coefs):
        mism = qn != parts[name + "_q"]
        ratio = parts[name + "_ratio"]
        near_tie = np.abs(np.abs(ratio - np.floor(ratio)) - 0.5) < 2e-3
        assert not (mism & ~near_tie).any(), f"{name}: coefficient differs away from a rounding tie"
        assert np.abs(qn - parts[name + "_q"]).max() <= 1
        flips += int(mism.sum())
        blk = mism.any((2, 3))
        flipped |= blk.reshape(b, mh, 2, mw, 2).any((2, 4)) if name == "y" else blk.reshape(b, mh, mw)
    clean = ~np.repeat(np.repeat(flipped, 16, 1), 16, 2)[:, None, :h, :w]
    d = np.abs(y.astype(np.float64) - ref) * clean
    assert d.max() <= TOL, float(d.max())
    return flips, int(flipped.sum())


@pytest.mark.parametrize("h", JPEG_SIDES)
def test_jpeg_sizes(h):
    """Every H crossed with every W of JPEG_SIDES: partial MCUs, partial 8-column lane groups, both row-access forms."""
    for w in JPEG_SIDES:
        b = 2
        assert _jpeg_path(b, h, w) == ("jpeg vec" if w % 4 == 0 else "jpeg scalar")
        rng = _rng(f"jpeg{h}x{w}")
        x = rng.random((b, 3, h, w), dtype=f32)
        q = rng.uniform(20, 90, b).astype(f32)
        y, factor, coefs = _jpeg_run(x, q)
        _jpeg_verify(x, q, y, factor, coefs)


@pytest.mark.parametrize("h, w", [(33, 50), (40, 48)])
def test_jpeg_quality_per_sample(h, w):
    """One sample per quality around the q = 50 switch of quality_to_factor (imgproc.py:1124-1141) and at the ends."""
    b = len(JPEG_QUALITIES)
    x = _rng(f"jq{h}x{w}").random((b, 3, h, w), dtype=f32)
    y, factor, coefs = _jpeg_run(x, JPEG_QUALITIES)
    flips, mcus = _jpeg_verify(x, JPEG_QUALITIES, y, factor, coefs)
    print(f"jpeg qualities {h}x{w}: {flips} tie flips in {mcus} MCUs")


def test_jpeg_many_mcus_warps_loop():
    b, h, w = 4, 784, 784
    assert _jpeg_path(b, h, w) == "jpeg vec loop"
    rng = _rng("jpeg-big")
    x = rng.random((b, 3, h, w), dtype=f32)
    q = np.array([10, 45, 70, 92], f32)
    y, factor, coefs = _jpeg_run(x, q)
    flips, mcus = _jpeg_verify(x, q, y, factor, coefs)
    print(f"jpeg {b}x3x{h}x{w}: {flips} tie flips in {mcus} of {b * 49 * 49} MCUs")


@pytest.mark.parametrize("w", [52, 45])
def test_jpeg_clamp_input(w):
    b, h = 2, 37
    rng = _rng(f"jpeg-clamp{w}")
    x = rng.uniform(-0.2, 1.2, (b, 3, h, w)).astype(f32)
    q = np.array([35, 80], f32)
    y, factor, coefs = _jpeg_run(x, q, clamp=1)
    _jpeg_verify(np.clip(x, 0, 1), q, y, factor, coefs)


@pytest.mark.parametrize("x_off, out_off", [(1, 0), (0, 3), (2, 1)])
def test_jpeg_unaligned_pointers(x_off, out_off):
    """W % 4 == 0 with an image or output base that is not 16-byte aligned takes the scalar rows, same result."""
    b, h, w = 2, 40, 48
    assert _jpeg_path(b, h, w, aligned=False) == "jpeg scalar"
    rng = _rng("jpeg-unaligned")
    x = rng.random((b, 3, h, w), dtype=f32)
    q = np.array([40, 75], f32)
    ya, fa, ca = _jpeg_run(x, q)
    yu, fu, cu = _jpeg_run(x, q, x_off=x_off, out_off=out_off)
    assert np.array_equal(ya, yu) and np.array_equal(fa, fu) and all(np.array_equal(a, u) for a, u in zip(ca, cu))


def test_diffjpeg_on_a_view_with_storage_offset():
    import resr_b200
    b, h, w = 2, 32, 64
    base = torch.rand(1 + b * 3 * h * w, generator=torch.Generator().manual_seed(0)).cuda()
    view = base[1:].view(b, 3, h, w)
    assert view.is_contiguous() and view.data_ptr() % 16 == 4
    j = resr_b200.imgproc.DiffJPEG(False)
    q = torch.tensor([30.0, 85.0], device="cuda")
    assert torch.equal(j(view, q.clone()), j(view.clone(), q.clone()))


# ============================================================================================== noise apply
NOISE_CAP = RESIZE_CAP


def _noise_path(kind, clip, rounds, elements):
    return {f"{kind} clip{clip} rounds{rounds}"} | ({f"{kind} stride"} if elements > NOISE_CAP else set())


def _tie_values():
    """fp32 values v with fl(v * 255) == k + 0.5 exactly, k = -1 .. 255: round-half-even decides them."""
    vals = []
    for k in range(-1, 256):
        v = f32((k + 0.5) / 255)
        for cand in (v, np.nextafter(v, f32(2)), np.nextafter(v, f32(-2))):
            if f32(cand) * f32(255) == f32(k + 0.5):
                vals.append(f32(cand))
                break
    assert len(vals) > 200
    return np.array(vals, f32)


def _noise_input(name, b, h, w):
    rng = _rng(name)
    x = rng.uniform(-0.05, 1.05, (b, 3, h, w)).astype(f32)
    ties = rng.random((h, w)) < 0.3         # pixels that stay on a u8 half-step: zero noise there
    tv = _tie_values()
    x[:, :, ties] = rng.choice(tv, (b, 3, int(ties.sum())))
    return rng, x, ties


# (id, kind, b, h, w, gray flags or None)
NOISE_GEOMS = [("small", 3, 24, 40, [1, 0, 1]), ("small-nogray", 2, 17, 33, None), ("stride", 2, 800, 800, [0, 1])]
NOISE_CASES = [(g, kind, clip, rounds) for g in NOISE_GEOMS for kind in ("gaussian", "poisson")
               for clip in (0, 1) for rounds in (0, 1) if g[0] != "stride" or (clip, rounds) == (1, 0)]


@pytest.mark.parametrize("geom, kind, clip, rounds", NOISE_CASES,
                         ids=[f"{g[0]}-{k}-clip{c}-rounds{r}" for g, k, c, r in NOISE_CASES])
def test_noise_apply_clip_rounds(geom, kind, clip, rounds):
    """Both noise ops restate the reference in fp32 op for op, so the kernel is bit-exact against the oracle."""
    from oracle import degrade as od
    name, b, h, w, gray = geom
    elements = b * 3 * h * w if kind == "gaussian" else b * h * w
    assert f"{kind} clip{clip} rounds{rounds}" in _noise_path(kind, clip, rounds, elements)
    assert (f"{kind} stride" in _noise_path(kind, clip, rounds, elements)) == (name == "stride")
    rng, x, ties = _noise_input(f"{name}-{kind}", b, h, w)
    gflags = None if gray is None else np.array(gray, f32)
    L = _L()
    out = Guarded(x.shape)
    if kind == "gaussian":
        sigma = rng.uniform(1, 30, b).astype(f32)
        nc = rng.standard_normal(x.shape, dtype=f32)
        nc[:, :, ties] = 0
        ng = None
        if gflags is not None:
            ng = rng.standard_normal((h, w), dtype=f32)
            ng[ties] = 0
        dev = [None if a is None else _t(a) for a in (x, sigma, gflags, nc, ng)]   # alive until the launch is queued
        L.check(L.lib().resr_gaussian_noise_apply(_p(dev[0]), out.ptr(), *(_p(d) for d in dev[1:]), b, 3, h, w, clip, rounds,
                                                  L.stream_ptr()))
        ref = od.gaussian_noise_apply(x, sigma, gflags, nc, ng, clip=bool(clip), rounds=bool(rounds))
    else:
        scale = rng.uniform(0.05, 3, b).astype(f32)
        r = od.poisson_rates(x, gflags is not None)
        sc = rng.poisson(r["rate"]).astype(f32)
        sc[:, :, ties] = r["rate"][:, :, ties]           # draw == rate: zero noise
        sg = None
        if gflags is not None:
            sg = rng.poisson(r["rate_g"]).astype(f32)
            sg[:, :, ties] = r["rate_g"][:, :, ties]
        need = L.lib().resr_poisson_workspace_bytes(b)
        ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        dev = [None if a is None else _t(a) for a in (x, scale, gflags, sc, sg)]
        L.check(L.lib().resr_poisson_noise_apply(_p(dev[0]), out.ptr(), *(_p(d) for d in dev[1:]), b, 3, h, w, clip, rounds, _p(ws),
                                                 need, 0, L.stream_ptr()))
        ref = od.poisson_noise_apply(x, scale, gflags, sc, sg, clip=bool(clip), rounds=bool(rounds))
    y = out.check(f"{kind} noise {name}")
    assert np.array_equal(y, ref), float(np.abs(y.astype(np.float64) - ref).max())
    if rounds:   # the half-step pixels went through round-half-even
        assert np.array_equal(y[:, :, ties], od.noise_post(x[:, :, ties], bool(clip), True))


# ============================================================================================== crop / round
def _crop_path(round_to_u8, hi, wi, ho, wo, elements):
    path = "crop copy" if not round_to_u8 and (ho, wo) == (hi, wi) else f"crop kernel round{round_to_u8}"
    return path + (" stride" if elements > RESIZE_CAP and path != "crop copy" else "")


# (id, b, c, hi, wi, top, left, ho, wo)
CROP_GEOMS = [("top-left", 2, 3, 37, 45, 0, 0, 10, 12), ("bottom-right", 2, 3, 37, 45, 27, 33, 10, 12),
              ("whole", 2, 3, 37, 45, 0, 0, 37, 45), ("one-pixel-corner", 1, 3, 9, 7, 8, 6, 1, 1),
              ("stride", 2, 3, 700, 600, 40, 7, 650, 590)]
CROP_CASES = [(g, r) for g in CROP_GEOMS for r in (0, 1)]


@pytest.mark.parametrize("geom, round_to_u8", CROP_CASES, ids=[f"{g[0]}-round{r}" for g, r in CROP_CASES])
def test_crop_paths(geom, round_to_u8):
    from oracle import degrade as od
    name, b, c, hi, wi, top, left, ho, wo = geom
    path = _crop_path(round_to_u8, hi, wi, ho, wo, b * c * ho * wo)
    assert path == {("whole", 0): "crop copy", ("stride", 0): "crop kernel round0 stride",
                    ("stride", 1): "crop kernel round1 stride"}.get((name, round_to_u8), f"crop kernel round{round_to_u8}")
    rng = _rng(f"crop{name}")
    x = rng.uniform(-0.05, 1.05, (b, c, hi, wi)).astype(f32)
    tie = rng.random((b, c, hi, wi)) < 0.3
    x[tie] = rng.choice(_tie_values(), int(tie.sum()))
    L = _L()
    xd = _t(x)
    out = Guarded((b, c, ho, wo))
    L.check(L.lib().resr_crop(_p(xd), out.ptr(), b * c, hi, wi, top, left, ho, wo, round_to_u8, L.stream_ptr()))
    y = out.check(f"crop {name}")
    ref = x[:, :, top:top + ho, left:left + wo]
    if round_to_u8:
        ref = od.round_u8(ref)
    assert np.array_equal(y, ref)


# ============================================================================================== coverage
REQUIRED = (
    {f"filter2d R{r}" for r in (2, 4, 8, 16)} | {"filter2d P85", "filter2d P127", "filter2d KSgen", "filter2d KSgen off>0"}
    | {f"filter2d KS{s}" for s in range(1, 22, 2)}
    | {"usm fused", "usm split", "usm generic", "usm-backward split", "usm-backward generic"}
    | {f"{m} {g}" for m in MODES for g in ("grid", "stride")}
    | {"jpeg vec", "jpeg scalar", "jpeg vec loop"}
    | {f"{k} clip{c} rounds{r}" for k in ("gaussian", "poisson") for c in (0, 1) for r in (0, 1)}
    | {"gaussian stride", "poisson stride"}
    | {"crop copy", "crop kernel round0", "crop kernel round1", "crop kernel round0 stride", "crop kernel round1 stride"}
)


def test_every_path_has_a_case():
    """Every path of the dispatch table is reached by at least one case above (paths recomputed from the selection
    formulas, so a changed threshold that empties a path fails here)."""
    seen = set()
    for (name, b, c, h, w, k, exts, side, kb, _) in F2D_CASES:
        seen |= _f2d_tags(_f2d_path(b, c, h, w, k, exts), k, exts)
    for (name, b, c, h, w, k, exts, side, kb, _) in F2D_R16_CASES:
        seen |= _f2d_tags(_f2d_path(b, c, h, w, k, exts, r16=True), k, exts)
    seen |= {"usm " + _usm_path(h, r) for (b, c, h, w, r, s, _) in USM_CASES}
    seen.add("usm " + _usm_path(USM_EQ_SHAPE[2], 50, fused_env=False))
    seen |= {"usm-backward " + _usm_path(h, r) for (b, c, h, w, r, _) in USM_BWD_CASES}
    seen |= {_resize_path(m, g[1] * g[2], g[5], g[6]) for g, m in RESIZE_CASES}
    seen |= {_jpeg_path(2, h, w) for h in JPEG_SIDES for w in JPEG_SIDES}
    seen |= {_jpeg_path(4, 784, 784), _jpeg_path(2, 40, 48, aligned=False)}
    for g, kind, clip, rounds in NOISE_CASES:
        seen |= _noise_path(kind, clip, rounds, g[1] * 3 * g[2] * g[3] if kind == "gaussian" else g[1] * g[2] * g[3])
    seen |= {_crop_path(r, g[3], g[4], g[7], g[8], g[1] * g[2] * g[7] * g[8]) for g, r in CROP_CASES}
    missing = REQUIRED - seen
    assert not missing, sorted(missing)
