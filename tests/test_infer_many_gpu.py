"""GPU: Generator.infer_many / infer_u8_many (C ABI resr_generator_forward_many[_u8]) run a list of differently sized
images as one packed canvas per forward. Each result must be its image's own forward: within the oracle contract of a
single-image forward (max-abs <= 2e-2, PSNR >= 45 dB), equal to infer() on that image alone, and untouched by the other
images of the canvas. Nonzero biases (oracle.generator.rich_state_dict) put nonzero values wherever a gutter pixel were
not forced back to zero.

"Equal to infer()": with the single-CTA convolution kernel (policy 0) the canvas result is bit-identical to the
image's own forward. The CTA-pair kernel sums the rows at ring positions 0 and 1 from two accumulator slots, and which
rows those are depends on where the image's rows fall in a CTA's strip, so there the fp32 summation order moves with the
image's place: on a B200 the largest difference from infer() was 1.3e-3 (fp16 recipe) and 8.3e-3 (bf16 recipe, whose
stored activations keep 8 mantissa bits), while the error against the oracle stayed that of infer(), in the border band
of each image as much as inside. So under pairs the test bounds the difference from infer() by those spreads and
requires the oracle error in each image's border band, where a leak across a gutter would show first, to stay within
3e-3 of infer()'s."""
import ctypes
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

MAX_ABS, MIN_PSNR = 2e-2, 45.0
PAIR_SPREAD = {"fp16": 2.5e-3, "bf16": 1.5e-2}    # infer_many vs infer() under the CTA-pair kernel (see above)
BORDER, BORDER_SLACK = 8, 3e-3
SIZES = [(1, 7), (5, 3), (17, 129), (64, 64), (128, 128), (130, 77), (200, 31), (33, 65), (9, 255), (3, 1), (41, 3)]


def _psnr(a, b):
    mse = torch.mean((a.double() - b.double()) ** 2).item()
    return 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)


@pytest.fixture(scope="module")
def case():
    """The seeded u8 images, their fp32 form (u8 / 255 on the device, an IEEE division) and the fp32 oracle outputs.
    The oracle runs on the GPU with TF32 off: the same fp32 restatement as on the CPU, in a fraction of the time."""
    from oracle import generator as og
    sd = og.rich_state_dict(5)
    rng = np.random.default_rng(11)
    imgs = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).cuda() for h, w in SIZES]
    xs = [(im.permute(2, 0, 1).float() / torch.full((3,) + im.shape[:2], 255.0, device="cuda")).unsqueeze(0).contiguous()
          for im in imgs]
    sd_gpu = {k: v.cuda() for k, v in sd.items()}
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        refs = [og.generator_forward(x, sd_gpu).cpu() for x in xs]
        torch.backends.cuda.matmul.allow_tf32 = prev
    return sd, imgs, xs, refs


def _border(t):
    m = torch.zeros_like(t, dtype=torch.bool)
    m[..., :BORDER, :] = True
    m[..., -BORDER:, :] = True
    m[..., :, :BORDER] = True
    m[..., :, -BORDER:] = True
    return m


def _gen(sd, recipe):
    import resr_b200
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    return g.cuda().eval().set_precision(recipe)


@pytest.fixture(params=[("fp16", 0), ("fp16", 2), ("bf16", 0), ("bf16", 2)], ids=lambda p: f"{p[0]}-policy{p[1]}")
def setup(request):
    import resr_b200
    lib = resr_b200._lib.lib()
    recipe, policy = request.param
    prev = lib.resr_set_conv_pair_policy(policy)
    yield recipe, policy
    lib.resr_set_conv_pair_policy(prev)


def test_infer_many_parity_alone_isolation_u8(case, setup):
    sd, imgs, xs, refs = case
    recipe, policy = setup
    g = _gen(sd, recipe)
    ys = g.infer_many(xs)
    assert [tuple(y.shape) for y in ys] == [(1, 3, 4 * h, 4 * w) for h, w in SIZES]
    worst_ref, worst_alone = 0.0, 0.0
    for (h, w), x, y, ref in zip(SIZES, xs, ys, refs):
        yc = y.cpu()
        err, ps = (yc - ref).abs().max().item(), _psnr(yc, ref)
        a = g.infer(x)
        alone = (y - a).abs().max().item()
        worst_ref, worst_alone = max(worst_ref, err), max(worst_alone, alone)
        assert err <= MAX_ABS and ps >= MIN_PSNR, ((h, w), err, ps)
        if policy == 0:
            assert torch.equal(y, a), ((h, w), alone)
        else:
            assert alone <= PAIR_SPREAD[recipe], ((h, w), alone)
            m = _border(ref)
            e_many, e_alone = (yc - ref).abs()[m].max().item(), (a.cpu() - ref).abs()[m].max().item()
            assert e_many <= e_alone + BORDER_SLACK, ((h, w), e_many, e_alone)
    print(f"{recipe} policy {policy}: max-abs vs oracle {worst_ref:.2e}, vs infer() alone {worst_alone:.2e}")

    # isolation: new pixels in one image, same canvas geometry -> every other output bit for bit the same
    k = SIZES.index((64, 64))
    xs2 = list(xs)
    xs2[k] = torch.rand_like(xs[k])
    ys2 = g.infer_many(xs2)
    for i, (a, b) in enumerate(zip(ys, ys2)):
        if i != k:
            assert torch.equal(a, b), SIZES[i]
    assert not torch.equal(ys[k], ys2[k])

    # u8: the reference conversion (mul(255).clamp(0, 255), truncation) of the fp32 outputs, bit for bit
    yu = g.infer_u8_many(imgs)
    for im, y, y8 in zip(imgs, ys, yu):
        want = y[0].permute(1, 2, 0).mul(255).clamp(0, 255).cpu().numpy().astype("uint8")
        assert y8.shape == (4 * im.shape[0], 4 * im.shape[1], 3) and y8.dtype == torch.uint8
        assert np.array_equal(y8.cpu().numpy(), want)


def test_edges_single_empty_and_split(case):
    """Under the single-CTA kernel, where placement does not change a result, a single image and a list the budget
    splits into several canvases give exactly the results of one canvas."""
    import resr_b200
    sd, imgs, xs, refs = case
    lib = resr_b200._lib.lib()
    prev = lib.resr_set_conv_pair_policy(0)
    try:
        g = _gen(sd, "fp16")
        assert g.infer_many([]) == [] and g.infer_u8_many([]) == []
        k = SIZES.index((130, 77))
        one = g.infer_many([xs[k][0]])               # a [3, h, w] image gives a [3, 4h, 4w] result
        assert one[0].shape == (3, 520, 308)
        assert torch.equal(one[0], g.infer(xs[k])[0])
        whole = g.infer_many(xs)
        parts = g.infer_many(xs, max_pixels=20000)  # several canvases
        assert len(_canvases(xs, 20000)) > 1
        for (h, w), a, b in zip(SIZES, whole, parts):
            assert torch.equal(a, b), (h, w)
        y8 = g.infer_u8_many(imgs, max_pixels=20000)
        assert all(torch.equal(a, b) for a, b in zip(y8, g.infer_u8_many(imgs)))
        # alternating with single-image calls keeps both kinds of plan valid and the results unchanged
        again = g.infer_many(xs)
        assert all(torch.equal(a, b) for a, b in zip(whole, again))
    finally:
        lib.resr_set_conv_pair_policy(prev)


def _canvases(xs, max_pixels):
    """Canvas sizes infer_many uses for `xs` under `max_pixels` (consecutive images up to the budget)."""
    import resr_b200
    groups, cur, px = [], [], 0
    for x in xs:
        h, w = x.shape[-2:]
        if cur and px + h * w > max_pixels:
            groups.append(cur)
            cur, px = [], 0
        cur.append((h, w))
        px += h * w
    groups.append(cur)
    return [resr_b200._lib.canvas_pack(gr)[1] for gr in groups]


def test_errors(case):
    import resr_b200
    L = resr_b200._lib
    sd, imgs, xs, refs = case
    g = _gen(sd, "fp16")
    with pytest.raises(ValueError):
        g.infer_many([xs[0][:, :2]])
    with pytest.raises(ValueError):
        g.infer_u8_many([imgs[0][..., :2]])
    with pytest.raises(L.ResrError):
        g.infer_many([xs[0].cpu()])
    # C ABI: a too-small workspace and a bad size
    g.infer_many(xs[:2])
    h = g._native()
    n = 2
    hs, ws = (ctypes.c_int * n)(*[s[0] for s in SIZES[:2]]), (ctypes.c_int * n)(*[s[1] for s in SIZES[:2]])
    need = L.lib().resr_generator_forward_many_workspace_bytes(h, hs, ws, n)
    assert need > 0
    y = [torch.empty(1, 3, 4 * a, 4 * b, device="cuda") for a, b in SIZES[:2]]
    xp, yp = (ctypes.c_void_p * n)(*[x.data_ptr() for x in xs[:2]]), (ctypes.c_void_p * n)(*[t.data_ptr() for t in y])
    wp, _ = g._aligned(g._workspace)
    assert L.lib().resr_generator_forward_many(h, xp, yp, hs, ws, n, wp, need - 1, L.stream_ptr()) == 3
    hs[0] = 0
    assert L.lib().resr_generator_forward_many(h, xp, yp, hs, ws, n, wp, need, L.stream_ptr()) == 1
    assert L.lib().resr_generator_forward_many_workspace_bytes(h, hs, ws, n) == 0
    torch.cuda.synchronize()
