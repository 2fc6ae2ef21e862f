"""GPU: model.MultiDeviceInference deals one image's halo bands, or a list's canvases, to several Generator replicas, one
host thread each. Every band and every canvas is the forward one GPU runs, so the results must be torch.equal to the
single-GPU calls: infer_tiled for a large image (and the same bands through infer_u8 for a u8 image), Generator.infer_many
/ infer_u8_many for a list. On one B200 the replicas share cuda:0 ([0, 0] and [0, 0, 0]); with two or more visible GPUs
the same equalities are checked on all of them."""
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

H, W, BAND = 70, 48, 12            # 6 bands, the last one ragged (10 rows)
SIZES = [(1, 7), (17, 129), (64, 64), (130, 77), (9, 255), (3, 1), (41, 3), (33, 65)]
BUDGET = 9000                      # several canvases to deal


@pytest.fixture(scope="module")
def sd():
    from oracle import generator as og
    return og.rich_state_dict(5)


def _gen(sd, recipe="fp16"):
    import resr_b200
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    return g.cuda().eval().set_precision(recipe)


@pytest.fixture(params=[0, 2], ids=lambda p: f"policy{p}")
def policy(request):
    import resr_b200
    lib = resr_b200._lib.lib()
    prev = lib.resr_set_conv_pair_policy(request.param)
    yield request.param
    lib.resr_set_conv_pair_policy(prev)


def _images(seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(1, 3, H, W, generator=g)
    img = torch.randint(0, 256, (H, W, 3), generator=g, dtype=torch.uint8)
    return x, img


def _tiled_u8(gen, img, band_rows, halo=16):
    """infer_tiled's assembly, with Generator.infer_u8 per band."""
    import resr_b200
    h, w, _ = img.shape
    out = torch.empty((4 * h, 4 * w, 3), dtype=torch.uint8, device="cuda")
    src = img.cuda()
    for y0, y1, _, _, wy0, wy1, _, _ in resr_b200.model.plan_tiles(h, w, band_rows, w, halo):
        sr = gen.infer_u8(src[None, wy0:wy1])
        out[4 * y0:4 * y1] = sr[0, 4 * (y0 - wy0):4 * (y0 - wy0) + 4 * (y1 - y0)]
    return out.cpu()


def _sources(t, devices):
    """The same tensor from pageable host memory, pinned host memory and every device in use."""
    return [t, t.pin_memory()] + [t.to(d) for d in sorted({torch.device(d) for d in devices}, key=str)]


def _check_large(gen, md, devices):
    import resr_b200
    M = resr_b200.model
    x, img = _images()
    ref = M.infer_tiled(gen, x.cuda(), BAND, W, 16)[0].cpu()
    ref8 = _tiled_u8(gen, img, BAND)
    for src in _sources(x, devices):
        y = md.infer_large(src, band_rows=BAND)
        assert y.is_pinned() and y.shape == (1, 3, 4 * H, 4 * W)
        assert torch.equal(y, ref), src.device
    for src in _sources(img, devices):
        y8 = md.infer_u8_large(src, band_rows=BAND)
        assert y8.is_pinned() and y8.shape == (4 * H, 4 * W, 3) and y8.dtype == torch.uint8
        assert torch.equal(y8, ref8), src.device
    # the default plan: at least two bands per replica
    rows = M.default_band_rows(H, W, len(md.devices))
    assert torch.equal(md.infer_large(x), M.infer_tiled(gen, x.cuda(), rows, W, 16)[0].cpu())
    assert torch.equal(md.infer_u8_large(img), _tiled_u8(gen, img, rows))
    return x, ref


def _check_many(gen, md, devices):
    rng = np.random.default_rng(11)
    imgs = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)) for h, w in SIZES]
    xs = [(im.permute(2, 0, 1).float() / 255.0) for im in imgs]
    xs = [x.unsqueeze(0) if i % 2 else x for i, x in enumerate(xs)]      # [1, 3, h, w] and [3, h, w] mixed
    for budget in (BUDGET, None):
        kw = {} if budget is None else {"max_pixels": budget}
        ref = [y.cpu() for y in gen.infer_many([x.cuda() for x in xs], **kw)]
        ref8 = [y.cpu() for y in gen.infer_u8_many([im.cuda() for im in imgs], **kw)]
        dev = sorted({torch.device(d) for d in devices}, key=str)[-1]
        for src in (xs, [x.pin_memory() for x in xs], [x.to(dev) for x in xs]):
            ys = md.infer_many(src, **kw)
            assert len(ys) == len(xs)
            for a, b in zip(ys, ref):
                assert a.is_pinned() and a.shape == b.shape and torch.equal(a, b)
        for src in (imgs, [im.to(dev) for im in imgs]):
            for a, b in zip(md.infer_u8_many(src, **kw), ref8):
                assert a.is_pinned() and a.dtype == torch.uint8 and torch.equal(a, b)


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]], ids=["2x0", "3x0"])
def test_large_and_lists_equal_single_gpu(sd, policy, devices):
    import resr_b200
    gen = _gen(sd)
    threads = threading.active_count()
    md = resr_b200.model.MultiDeviceInference(gen, devices)
    _check_large(gen, md, ["cuda:0"])
    _check_many(gen, md, ["cuda:0"])
    assert threading.active_count() == threads
    assert [e[0] for e in md.last_enqueue] == [torch.device("cuda", 0)] * len(devices)


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]], ids=["2x0", "3x0"])
def test_bf16_recipe(sd, devices):
    import resr_b200
    M = resr_b200.model
    gen = _gen(sd, "bf16")
    md = M.MultiDeviceInference(gen, devices)
    x, img = _images(1)
    assert torch.equal(md.infer_large(x, band_rows=BAND), M.infer_tiled(gen, x.cuda(), BAND, W, 16)[0].cpu())
    assert torch.equal(md.infer_u8_large(img, band_rows=BAND), _tiled_u8(gen, img, BAND))
    xs = [torch.rand(1, 3, h, w) for h, w in SIZES]
    for a, b in zip(md.infer_many(xs, max_pixels=BUDGET), gen.infer_many([t.cuda() for t in xs], max_pixels=BUDGET)):
        assert torch.equal(a, b.cpu())


def test_weight_changes_and_reused_out(sd):
    import resr_b200
    M = resr_b200.model
    gen = _gen(sd)
    md = M.MultiDeviceInference(gen, [0, 0])
    x, _ = _images(2)
    out = torch.empty((1, 3, 4 * H, 4 * W)).pin_memory()
    first = md.infer_large(x, out=out, band_rows=BAND).clone()
    assert md.infer_large(x, out=out, band_rows=BAND) is out and torch.equal(out, first)
    # an in-place optimizer-style update
    with torch.no_grad():
        gen.conv4.bias.add_(0.05)
    second = md.infer_large(x, out=out, band_rows=BAND).clone()
    assert not torch.equal(second, first)
    assert torch.equal(second, M.infer_tiled(gen, x.cuda(), BAND, W, 16)[0].cpu())
    # EMA.apply_shadow style: new storage behind a parameter
    gen.conv3[0].weight.data = gen.conv3[0].weight.data * 1.01
    third = md.infer_large(x, out=out, band_rows=BAND).clone()
    assert not torch.equal(third, second)
    assert torch.equal(third, M.infer_tiled(gen, x.cuda(), BAND, W, 16)[0].cpu())
    # a precision change
    gen.set_precision("bf16")
    assert torch.equal(md.infer_large(x, band_rows=BAND), M.infer_tiled(gen, x.cuda(), BAND, W, 16)[0].cpu())
    gen.set_precision("fp16")
    # static weights: the walk is skipped until invalidate()
    gen.assume_static_weights(True)
    assert torch.equal(md.infer_large(x, band_rows=BAND), third)
    with torch.no_grad():
        gen.conv4.bias.sub_(0.05)
    assert torch.equal(md.infer_large(x, band_rows=BAND), third)
    md.invalidate()
    assert torch.equal(md.infer_large(x, band_rows=BAND), M.infer_tiled(gen, x.cuda(), BAND, W, 16)[0].cpu())


def test_a_failing_replica_is_reported_after_all_threads_joined(sd):
    import resr_b200
    M = resr_b200.model
    gen = _gen(sd)
    md = M.MultiDeviceInference(gen, [0, 0, 0])
    x, _ = _images(3)
    good = md.infer_large(x, band_rows=BAND)
    threads = threading.active_count()

    def boom(*a, **k):
        raise RuntimeError("boom")

    md._replicas[1].infer = boom
    with pytest.raises(resr_b200._lib.ResrError, match=r"replica 1 on cuda:0 failed: RuntimeError: boom"):
        md.infer_large(x, band_rows=BAND)
    assert threading.active_count() == threads
    del md._replicas[1].infer
    assert torch.equal(md.infer_large(x, band_rows=BAND), good)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more visible GPUs")
def test_all_visible_gpus(sd, policy):
    import resr_b200
    gen = _gen(sd)
    threads = threading.active_count()
    md = resr_b200.model.MultiDeviceInference(gen)
    devices = [f"cuda:{i}" for i in range(torch.cuda.device_count())]
    _check_large(gen, md, devices)
    _check_many(gen, md, devices)
    assert threading.active_count() == threads
    assert len(md.devices) == torch.cuda.device_count()
