"""CPU: the VGG19 content loss (resr_b200.model.ContentLoss, C ABI resr_vgg_*) -- node parsing, argument checks of the C
ABI before any device work, the workspace formula, and the no-download rule of vgg=None."""
import ctypes
import socket

import pytest
import torch

REALESRGAN_NODES = ["features.2", "features.7", "features.16", "features.25", "features.34"]
MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
CONV_FEATURES = (0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34)
CIN = (3, 64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512)
COUT = (64, 64, 128, 128, 256, 256, 256, 256, 512, 512, 512, 512, 512, 512, 512, 512)
POOL_AFTER = (1, 3, 7, 11)


def _vgg_sd():
    from torchvision.models import vgg19
    torch.manual_seed(0)
    return vgg19(weights=None).state_dict()


def _create(features, mean=MEAN, std=STD):
    import resr_b200
    L = resr_b200._lib
    h = ctypes.c_void_p()
    arr = (ctypes.c_int * max(len(features), 1))(*features)
    rc = L.lib().resr_vgg_create(ctypes.byref(h), arr, len(features), (ctypes.c_float * 3)(*mean), (ctypes.c_float * 3)(*std))
    return rc, h


def test_node_names_parse_in_order_and_bad_ones_raise():
    import resr_b200
    parse = resr_b200.model.parse_vgg19_nodes
    assert parse(REALESRGAN_NODES) == [2, 7, 16, 25, 34]
    assert parse(["features.34", "features.0"]) == [34, 0]
    for bad in (["features.3"], ["features.36"], ["features.02"], ["classifier.0"], ["features.2", "features.2"], [],
                ["features.-2"], ["features"]):
        with pytest.raises(ValueError) as e:
            parse(bad)
        if bad and bad[0] == "features.3":
            assert "features.34" in str(e.value)   # the message lists the supported nodes
    sd = _vgg_sd()
    with pytest.raises(ValueError):
        resr_b200.model.ContentLoss(["features.4"], MEAN, STD, vgg=sd)
    with pytest.raises(ValueError):
        resr_b200.model.ContentLoss(["features.2"], MEAN, [0.2, 0.0, 0.2], vgg=sd)
    m = resr_b200.model.ContentLoss(REALESRGAN_NODES, MEAN, STD, vgg=sd)
    assert all(torch.equal(m.state_dict()[k], sd[k]) for k in m.state_dict())   # torchvision keys load unchanged
    assert not any(p.requires_grad for p in m.parameters())
    assert sum(p.numel() for p in m.parameters()) == resr_b200._lib.lib().resr_vgg_num_params() == 20024384
    with pytest.raises(resr_b200._lib.ResrError):   # no CPU path
        m(torch.rand(1, 3, 32, 32), torch.rand(1, 3, 32, 32))


def test_c_abi_rejects_bad_arguments_before_device_work():
    import resr_b200
    L = resr_b200._lib
    lib = L.lib()
    assert _create([3])[0] == 1
    assert b"features.3" in lib.resr_last_error()
    assert _create([2, 2])[0] == 1
    assert _create([])[0] == 1
    assert _create([2], std=[0.2, 0.0, 0.2])[0] == 1
    assert _create([2], mean=[float("nan"), 0, 0])[0] == 1
    assert lib.resr_vgg_create(None, None, 1, None, None) == 1
    rc, h = _create([2, 34])
    assert rc == 0   # creation is host-only
    try:
        # Never dereferenced, with or without a device: the handle's weights are never loaded and it holds no forward, so
        # every call below fails its host checks before any device work.
        ws = ctypes.c_void_p(1 << 20)
        big = lib.resr_vgg_workspace_bytes(h, 2, 64, 64)
        p = ctypes.c_void_p(4096)
        assert lib.resr_vgg_forward(h, None, p, p, 2, 64, 64, ws, big, None) == 1
        assert lib.resr_vgg_forward(h, p, p, p, 0, 64, 64, ws, big, None) == 1
        assert lib.resr_vgg_forward(h, p, p, p, 2, 15, 64, ws, big, None) == 1   # no pixel left at features.34
        assert b"features.34" in lib.resr_last_error()
        assert lib.resr_vgg_forward(h, p, p, p, 2, 64, 64, ws, big - 1, None) == 1
        assert lib.resr_vgg_forward(h, p, p, p, 2, 64, 64, ctypes.c_void_p((1 << 20) + 16), big, None) == 1
        assert lib.resr_vgg_forward(h, p, p, p, 2, 64, 64, ws, big, None) == 1   # weights never loaded
        assert lib.resr_vgg_backward(h, p, p, 2, 64, 64, ws, big, None) == 1     # no forward in this workspace
        assert lib.resr_vgg_backward(h, None, p, 2, 64, 64, ws, big, None) == 1
        assert lib.resr_vgg_load_params(h, None, None) == 1
    finally:
        lib.resr_vgg_destroy(h)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device error; with a device the call would pack weights")
def test_loading_weights_without_a_device_fails_with_resr_e_cuda():
    import resr_b200
    lib = resr_b200._lib.lib()
    rc, h = _create([2, 34])
    assert rc == 0
    try:
        # the pointer is never dereferenced: without a CUDA device the call stops at the device query
        assert lib.resr_vgg_load_params(h, ctypes.c_void_p(4096), None) == 2
        assert b"device" in lib.resr_last_error()
    finally:
        lib.resr_vgg_destroy(h)


def _ws_formula(features, n, h, w):
    """Restatement of the workspace layout: 1024-aligned buffers in this order -- the 8-channel fp16 input of the 2n batch,
    per conv its fp16 output (2n) and the pooled map after it, one fp32 split-K partial, two bf16 gradient buffers, the
    fp64 loss partial sums."""
    up = lambda v: (v + 1023) // 1024 * 1024
    deepest = max(CONV_FEATURES.index(f) for f in features)
    total = up(2 * n * h * w * 8 * 2)
    partial = g = 0
    for i in range(deepest + 1):
        p = n * h * w
        total += up(2 * p * COUT[i] * 2)
        if CIN[i] > 256:
            partial = max(partial, 2 * p * COUT[i] * 4)
        if COUT[i] > 256:
            partial = max(partial, p * CIN[i] * 4)
        g = max(g, p * COUT[i] * 2, p * CIN[i] * 2 if i else 0)
        if i in POOL_AFTER and i < deepest:
            h, w = h // 2, w // 2
            total += up(2 * n * h * w * COUT[i] * 2)
    total += (up(partial) if partial else 0) + 2 * up(g) + up(16 * 296 * 8)
    return total


@pytest.mark.parametrize("features", [[2, 7, 16, 25, 34], [0], [34], list(CONV_FEATURES), [19, 5]])
def test_workspace_formula(features):
    import resr_b200
    lib = resr_b200._lib.lib()
    rc, h = _create(features)
    assert rc == 0
    try:
        need = 1 << [0, 0, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4][max(CONV_FEATURES.index(f) for f in features)]
        for n, hh, ww in [(16, 256, 256), (1, 37, 53), (3, 16, 24), (2, 19, 200), (1, need, need)]:
            assert lib.resr_vgg_workspace_bytes(h, n, hh, ww) == _ws_formula(features, n, hh, ww)
        if need > 1:   # one row / column short of a pixel at the deepest node
            assert lib.resr_vgg_workspace_bytes(h, 1, need, need - 1) == 0
            assert lib.resr_vgg_workspace_bytes(h, 1, need - 1, need) == 0
        assert lib.resr_vgg_workspace_bytes(h, 0, 64, 64) == 0
    finally:
        lib.resr_vgg_destroy(h)


def test_default_weights_are_never_downloaded(tmp_path, monkeypatch):
    import resr_b200
    monkeypatch.setenv("TORCH_HOME", str(tmp_path))
    monkeypatch.setattr(torch.hub, "_hub_dir", None, raising=False)

    def no_network(*a, **k):
        raise AssertionError("ContentLoss(vgg=None) tried to open a network connection")

    monkeypatch.setattr(socket, "create_connection", no_network)
    monkeypatch.setattr(socket.socket, "connect", no_network)
    with pytest.raises(FileNotFoundError) as e:
        resr_b200.model.ContentLoss(REALESRGAN_NODES, MEAN, STD)
    assert "vgg19-dcbb9e9d.pth" in str(e.value) and str(tmp_path) in str(e.value)
    # the same file, present, is what vgg=None loads
    ckpt = tmp_path / "hub" / "checkpoints"
    ckpt.mkdir(parents=True)
    sd = _vgg_sd()
    torch.save(sd, ckpt / "vgg19-dcbb9e9d.pth")
    m = resr_b200.model.ContentLoss(REALESRGAN_NODES, MEAN, STD)
    assert torch.equal(m.features["34"].weight, sd["features.34.weight"])
