"""CPU: the shelf packer of the packed-canvas forward (resr_canvas_pack) and the argument checks of
Generator.infer_many / infer_u8_many that run before any device work."""
import numpy as np
import pytest
import torch


def _pack(sizes, max_width=0):
    import resr_b200
    return resr_b200._lib.canvas_pack(sizes, max_width)


def _check_layout(sizes, pos, canvas, max_width=0):
    ch, cw = canvas
    assert ch % 16 == 0 and cw % 128 == 0 and ch > 0 and cw > 0
    h = np.array([s[0] for s in sizes], np.int64)
    w = np.array([s[1] for s in sizes], np.int64)
    x0 = np.array([p[0] for p in pos], np.int64)
    y0 = np.array([p[1] for p in pos], np.int64)
    assert (x0 >= 0).all() and (y0 >= 0).all() and (x0 + w <= cw).all() and (y0 + h <= ch).all()
    if max_width > 0:
        assert (x0 + w <= max_width).all()
    # every pair is separated by a gutter of at least one pixel along x or along y
    gap_x = np.maximum(x0[:, None] - (x0 + w)[None, :], x0[None, :] - (x0 + w)[:, None])
    gap_y = np.maximum(y0[:, None] - (y0 + h)[None, :], y0[None, :] - (y0 + h)[:, None])
    sep = (gap_x >= 1) | (gap_y >= 1)
    np.fill_diagonal(sep, True)
    assert sep.all()


@pytest.mark.parametrize("seed", range(8))
def test_packer_random_lists(seed):
    rng = np.random.default_rng(seed)
    count = int(rng.integers(1, 300))
    if seed % 2:
        sizes = [(int(rng.integers(1, 601)), int(rng.integers(1, 41))) for _ in range(count)]
    else:
        sizes = [(int(rng.integers(1, 41)), int(rng.integers(1, 601))) for _ in range(count)]
    pos, canvas = _pack(sizes)
    _check_layout(sizes, pos, canvas)
    assert _pack(sizes) == (pos, canvas)                         # deterministic
    area = sum((h + 1) * (w + 1) for h, w in sizes)
    assert canvas[0] * canvas[1] <= 4 * area + 16 * 128 * 8      # a packing, not a diagonal
    mw = max(w for _, w in sizes) + int(rng.integers(0, 200))
    pos2, canvas2 = _pack(sizes, mw)
    _check_layout(sizes, pos2, canvas2, mw)


def test_packer_buckets_and_small_cases():
    pos, canvas = _pack([(1, 1)])
    assert pos == [(0, 0)] and canvas == (16, 128)
    sizes = [(1, 7), (5, 3), (17, 129), (64, 64), (128, 128), (130, 77), (200, 31), (33, 65), (9, 255)]
    pos, canvas = _pack(sizes)
    _check_layout(sizes, pos, canvas)
    # one shelf: images side by side with exactly one gutter column
    pos, canvas = _pack([(10, 10)] * 3, 128)
    assert pos == [(0, 0), (11, 0), (22, 0)] and canvas == (16, 128)
    pos, canvas = _pack([(10, 10)] * 3, 21)
    assert pos == [(0, 0), (11, 0), (0, 11)] and canvas == (32, 128)


def test_packer_rejects_bad_sizes():
    import resr_b200
    L = resr_b200._lib
    for sizes, mw in (([(0, 3)], 0), ([(3, -1)], 0), ([(3, 300)], 100), ([(20000, 3)], 0)):
        with pytest.raises(L.ResrError):
            _pack(sizes, mw)
    assert L.lib().resr_canvas_pack(None, None, 0, 0, None, None, None, None) == 1


def test_infer_many_argument_checks_without_device_work():
    import resr_b200
    g = resr_b200.model.Generator(3, 3, 4)
    assert g.infer_many([]) == [] and g.infer_u8_many([]) == []
    with pytest.raises(ValueError):
        g.infer_many([torch.rand(1, 4, 8, 8)])
    with pytest.raises(ValueError):
        g.infer_many([torch.rand(2, 3, 8, 8)])
    with pytest.raises(ValueError):
        g.infer_u8_many([torch.zeros(8, 8, 4, dtype=torch.uint8)])
    with pytest.raises(ValueError):
        g.infer_u8_many([torch.zeros(8, 8, 3)])
    with pytest.raises(resr_b200._lib.ResrError):
        g.infer_many([torch.rand(1, 3, 8, 8)])     # a CPU tensor: there is no CPU path
    with pytest.raises(resr_b200._lib.ResrError):
        g.infer_u8_many([torch.zeros(8, 8, 3, dtype=torch.uint8)])
