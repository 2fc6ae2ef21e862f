"""CPU: the host side of model.MultiDeviceInference. The band plan of a large image, the grouping and dealing of a list,
replica parameter layout, and input checks that raise before any device work."""
import random

import pytest
import torch

import resr_b200
from resr_b200 import model as M


def _groups_of_infer_many(sizes, max_pixels):
    """The grouping loop Generator._run_many ran before it moved into canvas_groups: consecutive images, up to
    max_pixels LR pixels per canvas."""
    groups, cur, px = [], [], 0
    for i, (hh, ww) in enumerate(sizes):
        if cur and px + hh * ww > max_pixels:
            groups.append(cur)
            cur, px = [], 0
        cur.append(i)
        px += hh * ww
    groups.append(cur)
    return groups


@pytest.mark.parametrize("h,w", [(1, 1), (5, 7), (16, 3), (100, 48), (2048, 2048), (8192, 8192), (3000, 20000), (997, 1)])
@pytest.mark.parametrize("replicas", [1, 2, 3, 8])
def test_default_band_plan_covers_once_and_feeds_every_replica(h, w, replicas):
    rows = M.default_band_rows(h, w, replicas)
    assert rows >= 1
    bands = M.plan_tiles(h, w, rows, w, 16)
    hit = [0] * h
    for y0, y1, x0, x1, wy0, wy1, wx0, wx1 in bands:
        assert (x0, x1, wx0, wx1) == (0, w, 0, w)          # full-width bands
        assert wy0 == max(y0 - 16, 0) and wy1 == min(y1 + 16, h)
        for y in range(y0, y1):
            hit[y] += 1
    assert hit == [1] * h
    per_replica = [len(bands[r::replicas]) for r in range(replicas)]
    if h >= 2 * replicas:
        assert min(per_replica) >= 2, per_replica
    assert rows * w <= max(M.CANVAS_MAX_PIXELS, w)        # the workspace of a band stays bounded


def test_canvas_groups_are_the_infer_many_canvases():
    rng = random.Random(3)
    for _ in range(200):
        sizes = [(rng.randint(1, 300), rng.randint(1, 300)) for _ in range(rng.randint(1, 40))]
        budget = rng.choice([1, 1000, 20000, 90000, M.CANVAS_MAX_PIXELS])
        assert M.canvas_groups(sizes, budget) == _groups_of_infer_many(sizes, budget)
    assert M.canvas_groups([]) == []


@pytest.mark.parametrize("replicas", [1, 2, 3, 8])
def test_deal_groups_every_image_once_largest_first_deterministic(replicas):
    rng = random.Random(replicas)
    for _ in range(50):
        sizes = [(rng.randint(1, 200), rng.randint(1, 200)) for _ in range(rng.randint(1, 64))]
        budget = rng.choice([5000, 40000, M.CANVAS_MAX_PIXELS])
        groups, dealt = M.deal_groups(sizes, replicas, budget)
        assert groups == _groups_of_infer_many(sizes, budget)
        assert sorted(k for d in dealt for k in d) == list(range(len(groups)))       # every canvas on one replica
        assert sorted(i for d in dealt for k in d for i in groups[k]) == list(range(len(sizes)))
        assert (groups, dealt) == M.deal_groups(list(sizes), replicas, budget)       # deterministic
        # the rule, replayed: largest canvas first onto the least loaded replica (ties: earlier canvas, lower replica)
        work = [sum(sizes[i][0] * sizes[i][1] for i in g) for g in groups]
        load, owner = [0] * replicas, {}
        for k in sorted(range(len(groups)), key=lambda k: (-work[k], k)):
            r = min(range(replicas), key=lambda r: (load[r], r))
            owner[k] = r
            load[r] += work[k]
        assert all(owner[k] == r for r, d in enumerate(dealt) for k in d)
        assert all(work[a] >= work[b] for d in dealt for a, b in zip(d, d[1:]))     # each replica runs largest first


def test_deal_groups_spreads_equal_canvases():
    groups, dealt = M.deal_groups([(100, 100)] * 8, 4, 20000)
    assert groups == [[0, 1], [2, 3], [4, 5], [6, 7]]
    assert dealt == [[0], [1], [2], [3]]


def test_replica_parameters_are_views_of_one_flat_vector():
    """A replica packs straight from its flat vector: the views must follow flat_parameters() order."""
    rep = M.MultiDeviceInference._replica(torch.device("cpu"))
    rep._flat_master.copy_(torch.arange(rep._flat_master.numel(), dtype=torch.float32))
    assert torch.equal(rep.flat_parameters(), rep._flat_master)
    assert next(rep.parameters()).data_ptr() == rep._flat_master.data_ptr()
    assert rep._static_weights and not any(p.requires_grad for p in rep.parameters())


def test_replicas_do_not_draw_from_the_global_rng():
    state = torch.random.get_rng_state()
    M.MultiDeviceInference._replica(torch.device("cpu"))
    assert torch.equal(state, torch.random.get_rng_state())


def test_bad_input_raises_before_device_work(monkeypatch):
    calls = []
    monkeypatch.setattr(M.MultiDeviceInference, "_check_devices", lambda self: calls.append(1))
    md = M.MultiDeviceInference(M.Generator(3, 3, 4), [0, 0])
    bad = [
        lambda: md.infer_many([]),
        lambda: md.infer_u8_many([]),
        lambda: md.infer_many([torch.zeros(2, 3, 8, 8)]),
        lambda: md.infer_many([torch.zeros(1, 4, 8, 8)]),
        lambda: md.infer_many([torch.zeros(1, 3, 8, 8, dtype=torch.uint8)]),
        lambda: md.infer_many([torch.zeros(1, 3, 0, 8)]),
        lambda: md.infer_u8_many([torch.zeros(8, 8, 3)]),
        lambda: md.infer_u8_many([torch.zeros(8, 8, 4, dtype=torch.uint8)]),
        lambda: md.infer_many([torch.zeros(3, 8, 8)], max_pixels=0),
        lambda: md.infer_large(torch.zeros(3, 8, 8)),
        lambda: md.infer_large(torch.zeros(2, 3, 8, 8)),
        lambda: md.infer_large(torch.zeros(1, 3, 8, 8, dtype=torch.float64)),
        lambda: md.infer_large(torch.zeros(1, 3, 0, 8)),
        lambda: md.infer_large(torch.zeros(1, 3, 8, 8), band_rows=0),
        lambda: md.infer_large(torch.zeros(1, 3, 8, 8), halo=-1),
        lambda: md.infer_large(torch.zeros(1, 3, 8, 8), out=torch.zeros(1, 3, 32, 31)),
        lambda: md.infer_large(torch.zeros(1, 3, 8, 8), out=torch.zeros(1, 3, 32, 32, dtype=torch.float16)),
        lambda: md.infer_u8_large(torch.zeros(8, 8, 3)),
        lambda: md.infer_u8_large(torch.zeros(1, 8, 8, 3, dtype=torch.uint8)),
        lambda: md.infer_u8_large(torch.zeros(8, 8, 3, dtype=torch.uint8), out=torch.zeros(32, 32, 3)),
    ]
    for f in bad:
        with pytest.raises(ValueError):
            f()
    assert calls == []
    for devices in ([], ["cpu"], [torch.device("cuda")]):
        with pytest.raises(ValueError):
            M.MultiDeviceInference(M.Generator(3, 3, 4), devices)
    with pytest.raises(ValueError):
        M.MultiDeviceInference(torch.nn.Conv2d(3, 3, 3))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the machine without a CUDA device")
def test_no_device_raises_resr_error():
    md = M.MultiDeviceInference(M.Generator(3, 3, 4))
    with pytest.raises(resr_b200._lib.ResrError):
        md.infer_large(torch.zeros(1, 3, 8, 8))
    with pytest.raises(resr_b200._lib.ResrError):
        md.infer_u8_many([torch.zeros(8, 8, 3, dtype=torch.uint8)])
    assert md._replicas is None
