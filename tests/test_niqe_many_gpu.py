"""NIQE of a list of differently sized images in one call (resr_niqe_features_many, iqa.niqe_features_many / niqe_many /
NIQE.forward_many) against the single-image path (bit for bit), the reference golden scores and the numpy oracle."""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# Block 96 after cropping: odd sides, one pixel above / below a block multiple, exactly one block, one much larger image.
SIZES = {
    4: [(104, 104), (201, 297), (199, 105), (105, 199), (200, 304), (297, 391), (611, 803), (193, 201), (392, 104)],
    0: [(96, 96), (97, 193), (191, 289), (192, 287), (193, 97), (289, 385), (500, 700), (96, 481)],
}


def _rows(a):
    return np.array(sorted(map(tuple, a)))


def _pristine(seed):
    rng = np.random.default_rng(seed)
    a = rng.normal(0, 0.3, (36, 36))
    return rng.normal(0, 1, 36), a @ a.T + 0.05 * np.eye(36)


def _images(sizes, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = []
    for i, (h, w) in enumerate(sizes):
        x = torch.rand(1, 3, h, w, device="cuda", generator=g)
        out.append(x if i % 2 == 0 else x[0])     # both accepted forms: [1, 3, h, w] and [3, h, w]
    return out


@pytest.mark.parametrize("border", [0, 4])
def test_list_features_equal_single_image_features_bit_for_bit(border):
    import resr_b200
    iqa = resr_b200.iqa
    xs = _images(SIZES[border], 10 + border)
    many = iqa.niqe_features_many(xs, border)
    assert len(many) == len(xs)
    base = many[0]._base if many[0]._base is not None else many[0]
    for i, (x, f) in enumerate(zip(xs, many)):
        single = iqa.niqe_features(x.reshape(1, *x.shape[-3:]), border)[0]
        assert f.dtype == torch.float64 and f.shape == single.shape, (i, f.shape, single.shape)
        assert (f._base if f._base is not None else f) is base       # views of one device tensor
        assert torch.equal(f, single), f"image {i} {tuple(x.shape)}: list features differ from the single-image call"


def test_list_scores_match_the_single_image_metric():
    """Images with at least two blocks: the covariance of a single block row is 0 / 0 (as in the reference's nancov), and
    torch.linalg.pinv refuses it."""
    import resr_b200
    iqa = resr_b200.iqa
    lib = resr_b200._lib.lib()
    mu, cov = _pristine(5)
    for border in (0, 4):
        sizes = [(h, w) for h, w in SIZES[border] if lib.resr_niqe_num_blocks(h, w, border, 96) >= 2]
        xs = _images(sizes, 20 + border)
        got = iqa.niqe_many(xs, border, (mu, cov))
        metric = iqa.NIQE(border, (mu, cov))
        assert got.dtype == torch.float64 and got.shape == (len(xs),) and got.is_cuda
        assert torch.equal(metric.forward_many(xs), got)
        for i, x in enumerate(xs):
            want = metric(x.reshape(1, *x.shape[-3:])).item()
            assert abs(got[i].item() - want) <= 1e-6 * abs(want), (border, i, got[i].item(), want)


def test_golden_images_as_lists_meet_the_reference_bounds():
    """crop_border belongs to a call, so the golden images go in one list per border: the two images of case 0 and the
    image of case 2 (border 4), the image of case 1 (border 0)."""
    import resr_b200
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "niqe.npz"))
    mu, cov = g["mu_prisparam"], g["cov_prisparam"]
    imgs, feats, scores, borders = [], [], [], []
    for ci in range(3):
        x = torch.from_numpy(g[f"x{ci}"].astype(np.float32) / np.float32(255.0)).cuda()
        for b in range(x.shape[0]):
            imgs.append(x[b])
            feats.append(g[f"feat{ci}"][b])
            scores.append(g[f"niqe{ci}"][b])
            borders.append(int(g[f"border{ci}"]))
    for border in sorted(set(borders)):
        idx = [i for i, bd in enumerate(borders) if bd == border]
        got_f = resr_b200.iqa.niqe_features_many([imgs[i] for i in idx], border)
        got_s = resr_b200.iqa.niqe_many([imgs[i] for i in idx], border, (mu, cov)).cpu().numpy()
        for k, i in enumerate(idx):
            assert np.abs(_rows(got_f[k].cpu().numpy()) - _rows(feats[i])).max() <= 1e-6
            assert abs(got_s[k] - scores[i]) <= 1e-6 * scores[i], (i, got_s[k], scores[i])


def test_list_with_the_large_oracle_image_matches_the_oracle():
    import resr_b200
    from oracle import niqe as on
    rng = np.random.default_rng(3)
    big = rng.integers(0, 256, (1, 3, 400, 520)).astype(np.float32) / np.float32(255.0)   # as in test_niqe_gpu.py
    a = rng.normal(0, 0.3, (36, 36))
    mu, cov = rng.normal(0, 1, 36), a @ a.T + 0.05 * np.eye(36)
    others = [rng.integers(0, 256, (1, 3, h, w)).astype(np.float32) / np.float32(255.0) for h, w in [(113, 205), (211, 107)]]
    xs = [others[0], big, others[1]]
    got_f = resr_b200.iqa.niqe_features_many([torch.from_numpy(x).cuda() for x in xs], 4)
    got_s = resr_b200.iqa.niqe_many([torch.from_numpy(x).cuda() for x in xs], 4, (mu, cov)).cpu().numpy()
    for i, x in enumerate(xs):
        score, feat = on.niqe(x, 4, mu, cov)
        assert np.abs(_rows(got_f[i].cpu().numpy()) - _rows(feat[0])).max() <= 1e-6, i
        assert abs(got_s[i] - score[0]) <= 1e-6 * score[0], (i, got_s[i], score[0])


def test_changing_one_image_leaves_the_others_bit_identical():
    import resr_b200
    iqa = resr_b200.iqa
    xs = _images(SIZES[4], 30)
    before = [f.clone() for f in iqa.niqe_features_many(xs, 4)]
    k = 3
    xs[k] = torch.rand_like(xs[k])
    after = iqa.niqe_features_many(xs, 4)
    for i in range(len(xs)):
        if i == k:
            assert not torch.equal(after[i], before[i])
        else:
            assert torch.equal(after[i], before[i]), i


def test_constant_blocks_match_the_single_image_path():
    """Blocks of one colour each (flat MSCN coefficients: the AGGD fit meets 0 / 0) next to a textured image."""
    import resr_b200
    iqa = resr_b200.iqa
    mu, cov = _pristine(7)
    flat = torch.empty(1, 3, 2 * 96, 3 * 96, device="cuda")
    colours = torch.tensor([[0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [0.2, 0.5, 0.7], [0.9, 0.1, 0.3], [0.5, 0.5, 0.5], [0.3, 0.3, 0.0]])
    for b in range(6):
        r, c = divmod(b, 3)
        flat[0, :, r * 96:(r + 1) * 96, c * 96:(c + 1) * 96] = colours[b].view(3, 1, 1).to("cuda")
    xs = [torch.rand(1, 3, 200, 210, device="cuda"), flat]
    many = iqa.niqe_features_many(xs, 0)
    single = iqa.niqe_features(flat, 0)[0]
    torch.testing.assert_close(many[1], single, rtol=0, atol=0, equal_nan=True)
    got = iqa.niqe_many(xs, 0, (mu, cov))[1].item()
    want = iqa.NIQE(0, (mu, cov))(flat).item()
    assert (np.isnan(got) and np.isnan(want)) or abs(got - want) <= 1e-6 * abs(want), (got, want)


def test_errors_and_empty_lists():
    import resr_b200
    iqa, L = resr_b200.iqa, resr_b200._lib
    xs = _images([(200, 200), (104, 104), (103, 300), (300, 300)], 40)
    with pytest.raises(ValueError, match="image 2"):
        iqa.niqe_features_many(xs, 4)
    with pytest.raises(ValueError, match="image 2"):
        iqa.niqe_many(xs, 4, _pristine(1))
    assert iqa.niqe_features_many([], 4) == []
    assert iqa.niqe_many([], 4, _pristine(1)).shape == (0,)
    # a workspace one byte short is refused through the C ABI
    lib = L.lib()
    ok = [xs[0], xs[1], xs[3]]
    n = len(ok)
    hs = (ctypes.c_int * n)(*[x.shape[-2] for x in ok])
    ws = (ctypes.c_int * n)(*[x.shape[-1] for x in ok])
    ptrs = (ctypes.c_void_p * n)(*[x.data_ptr() for x in ok])
    offs = (ctypes.c_int * (n + 1))()
    need = lib.resr_niqe_many_workspace_bytes(hs, ws, n, 4, 96)
    work = torch.empty(need, dtype=torch.uint8, device="cuda")
    feat = torch.empty(4 + 1 + 9, 36, dtype=torch.float64, device="cuda")
    stream = L.stream_ptr()
    assert lib.resr_niqe_features_many(ptrs, hs, ws, n, 4, 96, L.ptr(feat), offs, L.ptr(work), need - 1, stream) == 3
    assert lib.resr_niqe_features_many(ptrs, hs, ws, n, 4, 96, L.ptr(feat), offs, L.ptr(work), need, stream) == 0
    assert list(offs) == [0, 4, 5, 14]
    torch.cuda.synchronize()
