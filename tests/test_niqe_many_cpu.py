"""CPU: the list form of NIQE. Argument rejection of resr_niqe_many_workspace_bytes / resr_niqe_features_many before any
device work, and the batched Gaussian fit of iqa.py against the per-image loop it replaced."""
import ctypes

import numpy as np
import pytest
import torch


def _ints(v):
    return (ctypes.c_int * len(v))(*v)


def _loop_fit(feat, mu_pris, cov_pris):
    """The per-image fit as iqa.niqe_from_features computed it before the fit was batched (one image at a time)."""
    mu_pris, cov_pris = mu_pris.to(feat), cov_pris.to(feat)
    out = []
    for f in feat:
        nan_rows = torch.isnan(f).any(dim=1)
        nan = torch.isnan(f)
        mu = torch.where(nan, torch.zeros_like(f), f).sum(0) / (~nan).to(f).sum(0)
        g = f[~nan_rows]
        g = g - g.mean(0, keepdim=True)
        cov = g.t() @ g / (g.shape[0] - 1)
        inv = torch.linalg.pinv((cov_pris + cov) / 2)
        d = (mu_pris - mu).unsqueeze(0)
        out.append(torch.sqrt(d @ inv @ d.t()).reshape(()))
    return torch.stack(out)


def _pristine(rng):
    a = rng.normal(0, 0.3, (36, 36))
    return torch.from_numpy(rng.normal(0, 1, 36)), torch.from_numpy(a @ a.T + 0.05 * np.eye(36))


def test_many_workspace_bytes_rejects_bad_arguments():
    import resr_b200
    lib = resr_b200._lib.lib()
    ok = lib.resr_niqe_many_workspace_bytes(_ints([200, 104]), _ints([304, 104]), 2, 4, 96)
    assert ok > 0
    assert ok >= lib.resr_niqe_many_workspace_bytes(_ints([200]), _ints([304]), 1, 4, 96)
    bad = [
        (_ints([200, 90]), _ints([304, 200]), 2, 0, 96),     # image 1 holds no block
        (_ints([200, 0]), _ints([304, 200]), 2, 0, 96),      # empty
        (_ints([200, -5]), _ints([304, 200]), 2, 0, 96),     # negative
        (_ints([200]), _ints([304]), 0, 0, 96),              # no image
        (_ints([200]), _ints([304]), -1, 0, 96),
        (_ints([200]), _ints([304]), 1, 0, 95),              # odd block
        (_ints([200]), _ints([304]), 1, 0, 0),
        (_ints([200]), _ints([304]), 1, -1, 96),
        (None, _ints([304]), 1, 0, 96),
        (_ints([200]), None, 1, 0, 96),
    ]
    for args in bad:
        assert lib.resr_niqe_many_workspace_bytes(*args) == 0, args


def test_features_many_rejects_bad_arguments_without_a_device():
    """Every rejection returns RESR_E_INVALID before the device is touched, so it runs without a GPU; the message names
    the offending image."""
    import resr_b200
    lib = resr_b200._lib.lib()
    fake = ctypes.c_void_p(0x10000)                          # never dereferenced: the call must fail before any device work
    imgs = (ctypes.c_void_p * 3)(0x10000, 0x20000, 0x30000)
    offs = (ctypes.c_int * 4)()

    def call(images, hs, ws, n, border=4, block=96, feat=fake, offsets=offs):
        return lib.resr_niqe_features_many(images, hs, ws, n, border, block, feat, offsets, fake, 1 << 30, None)

    def msg():
        return lib.resr_last_error().decode()

    assert call(imgs, _ints([200, 104, 90]), _ints([304, 104, 200]), 3) == 1
    assert "image 2" in msg()
    assert call(imgs, _ints([200, 0, 200]), _ints([304, 104, 200]), 3) == 1
    assert "image 1" in msg()
    assert call(imgs, _ints([200, 104, 200]), _ints([-3, 104, 200]), 3) == 1
    assert "image 0" in msg()
    assert call(imgs, _ints([200]), _ints([304]), 0) == 1
    assert call(imgs, _ints([200]), _ints([304]), 1, block=97) == 1
    assert call(imgs, _ints([200]), _ints([304]), 1, border=-1) == 1
    assert call(None, _ints([200]), _ints([304]), 1) == 1
    assert call(imgs, None, _ints([304]), 1) == 1
    assert call(imgs, _ints([200]), _ints([304]), 1, feat=None) == 1
    assert call(imgs, _ints([200]), _ints([304]), 1, offsets=None) == 1
    nul = (ctypes.c_void_p * 2)(0x10000, None)
    assert call(nul, _ints([200, 200]), _ints([304, 304]), 2) == 1
    assert "image pointer 1" in msg()


def test_many_workspace_is_the_batch_workspace_for_equal_images():
    import resr_b200
    lib = resr_b200._lib.lib()
    for b, h, w, border in [(1, 200, 304, 4), (3, 97, 193, 0), (2, 400, 520, 4)]:
        assert lib.resr_niqe_many_workspace_bytes(_ints([h] * b), _ints([w] * b), b, border, 96) == \
            lib.resr_niqe_workspace_bytes(b, h, w, border, 96)


def test_batched_fit_matches_the_per_image_loop():
    import resr_b200
    iqa = resr_b200.iqa
    rng = np.random.default_rng(11)
    mu, cov = _pristine(rng)
    feats = []
    for nb in [3, 6, 40, 17, 2, 9, 9]:
        f = torch.from_numpy(rng.normal(0.5, 0.2, (nb, 36)) * rng.uniform(0.5, 2.0, 36))
        feats.append(f)
    feats[1][2, 5] = float("nan")                            # one NaN row
    feats[2][[0, 3, 39], 7] = float("nan")                   # several NaN rows, one column
    feats[2][10, :] = float("nan")                           # a row that is NaN everywhere
    feats[3][4, [1, 30]] = float("nan")
    feats[5][:, 0] = float("nan")                            # every block NaN in one column: the column mean is NaN
    feats[6][range(9), range(9)] = float("nan")              # every block has a NaN, no column is all NaN: covariance -0
    got = iqa.niqe_from_feature_list(feats, mu, cov)
    want = torch.cat([_loop_fit(f.unsqueeze(0), mu, cov) for f in feats])
    assert got.dtype == torch.float64 and got.shape == (len(feats),)
    assert torch.isnan(got[5]) and torch.isnan(want[5])
    keep = [i for i in range(len(feats)) if i != 5]
    rel = ((got[keep] - want[keep]).abs() / want[keep].abs()).max().item()
    assert rel <= 1e-12, rel
    # a batch of equally sized images through niqe_from_features is the same fit
    batch = torch.stack([feats[4], torch.from_numpy(rng.normal(0.5, 0.2, (2, 36)))])
    got_b = iqa.niqe_from_features(batch, mu, cov)
    want_b = _loop_fit(batch, mu, cov)
    assert ((got_b - want_b).abs() / want_b.abs()).max().item() <= 1e-12


def test_list_entry_points_reject_cpu_tensors():
    import resr_b200
    iqa = resr_b200.iqa
    with pytest.raises(resr_b200._lib.ResrError):
        iqa.niqe_features_many([torch.zeros(1, 3, 100, 100)], 0)
    with pytest.raises(resr_b200._lib.ResrError):
        iqa.niqe_many([torch.zeros(3, 100, 100)], 0, (np.zeros(36), np.eye(36)))
    assert iqa.niqe_features_many([], 4) == []
    out = iqa.NIQE(4, (np.zeros(36), np.eye(36))).forward_many([])
    assert out.dtype == torch.float64 and out.shape == (0,)
