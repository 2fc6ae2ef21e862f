"""NIQE on the device: mirror of the reference's `NIQE` module (image_quality_assessment.py:1001-1033 -> `_niqe_torch`
:886-998). The per-block feature extraction (Y channel, MSCN coefficients, AGGD fits at two scales, MATLAB-style
half-size resize) runs in libresr.so (`resr_niqe_features`, csrc/niqe.cu, float64 like the reference); the 36-dimensional
Gaussian fit against the pristine statistics is a handful of torch.linalg calls on the same device. A list of
differently sized images (the per-image loops of test.py / validate()) runs as one feature call
(`resr_niqe_features_many`) and one batched fit: `niqe_many`, `NIQE.forward_many`.

The pristine statistics (`niqe_model.mat`, config.py:72) are a download: pass the path of the .mat file exactly as the
reference does, or the arrays themselves (`mu_prisparam` [36], `cov_prisparam` [36, 36])."""
import ctypes

import torch
from torch import nn

from . import _lib


def _load_pristine(model):
    if isinstance(model, (tuple, list)):
        mu, cov = model
    else:
        import numpy as np
        import scipy.io                                           # image_quality_assessment.py:976-979
        m = scipy.io.loadmat(model)
        mu, cov = np.ravel(m["mu_prisparam"]), m["cov_prisparam"]
    mu = torch.as_tensor(mu, dtype=torch.float64).reshape(-1)
    cov = torch.as_tensor(cov, dtype=torch.float64)
    if mu.numel() != 36 or tuple(cov.shape) != (36, 36):
        raise ValueError("pristine statistics must be a 36-vector and a 36 x 36 matrix")
    return mu, cov


def niqe_features(raw_tensor: torch.Tensor, crop_border: int, block_size: int = 96) -> torch.Tensor:
    """[b, 3, h, w] fp32 CUDA tensor in [0, 1] -> float64 [b, blocks, 36] (C ABI resr_niqe_features)."""
    if not raw_tensor.is_cuda:
        raise _lib.ResrError("resr_b200.iqa runs on CUDA tensors only; there is no CPU path")
    if raw_tensor.dim() != 4 or raw_tensor.size(1) != 3:
        raise ValueError("expected an RGB tensor [b, 3, h, w]")
    x = raw_tensor.detach().contiguous().float()
    b, _, h, w = x.shape
    lib = _lib.lib()
    nb = lib.resr_niqe_num_blocks(h, w, int(crop_border), int(block_size))
    if nb <= 0:
        raise ValueError(f"image {h}x{w} holds no {block_size}x{block_size} block after cropping {crop_border} pixels")
    with torch.cuda.device(x.device):
        need = lib.resr_niqe_workspace_bytes(b, h, w, int(crop_border), int(block_size))
        ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        feat = torch.empty(b, nb, 36, dtype=torch.float64, device=x.device)
        _lib.check(lib.resr_niqe_features(_lib.ptr(x), _lib.ptr(feat), b, h, w, int(crop_border), int(block_size), _lib.ptr(ws), need,
                                          _lib.stream_ptr(x.device)))
    return feat


def niqe_features_many(images, crop_border: int, block_size: int = 96):
    """Features of a list of differently sized images ([1, 3, h, w] or [3, h, w] fp32 CUDA tensors in [0, 1]) in one call
    (C ABI resr_niqe_features_many): a list of float64 [blocks_i, 36] views of one device tensor, in input order. Each equals
    niqe_features(image)[0] bit for bit."""
    xs = []
    for i, x in enumerate(images):
        if not x.is_cuda:
            raise _lib.ResrError("resr_b200.iqa runs on CUDA tensors only; there is no CPU path")
        if x.dim() not in (3, 4) or x.size(-3) != 3 or (x.dim() == 4 and x.size(0) != 1):
            raise ValueError(f"image {i}: expected a [1, 3, H, W] or [3, H, W] image, got {tuple(x.shape)}")
        if xs and x.device != xs[0].device:
            raise ValueError(f"image {i} is on {x.device}, image 0 on {xs[0].device}")
        xs.append(x.detach().float().contiguous())
    if not xs:
        return []
    lib = _lib.lib()
    n, dev = len(xs), xs[0].device
    sizes = [tuple(x.shape[-2:]) for x in xs]
    total = 0
    for i, (h, w) in enumerate(sizes):
        nb = lib.resr_niqe_num_blocks(h, w, int(crop_border), int(block_size))
        if nb <= 0:
            raise ValueError(f"image {i} ({h}x{w}) holds no {block_size}x{block_size} block after cropping {crop_border} pixels")
        total += nb
    hs = (ctypes.c_int * n)(*[h for h, _ in sizes])
    ws_ = (ctypes.c_int * n)(*[w for _, w in sizes])
    ptrs = (ctypes.c_void_p * n)(*[x.data_ptr() for x in xs])
    offsets = (ctypes.c_int * (n + 1))()
    with torch.cuda.device(dev):
        need = lib.resr_niqe_many_workspace_bytes(hs, ws_, n, int(crop_border), int(block_size))
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        feat = torch.empty(total, 36, dtype=torch.float64, device=dev)
        _lib.check(lib.resr_niqe_features_many(ptrs, hs, ws_, n, int(crop_border), int(block_size), _lib.ptr(feat), offsets,
                                               _lib.ptr(ws), need, _lib.stream_ptr(dev)))
    return [feat[offsets[i]:offsets[i + 1]] for i in range(n)]


def _gaussian_fit(feat: torch.Tensor, valid: torch.Tensor, mu_pris: torch.Tensor, cov_pris: torch.Tensor) -> torch.Tensor:
    """The multivariate-Gaussian distance of image_quality_assessment.py:879-884 (nanmean / nancov / pinv) for every image
    at once. feat: [n, m, 36]; valid: [n, m], False on the padding rows of images with fewer than m blocks. Rows with a NaN
    are dropped from the covariance (:631-644); the mean is taken per column over the values that are not NaN."""
    mu_pris, cov_pris = mu_pris.to(feat), cov_pris.to(feat)
    ok = ~torch.isnan(feat) & valid.unsqueeze(-1)
    mu = torch.where(ok, feat, 0.0).sum(1) / ok.sum(1).to(feat)
    rows = ok.all(-1, keepdim=True)
    nrows = rows.sum(1, keepdim=True).to(feat)
    g = torch.where(rows, feat - torch.where(rows, feat, 0.0).sum(1, keepdim=True) / nrows, 0.0)
    cov = g.transpose(1, 2) @ g / (nrows - 1)
    inv = torch.linalg.pinv((cov_pris + cov) / 2)
    d = (mu_pris - mu).unsqueeze(1)
    return torch.sqrt(d @ inv @ d.transpose(1, 2)).reshape(-1)


def niqe_from_features(feat: torch.Tensor, mu_pris: torch.Tensor, cov_pris: torch.Tensor) -> torch.Tensor:
    """NIQE per image of a batch of features [b, blocks, 36] -> float64 [b]."""
    return _gaussian_fit(feat, torch.ones(feat.shape[:2], dtype=torch.bool, device=feat.device), mu_pris, cov_pris)


def niqe_from_feature_list(feats, mu_pris: torch.Tensor, cov_pris: torch.Tensor) -> torch.Tensor:
    """NIQE per image of a list of [blocks_i, 36] feature tensors -> float64 [len(feats)]: the images are padded to the
    largest block count and fitted together (one batched pinv)."""
    counts = [f.shape[0] for f in feats]
    flat = torch.cat(list(feats))
    dev = flat.device
    cnt = torch.tensor(counts, device=dev)
    img = torch.repeat_interleave(torch.arange(len(counts), device=dev), cnt)
    pos = torch.arange(flat.shape[0], device=dev) - (torch.cumsum(cnt, 0) - cnt)[img]
    padded = flat.new_zeros(len(counts), max(counts), 36)
    padded[img, pos] = flat
    valid = torch.arange(max(counts), device=dev).unsqueeze(0) < cnt.unsqueeze(1)
    return _gaussian_fit(padded, valid, mu_pris, cov_pris)


def niqe_many(images, crop_border: int, pristine, block_size: int = 96) -> torch.Tensor:
    """NIQE of a list of differently sized images ([1, 3, h, w] or [3, h, w] fp32 CUDA tensors in [0, 1]) -> float64 scores
    in input order, on the images' device (an empty list gives an empty CPU tensor). `pristine`: the path of
    niqe_model.mat or (mu_prisparam, cov_prisparam), as for NIQE. One feature call and one Gaussian fit for the list."""
    feats = niqe_features_many(images, crop_border, block_size)
    if not feats:
        return torch.empty(0, dtype=torch.float64)
    return niqe_from_feature_list(feats, *_load_pristine(pristine))


class NIQE(nn.Module):
    """Same constructor and call as the reference (image_quality_assessment.py:1001-1033); block height and width must be
    equal and even here."""

    def __init__(self, crop_border: int, niqe_model_path, block_size_height: int = 96, block_size_width: int = 96) -> None:
        super().__init__()
        if block_size_height != block_size_width:
            raise ValueError("resr_b200.iqa.NIQE implements square blocks (the reference's default 96 x 96)")
        self.crop_border = crop_border
        self.niqe_model_path = niqe_model_path
        self.block_size = block_size_height
        self._pristine = None

    def forward(self, raw_tensor: torch.Tensor) -> torch.Tensor:
        if self._pristine is None:
            self._pristine = _load_pristine(self.niqe_model_path)
        feat = niqe_features(raw_tensor, self.crop_border, self.block_size)
        return niqe_from_features(feat, *self._pristine).squeeze()

    def forward_many(self, images) -> torch.Tensor:
        """Scores of a list of differently sized images in input order (float64 [len(images)]), as niqe_many: what the
        per-image loops of test.py / validate() compute, in one feature call and one fit."""
        if self._pristine is None:
            self._pristine = _load_pristine(self.niqe_model_path)
        return niqe_many(images, self.crop_border, self._pristine, self.block_size)
