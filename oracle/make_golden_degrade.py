"""Golden vectors for hot path 2 from the UNMODIFIED reference (build container only; called by oracle/make_golden.py).

degrade_ops.npz    per-op input/output pairs of imgproc.filter2d_torch / USMSharp / DiffJPEG / F.interpolate /
                   random_add_{gaussian,poisson}_noise_torch with the random tensors recorded
degrade_block.npz  whole-block executions of train_realesrnet.py:267-377 (exec of the literal source lines) for
                   several seeds: blur kernels, recorded plan, every stage output, final lr

Each file stays under 1 MB. The input images are not stored: smooth_image regenerates them from their seeds, and
load_ops / load_block check them bit for bit against the SHA-256 digest stored beside. The stage outputs of the block
are stored on the sub-grid STAGE_GRID (every second row and column). The reference's hr crop is not stored either:
it is hr[..., hr_top:hr_top + image_size, hr_left:hr_left + image_size] of the recorded plan.
"""
import hashlib
import math
import os
import random

import numpy as np
import torch
import torch.nn.functional as F

from . import degrade as od
from . import plan as oplan


def ref_kernels(imgproc, config, seed):
    """kernel1, kernel2, sinc_kernel for one sample, sequenced as dataset.py:81-141 does."""
    P = config.degradation_model_parameters_dict
    random.seed(seed)
    np.random.seed(seed)

    def one(prob_key, sig_key, bg_key, bp_key, sinc_key):
        ks = random.choice(P["gaussian_kernel_range"])
        if np.random.uniform() < P[sinc_key]:
            if ks < int(np.median(P["gaussian_kernel_range"])):
                om = np.random.uniform(np.pi / 3, np.pi)
            else:
                om = np.random.uniform(np.pi / 5, np.pi)
            k = imgproc.generate_sinc_kernel(om, ks, padding=False)
        else:
            k = imgproc.random_mixed_kernels(P["gaussian_kernel_type"], P[prob_key], ks, P[sig_key], P[sig_key],
                                             [-math.pi, math.pi], P[bg_key], P[bp_key], noise_range=None)
        pad = (P["gaussian_kernel_range"][-1] - ks) // 2
        return np.pad(k, ((pad, pad), (pad, pad)))

    k1 = one("gaussian_kernel_probability1", "gaussian_sigma_range1", "generalized_kernel_beta_range1",
             "plateau_kernel_beta_range1", "sinc_kernel_probability1")
    k2 = one("gaussian_kernel_probability2", "gaussian_sigma_range2", "generalized_kernel_beta_range2",
             "plateau_kernel_beta_range2", "sinc_kernel_probability2")
    if np.random.uniform() < P["sinc_kernel_probability3"]:
        ks = random.choice(P["gaussian_kernel_range"])
        om = np.random.uniform(np.pi / 3, np.pi)
        sk = imgproc.generate_sinc_kernel(om, ks, padding=P["sinc_kernel_size"])
    else:
        sk = np.zeros((21, 21), np.float32)
        sk[10, 10] = 1
    return (torch.FloatTensor(k1), torch.FloatTensor(k2), torch.FloatTensor(sk))


def batch_kernels(imgproc, config, b, seed):
    ks = [ref_kernels(imgproc, config, seed * 100 + i) for i in range(b)]
    return tuple(torch.stack([k[j] for k in ks]) for j in range(3))


def smooth_image(b, h, w, seed):
    """Natural-ish synthetic image in [0,1]: low-pass noise + edges (keeps USM masks / JPEG ties realistic)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(b, 3, h // 4 + 2, w // 4 + 2, generator=g)
    x = F.interpolate(x, size=(h, w), mode="bicubic", align_corners=False).clamp(0, 1)
    x = 0.8 * x + 0.2 * torch.rand(b, 3, h, w, generator=g)
    x[:, :, h // 3:h // 2, w // 4:w // 2] *= 0.3
    return x.clamp(0, 1).contiguous()


STAGE_GRID = (Ellipsis, slice(None, None, 2), slice(None, None, 2))
OPS_INPUTS = {"f2d_x": (2, 48, 56, 1), "usm_x": (1, 72, 88, 2), "jpeg_x": (3, 40, 52, 4)}   # key: smooth_image arguments


def digest(a):
    return np.array(hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest())


def _regenerated(z, key, args):
    x = smooth_image(*args).numpy()
    if str(digest(x)) != str(z[key + "_sha256"]):
        raise AssertionError(f"{key}: smooth_image{args} no longer reproduces the stored input")
    return x


def load_ops(path):
    """degrade_ops.npz as a dict, with the input images regenerated and checked."""
    z = dict(np.load(path))
    for key, args in OPS_INPUTS.items():
        z[key] = _regenerated(z, key, args)
    return z


def load_block(path):
    """degrade_block.npz as a dict, with every seed's hr regenerated and checked and its hr crop cut out of it."""
    z = dict(np.load(path))
    for seed in z["seeds"]:
        tag = f"s{seed}."
        hr = _regenerated(z, tag + "hr", (2, 64, 72, 100 + int(seed)))
        top, left, size = (int(z[tag + "plan.crop." + k]) for k in ("hr_top", "hr_left", "image_size"))
        z[tag + "hr"], z[tag + "hr_crop"] = hr, hr[:, :, top:top + size, left:left + size]
    return z


def make_ops(imgproc, config, out_dir):
    z = {}
    torch.manual_seed(11)
    img = smooth_image(2, 48, 56, 1)
    k1, k2, sk = batch_kernels(imgproc, config, 2, 3)
    z["f2d_x"], z["f2d_k"] = img.numpy(), k1.numpy()
    z["f2d_y"] = imgproc.filter2d_torch(img, k1).numpy()
    z["f2d_sk"] = sk[:1].numpy()
    z["f2d_y_shared"] = imgproc.filter2d_torch(img, sk[:1]).numpy()
    usm = imgproc.USMSharp(50, 0)
    big = smooth_image(1, 72, 88, 2)
    z["usm_x"], z["usm_y"] = big.numpy(), usm(big, 0.5, 10).numpy()
    rs = []
    for mode in ("area", "bilinear", "bicubic"):
        for s in (0.37, 1.37, 0.15):
            y = F.interpolate(img, scale_factor=s, mode=mode)
            rs.append((od.MODE_ID[mode], s, y.shape[2], y.shape[3]))
            z[f"rs_sf_{mode}_{s}"] = y.numpy()
        for size in ((12, 14), (30, 17), (60, 70)):
            z[f"rs_sz_{mode}_{size[0]}x{size[1]}"] = F.interpolate(img, size=size, mode=mode).numpy()
    j = imgproc.DiffJPEG(False)
    xj = smooth_image(3, 40, 52, 4)
    q = torch.tensor([31.7, 49.99, 94.2])
    z["jpeg_x"], z["jpeg_q"] = xj.numpy(), q.numpy().copy()
    z["jpeg_y"] = np.ascontiguousarray(j(xj, q.clone()).detach().numpy())
    qq = q.clone()
    j(xj, qq)
    z["jpeg_factor"] = qq.numpy()
    _, parts = od.jpeg(xj.numpy(), q.numpy(), return_parts=True)
    z["jpeg_qy_oracle"], z["jpeg_qcb_oracle"], z["jpeg_qcr_oracle"] = parts["y_q"], parts["cb_q"], parts["cr_q"]
    for key in OPS_INPUTS:
        z[key + "_sha256"] = digest(z.pop(key))
    np.savez_compressed(os.path.join(out_dir, "degrade_ops.npz"), **z)
    print("degrade_ops.npz written")


def flatten_plan(prefix, plan, z):
    for k, v in plan.items():
        if isinstance(v, dict):
            flatten_plan(f"{prefix}{k}.", v, z)
        elif v is None:
            z[f"{prefix}{k}"] = np.array("None")
        else:
            z[f"{prefix}{k}"] = np.asarray(v)


def unflatten_plan(z, prefix):
    plan = {}
    for key in z:
        if not key.startswith(prefix):
            continue
        parts = key[len(prefix):].split(".")
        d = plan
        for p in parts[:-1]:
            d = d.setdefault(p, {})
        v = z[key]
        if v.dtype.kind == "U":
            v = None if str(v) == "None" else str(v)
        elif v.ndim == 0:
            v = v.item()
        d[parts[-1]] = v
    return plan


def make_block(imgproc, config, out_dir):
    z = {}
    config.image_size = 48  # crop size (config.py:89); the literal block reads it — smaller than 256 keeps fixtures small
    seeds = [0, 1, 5, 6]
    kept = []
    for seed in seeds:
        b, h, w = 2, 64, 72
        hr = smooth_image(b, h, w, 100 + seed)
        k1, k2, sk = batch_kernels(imgproc, config, b, seed)
        plan, stages, lr, hr_c = oplan.record_reference_plan(hr, k1, k2, sk, seed)
        tag = f"s{seed}."
        assert np.array_equal(hr_c, hr.numpy()[:, :, plan["crop"]["hr_top"]:plan["crop"]["hr_top"] + config.image_size,
                                               plan["crop"]["hr_left"]:plan["crop"]["hr_left"] + config.image_size])
        z[tag + "hr_sha256"], z[tag + "k1"], z[tag + "k2"], z[tag + "sk"] = digest(hr.numpy()), k1.numpy(), k2.numpy(), sk.numpy()
        flatten_plan(tag + "plan.", plan, z)
        z[tag + "stage_names"] = np.array([s[0] for s in stages])
        for name, xin, yout in stages:
            z[tag + "out." + name] = np.ascontiguousarray(yout.astype(np.float32)[STAGE_GRID])
        z[tag + "lr"] = lr
        kept.append(seed)
        print(f"seed {seed}: blur1={plan['blur1']} r1={plan['resize1']['mode']}/{plan['resize1']['out_h']}x{plan['resize1']['out_w']} "
              f"n1={plan['noise1']['type']} blur2={plan['blur2']} r2={plan['resize2']['mode']}/{plan['resize2']['out_h']}x{plan['resize2']['out_w']} "
              f"n2={plan['noise2']['type']} order={plan['final_order']} r3={plan['resize3']['mode']} crop={plan['crop']['hr_top']},{plan['crop']['hr_left']}")
    z["seeds"] = np.array(kept)
    np.savez_compressed(os.path.join(out_dir, "degrade_block.npz"), **z)
    print("degrade_block.npz written")


def make(imgproc, config, out_dir):
    make_ops(imgproc, config, out_dir)
    make_block(imgproc, config, out_dir)
