"""CPU: the oracle (oracle/) reproduces the committed outputs of the unmodified reference (tests/golden/*.npz).
This is what pins the oracle; the GPU parity tests then compare the CUDA path against oracle + golden vectors."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import degrade as od
from oracle import generator as og
from oracle import make_golden_degrade as mg
from oracle import plan as oplan


@pytest.fixture(scope="module")
def ops(golden_dir):
    return mg.load_ops(os.path.join(golden_dir, "degrade_ops.npz"))


@pytest.fixture(scope="module")
def block(golden_dir):
    return mg.load_block(os.path.join(golden_dir, "degrade_block.npz"))


def test_generator_oracle_matches_reference_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "generator.npz"))
    for tag in ("a", "b"):
        sd = og.random_state_dict(int(z[f"{tag}_seed"]))
        y = og.generator_forward(torch.from_numpy(z[f"{tag}_x"]), sd).numpy()
        assert np.abs(y - z[f"{tag}_y"]).max() <= 1e-6


def test_random_state_dict_layout():
    sd = og.random_state_dict(0)
    assert len(sd) == 702
    assert sum(v.numel() for v in sd.values()) == 16697987
    assert sd["trunk.22.rdb3.conv5.weight"].shape == (64, 192, 3, 3)
    assert float(sd["trunk.0.rdb1.conv1.bias"].abs().max()) == 0.0


def test_filter2d_usm_oracle(ops):
    assert np.abs(od.filter2d(ops["f2d_x"], ops["f2d_k"]) - ops["f2d_y"]).max() <= 2e-6
    assert np.abs(od.filter2d(ops["f2d_x"], ops["f2d_sk"]) - ops["f2d_y_shared"]).max() <= 2e-6
    assert np.abs(od.usm_sharp(ops["usm_x"], 0.5, 10) - ops["usm_y"]).max() <= 5e-6
    with pytest.raises(ValueError):
        od.filter2d(ops["f2d_x"], np.ones((1, 4, 4), np.float32))


def test_resize_oracle(ops):
    x = ops["f2d_x"]
    n = 0
    for key in ops:
        if key.startswith("rs_sf_"):
            _, _, mode, s = key.split("_")
            s = float(s)
            y = od.resize(x, od.interp_out_size(x.shape[2], s), od.interp_out_size(x.shape[3], s), mode, s, s)
        elif key.startswith("rs_sz_"):
            _, _, mode, sz = key.split("_")
            hh, ww = (int(v) for v in sz.split("x"))
            y = od.resize(x, hh, ww, mode)
        else:
            continue
        assert y.shape == ops[key].shape
        assert np.abs(y - ops[key]).max() <= 2e-6, key
        n += 1
    assert n == 18


def test_jpeg_oracle(ops):
    y, parts = od.jpeg(ops["jpeg_x"], ops["jpeg_q"], return_parts=True)
    assert np.array_equal(parts["factor"], ops["jpeg_factor"])  # fp32 factor arithmetic, bit for bit
    assert np.abs(y - ops["jpeg_y"]).max() <= 1e-6
    assert np.array_equal(parts["y_q"], ops["jpeg_qy_oracle"])
    # tables: transposed Annex-K luma, symmetric chroma (imgproc.py:40-49)
    assert od.Y_TABLE[0, 1] == 12 and od.Y_TABLE[1, 0] == 11 and od.C_TABLE[3, 3] == 99 and od.C_TABLE[4, 0] == 99


def test_block_replay_matches_reference(block):
    for seed in block["seeds"]:
        tag = f"s{seed}."
        plan = mg.unflatten_plan(block, tag + "plan.")
        stages = []
        lr, hr = od.degrade_batch(block[tag + "hr"], block[tag + "k1"], block[tag + "k2"], block[tag + "sk"], plan, stages)
        assert np.array_equal(hr, block[tag + "hr_crop"])
        assert np.array_equal(np.rint(lr * 255), np.rint(block[tag + "lr"] * 255)), f"seed {seed}: lr differs on the u8 grid"
        for name, t in stages:   # the reference's stage outputs are stored on mg.STAGE_GRID
            assert np.abs(t[mg.STAGE_GRID] - block[tag + "out." + name]).max() <= 5e-6, (seed, name)


def test_noise_edge_cases():
    rng = np.random.default_rng(0)
    x = rng.random((2, 3, 8, 8), dtype=np.float32)
    # gray flags all zero with no gray field == colour noise only
    nc = rng.standard_normal((2, 3, 8, 8), dtype=np.float32)
    s = np.array([5, 10], np.float32)
    a = od.gaussian_noise_apply(x, s, np.zeros(2, np.float32), nc, None)
    assert np.abs(a - np.clip(x + nc * s.reshape(2, 1, 1, 1) / 255, 0, 1)).max() <= 1e-7
    # unique counts -> power of two
    assert list(od.poisson_vals(np.array([1, 2, 3, 128, 129, 256]))) == [1, 2, 4, 128, 256, 256]
    q = od.round_u8(np.array([[0.5 / 255, 1.5 / 255, 2.5 / 255]], np.float32))  # half to even on the u8 grid
    assert np.allclose(q * 255, [[0, 2, 2]])


def test_synth_and_canonical_plans_are_replayable():
    rng = np.random.default_rng(1)
    hr = rng.random((2, 3, 64, 64), dtype=np.float32)
    k = np.zeros((2, 21, 21), np.float32)
    k[:, 9:12, 9:12] = 1 / 9
    for plan in (oplan.synth_plan(2, 64, 64, 3, image_size=64), oplan.canonical_plan_s0(2, 64, 64)):
        for key in ("noise1", "noise2"):
            if plan[key]["type"] == "poisson":  # draws depend on the image: fill in lazily, as the GPU path does
                plan[key]["samples_color"] = None
        # fill Poisson draws through the oracle's own rates
        def fill(x, p):
            if p["type"] == "poisson" and p["samples_color"] is None:
                r = od.poisson_rates(x, p["gray"].sum() > 0)
                p["samples_color"] = rng.poisson(r["rate"]).astype(np.float32)
                if p["gray"].sum() > 0:
                    p["samples_gray"] = rng.poisson(r["rate_g"]).astype(np.float32)
        # walk the chain once to materialise the Poisson tensors, then replay
        out = od.usm_sharp(hr, 0.5, 10)
        out = od.filter2d(out, k) if plan["blur1"] else out
        r = plan["resize1"]
        out = od.resize(out, r["out_h"], r["out_w"], r["mode"], r["scale"], r["scale"])
        fill(out, plan["noise1"])
        stages = []
        # second noise needs the chain up to there: easiest is a first replay that stops at noise2
        p2 = dict(plan)
        if plan["noise2"]["type"] == "poisson":
            tmp = dict(plan["noise2"])
            tmp.update(type="gaussian", sigma=np.zeros(2, np.float32), noise_color=np.zeros((2, 3, plan["resize2"]["out_h"], plan["resize2"]["out_w"]), np.float32))
            p2["noise2"] = tmp
            od.degrade_batch(hr, k, k, k[:1], p2, stages)
            x2 = dict(stages)["resize2"]
            fill(x2, plan["noise2"])
        lr, hrc = od.degrade_batch(hr, k, k, k[:1], plan)
        assert lr.shape == (2, 3, 16, 16) and hrc.shape == (2, 3, 64, 64)
        assert np.abs(lr * 255 - np.rint(lr * 255)).max() < 1e-4


from oracle.plan import DEGRADATION_MODEL_PARAMETERS as MODEL_PARAMS  # noqa: E402


def test_kernel_synthesis_oracle_and_rng_order(golden_dir):
    """Replaying the reference's seeds through the host-side draw mirror + the numpy oracle reproduces the reference
    kernels (imgproc.py:492-603) to float64 round-off: checks both the formulas and the RNG consumption order."""
    import math
    import random

    import resr_b200
    from oracle import kernels as ok
    z = np.load(os.path.join(golden_dir, "kernels.npz"))
    P = MODEL_PARAMS
    for seed in range(16):
        ks = int(z[f"mixed_{seed}_ks"])
        random.seed(seed)
        np.random.seed(seed)
        p, _ = resr_b200.imgproc.draw_mixed_kernel_params(
            P["gaussian_kernel_type"], P["gaussian_kernel_probability1"], ks, P["gaussian_sigma_range1"],
            P["gaussian_sigma_range1"], [-math.pi, math.pi], P["generalized_kernel_beta_range1"],
            P["plateau_kernel_beta_range1"])
        assert np.abs(ok.from_params(p) - z[f"mixed_{seed}"]).max() <= 1e-15
    for i in range(4):
        om, ks, pad = z[f"sinc_{i}_args"]
        assert np.abs(ok.sinc(float(om), int(ks), int(pad)) - z[f"sinc_{i}"]).max() <= 1e-15


def test_filter2d_fft_path_equals_direct_definition():
    """The FFT evaluation used for BASELINE-size inputs is the same float64 cross-correlation as the tap-by-tap sum."""
    from oracle import degrade as od
    rng = np.random.default_rng(4)
    x = rng.random((2, 3, 61, 83), dtype=np.float32)
    k = rng.random((2, 21, 21)).astype(np.float32)
    k[:, :3] = 0
    k /= k.sum((1, 2), keepdims=True)
    assert np.abs(od.filter2d(x, k, "direct").astype(np.float64) - od.filter2d(x, k, "fft")).max() <= 1e-7
    ku = od.usm_kernel_2d()
    assert np.abs(od.filter2d(x, ku, "direct").astype(np.float64) - od.filter2d(x, ku, "fft")).max() <= 1e-7


def test_augment_oracle_matches_reference_golden():
    """dataset.py:67-79 (rotate / flips / BGR->RGB / image_to_tensor): the numpy restatement reproduces the reference's own
    functions bit for bit on every (angle, hflip, vflip) of six image shapes (odd, even, non-square)."""
    import numpy as np
    from oracle import augment as oa
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "augment.npz"))
    n = 0
    for idx in range(6):
        img = gold[f"img{idx}"]
        for ai in range(4):
            for hf in (0, 1):
                for vf in (0, 1):
                    assert np.array_equal(oa.augment(img, ai, hf, vf), gold[f"out{idx}_{ai}_{hf}_{vf}"])
                    n += 1
    assert n == 96


def test_draw_augment_ops_keeps_the_reference_rng_order():
    import random
    import resr_b200
    random.seed(5)
    ops = resr_b200.imgproc.draw_augment_ops(6).tolist()
    random.seed(5)
    for op in ops:
        assert [0, 90, 180, 270][op & 3] == random.choice([0, 90, 180, 270])
        assert bool(op & 4) == (random.random() < 0.5)
        assert bool(op & 8) == (random.random() < 0.5)


def test_niqe_oracle_matches_reference_golden():
    """image_quality_assessment.py:886-998 restated in numpy (oracle/niqe.py) against the unmodified reference run with
    synthetic pristine statistics (tests/golden/niqe.npz): per-block features and the final score."""
    import numpy as np
    from oracle import niqe as on
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "niqe.npz"))
    for ci in range(3):
        x = g[f"x{ci}"].astype(np.float32) / np.float32(255.0)
        score, feat = on.niqe(x, int(g[f"border{ci}"]), g["mu_prisparam"], g["cov_prisparam"])
        ref_feat = g[f"feat{ci}"]
        for b in range(feat.shape[0]):      # block order differs (the reference stores blocks column-first): compare as sets
            a = np.array(sorted(map(tuple, feat[b])))
            r = np.array(sorted(map(tuple, ref_feat[b])))
            assert np.abs(a - r).max() <= 1e-6
        assert np.abs(score - g[f"niqe{ci}"]).max() <= 1e-5 * g[f"niqe{ci}"].max()


def test_oracle_grads_without_formats_is_float64_autograd():
    """grads() with no formats is float64 autograd of the oracle forward (l1_loss_and_grads casts to float32, so it is
    only checked to fp32 accuracy)."""
    sd = og.rich_state_dict(5)
    torch.manual_seed(5)
    x, hr = torch.rand(1, 3, 4, 6), torch.rand(1, 3, 16, 24)
    loss, g, sr = og.grads(x, sd, lambda y: torch.nn.functional.l1_loss(y, hr.double()))
    params = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    sr64 = og._forward(x.double(), params, 23)
    loss64 = torch.nn.functional.l1_loss(sr64, hr.double())
    loss64.backward()
    assert loss.dtype == torch.float64 and torch.equal(loss, loss64.detach()) and torch.equal(sr, sr64.detach())
    assert list(g) == list(sd) and all(torch.equal(g[k], params[k].grad) for k in sd)
    loss32, g32, _ = og.l1_loss_and_grads(x, hr, sd)
    assert abs(loss32.item() - loss.item()) <= 1e-5 * loss.item()
    flat, flat32 = torch.cat([g[k].reshape(-1) for k in sd]), torch.cat([g32[k].reshape(-1).double() for k in sd])
    assert float((flat32 - flat).norm() / flat.norm()) <= 1e-4


def test_oracle_recipe_rounding_points():
    """On one convolution: the forward multiplies operands rounded to the operand format (the bias is not rounded); the
    output gradient is rounded to the gradient format, and the data and weight gradients multiply it with the weights
    and the input rounded to the backward format."""
    torch.manual_seed(6)
    x = (torch.randn(2, 5, 6, 7, dtype=torch.float64) * 3).requires_grad_(True)
    p = {"c.weight": torch.randn(4, 5, 3, 3, dtype=torch.float64).requires_grad_(True),
         "c.bias": torch.randn(4, dtype=torch.float64).requires_grad_(True)}
    r = torch.randn(2, 4, 6, 7, dtype=torch.float64)
    q = lambda t, fmt: t.detach().to(fmt).double()
    for ofmt, bfmt in ((torch.float16, torch.bfloat16), (torch.bfloat16, torch.bfloat16), (torch.float16, torch.float16)):
        for t in (x, *p.values()):
            t.grad = None
        y = og.recipe_conv(ofmt, torch.bfloat16, bfmt)(x, p, "c")
        (y * r).sum().backward()
        rq = q(r, torch.bfloat16)
        assert not torch.equal(q(x, ofmt), x.detach()) and not torch.equal(rq, r)
        assert torch.allclose(y, F.conv2d(q(x, ofmt), q(p["c.weight"], ofmt), p["c.bias"].detach(), padding=1), rtol=1e-14, atol=1e-12)
        gx = torch.nn.grad.conv2d_input(x.shape, q(p["c.weight"], bfmt), rq, padding=1)
        gw = torch.nn.grad.conv2d_weight(q(x, bfmt), p["c.weight"].shape, rq, padding=1)
        assert torch.allclose(x.grad, gx, rtol=1e-12, atol=1e-12)
        assert torch.allclose(p["c.weight"].grad, gw, rtol=1e-12, atol=1e-12)
        assert torch.equal(p["c.bias"].grad, rq.sum((0, 2, 3)))
        if bfmt != ofmt:   # the backward format is not the forward one
            assert not torch.allclose(x.grad, torch.nn.grad.conv2d_input(x.shape, q(p["c.weight"], ofmt), rq, padding=1), rtol=1e-6)
    # backward format defaults to the operand format; no formats: the plain convolution
    for t in (x, *p.values()):
        t.grad = None
    (og.recipe_conv(torch.float16, torch.bfloat16)(x, p, "c") * r).sum().backward()
    assert torch.allclose(x.grad, torch.nn.grad.conv2d_input(x.shape, q(p["c.weight"], torch.float16), q(r, torch.bfloat16), padding=1),
                          rtol=1e-12, atol=1e-12)
    y = og.recipe_conv()(x, p, "c")
    assert torch.equal(y, F.conv2d(x, p["c.weight"], p["c.bias"], padding=1))


def test_rich_state_dict_adds_nonzero_biases_only():
    sd0, sd = og.random_state_dict(3), og.rich_state_dict(3)
    assert list(sd) == list(sd0)
    for k in sd:
        assert sd[k].dtype == torch.float32 and sd[k].shape == sd0[k].shape
        if k.endswith(".weight"):
            assert torch.equal(sd[k], sd0[k])
        else:
            cin = sd[k[:-len("bias")] + "weight"].shape[1]
            assert bool((sd[k] != 0).all()), k
            assert float(sd[k].abs().max()) <= 1.0 / (9 * cin) ** 0.5 or k == "conv4.bias"
    assert sd["conv4.bias"].tolist() == pytest.approx([-0.02, 0.5, 1.02])
    assert float(og.random_state_dict(3)["trunk.0.rdb1.conv1.bias"].abs().max()) == 0.0
    assert not torch.equal(og.rich_state_dict(4)["trunk.0.rdb1.conv1.bias"], sd["trunk.0.rdb1.conv1.bias"])
