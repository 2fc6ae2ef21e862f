"""GPU parity of the degradation kernels (C ABI behind resr_b200.imgproc) against (i) the committed outputs of the
unmodified reference (tests/golden/degrade_*.npz) and (ii) the numpy oracle on fresh seeded inputs.

Contract (BASELINE.json north_star): <= 1e-5 in fp32 per stage on identical stage inputs; integer work (unique
counts, quantisation factors, quantised JPEG coefficients, crop indexing, u8 rounding) bit-exact. Discontinuous
decisions (USM mask, JPEG rounding ties, final u8 rounding) may flip where the reference's own pre-decision value
sits within fp32 noise of the threshold (SURVEY.md §7.3-4); those are counted, bounded and printed."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _maxdiff(a, b):
    return float(np.abs(a.cpu().numpy().astype(np.float64) - b.astype(np.float64)).max())


@pytest.fixture(scope="module")
def ops(golden_dir):
    from oracle import make_golden_degrade as mg
    return mg.load_ops(os.path.join(golden_dir, "degrade_ops.npz"))


@pytest.fixture(scope="module")
def block(golden_dir):
    from oracle import make_golden_degrade as mg
    return mg.load_block(os.path.join(golden_dir, "degrade_block.npz"))


def test_filter2d_golden(ops):
    import resr_b200
    y = resr_b200.imgproc.filter2d_torch(_t(ops["f2d_x"]), _t(ops["f2d_k"]))
    assert _maxdiff(y, ops["f2d_y"]) <= TOL
    y = resr_b200.imgproc.filter2d_torch(_t(ops["f2d_x"]), _t(ops["f2d_sk"]))
    assert _maxdiff(y, ops["f2d_y_shared"]) <= TOL


def test_filter2d_vs_oracle_shapes_and_errors():
    import resr_b200
    from oracle import degrade as od
    rng = np.random.default_rng(0)
    for (b, c, h, w, k, kb) in [(3, 3, 37, 45, 21, 3), (2, 1, 64, 33, 7, 1), (1, 3, 100, 130, 13, 1), (2, 3, 30, 30, 21, 2)]:
        x = rng.random((b, c, h, w), dtype=np.float32)
        kern = rng.random((kb, k, k), dtype=np.float32)
        kern[:, :2] = 0  # trimmed support
        kern /= kern.sum((1, 2), keepdims=True)
        y = resr_b200.imgproc.filter2d_torch(_t(x), _t(kern))
        assert _maxdiff(y, od.filter2d(x, kern)) <= TOL
    with pytest.raises(ValueError):
        resr_b200.imgproc.filter2d_torch(_t(x), _t(np.ones((1, 4, 4), np.float32)))


def test_usm_golden(ops):
    import resr_b200
    usm = resr_b200.imgproc.USMSharp(50, 0).cuda()
    y = usm(_t(ops["usm_x"]), 0.5, 10)
    d = np.abs(y.cpu().numpy() - ops["usm_y"])
    frac = float((d > TOL).mean())
    print(f"usm: max {d.max():.3e}, fraction > 1e-5: {frac:.2e}")
    assert frac <= 1e-3  # mask flips at |residual|*255 == 10 +- fp32 noise
    assert np.median(d) <= 1e-6
    from oracle import degrade as od
    assert np.abs(usm.kernel.cpu().numpy() - od.usm_kernel_2d()).max() <= 1e-9


def test_resize_golden(ops):
    import resr_b200
    x = _t(ops["f2d_x"])
    n = 0
    for key in ops:
        if key.startswith("rs_sf_"):
            _, _, mode, s = key.split("_")
            y = resr_b200.imgproc.interpolate(x, scale_factor=float(s), mode=mode)
        elif key.startswith("rs_sz_"):
            _, _, mode, sz = key.split("_")
            hh, ww = (int(v) for v in sz.split("x"))
            y = resr_b200.imgproc.interpolate(x, size=(hh, ww), mode=mode)
        else:
            continue
        assert tuple(y.shape) == ops[key].shape, key
        assert _maxdiff(y, ops[key]) <= TOL, key
        n += 1
    assert n == 18
    for mode in ("area", "bilinear", "bicubic"):  # same-size resize is the identity, bit-exactly (SURVEY a12b)
        assert torch.equal(resr_b200.imgproc.interpolate(x, size=tuple(x.shape[2:]), mode=mode), x)
        assert torch.equal(resr_b200.imgproc.interpolate(x, scale_factor=1, mode=mode), x)


def _jpeg_check(y, factor, q_native, x_np, quality_np, ref_y):
    """Returns (#coefficient flips, #flips not explained by a tie)."""
    from oracle import degrade as od
    _, parts = od.jpeg(x_np, quality_np, return_parts=True)
    assert np.array_equal(factor.cpu().numpy(), parts["factor"]), "quantisation factor must be bit-exact"
    flips = unexplained = 0
    for name, qn in zip(("y", "cb", "cr"), q_native):
        qn = qn.cpu().numpy()
        mism = qn != parts[name + "_q"]
        flips += int(mism.sum())
        ratio = parts[name + "_ratio"]
        near_tie = np.abs(np.abs(ratio - np.floor(ratio)) - 0.5) < 2e-3
        unexplained += int((mism & ~near_tie).sum())
        assert np.abs(qn - parts[name + "_q"]).max() <= 1
    d = np.abs(y.cpu().numpy() - ref_y)
    return flips, unexplained, float(d.max()), float((d > TOL).mean())


def test_jpeg_golden(ops):
    import resr_b200
    j = resr_b200.imgproc.DiffJPEG(False)
    q = _t(ops["jpeg_q"])
    y, factor, qy, qcb, qcr = j(_t(ops["jpeg_x"]), q, return_coefficients=True)
    assert np.array_equal(q.cpu().numpy(), ops["jpeg_factor"]), "quality tensor is overwritten with the factor, as in the reference"
    flips, unexplained, dmax, frac = _jpeg_check(y, factor, (qy, qcb, qcr), ops["jpeg_x"], ops["jpeg_q"], ops["jpeg_y"])
    print(f"jpeg: {flips} coefficient flips ({unexplained} not at a tie), max diff {dmax:.3e}, frac>1e-5 {frac:.2e}")
    assert unexplained == 0
    if flips == 0:
        assert dmax <= TOL
    assert frac <= 64.0 * max(flips, 0) / y.numel() * 4 + 1e-12


def test_unique_count_bit_exact():
    import resr_b200
    from oracle import degrade as od
    rng = np.random.default_rng(3)
    x = rng.random((4, 3, 40, 56), dtype=np.float32)
    x[1] = np.round(x[1] * 6) / 6          # few levels
    x[2] = 0.25                             # one level
    x[3, :, :20] = np.round(x[3, :, :20] * 40) / 255
    cc, cg = resr_b200.imgproc.unique_count_u8(_t(x))
    assert np.array_equal(cc.cpu().numpy(), od.unique_count_u8(od.round_u8(x)))
    assert np.array_equal(cg.cpu().numpy(), od.unique_count_u8(od.round_u8(od.rgb_to_gray(x))))


def test_noise_vs_oracle_all_flag_combinations():
    import resr_b200
    from oracle import degrade as od
    rng = np.random.default_rng(5)
    b, h, w = 3, 24, 40
    x = rng.random((b, 3, h, w), dtype=np.float32)
    sigma = rng.uniform(1, 30, b).astype(np.float32)
    gray = np.array([1, 0, 1], np.float32)
    nc = rng.standard_normal((b, 3, h, w), dtype=np.float32)
    ng = rng.standard_normal((h, w), dtype=np.float32)
    for use_gray in (True, False):
        y = resr_b200.imgproc.gaussian_noise_apply(_t(x), _t(sigma), _t(gray), _t(nc), _t(ng) if use_gray else None)
        ref = od.gaussian_noise_apply(x, sigma, gray, nc, ng if use_gray else None)
        assert _maxdiff(y, ref) <= 1e-7
    scale = rng.uniform(0.05, 3, b).astype(np.float32)
    for use_gray in (True, False):
        rates = od.poisson_rates(x, use_gray)
        rc, rg = resr_b200.imgproc.poisson_rates(_t(x), use_gray)
        assert np.array_equal(rc.cpu().numpy(), rates["rate"])
        sc = rng.poisson(rates["rate"]).astype(np.float32)
        sg = None
        if use_gray:
            assert np.array_equal(rg.cpu().numpy(), rates["rate_g"])
            sg = rng.poisson(rates["rate_g"]).astype(np.float32)
        y = resr_b200.imgproc.poisson_noise_apply(_t(x), _t(scale), _t(gray), _t(sc), None if sg is None else _t(sg))
        ref = od.poisson_noise_apply(x, scale, gray, sc, sg)
        assert _maxdiff(y, ref) <= 1e-7


def _plan(block, seed):
    from oracle import make_golden_degrade as mg
    return mg.unflatten_plan(block, f"s{seed}.plan.")


def test_block_per_stage_on_reference_inputs(block):
    """Every stage of the recorded reference executions reproduces the reference's stage output (stored on
    mg.STAGE_GRID). The first stage is fed the reference's own input; every later stage is fed the numpy oracle's replay
    of the reference's stage input, which test_oracle_cpu pins to within 5e-6 of the reference at every stored pixel."""
    import resr_b200
    from oracle import degrade as od
    from oracle import make_golden_degrade as mg
    ip = resr_b200.imgproc
    for seed in block["seeds"]:
        tag = f"s{seed}."
        plan = _plan(block, seed)
        names = [str(n) for n in block[tag + "stage_names"]]
        replay = []
        od.degrade_batch(block[tag + "hr"], block[tag + "k1"], block[tag + "k2"], block[tag + "sk"], _plan(block, seed), replay)
        assert [n for n, _ in replay] == names
        prev = block[tag + "hr"]
        for name, replayed in replay:
            ref = block[tag + "out." + name]
            x = _t(prev)
            flips_ok = 0.0
            if name == "usm":
                y = ip.USMSharp(50, 0)(x, 0.5, 10)
                flips_ok = 1e-3
            elif name in ("blur1", "blur2", "sinc"):
                y = ip.filter2d_torch(x, _t(block[tag + {"blur1": "k1", "blur2": "k2", "sinc": "sk"}[name]]))
            elif name.startswith("resize"):
                r = plan[name]
                mode = ("area", "bilinear", "bicubic")[r["mode"]]
                y = ip.interpolate(x, scale_factor=r["scale"], mode=mode) if r.get("scale") is not None else \
                    ip.interpolate(x, size=(r["out_h"], r["out_w"]), mode=mode)
            elif name.startswith("noise"):
                y = ip._noise(x, plan[name])
            elif name.startswith("jpeg"):
                y = ip.DiffJPEG(False)(x, _t(plan[name + "_quality"]), clamp_input=True)
                flips_ok = 2e-2
            d = np.abs(y.cpu().numpy()[mg.STAGE_GRID] - ref)
            frac = float((d > TOL).mean())
            print(f"seed {seed} {name:8s} {tuple(ref.shape)} max {d.max():.2e} frac>1e-5 {frac:.1e}")
            assert frac <= flips_ok, (seed, name, d.max())
            prev = replayed


def test_block_end_to_end(block):
    """Whole block through the native path vs the reference's final (lr, hr): hr crop exact, lr on the u8 grid with
    the count of differing u8 values reported (tie flips upstream move a handful of pixels by one level)."""
    import resr_b200
    tot = bad = 0
    for seed in block["seeds"]:
        tag = f"s{seed}."
        lr, hr = resr_b200.imgproc.degrade_batch(_t(block[tag + "hr"]), _t(block[tag + "k1"]), _t(block[tag + "k2"]),
                                                 _t(block[tag + "sk"]), _plan(block, seed))
        assert np.array_equal(hr.cpu().numpy(), block[tag + "hr_crop"])
        lv = np.rint(lr.cpu().numpy() * 255)
        assert np.abs(lr.cpu().numpy() - lv / 255).max() < 1e-7, "lr must sit on the u8 grid"
        ref = np.rint(block[tag + "lr"] * 255)
        diff = np.abs(lv - ref)
        tot += diff.size
        bad += int((diff > 0).sum())
        print(f"seed {seed}: {int((diff > 0).sum())}/{diff.size} u8 values differ, max {int(diff.max())} levels")
        assert diff.max() <= 2
    assert bad <= 0.02 * tot


def test_block_one_call_abi_equals_op_sequence(block):
    """resr_degrade_batch (the whole block behind ONE C-ABI call, POD plan) is bit-identical to the same block sequenced
    from Python through the op-level entry points, on the recorded reference plans (host-fed draws) and on a synthetic
    plan whose first resize goes through the scale_factor path."""
    import resr_b200
    ip = resr_b200.imgproc
    for seed in block["seeds"]:
        tag = f"s{seed}."
        args = (_t(block[tag + "hr"]), _t(block[tag + "k1"]), _t(block[tag + "k2"]), _t(block[tag + "sk"]), _plan(block, seed))
        lr_a, hr_a = ip.degrade_batch(*args)
        lr_b, hr_b = ip.degrade_batch_native(*args)
        assert torch.equal(lr_a, lr_b) and torch.equal(hr_a, hr_b)
    plan = resr_b200.plan.synth_plan(3, 96, 80, seed=11, image_size=64)
    for name in ("noise1", "noise2"):  # make every draw host-fed so that both paths see the same numbers
        n = plan[name]
        if n["type"] == "poisson":
            r = plan["resize1"] if name == "noise1" else plan["resize2"]
            rng = np.random.default_rng(5)
            n["samples_color"] = rng.poisson(20.0, (3, 3, r["out_h"], r["out_w"])).astype(np.float32)
            n["samples_gray"] = rng.poisson(20.0, (3, 1, r["out_h"], r["out_w"])).astype(np.float32)
    g = torch.Generator().manual_seed(0)
    hr = torch.rand(3, 3, 96, 80, generator=g).cuda()
    k = torch.zeros(3, 21, 21)
    k[:, 7:14, 7:14] = 1 / 49
    k = k.cuda()
    sk = torch.zeros(1, 21, 21)
    sk[0, 10, 10] = 1
    sk = sk.cuda()
    lr_a, hr_a = ip.degrade_batch(hr, k, k, sk, plan)
    lr_b, hr_b = ip.degrade_batch_native(hr, k, k, sk, plan)
    assert torch.equal(lr_a, lr_b) and torch.equal(hr_a, hr_b)


def test_kernel_synthesis_device(golden_dir):
    """Device float64 synthesis (resr_synthesize_kernels) vs the reference kernels: same seeds, same RNG order."""
    import math
    import random

    import resr_b200
    from oracle.plan import DEGRADATION_MODEL_PARAMETERS as P
    z = np.load(os.path.join(golden_dir, "kernels.npz"))
    ip = resr_b200.imgproc
    for seed in range(16):
        ks = int(z[f"mixed_{seed}_ks"])
        random.seed(seed)
        np.random.seed(seed)
        k = ip.random_mixed_kernels(P["gaussian_kernel_type"], P["gaussian_kernel_probability1"], ks,
                                    P["gaussian_sigma_range1"], P["gaussian_sigma_range1"], [-math.pi, math.pi],
                                    P["generalized_kernel_beta_range1"], P["plateau_kernel_beta_range1"], noise_range=None)
        assert k.dtype == np.float64 and k.shape == (ks, ks)
        assert np.abs(k - z[f"mixed_{seed}"]).max() <= 1e-12
    for i in range(4):
        om, ks, pad = z[f"sinc_{i}_args"]
        k = ip.generate_sinc_kernel(float(om), int(ks), padding=int(pad))
        assert k.shape == z[f"sinc_{i}"].shape
        assert np.abs(k - z[f"sinc_{i}"]).max() <= 1e-12
    with pytest.raises(AssertionError):
        ip.generate_sinc_kernel(1.0, 8)
    # batched: sequencing of dataset.py:81-141 for a whole batch in one launch
    from oracle import kernels as ok
    random.seed(3)
    np.random.seed(3)
    k1, k2, sk = ip.synthesize_degradation_kernels(6, P)
    assert k1.shape == (6, 21, 21) and k1.dtype == torch.float32
    for t in (k1, k2, sk):
        assert np.abs(t.sum((1, 2)).cpu().numpy() - 1).max() < 1e-5


@pytest.mark.gpu
def test_poisson_sampled_in_kernel_statistics():
    """resr_poisson_noise_sampled: the draws made inside the fused kernel are Poisson(q * vals) (imgproc.py:895, 906) in
    the small-rate and in the large-rate regime of the sampler, the luma branch is shared by the three channels, and
    consecutive calls draw fresh samples."""
    import scipy.stats as st
    import resr_b200
    ip = resr_b200.imgproc
    dev = "cuda"
    b, h, w = 2, 160, 256
    levels = torch.empty(b, 3, h, w)
    levels[:, :, :40] = 3.0
    levels[:, :, 40:80] = 10.0
    levels[:, :, 80:] = 200.0
    levels[:, :, 0, :256] = torch.arange(256.0)          # all 256 levels present -> vals = 256 (colour and luma)
    x = (levels / 255.0).to(dev)
    scale = torch.ones(b, device=dev)
    out = ip.poisson_noise_sampled(x, scale, None, seed=1234, clip=False)
    draws = ((out - x) + x) * 256.0                        # n = draw / vals - q, scale = 1, q = x on the u8 grid
    for lv, rows in ((3.0, slice(1, 40)), (10.0, slice(40, 80)), (200.0, slice(80, 160))):
        lam = lv / 255.0 * 256.0
        d = draws[:, :, rows].reshape(-1).double().cpu().numpy()
        assert abs(d - d.round()).max() < 2e-2            # integers up to fp32 rounding of the affine map
        d = d.round()
        n = d.size
        assert abs(d.mean() - lam) < 5 * (lam / n) ** 0.5
        assert abs(d.var() - lam) < 0.05 * lam
        ks = st.kstest(d + np.random.default_rng(0).uniform(-0.5, 0.5, n), lambda t: _pois_cont_cdf(t, lam, st)).statistic
        assert ks < 0.02, ks
    out2 = ip.poisson_noise_sampled(x, scale, None, seed=1234, clip=False)
    assert not torch.equal(out, out2)                     # the call counter advanced
    gray = torch.ones(b, device=dev)
    og = ip.poisson_noise_sampled(x, scale, gray, seed=7, clip=False)
    nz = og - x
    assert (nz[:, 0] - nz[:, 1]).abs().max().item() < 1e-6 and (nz[:, 0] - nz[:, 2]).abs().max().item() < 1e-6


def _pois_cont_cdf(t, lam, st):
    """CDF of Poisson(lam) + Uniform(-0.5, 0.5) (continuity-smoothed, so the KS statistic is meaningful)."""
    k = np.floor(t + 0.5)
    frac = t + 0.5 - k
    return st.poisson.cdf(k - 1, lam) + frac * st.poisson.pmf(k, lam)


@pytest.mark.gpu
def test_gaussian_noise_sampled_in_kernel_statistics():
    """resr_gaussian_noise_sampled: N(0, (sigma/255)^2) colour noise per element, ONE gray field shared by the batch
    (imgproc.py:853-861), fresh draws on every call."""
    import scipy.stats as st
    import resr_b200
    ip = resr_b200.imgproc
    dev = "cuda"
    b, h, w = 3, 128, 192
    x = torch.full((b, 3, h, w), 0.5, device=dev)
    sigma = torch.tensor([5.0, 10.0, 20.0], device=dev)
    out = ip.gaussian_noise_sampled(x, sigma, None, seed=99, clip=False)
    for i in range(b):
        z = ((out[i] - 0.5) * 255.0 / sigma[i]).reshape(-1).double().cpu().numpy()
        assert abs(z.mean()) < 5 / np.sqrt(z.size) and abs(z.std() - 1) < 0.01
        assert st.kstest(z, "norm").statistic < 0.01
    c01 = np.corrcoef(((out[0, 0] - 0.5)).reshape(-1).cpu().numpy(), ((out[0, 1] - 0.5)).reshape(-1).cpu().numpy())[0, 1]
    assert abs(c01) < 0.02                                        # channels are independent
    assert not torch.equal(out, ip.gaussian_noise_sampled(x, sigma, None, seed=99, clip=False))
    gray = torch.tensor([1.0, 1.0, 0.0], device=dev)
    og = ip.gaussian_noise_sampled(x, sigma, gray, seed=5, clip=False)
    n0, n1 = (og[0] - 0.5) / sigma[0], (og[1] - 0.5) / sigma[1]
    assert (n0[0] - n0[1]).abs().max().item() < 1e-6              # gray: same field on the three channels ...
    assert (n0 - n1).abs().max().item() < 1e-6                    # ... and on every gray sample of the batch
    assert (og[2, 0] - og[2, 1]).abs().max().item() > 1e-3        # colour sample keeps independent channels


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2, 3, 4, 5])
def test_pipeline_graph_with_device_drawn_noise(seed):
    """Random plans (every branch mix the seeds reach) with ALL noise drawn inside the kernels, through the CUDA-graph
    pipeline, the Python-sequenced block and the one-call C ABI: shapes, u8 grid, finite values, fresh draws per replay."""
    import resr_b200
    ip = resr_b200.imgproc
    b, h, w = 4, 128, 160
    plan = resr_b200.plan.synth_plan(b, h, w, seed=seed, image_size=96, device_noise=True)
    g = torch.Generator().manual_seed(seed)
    hr = torch.rand(b, 3, h, w, generator=g).cuda()
    k = torch.zeros(b, 21, 21)
    k[:, 8:13, 8:13] = 1 / 25
    k = k.cuda()
    sk = torch.zeros(b, 21, 21)
    sk[:, 10, 10] = 1
    sk = sk.cuda()
    pipe = ip.DegradePipeline(hr, k, k, sk, plan)
    outs = []
    for _ in range(2):
        lr, hrc = pipe()
        outs.append(lr.clone())
        assert lr.shape == (b, 3, 24, 24) and hrc.shape == (b, 3, 96, 96)
        assert torch.isfinite(lr).all() and lr.min().item() >= 0 and lr.max().item() <= 1
        assert (lr * 255 - torch.round(lr * 255)).abs().max().item() < 1e-4
    assert not torch.equal(outs[0], outs[1])               # replays draw fresh noise
    for fn in (ip.degrade_batch, ip.degrade_batch_native):
        lr, hrc = fn(hr, k, k, sk, plan)
        assert lr.shape == (b, 3, 24, 24) and torch.isfinite(lr).all()
        assert torch.equal(hrc, outs and pipe()[1])


@pytest.mark.gpu
def test_device_side_kernel_parameter_draws_follow_the_reference_distributions():
    """f3: resr_draw_degradation_kernel_params replaces the per-sample host loop of dataset.py:81-141. The draws come from
    another RNG stream than the reference's, so they are checked as DISTRIBUTIONS (config.py:20-39), and the kernels made
    from them against the float64 oracle evaluated on the same parameters."""
    import ctypes
    import resr_b200
    from oracle import kernels as ok
    ip, L = resr_b200.imgproc, resr_b200._lib
    P = resr_b200.plan.DEGRADATION_MODEL_PARAMETERS
    n = 30000
    k1, k2, sk, params = ip.draw_degradation_kernels_device(n, P, seed=123, return_params=True)
    assert k1.shape == (n, 21, 21) and k1.dtype == torch.float32
    for t in (k1, k2, sk):
        assert np.abs(t.sum((1, 2)).cpu().numpy() - 1).max() < 1e-5
    raw = params.cpu().numpy().tobytes()
    arr = (L.KernelParams * (3 * n)).from_buffer_copy(raw)
    names = {0: "gaussian", 1: "generalized", 2: "plateau", 3: "sinc", 4: "delta"}
    tol = 4.5 / np.sqrt(n)   # ~4.5 sigma of a binomial proportion (p(1-p) <= 1/4 -> sigma <= 0.5/sqrt(n))
    for which, probs, srange in ((0, P["gaussian_kernel_probability1"], P["gaussian_sigma_range1"]),
                                 (1, P["gaussian_kernel_probability2"], P["gaussian_sigma_range2"])):
        ps = [arr[3 * i + which] for i in range(n)]
        types = np.array([p.type for p in ps])
        sizes = np.array([p.kernel_size for p in ps])
        iso = np.array([p.isotropic for p in ps])
        assert set(np.unique(sizes)) == set(P["gaussian_kernel_range"])
        for s in P["gaussian_kernel_range"]:
            assert abs((sizes == s).mean() - 1 / 8) < tol
        assert abs((types == 3).mean() - 0.1) < tol                     # sinc_kernel_probability
        mixed = types != 3
        want = {(0, 1): probs[0], (0, 0): probs[1], (1, 1): probs[2], (1, 0): probs[3], (2, 1): probs[4], (2, 0): probs[5]}
        for (ty, is_iso), pr in want.items():
            got = ((types == ty) & (iso == is_iso)).sum() / mixed.sum()
            assert abs(got - pr) < 1.5 * tol, (ty, is_iso, got, pr)
        sx = np.array([p.sigma_x for p in ps])[mixed]
        assert sx.min() >= srange[0] and sx.max() <= srange[1] and abs(sx.mean() - sum(srange) / 2) < 0.03
        aniso = mixed & (iso == 0)
        th = np.array([p.theta for p in ps])[aniso]
        assert th.min() >= -np.pi and th.max() <= np.pi and abs(th.mean()) < 0.08
        beta_g = np.array([p.beta for p in ps])[types == 1]
        assert beta_g.min() >= 0.5 and beta_g.max() <= 4 and abs((beta_g < 1).mean() - 0.5) < 3 * tol
        beta_p = np.array([p.beta for p in ps])[types == 2]
        assert beta_p.min() >= 1 and beta_p.max() <= 2
        cut = np.array([p.cutoff for p in ps])[types == 3]
        small = sizes[types == 3] < 13
        assert cut[small].min() >= np.pi / 3 - 1e-12 and cut[~small].min() >= np.pi / 5 - 1e-12 and cut.max() <= np.pi + 1e-12
    third = [arr[3 * i + 2] for i in range(n)]
    t3 = np.array([p.type for p in third])
    assert set(np.unique(t3)) == {3, 4} and abs((t3 == 3).mean() - 0.8) < tol
    assert all(p.kernel_size == 21 for p in third if p.type == 4)
    # kernels evaluated from the drawn parameters == float64 oracle on the same parameters
    for idx in range(0, 60):
        p = arr[idx]
        d = {"type": names[p.type], "kernel_size": p.kernel_size, "isotropic": bool(p.isotropic), "sigma_x": p.sigma_x,
             "sigma_y": p.sigma_y, "theta": p.theta, "beta": p.beta, "cutoff": p.cutoff}
        ref = ok.from_params(d, 21)
        got = (k1, k2, sk)[idx % 3][idx // 3].cpu().numpy()
        assert np.abs(got - ref).max() <= 1e-7
    # fresh draws per call for a fixed seed
    k1b, _, _ = ip.draw_degradation_kernels_device(16, P, seed=123)
    k1c, _, _ = ip.draw_degradation_kernels_device(16, P, seed=123)
    assert not torch.equal(k1b, k1c)


@pytest.mark.gpu
def test_augment_batch_is_the_reference_chain_bit_for_bit():
    """SURVEY.md §8 f3 (data path): rotate / flip / BGR->RGB / image_to_tensor of dataset.py:67-79 as one device gather,
    against the golden outputs of the reference's own functions and against the oracle on a 400 x 400 batch."""
    import os
    import numpy as np
    import resr_b200
    from oracle import augment as oa
    ip = resr_b200.imgproc
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "augment.npz"))
    for idx in range(6):
        img = gold[f"img{idx}"]
        combos = [(ai, hf, vf) for ai in range(4) for hf in (0, 1) for vf in (0, 1)]
        batch = torch.from_numpy(np.stack([img] * len(combos))).cuda()
        ops = torch.tensor([oa.pack_op(*c) for c in combos], dtype=torch.int32)
        out = ip.augment_batch(batch, ops).cpu().numpy()
        for k, (ai, hf, vf) in enumerate(combos):
            assert np.array_equal(out[k], gold[f"out{idx}_{ai}_{hf}_{vf}"]), (idx, ai, hf, vf)
    rng = np.random.default_rng(3)
    imgs = rng.integers(0, 256, (16, 400, 400, 3), dtype=np.uint8)   # the reference's dataset images are 400 x 400
    import random
    random.seed(9)
    ops = ip.draw_augment_ops(16)
    out = ip.augment_batch(torch.from_numpy(imgs).cuda(), ops).cpu().numpy()
    for k in range(16):
        op = int(ops[k])
        assert np.array_equal(out[k], oa.augment(imgs[k], op & 3, bool(op & 4), bool(op & 8)))


@pytest.mark.gpu
def test_degrade_pipeline_fed_with_u8_images():
    """DegradePipeline(u8_images=True): the augmentation gather is the first node of the captured graph; the result equals
    augment_batch followed by the plain pipeline."""
    import random
    import resr_b200
    ip = resr_b200.imgproc
    B, H, W = 4, 64, 72
    plan = resr_b200.plan.canonical_plan_s0(B, H, W, seed=2)
    rng = np.random.default_rng(5)   # host-fed second noise: the in-kernel Poisson draws advance a per-device call counter
    plan["noise2"] = {"type": "gaussian", "sigma": rng.uniform(1, 25, size=B).astype(np.float32), "gray": plan["noise1"]["gray"],
                      "noise_color": rng.standard_normal((B, 3, H // 4, W // 4), dtype=np.float32),
                      "noise_gray": rng.standard_normal((H // 4, W // 4), dtype=np.float32)}
    torch.manual_seed(0)
    k = torch.zeros(B, 21, 21)
    k[:, 8:13, 8:13] = 1.0 / 25
    sk = torch.zeros(B, 21, 21)
    sk[:, 10, 10] = 1
    k, sk = k.cuda(), sk.cuda()
    imgs = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8).cuda()
    random.seed(4)
    ops = ip.draw_augment_ops(B)
    hr = ip.augment_batch(imgs, ops)
    ref = ip.DegradePipeline(hr, k, k, sk, plan)
    lr_ref, hrc_ref = ref()
    pipe = ip.DegradePipeline(torch.zeros_like(hr), k, k, sk, plan, u8_images=True)
    pipe.images_u8.copy_(imgs)
    pipe.augment_ops.copy_(ops)
    for _ in range(2):
        lr, hrc = pipe()
    torch.cuda.synchronize()
    assert torch.equal(lr, lr_ref) and torch.equal(hrc, hrc_ref)
