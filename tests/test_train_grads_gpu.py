"""Per-tensor parity of every generator gradient, biases included, against float64 autograd of the oracle, with a
nonzero bias on every convolution (oracle.generator.rich_state_dict) so that the bias paths of the forward, the data
gradient and the weight gradient all carry signal.

For each of the 702 tensors, e_k is the relative L2 error of the kernel's gradient against plain float64 autograd and
d_k that of the recipe's noise model (oracle.generator.grads: 16-bit operands and bf16 output gradients at every
convolution) against the same reference. Every tensor must meet e_k <= 3 d_k + 1e-3: an error confined to one layer, or
to one bias, that the whole-network cosine cannot see fails here. The median of e_k / d_k must stay <= 1.5, which
catches an extra error spread evenly over all layers."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# forward operand, output-gradient and backward operand format. The fp16 recipe's backward kernels read bf16 operands
# only: the data-gradient convolutions use bf16 transposed weight packs and the weight gradient converts the saved fp16
# activations to bf16. Modelling its backward with fp16 operands instead leaves its L1-loss gradients ~2x noisier than
# the model (median e_k / d_k ~1.6-2.0 on the B200) while the bf16 recipe sits at ~1.0.
RECIPES = {"fp16": (torch.float16, torch.bfloat16, torch.bfloat16), "bf16": (torch.bfloat16, torch.bfloat16, torch.bfloat16)}
FACTOR, FLOOR, MEDIAN_MAX = 3.0, 1e-3, 1.5
MAX_ABS, MIN_PSNR = 2e-2, 45.0


def _inputs(case):
    """case = (seed, shape, loss): the LR batch and the loss target. "l1" is the training loss against a random HR image;
    "dot" is sum(sr * R) with a fixed random R, a smooth upstream gradient that is nonzero at every output pixel."""
    seed, shape, loss = case
    gen = torch.Generator().manual_seed(700 + seed)
    x = torch.rand(shape, generator=gen)
    out = (shape[0], 3, 4 * shape[2], 4 * shape[3])
    if loss == "l1":
        return x, torch.rand(out, generator=gen)
    return x, torch.randn(out, generator=gen) / math.prod(out)


def _loss_fn(loss, target):
    t = target.double()
    return (lambda sr: F.l1_loss(sr, t)) if loss == "l1" else (lambda sr: (sr * t).sum())


@pytest.fixture(scope="module")
def oracle():
    """Flat float64 gradients of a case, cached by (case, recipe); recipe None is the plain float64 reference."""
    from oracle import generator as og
    sds, runs = {}, {}

    def state_dict(seed):
        if seed not in sds:
            sds[seed] = og.rich_state_dict(seed)
        return sds[seed]

    def grads(case, recipe=None):
        if (case, recipe) not in runs:
            sd = state_dict(case[0])
            x, target = _inputs(case)
            fmts = RECIPES[recipe] if recipe else (None, None, None)
            _, g, sr = og.grads(x, sd, _loss_fn(case[2], target), *fmts)
            if recipe is None:
                lo, hi = (sr == 0).double().mean((0, 2, 3)), (sr == 1).double().mean((0, 2, 3))
                print(f"{case}: output clamped at 0 per channel {lo.tolist()}, at 1 {hi.tolist()}")
            runs[(case, recipe)] = torch.cat([g[k].reshape(-1) for k in sd])
        return runs[(case, recipe)]

    grads.state_dict = state_dict
    return grads


def _generator(sd, precision):
    import resr_b200
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    return g.cuda().train().set_precision(precision)


def _cos(a, b):
    return float(torch.dot(a.double(), b.double()) / (a.double().norm() * b.double().norm() + 1e-300))


def _per_tensor_gate(label, sd, got, ref, model):
    """e_k <= FACTOR * d_k + FLOOR for every tensor and median(e_k / d_k) <= MEDIAN_MAX; prints the ten worst ratios."""
    got = got.detach().cpu().double()
    assert got.shape == ref.shape and torch.isfinite(got).all()
    rows, pos = [], 0
    for name, v in sd.items():
        sl = slice(pos, pos + v.numel())
        pos += v.numel()
        r = float(ref[sl].norm())
        assert r > 0, name
        e, d = float((got[sl] - ref[sl]).norm()) / r, float((model[sl] - ref[sl]).norm()) / r
        rows.append((e / d, e, d, name))
    rows.sort(reverse=True)
    ratios = sorted(row[0] for row in rows)
    median = ratios[len(ratios) // 2]
    print(f"\n{label}: median e/d {median:.3f}; worst e/d:")
    for ratio, e, d, name in rows[:10]:
        print(f"    {ratio:7.3f}  e {e:.3e}  d {d:.3e}  {name}")
    bad = [(name, e, d) for _, e, d, name in rows if e > FACTOR * d + FLOOR]
    assert not bad, f"{len(bad)} tensors over {FACTOR} d + {FLOOR}: {bad[:10]}"
    assert median <= MEDIAN_MAX


@pytest.fixture
def pair_policy(request):
    import resr_b200
    lib = resr_b200._lib.lib()
    prev = lib.resr_set_conv_pair_policy(request.param)
    yield request.param
    lib.resr_set_conv_pair_policy(prev)


SHAPES = [(1, 3, 16, 24), (2, 3, 16, 64), (3, 3, 5, 8), (1, 3, 1, 8), (1, 3, 9, 136), (2, 3, 7, 13), (1, 3, 3, 257)]
# every shape in both recipes; the fp16 cases with W % 8 != 0 come last so that each earlier case keeps its test id
CASES = [("fp16", s) for s in SHAPES[:5]] + [("bf16", s) for s in SHAPES] + [("fp16", s) for s in SHAPES[5:]]


@pytest.mark.parametrize("pair_policy", [1, 2], indirect=True)
@pytest.mark.parametrize("precision,shape", CASES)
def test_l1_gradients_per_tensor_vs_float64(oracle, precision, shape, pair_policy):
    """The fused training step (autograd.l1_loss_backward: resr_generator_forward_train + resr_generator_backward_l1)."""
    import resr_b200
    case = (SHAPES.index(shape), shape, "l1")
    sd = oracle.state_dict(case[0])
    x, hr = _inputs(case)
    g = _generator(sd, precision)
    _, _, flat = resr_b200.autograd.l1_loss_backward(g, x.cuda(), hr.cuda())
    torch.cuda.synchronize()
    _per_tensor_gate(f"[{precision} policy {pair_policy} {shape} l1]", sd, flat, oracle(case), oracle(case, precision))


@pytest.mark.parametrize("precision,shape,pair_policy", [("fp16", (1, 3, 16, 24), 2), ("bf16", (3, 3, 5, 8), 1)],
                         indirect=["pair_policy"])
def test_autograd_function_gradients_per_tensor_vs_float64(oracle, precision, shape, pair_policy):
    """Generator.forward + sum(sr * R).backward(): resr_generator_backward with a smooth upstream gradient that crosses
    the output clamp."""
    case = (10, shape, "dot")
    sd = oracle.state_dict(case[0])
    x, r = _inputs(case)
    g = _generator(sd, precision)
    g.zero_grad(set_to_none=True)
    (g(x.cuda()) * r.cuda()).sum().backward()
    flat = torch.cat([p.grad.reshape(-1) for p in g.parameters()])
    _per_tensor_gate(f"[{precision} policy {pair_policy} {shape} sum(sr*R)]", sd, flat, oracle(case), oracle(case, precision))


def test_precision_switch_on_a_live_train_step(oracle):
    """Generator.set_precision between TrainStep.step calls: the captured step graph belongs to the old recipe and must
    not be replayed against weights repacked for the new one. Each step matches the eager step of the current recipe
    and the float64 reference, and the step runs as a graph again after each switch."""
    import resr_b200
    case = (11, (2, 3, 16, 32), "l1")
    sd = oracle.state_dict(case[0])
    x, hr = (t.cuda() for t in _inputs(case))
    g = _generator(sd, "fp16")
    ts = resr_b200.autograd.TrainStep(g, 2, 16, 32)
    for it, precision in enumerate(("fp16", "fp16", "bf16", "fp16")):
        g.set_precision(precision)
        loss_g, _, flat_g = ts.step(x, hr, scatter=False)
        loss_g, flat_g = loss_g.item(), flat_g.clone()
        assert ts.is_graph
        loss_e, _, flat_e = resr_b200.autograd.l1_loss_backward(g, x, hr)
        torch.cuda.synchronize()
        cos = _cos(flat_e, flat_g)
        print(f"step {it} [{precision}]: loss graph {loss_g:.7f} eager {loss_e.item():.7f}; cosine {cos:.8f}")
        assert abs(loss_e.item() - loss_g) <= 1e-6 and cos >= 0.999999
        _per_tensor_gate(f"[step {it} {precision}]", sd, flat_g, oracle(case), oracle(case, precision))


def _psnr(a, b):
    mse = torch.mean((a.double() - b.double()) ** 2).item()
    return 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)


@pytest.fixture(scope="module")
def forward_refs():
    from oracle import generator as og
    refs = {}

    def get(seed, shape):
        if (seed, shape) not in refs:
            x = torch.rand(shape, generator=torch.Generator().manual_seed(800 + seed))
            sd = og.rich_state_dict(seed)
            refs[(seed, shape)] = sd, x, og.generator_forward(x, sd)
        return refs[(seed, shape)]
    return get


@pytest.mark.parametrize("pair_policy", [1, 2], indirect=True)
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("seed,shape", [(1, (2, 3, 24, 40)), (3, (1, 3, 20, 128))])
def test_generator_forward_with_nonzero_biases_vs_oracle(forward_refs, seed, shape, precision, pair_policy):
    sd, x, ref = forward_refs(seed, shape)
    g = _generator(sd, precision).eval()
    with torch.no_grad():
        y = g(x.cuda()).cpu()
    err, ps = (y - ref).abs().max().item(), _psnr(y, ref)
    print(f"[{precision} policy {pair_policy}] {shape}: max-abs {err:.3e}  psnr {ps:.2f} dB")
    assert err <= MAX_ABS and ps >= MIN_PSNR


@pytest.mark.parametrize("pair_policy", [1, 2], indirect=True)
def test_dense_blocks_with_nonzero_biases_vs_oracle(pair_policy):
    """ResidualDenseBlock / ResidualResidualDenseBlock forwards (resr_conv3x3) with nonzero biases; same bound as
    tests/test_generator_gpu.py::test_dense_block_forwards_vs_oracle."""
    from oracle import generator as og
    sd = og.rich_state_dict(2)
    g = _generator(sd, "fp16").eval()
    torch.manual_seed(8)
    x = torch.randn(2, 64, 20, 136) * 0.5
    rrdb = g.trunk[3]
    with torch.no_grad():
        y_rdb = rrdb.rdb2(x.cuda()).cpu()
        y_rrdb = rrdb(x.cuda()).cpu()
    e1 = (y_rdb - og.rdb_forward(x, sd, "trunk.3.rdb2")).abs().max().item()
    e2 = (y_rrdb - og.rrdb_forward(x, sd, "trunk.3")).abs().max().item()
    print(f"[policy {pair_policy}] rdb max-abs {e1:.2e}, rrdb max-abs {e2:.2e}")
    assert e1 <= 4e-3 and e2 <= 4e-3
