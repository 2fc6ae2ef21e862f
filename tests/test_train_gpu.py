"""GPU parity of the training path (SURVEY.md row a5): tensor-core weight gradient, and loss + parameter gradients of
the whole generator against fp32 autograd of the oracle. BASELINE.json states no tolerance for the training step;
the gate proposed in SURVEY.md §8d is used: loss within 1e-3 relative, global gradient cosine >= 0.999 and global
relative L2 error <= 3 %."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,h,w,cin,xs,cout,ys", [(2, 12, 64, 64, 64, 32, 64), (1, 9, 128, 160, 192, 32, 64), (2, 16, 64, 192, 192, 64, 64),
                                                 (1, 8, 72, 64, 64, 3, 64), (3, 5, 16, 96, 192, 32, 192), (1, 7, 9, 3, 64, 64, 64),
                                                 (2, 6, 150, 192, 192, 192, 192), (1, 3, 1, 130, 136, 70, 72), (4, 32, 32, 128, 192, 128, 128)])
def test_wgrad_nhwc_kernel(n, h, w, cin, xs, cout, ys):
    """MN-major weight-gradient kernel (csrc/wgrad_mn.cu: both operands straight from NHWC bf16 buffers, pixel shifts as
    descriptor / TMA-coordinate shifts) vs torch's conv2d_weight in float64 on the same bf16-rounded operands. Ragged and odd
    widths, one-pixel rows, 3 input channels, 3 ci blocks x 2 co chunks (every unit shape), garbage in the unused channels."""
    import resr_b200
    L = resr_b200._lib
    torch.manual_seed(n + h + w + cin + cout)
    dev = "cuda"
    x = torch.randn(n, cin, h, w, device=dev).bfloat16().float()
    dy = torch.randn(n, cout, h, w, device=dev).bfloat16().float()
    x16 = torch.randn(n, h, w, xs, device=dev).bfloat16()
    x16[..., :cin] = x.permute(0, 2, 3, 1).bfloat16()
    dy16 = torch.randn(n, h, w, ys, device=dev).bfloat16()
    dy16[..., :cout] = dy.permute(0, 2, 3, 1).bfloat16()
    dy16[..., cout:(cout + 7) // 8 * 8] = 0
    dw = torch.full((cout, cin, 3, 3), float("nan"), device=dev)
    db = torch.full((cout,), float("nan"), device=dev)
    need = L.lib().resr_conv3x3_wgrad_nhwc_workspace_bytes()
    ws = torch.empty(need + 1024, dtype=torch.uint8, device=dev)
    wp = ws.data_ptr() + (-ws.data_ptr()) % 1024
    for _ in range(2):  # twice: the second call runs on a dirty partial buffer
        L.check(L.lib().resr_conv3x3_wgrad_nhwc(L.ptr(x16), xs, L.ptr(dy16), ys, n, h, w, cin, cout, L.ptr(dw), L.ptr(db),
                                                ctypes.c_void_p(wp), need, L.stream_ptr()))
    torch.cuda.synchronize()
    ref_w = torch.nn.grad.conv2d_weight(x.double(), (cout, cin, 3, 3), dy.double(), padding=1).float()
    ref_b = dy.double().sum((0, 2, 3)).float()
    scale = ref_w.abs().max().item()
    assert torch.isfinite(dw).all() and torch.isfinite(db).all()
    err = (dw - ref_w).abs().max().item()
    print(f"wgrad nhwc max err {err:.3e} (scale {scale:.3e})")
    assert err <= 1e-4 * scale + 1e-4
    assert (db - ref_b).abs().max().item() <= 1e-3 * ref_b.abs().max().item() + 1e-3


def _cos(a, b):
    return float(torch.dot(a.double(), b.double()) / (a.double().norm() * b.double().norm() + 1e-300))


@pytest.mark.parametrize("seed,shape", [(0, (1, 3, 16, 24)), (1, (2, 3, 16, 64)), (2, (3, 3, 5, 8)), (3, (1, 3, 9, 136))])
@pytest.mark.parametrize("policy,precision", [(1, "fp16"), (2, "fp16"), (1, "bf16"), (2, "bf16")])
def test_generator_loss_and_gradients_vs_oracle_autograd(seed, shape, policy, precision):
    import resr_b200
    from oracle import generator as og
    prev = resr_b200._lib.lib().resr_set_conv_pair_policy(policy)  # 2: forward / data-gradient convs on CTA pairs
    sd = og.random_state_dict(seed)
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    g = g.cuda()
    g.set_precision(precision)  # bf16: activations and gradients in one format, MN-major weight-gradient kernel (wgrad_mn.cu)
    torch.manual_seed(50 + seed)
    x = torch.rand(*shape)
    hr = torch.rand(shape[0], 3, 4 * shape[2], 4 * shape[3])
    ref_loss, ref_grads, ref_sr = og.l1_loss_and_grads(x, hr, sd)
    loss, sr, flat = resr_b200.autograd.l1_loss_backward(g, x.cuda(), hr.cuda())
    torch.cuda.synchronize()
    resr_b200._lib.lib().resr_set_conv_pair_policy(prev)
    assert (sr.cpu() - ref_sr).abs().max().item() <= 2e-2
    rel = abs(loss.item() - ref_loss.item()) / ref_loss.item()
    ref_flat = torch.cat([ref_grads[k].reshape(-1) for k in sd])
    got = flat.cpu()
    assert torch.isfinite(got).all()
    cos = _cos(got, ref_flat)
    rl2 = float((got - ref_flat).double().norm() / ref_flat.double().norm())
    worst = 1.0
    pos = 0
    for k in sd:
        nel = sd[k].numel()
        if nel >= 1024:
            worst = min(worst, _cos(got[pos:pos + nel], ref_flat[pos:pos + nel]))
        pos += nel
    print(f"[{precision}] loss rel err {rel:.2e}; grad cosine {cos:.5f}; rel-L2 {rl2:.3%}; worst per-tensor cosine {worst:.4f}")
    assert rel <= 1e-3 and cos >= 0.999 and rl2 <= 0.03 and worst >= 0.98
    # param.grad populated in state_dict order
    p0 = next(g.parameters())
    assert torch.allclose(p0.grad.cpu(), ref_grads["conv1.weight"], atol=5e-2 * ref_grads["conv1.weight"].abs().max().item() + 1e-7)


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_trains_on_widths_that_are_not_multiples_of_8(precision):
    """The NHWC weight-gradient path has no W % 8 restriction, in either recipe."""
    import resr_b200
    from oracle import generator as og
    sd = og.random_state_dict(4)
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    g = g.cuda()
    g.set_precision(precision)
    torch.manual_seed(54)
    x = torch.rand(2, 3, 7, 13)
    hr = torch.rand(2, 3, 28, 52)
    ref_loss, ref_grads, _ = og.l1_loss_and_grads(x, hr, sd)
    loss, _, flat = resr_b200.autograd.l1_loss_backward(g, x.cuda(), hr.cuda())
    ref_flat = torch.cat([ref_grads[k].reshape(-1) for k in sd])
    cos = _cos(flat.cpu(), ref_flat)
    rl2 = float((flat.cpu() - ref_flat).double().norm() / ref_flat.double().norm())
    print(f"13-wide {precision} step: grad cosine {cos:.5f}; rel-L2 {rl2:.3%}")
    assert abs(loss.item() - ref_loss.item()) / ref_loss.item() <= 1e-3 and cos >= 0.999 and rl2 <= 0.03


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_identical_steps_give_bit_identical_gradients(precision):
    """Weight and bias gradients are summed in a fixed order (no atomics): two eager steps on the same weights and inputs
    return the same flat gradient vector, bit for bit."""
    import resr_b200
    from oracle import generator as og
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.rich_state_dict(5))
    g = g.cuda().train()
    g.set_precision(precision)
    torch.manual_seed(55)
    lr = torch.rand(2, 3, 16, 40, device="cuda")
    hr = torch.rand(2, 3, 64, 160, device="cuda")
    loss_a, sr_a, flat_a = resr_b200.autograd.l1_loss_backward(g, lr, hr)
    loss_b, sr_b, flat_b = resr_b200.autograd.l1_loss_backward(g, lr, hr)
    torch.cuda.synchronize()
    assert torch.equal(sr_a, sr_b) and torch.equal(loss_a, loss_b)
    assert torch.isfinite(flat_a).all() and torch.equal(flat_a, flat_b)


def test_autograd_function_matches_fused_path():
    """`loss.backward()` through Generator.forward (torch autograd.Function) gives the same gradients as the fused call."""
    import resr_b200
    from oracle import generator as og
    sd = og.random_state_dict(3)
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    g = g.cuda().train()
    torch.manual_seed(7)
    x = torch.rand(1, 3, 16, 16, device="cuda")
    hr = torch.rand(1, 3, 64, 64, device="cuda")
    _, _, flat = resr_b200.autograd.l1_loss_backward(g, x, hr)
    g.zero_grad(set_to_none=True)
    sr = g(x)
    loss = F.l1_loss(sr, hr)
    loss.backward()
    got = torch.cat([p.grad.reshape(-1) for p in g.parameters()])
    assert _cos(got, flat) >= 0.99999


@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_train_step_graph_replay_matches_eager(precision):
    """The CUDA-graph training step (persistent buffers) reproduces the eager fused call, also after a weight update."""
    import resr_b200
    from oracle import generator as og
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.random_state_dict(2))
    g = g.cuda().train()
    g.set_precision(precision)
    torch.manual_seed(11)
    lr = torch.rand(2, 3, 16, 32, device="cuda")
    hr = torch.rand(2, 3, 64, 128, device="cuda")
    ts = resr_b200.autograd.TrainStep(g, 2, 16, 32)
    for it in range(3):
        loss_e, _, flat_e = resr_b200.autograd.l1_loss_backward(g, lr, hr)
        loss_g, _, flat_g = ts.step(lr, hr)
        torch.cuda.synchronize()
        assert abs(loss_e.item() - loss_g.item()) <= 1e-6
        assert _cos(flat_e.cpu(), flat_g.cpu()) >= 0.999999
        with torch.no_grad():  # SGD-like update: the packed (and transposed) weights must follow
            for p in g.parameters():
                p.add_(p.grad, alpha=-1e-3)
    assert ts.is_graph


@pytest.mark.gpu
def test_flat_adam_ema_matches_torch_adam_and_reference_ema():
    """SURVEY.md §8 row f1: resr_adam_ema_step vs torch.optim.Adam(lr, betas) (train_realesrnet.py:197-200) followed by the
    reference EMA update (model.py:42-49), five steps on the generator's real parameter layout."""
    import resr_b200
    torch.manual_seed(0)
    g = resr_b200.model.Generator(3, 3, 4).cuda()
    keys = list(g.state_dict().keys())
    ref_params = [p.detach().clone().requires_grad_(True) for p in g.parameters()]
    ref_opt = torch.optim.Adam(ref_params, 2e-4, (0.9, 0.99))
    shadow = [p.detach().clone() for p in ref_params]
    opt = resr_b200.optim.FlatAdamEMA(g, lr=2e-4, betas=(0.9, 0.99), ema_decay=0.999)
    assert list(g.state_dict().keys()) == keys and next(g.parameters()).data_ptr() == opt.flat.data_ptr()
    x = torch.rand(1, 3, 16, 24, device="cuda")
    with torch.no_grad():
        y0 = g(x).clone()
    n = opt.flat.numel()
    for step in range(5):
        grads = torch.randn(n, device="cuda") * (10.0 ** (step - 3))
        pos = 0
        for p in ref_params:
            p.grad = grads[pos:pos + p.numel()].view_as(p).clone()
            pos += p.numel()
        ref_opt.step()
        for s_, p in zip(shadow, ref_params):
            s_.copy_((1.0 - 0.999) * p.data + 0.999 * s_)
        opt.step(grads)
    ref_flat = torch.cat([p.detach().reshape(-1) for p in ref_params])
    ref_shadow = torch.cat([s_.reshape(-1) for s_ in shadow])
    assert (opt.flat - ref_flat).abs().max().item() <= 2e-7
    assert (opt.shadow - ref_shadow).abs().max().item() <= 2e-7
    torch.testing.assert_close(torch.cat([p.detach().reshape(-1) for p in g.parameters()]), opt.flat, rtol=0, atol=0)
    with torch.no_grad():
        y1 = g(x)                                    # weights were repacked from the master copy
    assert (y1 - y0).abs().max().item() > 0
    opt.apply_shadow()
    with torch.no_grad():
        y2 = g(x)
    opt.restore()
    with torch.no_grad():
        y3 = g(x)
    assert torch.equal(y3, y1) and not torch.equal(y2, y1)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
def test_training_loop_step_graph_plus_fused_optimizer_reduces_the_loss(precision):
    """The pieces together as train_realesrnet.py:383-394 uses them: TrainStep (one CUDA-graph replay per step), flat Adam +
    EMA, weights repacked from the flat master copy — eight iterations on one fixed batch must drive the L1 loss down, and
    the first step must equal a torch.optim.Adam step taken from the same gradients."""
    import resr_b200
    torch.manual_seed(3)
    g = resr_b200.model.Generator(3, 3, 4).cuda().train()
    g.set_precision(precision)
    opt = resr_b200.optim.FlatAdamEMA(g, lr=2e-4, betas=(0.9, 0.99))
    ts = resr_b200.autograd.TrainStep(g, 2, 16, 24)
    lr = torch.rand(2, 3, 16, 24, device="cuda")
    hr = torch.rand(2, 3, 64, 96, device="cuda")
    p_before = opt.flat.clone()
    losses = []
    for it in range(8):
        loss, _, flat = ts.step(lr, hr, scatter=False)
        losses.append(float(loss.item()))
        if it == 0:
            ref = p_before.clone().requires_grad_(True)
            ref.grad = flat.clone()
            torch.optim.Adam([ref], 2e-4, (0.9, 0.99)).step()
        opt.step(flat)
        if it == 0:
            assert (opt.flat - ref.detach()).abs().max().item() <= 2e-7
    assert ts.is_graph
    print(f"[{precision}] losses", [round(v, 5) for v in losses])
    assert losses[-1] < losses[0] * 0.9 and min(losses[4:]) < min(losses[:2])
    assert torch.isfinite(opt.flat).all() and torch.isfinite(opt.shadow).all()


def test_stale_backward_is_refused():
    """ADVICE r01: the saved activations live in ONE workspace per Generator; a second training-mode forward before the
    first backward must not silently produce gradients for the wrong activations."""
    import resr_b200
    from oracle import generator as og
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.random_state_dict(0))
    g = g.cuda().train()
    x1 = torch.rand(1, 3, 8, 16, device="cuda")
    x2 = torch.rand(1, 3, 8, 16, device="cuda")
    sr1 = g(x1)
    sr2 = g(x2)                      # overwrites the activations sr1's graph refers to
    with pytest.raises(resr_b200._lib.ResrError):
        sr1.mean().backward()
    sr2.mean().backward()            # the latest forward is still consistent
    assert next(g.parameters()).grad is not None
    # an inference forward (no_grad) in between is harmless: it uses the inference workspace
    g.zero_grad(set_to_none=True)
    sr3 = g(x1)
    with torch.no_grad():
        g(x2)
    sr3.mean().backward()
    assert torch.isfinite(next(g.parameters()).grad).all()


def test_checkpoint_round_trip_in_reference_format(tmp_path):
    """f4: the reference's .pth.tar layout (train_realesrnet.py:117-129): our file feeds torch.optim.Adam / a fresh
    Generator exactly like a reference file, and a resumed FlatAdamEMA continues bit-identically."""
    import resr_b200
    from oracle import generator as og
    ck = resr_b200.checkpoint
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(og.random_state_dict(0))
    g = g.cuda().train()
    opt = resr_b200.optim.FlatAdamEMA(g, lr=2e-4, betas=(0.9, 0.99))
    torch.manual_seed(0)
    grads = [torch.randn(opt.flat.numel(), device="cuda") * 1e-3 for _ in range(3)]
    for gr in grads[:2]:
        opt.step(gr)
    path = str(tmp_path / "g_epoch_1.pth.tar")
    ck.save_checkpoint(path, g, opt, epoch=1, best_niqe=7.5, scheduler_state={"last_epoch": 1})
    file = torch.load(path, map_location="cpu")
    assert set(file) >= {"epoch", "best_niqe", "state_dict", "ema_state_dict", "optimizer", "scheduler"}
    assert set(file["state_dict"]) == set(og.random_state_dict(0)) and all(k.startswith("model.") for k in file["ema_state_dict"])
    # (a) reference side: a plain torch Adam over a fresh generator accepts the optimizer state and takes the same step
    g_ref = resr_b200.model.Generator(3, 3, 4)
    g_ref.load_state_dict({k.replace("model.", ""): v for k, v in file["state_dict"].items()})   # inference.py:33
    g_ref = g_ref.cuda()
    adam = torch.optim.Adam(g_ref.parameters(), 2e-4, (0.9, 0.99))
    adam.load_state_dict(file["optimizer"])
    pos = 0
    for p in g_ref.parameters():
        p.grad = grads[2][pos:pos + p.numel()].view_as(p).clone()
        pos += p.numel()
    adam.step()
    # (b) our side: resume into a fresh generator + optimizer, take the same third step
    g2 = resr_b200.model.Generator(3, 3, 4).cuda().train()
    opt2 = resr_b200.optim.FlatAdamEMA(g2, lr=1.0, betas=(0.5, 0.5))
    ck.load_checkpoint(path, g2, opt2)
    assert opt2.step_count == 2 and opt2.lr == 2e-4 and tuple(opt2.betas) == (0.9, 0.99)
    assert torch.equal(opt2.shadow, opt.shadow) and torch.equal(opt2.flat, opt.flat)
    opt.step(grads[2])
    opt2.step(grads[2])
    assert torch.equal(opt2.flat, opt.flat) and torch.equal(opt2.shadow, opt.shadow)
    ref_flat = torch.cat([p.detach().reshape(-1) for p in g_ref.parameters()])
    assert (ref_flat - opt.flat).abs().max().item() <= 2e-7


def test_gradient_buckets_follow_the_backward_order():
    """Data-parallel plumbing (SURVEY.md §8e): four contiguous buckets of the flat gradient vector, cut at trunk.5 / 11 / 17 in
    state_dict order; after a step the completion events of buckets 3, 2, 1 can be waited on from another stream (bucket 0
    closes with the step). The 2- and 8-GPU runs of tools/ddp_overlap_check.py (profiles/r02_ddp_overlap.txt) check that the
    bucketed all-reduce is bit-identical to the single all-reduce after the step."""
    import resr_b200
    L = resr_b200._lib
    g = resr_b200.model.Generator(3, 3, 4).cuda().train()
    g.set_precision("bf16")
    offs = (ctypes.c_size_t * 5)()
    assert L.lib().resr_generator_grad_buckets(offs, 5) == 4
    offs = [int(o) for o in offs]
    pos, want = 0, {}
    for k, v in g.state_dict().items():
        if k in ("trunk.5.rdb1.conv1.weight", "trunk.11.rdb1.conv1.weight", "trunk.17.rdb1.conv1.weight"):
            want[k] = pos
        pos += v.numel()
    assert offs == [0, want["trunk.5.rdb1.conv1.weight"], want["trunk.11.rdb1.conv1.weight"], want["trunk.17.rdb1.conv1.weight"], pos]
    ts = resr_b200.autograd.TrainStep(g, 1, 8, 8)
    side = torch.cuda.Stream()
    for it in range(2):   # eager step, then the graph replay
        _, _, flat = ts.step(torch.rand(1, 3, 8, 8).cuda(), torch.rand(1, 3, 32, 32).cuda(), scatter=False)
        for k in (3, 2, 1, 0):
            L.check(L.lib().resr_generator_wait_grad_bucket(g._native(), k, ctypes.c_void_p(side.cuda_stream)))
        side.synchronize()
        assert torch.isfinite(flat).all()
