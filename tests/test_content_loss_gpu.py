"""The VGG19 content loss of the RealESRGAN generator step (resr_b200.model.ContentLoss; reference ContentLoss,
model.py:278-335) against float64 torchvision: vgg19(weights=None) under a fixed seed, create_feature_extractor,
Normalize, F.l1_loss per node and autograd for d/d sr. The guards are 2x the worst value measured on a B200 (DESIGN.md §8).

The gradient of an L1 loss is sign(f_sr - f_gt): wherever the fp16 features of the tensor-core forward land on the other
side of f_gt than the float64 ones, the seed flips. A deep node's features carry enough forward rounding for that to
move the gradient by ~10 % (rel-L2) against float64 torchvision, although the losses agree to ~1e-4. The backward itself
is therefore also checked against a float64 oracle that stores the same fp16-rounded activations as the forward does
(straight-through rounding), so that seeds and ReLU masks agree and only the backward's own arithmetic differs."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
NODE_SETS = {
    "realesrgan": ["features.2", "features.7", "features.16", "features.25", "features.34"],
    "shallow": ["features.0"],
    "deep": ["features.34"],
    "all16": [f"features.{i}" for i in (0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34)],
}
SHAPES = [(2, 3, 64, 64), (1, 3, 37, 53), (3, 3, 16, 24), (2, 3, 19, 200), (16, 3, 256, 256)]
# guards against float64 torchvision, per node set: loss relative error, gradient cosine (1 - cos) and relative L2
# (2x the worst value measured over the five shapes on a B200, DESIGN.md §8)
LOSS_RTOL = 7e-3
GUARDS = {"realesrgan": (0.013, 0.23), "shallow": (3e-5, 0.011), "deep": (0.027, 0.33), "all16": (0.017, 0.19)}
# against the oracle with the forward's fp16 storage points (1 - cosine, rel-L2), 2x the worst measured value
GUARDS_FP16 = {"realesrgan": (0.0085, 0.19), "shallow": (1e-6, 0.0014), "deep": (0.012, 0.22), "all16": (0.0038, 0.15)}


def _vgg(seed=0):
    from torchvision.models import vgg19
    torch.manual_seed(seed)
    v = vgg19(weights=None)
    with torch.no_grad():   # torchvision initialises the biases to 0: give them values so that the bias path is checked
        for m in v.features:
            if isinstance(m, torch.nn.Conv2d):
                m.bias.normal_(0, 0.05)
    return v.eval()


def _oracle(vgg, nodes, sr, gt, wgt):
    """float64 torchvision on the GPU: losses and d(sum(wgt * losses))/d sr."""
    from torchvision.models.feature_extraction import create_feature_extractor
    from torchvision import transforms
    fe = create_feature_extractor(vgg.double().cuda(), nodes)
    norm = transforms.Normalize(MEAN, STD)
    x = sr.double().cuda().requires_grad_(True)
    fs = fe(norm(x))
    with torch.no_grad():
        fg = fe(norm(gt.double().cuda()))
    losses = torch.stack([F.l1_loss(fs[k], fg[k]) for k in nodes])
    (losses * wgt.double().cuda()).sum().backward()
    vgg.float()
    return losses.detach().cpu(), x.grad.cpu()


def _metrics(got, ref):
    g, r = got.double().flatten(), ref.double().flatten()
    cos = float(torch.dot(g, r) / (g.norm() * r.norm()))
    rl2 = float((g - r).norm() / r.norm())
    return cos, rl2


def _run(mod, sr, gt, wgt):
    x = sr.cuda().requires_grad_(True)
    losses = mod(x, gt.cuda())
    (losses * wgt.cuda()).sum().backward()
    torch.cuda.synchronize()
    return losses.detach().cpu(), x.grad.cpu()


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("nodes", list(NODE_SETS), ids=str)
def test_losses_and_input_gradient_match_torchvision(shape, nodes):
    import resr_b200
    names = NODE_SETS[nodes]
    vgg = _vgg()
    mod = resr_b200.model.ContentLoss(names, MEAN, STD, vgg=vgg).cuda()
    torch.manual_seed(1)
    sr, gt = torch.rand(shape), torch.rand(shape)
    wgt = torch.rand(len(names)) + 0.5
    got_l, got_g = _run(mod, sr, gt, wgt)
    ref_l, ref_g = _oracle(vgg, names, sr, gt, wgt)
    lerr = ((got_l.double() - ref_l).abs() / ref_l.abs()).max().item()
    cos, rl2 = _metrics(got_g, ref_g)
    print(f"content loss {nodes} {shape}: loss rel err {lerr:.2e}; grad cosine {cos:.6f}, rel-L2 {rl2:.3%}")
    assert lerr <= LOSS_RTOL
    assert 1 - cos <= GUARDS[nodes][0] and rl2 <= GUARDS[nodes][1]


def _emulated_oracle(vgg, nodes, sr, gt, wgt):
    """float64 VGG19 with the forward's storage points: fp16 weights, the normalized input and every conv output rounded to
    fp16 (after the ReLU, as stored), pooling on the rounded maps; rounding is straight-through for autograd."""
    sd = {k: v.double().cuda() for k, v in vgg.state_dict().items()}
    feats = [int(n.split(".")[1]) for n in nodes]
    convs = [i for i in (0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34) if i <= max(feats)]
    mean = torch.tensor(MEAN, dtype=torch.float64, device="cuda").view(1, 3, 1, 1)
    std = torch.tensor(STD, dtype=torch.float64, device="cuda").view(1, 3, 1, 1)
    r16 = lambda t: t + (t.half().double() - t).detach()

    def run(x):
        xf = x.float()
        xn = (xf - mean.float()) / std.float()   # fp32 normalize, as the layout kernel computes it
        a = (x - mean) / std
        a = a + (xn.half().double() - a).detach()
        out = {}
        for i in convs:
            y = F.conv2d(a, sd[f"features.{i}.weight"].half().double(), sd[f"features.{i}.bias"], padding=1)
            if i != max(feats):
                y = F.relu(y)
            y = r16(y)
            out[i] = y
            a = F.max_pool2d(y, 2) if i in (2, 7, 16, 25) else y
        return out

    x = sr.double().cuda().requires_grad_(True)
    fs = run(x)
    with torch.no_grad():
        fg = run(gt.double().cuda())
    losses = torch.stack([F.l1_loss(fs[f], fg[f]) for f in feats])
    (losses * wgt.double().cuda()).sum().backward()
    return losses.detach().cpu(), x.grad.cpu()


@pytest.mark.parametrize("shape", [(2, 3, 64, 64), (1, 3, 37, 53), (16, 3, 256, 256)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("nodes", list(NODE_SETS), ids=str)
def test_input_gradient_matches_an_oracle_with_the_same_fp16_activations(shape, nodes):
    import resr_b200
    names = NODE_SETS[nodes]
    vgg = _vgg()
    mod = resr_b200.model.ContentLoss(names, MEAN, STD, vgg=vgg).cuda()
    torch.manual_seed(1)
    sr, gt = torch.rand(shape), torch.rand(shape)
    wgt = torch.rand(len(names)) + 0.5
    got_l, got_g = _run(mod, sr, gt, wgt)
    ref_l, ref_g = _emulated_oracle(vgg, names, sr, gt, wgt)
    lerr = ((got_l.double() - ref_l).abs() / ref_l.abs()).max().item()
    cos, rl2 = _metrics(got_g, ref_g)
    print(f"content loss vs fp16-storage oracle {nodes} {shape}: loss rel err {lerr:.2e}; grad cosine {cos:.8f}, rel-L2 {rl2:.3%}")
    assert lerr <= LOSS_RTOL
    assert 1 - cos <= GUARDS_FP16[nodes][0] and rl2 <= GUARDS_FP16[nodes][1]


def test_tied_pool_windows_route_the_gradient_like_torch():
    """Piecewise-constant images: the conv outputs inside a flat region are exactly equal, so most 2x2 pool windows tie;
    the gradient must go to the first element of each window, as max_pool2d's backward sends it."""
    import resr_b200
    names = ["features.2", "features.5", "features.10"]
    vgg = _vgg(3)
    mod = resr_b200.model.ContentLoss(names, MEAN, STD, vgg=vgg).cuda()
    torch.manual_seed(4)
    blocks = lambda: torch.rand(2, 3, 6, 7).repeat_interleave(8, 2).repeat_interleave(8, 3)[:, :, :45, :51].contiguous()
    sr, gt = blocks(), blocks()
    wgt = torch.tensor([1.0, 0.7, 1.3])
    got_l, got_g = _run(mod, sr, gt, wgt)
    ref_l, ref_g = _emulated_oracle(vgg, names, sr, gt, wgt)
    lerr = ((got_l.double() - ref_l).abs() / ref_l.abs()).max().item()
    cos, rl2 = _metrics(got_g, ref_g)
    print(f"tied windows: loss rel err {lerr:.2e}; grad cosine {cos:.6f}, rel-L2 {rl2:.3%}")
    assert lerr <= LOSS_RTOL and 1 - cos <= 5e-5 and rl2 <= 0.014


# ---- single parts of the VGG plan in isolation: every convolution but the ones under test is a channel permutation
# (one tap of weight 1 at the centre, zero bias), which the fp16 forward computes exactly. The oracle with the same fp16
# storage points then sees bit-identical activations, so ReLU masks, pool argmaxes and L1 signs agree, and what is left
# is the part under test plus the bf16 rounding of the gradients.
CONV_FEATURES = (0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34)


def _permuting_vgg(random_convs, seed=0):
    vgg = _vgg(seed)
    with torch.no_grad():
        for i in CONV_FEATURES:
            if i in random_convs:
                continue
            conv = vgg.features[i]
            cout, cin = conv.weight.shape[:2]
            conv.weight.zero_()
            conv.bias.zero_()
            co = torch.arange(cout)
            # a different source channel for co and co + cin, so that duplicated channels never line up across the two
            # 256-channel halves of a 512-channel input
            conv.weight[co, (7 * co + co // cin) % cin, 1, 1] = 1.0
    return vgg


@pytest.mark.parametrize("inputs", ["tied", "random"])
def test_max_pool_forward_and_backward_match_torch(inputs):
    """features.2 (a node followed by the first pool) and features.5 (after the pool), every convolution a permutation:
    the losses are L1 of exact fp16 maps and their max-pool, and the gradient's routing through the pool (ties to the first
    element of the window in row-major order) must land on exactly the pixels torch's max_pool2d backward picks."""
    import resr_b200
    names = ["features.2", "features.5"]
    vgg = _permuting_vgg(())
    mod = resr_b200.model.ContentLoss(names, MEAN, STD, vgg=vgg).cuda()
    torch.manual_seed(7)
    if inputs == "tied":   # flat 4 x 4 blocks at odd offsets: most 2x2 windows hold four equal values
        make = lambda: torch.rand(2, 3, 13, 15).repeat_interleave(4, 2).repeat_interleave(4, 3)[:, :, 1:46, 3:54].contiguous()
    else:
        make = lambda: torch.rand(1, 3, 37, 53)
    sr, gt = make(), make()
    wgt = torch.tensor([0.8, 1.3])
    got_l, got_g = _run(mod, sr, gt, wgt)
    ref_l, ref_g = _emulated_oracle(vgg, names, sr, gt, wgt)
    lerr = ((got_l.double() - ref_l).abs() / ref_l.abs()).max().item()
    cos, rl2 = _metrics(got_g, ref_g)
    support = int(((got_g != 0) != (ref_g != 0)).sum())
    print(f"max-pool {inputs}: loss rel err {lerr:.2e}; grad cosine {cos:.8f}, rel-L2 {rl2:.3%}; support mismatches {support}")
    assert lerr <= 7e-8   # guards: 2x the worst value measured on a B200 (DESIGN.md §8)
    assert support == 0
    assert 1 - cos <= 1.4e-6 and rl2 <= 0.0027


@pytest.mark.parametrize("shape", [(2, 3, 37, 53), (1, 3, 16, 130)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("node", ["features.21", "features.34"])
def test_512_channel_layers_of_the_vgg_plan(shape, node):
    """The split-K path as the VGG plan runs it: its weight slicing, both forward halves, the transposed half packs of the
    data-gradient convolutions and the fused ReLU' mask. The deepest node is a random 512 -> 512 convolution; everything
    before it is a permutation, so each 512-channel layer's halves must pick the right channels for the result to match."""
    import resr_b200
    vgg = _permuting_vgg((int(node.split(".")[1]),), seed=8)
    mod = resr_b200.model.ContentLoss([node], MEAN, STD, vgg=vgg).cuda()
    torch.manual_seed(9)
    sr, gt = torch.rand(shape), torch.rand(shape)
    wgt = torch.tensor([1.1])
    got_l, got_g = _run(mod, sr, gt, wgt)
    ref_l, ref_g = _emulated_oracle(vgg, [node], sr, gt, wgt)
    lerr = ((got_l.double() - ref_l).abs() / ref_l.abs()).max().item()
    cos, rl2 = _metrics(got_g, ref_g)
    print(f"512-channel layers {node} {shape}: loss rel err {lerr:.2e}; grad cosine {cos:.8f}, rel-L2 {rl2:.3%}")
    assert lerr <= 6e-5   # guards: 2x the worst value measured on a B200 (DESIGN.md §8)
    assert 1 - cos <= 1.2e-6 and rl2 <= 0.0036


# ---- the 512-channel split-K composition on its own: two 256-channel halves of resr_conv3x3, the second reading the
# channels at offset 256 and adding the first half's fp32 partial (EP_SKIP, zero bias), forward (fp16) and data gradient
# (bf16, transposed flipped weights), against float64 conv2d of the 16-bit-rounded operands.
GUARD = 64


def _framed(shape, dtype):
    """NaN-filled output with GUARD sentinel elements before and after."""
    buf = torch.full((GUARD * 2 + int(torch.tensor(shape).prod()),), float("nan"), dtype=dtype, device="cuda")
    buf[:GUARD] = 7.0
    buf[-GUARD:] = 7.0
    return buf, buf[GUARD:-GUARD].view(shape)


def _conv(L, x16, c_total, cin, cout, fmt, weight, bias, *, out16=None, outf=None, res1=None, ep_mode=0, ptr_off=0):
    d = L.ConvDesc()
    d.in16 = x16.data_ptr() + ptr_off
    n, h, w, _ = x16.shape
    d.n, d.h, d.w, d.c_total, d.cin, d.cout = n, h, w, c_total, cin, cout
    d.fmt_in, d.mode = fmt, -1
    d.weight, d.bias = weight.data_ptr(), bias.data_ptr()
    d.ep_mode = ep_mode
    if out16 is not None:
        d.out16, d.out16_fmt, d.out16_cstride = out16.data_ptr(), fmt, cout
    if outf is not None:
        d.outf, d.outf_cstride = outf.data_ptr(), cout
    if res1 is not None:
        d.res1, d.res_cstride = res1.data_ptr(), cout
    L.check(L.lib().resr_conv3x3(ctypes.byref(d), L.stream_ptr()))


@pytest.mark.parametrize("n,h,w", [(1, 5, 7), (3, 2, 130), (2, 17, 33), (5, 1, 1)])
@pytest.mark.parametrize("direction", ["forward", "data_gradient"])
def test_split_k_512_channel_convolution(n, h, w, direction):
    import resr_b200
    L = resr_b200._lib
    torch.manual_seed(n * 100 + h + w)
    fmt = 0 if direction == "forward" else 1
    dt = torch.float16 if fmt == 0 else torch.bfloat16
    cin, cout = 512, 256 if direction == "forward" else 512
    wt = torch.randn(cout, cin, 3, 3) * 0.02
    if direction == "data_gradient":   # the data-gradient convolution of a forward 512 -> 512 layer: W'[ci][co] = W[co][ci] flipped
        wt = wt.transpose(0, 1).flip(2, 3).contiguous()
        cin, cout = wt.shape[1], wt.shape[0]
    bias = torch.randn(cout) * 0.1 if direction == "forward" else torch.zeros(cout)
    x = torch.randn(n, h, w, cin).to(dt).cuda()
    wq = wt.to(dt).float()
    w0, w1 = wq[:, :256].contiguous().cuda(), wq[:, 256:].contiguous().cuda()
    pbuf, partial = _framed((n, h, w, cout), torch.float32)
    obuf, out = _framed((n, h, w, cout), dt)
    _conv(L, x, 512, 256, cout, fmt, w0, bias.cuda(), outf=partial)
    _conv(L, x, 512, 256, cout, fmt, w1, torch.zeros(cout).cuda(), out16=out, res1=partial, ep_mode=3, ptr_off=512)
    torch.cuda.synchronize()
    for buf in (pbuf, obuf):
        assert (buf[:GUARD] == 7).all() and (buf[-GUARD:] == 7).all(), "a sentinel changed"
        assert not torch.isnan(buf.float()).any(), "an output element was not written"
    ref = F.conv2d(x.double().permute(0, 3, 1, 2).cpu(), wq.double(), bias.double(), padding=1).permute(0, 2, 3, 1)
    got = out.double().cpu()
    half_ulp = ref.abs() * (2.0 ** -11 if fmt == 0 else 2.0 ** -8)
    err = ((got - ref).abs() - half_ulp).max().item()
    scale = ref.abs().max().item()
    print(f"split-K 512 {direction} {n}x{h}x{w}: max err beyond half an ulp {err:.2e} (scale {scale:.2e})")
    assert err <= 1e-4 * scale


def _usm_ref(x, kernel2d, weight, threshold):
    """USMSharp (imgproc.py:1526-1535) restated in torch: reflect pad + conv2d with the outer-product kernel."""
    b, c, h, w = x.shape
    K = kernel2d.shape[-1]
    R = K // 2
    k = kernel2d.to(x).view(1, 1, K, K)

    def blur(t):
        return F.conv2d(F.pad(t.reshape(b * c, 1, h, w), (R, R, R, R), mode="reflect"), k).view(b, c, h, w)

    residual = x - blur(x)
    soft = blur((torch.abs(residual) * 255 > threshold).to(x.dtype))
    out = torch.clip(x + weight * residual, 0, 1)
    return soft * out + (1 - soft) * x


def test_generator_gradients_through_usm_and_content_loss():
    """The content term of g_loss (train_realesrgan.py:477): ContentLoss(usm_sharpener(G(lr)), hr) back through
    resr_usm_sharp_backward and resr_generator_backward, all 702 generator gradients against fp32 autograd of the oracle
    generator + torchvision VGG19 + the restated USM."""
    import resr_b200
    from oracle import generator as og
    from torchvision.models.feature_extraction import create_feature_extractor
    from torchvision import transforms
    names = NODE_SETS["realesrgan"]
    wgt = torch.tensor([0.1, 0.1, 1.0, 1.0, 1.0])   # the reference's feature_loss_weights
    sd = og.random_state_dict(6)
    g = resr_b200.model.Generator(3, 3, 4)
    g.load_state_dict(sd)
    g = g.cuda().train()
    usm = resr_b200.imgproc.USMSharp(50, 0).cuda()
    vgg = _vgg(5)
    content = resr_b200.model.ContentLoss(names, MEAN, STD, vgg=vgg).cuda()
    torch.manual_seed(61)
    lr, hr = torch.rand(1, 3, 16, 16), torch.rand(1, 3, 64, 64)
    ref_params = {k: v.detach().clone().float().requires_grad_(True) for k, v in sd.items()}
    sr_ref = og._forward(lr, ref_params, 23)
    out_ref = _usm_ref(sr_ref, usm.kernel[0].cpu(), 0.5, 10)
    fe = create_feature_extractor(vgg.float(), names)
    norm = transforms.Normalize(MEAN, STD)
    fs, fg = fe(norm(out_ref)), fe(norm(hr))
    loss_ref = sum(wk * F.l1_loss(fs[k], fg[k].detach()) for wk, k in zip(wgt.tolist(), names))
    loss_ref.backward()
    ref_flat = torch.cat([ref_params[k].grad.reshape(-1) for k in sd])
    sr = g(lr.cuda())
    loss = (content(usm(sr, 0.5, 10), hr.cuda()) * wgt.cuda()).sum()
    loss.backward()
    got = torch.cat([p.grad.reshape(-1) for p in g.parameters()]).cpu()
    assert sum(1 for _ in g.parameters()) == 702
    cos, rl2 = _metrics(got, ref_flat)
    print(f"content loss through USM into the generator: loss {loss.item():.6f} vs {loss_ref.item():.6f}; "
          f"grad cosine {cos:.5f}; rel-L2 {rl2:.3%}")
    assert abs(loss.item() - loss_ref.item()) <= LOSS_RTOL * loss_ref.item()
    assert 1 - cos <= 2.2e-4 and rl2 <= 0.03


def test_two_identical_calls_are_bit_identical():
    import resr_b200
    mod = resr_b200.model.ContentLoss(NODE_SETS["all16"], MEAN, STD, vgg=_vgg()).cuda()
    torch.manual_seed(2)
    sr, gt = torch.rand(2, 3, 48, 40), torch.rand(2, 3, 48, 40)
    wgt = torch.rand(16)
    a_l, a_g = _run(mod, sr, gt, wgt)
    b_l, b_g = _run(mod, sr, gt, wgt)
    assert torch.equal(a_l, b_l) and torch.equal(a_g, b_g)


def test_stale_backward_shapes_and_gt_gradient():
    import resr_b200
    mod = resr_b200.model.ContentLoss(NODE_SETS["realesrgan"], MEAN, STD, vgg=_vgg()).cuda()
    sr = torch.rand(1, 3, 32, 32, device="cuda", requires_grad=True)
    gt = torch.rand(1, 3, 32, 32, device="cuda", requires_grad=True)
    first = mod(sr, gt).sum()
    mod(sr, gt).sum().backward()   # a later forward overwrote the saved activations of `first`
    assert gt.grad is None          # the gradient flows to sr only
    with pytest.raises(resr_b200._lib.ResrError, match="stale"):
        first.backward()
    with pytest.raises(ValueError):
        mod(sr, torch.rand(1, 3, 32, 31, device="cuda"))
    with pytest.raises(ValueError):
        mod(torch.rand(1, 3, 15, 32, device="cuda"), torch.rand(1, 3, 15, 32, device="cuda"))   # features.34 needs 16
    with pytest.raises(resr_b200._lib.ResrError):
        mod(sr.detach().cpu(), gt.detach().cpu())
    # new weights are repacked: a changed parameter changes the losses
    before = mod(sr, gt).detach().clone()
    with torch.no_grad():
        mod.features["0"].weight.mul_(2)
    assert not torch.equal(mod(sr, gt).detach(), before)
