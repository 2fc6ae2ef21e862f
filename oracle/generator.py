"""Oracle for hot path 1: plain torch fp32 restatement of the reference RRDBNet x4 forward. TEST INFRASTRUCTURE ONLY.

Follows /root/reference/model.py:
  ResidualDenseBlock.forward            model.py:87-98
  ResidualResidualDenseBlock.forward    model.py:123-132
  Generator._forward_impl               model.py:255-272
Takes a reference-format state_dict (model.py:223-252 key names). Pinned by tests/golden/generator_*.npz.
grads() is float64 autograd of the same forward, plain or with the rounding points of a training recipe.
"""
import torch
import torch.nn.functional as F


def _conv(x, sd, name):
    return F.conv2d(x, sd[name + ".weight"], sd[name + ".bias"], stride=1, padding=1)


def rdb_forward(x, sd, prefix, conv=_conv):
    feats = [x]
    for k in range(1, 5):  # model.py:90-93: dense concat, LeakyReLU(0.2)
        feats.append(F.leaky_relu(conv(torch.cat(feats, 1), sd, f"{prefix}.conv{k}"), 0.2))
    out5 = conv(torch.cat(feats, 1), sd, f"{prefix}.conv5")  # model.py:94
    return out5 * 0.2 + x  # model.py:95-96


def rrdb_forward(x, sd, prefix, conv=_conv):
    out = x
    for j in (1, 2, 3):  # model.py:126-128
        out = rdb_forward(out, sd, f"{prefix}.rdb{j}", conv)
    return out * 0.2 + x  # model.py:129-130


@torch.no_grad()
def generator_forward(x: torch.Tensor, sd: dict, num_rrdb: int = 23) -> torch.Tensor:
    """x: [N,3,H,W] fp32 in [0,1] -> [N,3,4H,4W] fp32 in [0,1]."""
    sd = {k: v.detach().to(torch.float32) for k, v in sd.items()}
    return _forward(x, sd, num_rrdb)


def l1_loss_and_grads(x: torch.Tensor, hr: torch.Tensor, sd: dict):
    """Reference training-step core under fp32 autograd (train_realesrnet.py:383-388 without AMP): returns
    (loss, {name: grad}) of loss = nn.L1Loss()(G(x), hr)."""
    params = {k: v.detach().clone().to(torch.float32).requires_grad_(True) for k, v in sd.items()}
    with torch.enable_grad():
        sr = _forward(x, params, 23)
        loss = torch.nn.functional.l1_loss(sr, hr)
        loss.backward()
    return loss.detach(), {k: p.grad for k, p in params.items()}, sr.detach()


def _forward(x, sd, num_rrdb=23, conv=_conv):
    out1 = conv(x, sd, "conv1")  # model.py:258 (PixelUnshuffle(1) is the identity at x4, model.py:257)
    out = out1
    for i in range(num_rrdb):  # model.py:259
        out = rrdb_forward(out, sd, f"trunk.{i}", conv)
    out = out1 + conv(out, sd, "conv2")  # model.py:260-262
    out = F.leaky_relu(conv(F.interpolate(out, scale_factor=2, mode="nearest"), sd, "upsampling1.0"), 0.2)  # :264
    out = F.leaky_relu(conv(F.interpolate(out, scale_factor=2, mode="nearest"), sd, "upsampling2.0"), 0.2)  # :265
    out = F.leaky_relu(conv(out, sd, "conv3.0"), 0.2)  # :267
    out = conv(out, sd, "conv4")  # :268
    return torch.clamp(out, 0.0, 1.0)  # :270 (clamp_ in the reference)


def _round(t, fmt):
    return t if fmt is None else t.to(fmt).to(t.dtype)


class _RecipeConv(torch.autograd.Function):
    """3x3 convolution (pad 1) with the rounding points of a training recipe: the forward multiplies operands rounded to
    `fwd_fmt`; the output gradient is rounded to `grad_fmt`, and the data- and weight-gradient convolutions multiply it
    with the weights / saved input rounded to `bwd_fmt` (the format the backward kernels read them in)."""

    @staticmethod
    def forward(ctx, x, w, b, fwd_fmt, bwd_fmt, grad_fmt):
        ctx.save_for_backward(x, w)
        ctx.fmts = bwd_fmt, grad_fmt
        return F.conv2d(_round(x, fwd_fmt), _round(w, fwd_fmt), b, stride=1, padding=1)

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        bwd_fmt, grad_fmt = ctx.fmts
        g = _round(g, grad_fmt)
        gx = torch.nn.grad.conv2d_input(x.shape, _round(w, bwd_fmt), g, padding=1)
        gw = torch.nn.grad.conv2d_weight(_round(x, bwd_fmt), w.shape, g, padding=1)
        return gx, gw, g.sum((0, 2, 3)), None, None, None


def recipe_conv(operand_fmt=None, grad_fmt=None, backward_fmt=None):
    """The convolution of the noise model (_RecipeConv); backward_fmt defaults to operand_fmt. Without formats it is the
    plain convolution."""
    if operand_fmt is None and grad_fmt is None and backward_fmt is None:
        return _conv
    bwd = operand_fmt if backward_fmt is None else backward_fmt

    def conv(x, sd, name):
        return _RecipeConv.apply(x, sd[name + ".weight"], sd[name + ".bias"], operand_fmt, bwd, grad_fmt)
    return conv


def grads(x: torch.Tensor, sd: dict, loss_fn, operand_fmt=None, grad_fmt=None, backward_fmt=None):
    """float64 autograd of the generator: returns (loss, {name: grad}, sr) of loss = loss_fn(G(x)), all float64.

    With no formats this is the plain high-precision reference. Otherwise it is the noise model of a training recipe:
    every convolution multiplies operands rounded to `operand_fmt` (a torch dtype) in the forward; its output gradient
    is rounded to `grad_fmt`, and its data and weight gradients multiply that with the weights and the input rounded to
    `backward_fmt` (default `operand_fmt`). It is not a bit-exact emulation of the kernels (they sum in other orders);
    it gives the rounding-noise scale of each gradient."""
    params = {k: v.detach().to(torch.float64).clone().requires_grad_(True) for k, v in sd.items()}
    with torch.enable_grad():
        sr = _forward(x.detach().to(torch.float64), params, 23, recipe_conv(operand_fmt, grad_fmt, backward_fmt))
        loss = loss_fn(sr)
        loss.backward()
    return loss.detach(), {k: p.grad for k, p in params.items()}, sr.detach()


def random_state_dict(seed: int) -> dict:
    """Random-init weights exactly as the reference constructor leaves them (model.py:100-106 + PyTorch defaults),
    drawn in the reference's RNG order, WITHOUT importing the reference: conv default init, then per-RDB
    kaiming_normal_ * 0.1 and zero bias."""
    from torch import nn
    torch.manual_seed(seed)
    sd = {}

    def conv(name, cin, cout):
        m = nn.Conv2d(cin, cout, 3, 1, 1)
        sd[name + ".weight"], sd[name + ".bias"] = m.weight.data, m.bias.data
        return m

    conv("conv1", 3, 64)
    for i in range(23):
        for j in (1, 2, 3):
            ms = [conv(f"trunk.{i}.rdb{j}.conv{k + 1}", 64 + 32 * k, 32 if k < 4 else 64) for k in range(5)]
            for m in ms:
                nn.init.kaiming_normal_(m.weight)
                m.weight.data *= 0.1
                nn.init.constant_(m.bias, 0)
    conv("conv2", 64, 64)
    conv("upsampling1.0", 64, 64)
    conv("upsampling2.0", 64, 64)
    conv("conv3.0", 64, 64)
    conv("conv4", 64, 3)
    return sd


def rich_state_dict(seed: int) -> dict:
    """random_state_dict(seed) with a nonzero bias on every convolution, as trained checkpoints have: each bias drawn
    from U(+-1/sqrt(9 cin)) (PyTorch's default bias scale) by a generator of its own, so the weights stay those of
    random_state_dict(seed). conv4's bias [-0.02, 0.5, 1.02] puts a share of the output below 0 and above 1, where the
    final clamp (model.py:270) cuts the gradient."""
    sd = random_state_dict(seed)
    gen = torch.Generator().manual_seed(1_000_003 + seed)
    for name in [k[:-len(".bias")] for k in sd if k.endswith(".bias")]:
        cout, cin = sd[name + ".weight"].shape[:2]
        bound = 1.0 / (9 * cin) ** 0.5
        sd[name + ".bias"] = (torch.rand(cout, generator=gen, dtype=torch.float64) * 2 - 1).mul_(bound).float()
    sd["conv4.bias"] = torch.tensor([-0.02, 0.5, 1.02])
    return sd
