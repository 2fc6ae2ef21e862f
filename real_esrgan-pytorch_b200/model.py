"""Host-side mirror of the reference generator API (/root/reference/model.py:64-132, 206-275).

`Generator(in_channels, out_channels, upscale_factor)` is an nn.Module whose parameters carry exactly the reference
names, shapes, initialisation and RNG consumption order (so `torch.manual_seed(s); Generator(3, 3, 4)` reproduces
the reference weights and reference checkpoints load unchanged), but whose forward is ONE call into the C ABI
(`resr_generator_forward`, include/resr.h) running hand-written sm_100a kernels. `ResidualDenseBlock.forward` and
`ResidualResidualDenseBlock.forward` (model.py:87-98, 123-132) run block by block through the same tensor-core
convolution (`resr_conv3x3`). There is no PyTorch fallback path.
"""
import ctypes
import threading
import time

import torch
from torch import nn

from . import _lib

__all__ = ["ResidualDenseBlock", "ResidualResidualDenseBlock", "Generator", "ContentLoss", "plan_tiles", "infer_tiled",
           "canvas_groups", "default_band_rows", "deal_groups", "MultiDeviceInference"]


_PRECISIONS = {"fp16": 0, "bf16": 1}
# LR pixels per packed canvas of infer_many: cfg3's 64 x 128 x 128 batch, about 8 GB of workspace in the fp16 recipe
CANVAS_MAX_PIXELS = 1 << 20


def canvas_groups(sizes, max_pixels: int = CANVAS_MAX_PIXELS):
    """The canvases of Generator.infer_many: lists of indices into `sizes` ((h, w) LR sizes), consecutive images up to
    `max_pixels` LR pixels per canvas (an image larger than that runs alone)."""
    groups, cur, px = [], [], 0
    for i, (hh, ww) in enumerate(sizes):
        if cur and px + hh * ww > max_pixels:
            groups.append(cur)
            cur, px = [], 0
        cur.append(i)
        px += hh * ww
    if cur:
        groups.append(cur)
    return groups


def _conv(cin: int, cout: int) -> nn.Conv2d:
    return nn.Conv2d(cin, cout, (3, 3), (1, 1), (1, 1))


def _conv_native(x16, conv: nn.Conv2d, *, lrelu=0, ep_mode=0, out16=None, out16_choff=0, outf=None, res1=None, res2=None):
    """One nn.Conv2d(3x3, pad 1) of a block through the tensor-core kernel (C ABI resr_conv3x3): NHWC fp16 operands,
    fp32 accumulation and epilogue, fp32 NHWC residuals."""
    n, h, w, c_total = x16.shape
    d = _lib.ConvDesc()
    d.in16 = x16.data_ptr()
    d.n, d.h, d.w, d.c_total, d.cin, d.cout = n, h, w, c_total, conv.in_channels, conv.out_channels
    d.fmt_in, d.mode = 0, -1
    wt = conv.weight.detach().float().contiguous()
    bs = conv.bias.detach().float().contiguous() if conv.bias is not None else None
    d.weight, d.bias = wt.data_ptr(), (bs.data_ptr() if bs is not None else None)
    d.ep_mode, d.lrelu, d.clamp01 = ep_mode, lrelu, 0
    if out16 is not None:
        d.out16, d.out16_fmt, d.out16_cstride, d.out16_choff, d.out16_up2 = out16.data_ptr(), 0, out16.shape[-1], out16_choff, 0
    if outf is not None:
        d.outf, d.outf_cstride, d.outf_choff = outf.data_ptr(), outf.shape[-1], 0
    if res1 is not None:
        d.res1, d.res_cstride, d.res_choff = res1.data_ptr(), res1.shape[-1], 0
    if res2 is not None:
        d.res2 = res2.data_ptr()
    with torch.cuda.device(x16.device):
        _lib.check(_lib.lib().resr_conv3x3(ctypes.byref(d), _lib.stream_ptr(x16.device)))


def _check_block_input(x: torch.Tensor, channels: int):
    if x.dim() != 4 or x.size(1) != channels:
        raise ValueError(f"expected [N, {channels}, H, W] input, got {tuple(x.shape)}")
    if not x.is_cuda:
        raise _lib.ResrError("resr_b200 blocks run on a CUDA (sm_100a) device only; there is no CPU path")
    if torch.is_grad_enabled() and x.requires_grad:
        raise _lib.ResrError("block-level forward is inference only; train through Generator (autograd.generator_apply)")


def _rdb_native(block, cat16: torch.Tensor, res_f32: torch.Tensor, *, ep_mode=1, res2=None, out16=None):
    """The five convolutions of one dense block on its in-place concat buffer `cat16` ([N,H,W,192] fp16, channels
    [0, 64) = block input). Returns the fp32 NHWC block output (and also writes it as fp16 into out16[..., :64])."""
    for k in range(4):  # model.py:90-93: out_k = lrelu(conv_k(cat[x, out_1..k-1])) written in place (no torch.cat copy)
        _conv_native(cat16, getattr(block, f"conv{k + 1}"), lrelu=1, out16=cat16, out16_choff=64 + 32 * k)
    outf = torch.empty(cat16.shape[:3] + (64,), dtype=torch.float32, device=cat16.device)
    _conv_native(cat16, block.conv5, ep_mode=ep_mode, res1=res_f32, res2=res2, outf=outf, out16=out16)  # model.py:94-96
    return outf


def _to_cat16(x_nhwc_f32: torch.Tensor) -> torch.Tensor:
    n, h, w, c = x_nhwc_f32.shape
    cat16 = torch.zeros((n, h, w, 192), dtype=torch.float16, device=x_nhwc_f32.device)
    cat16[..., :c] = x_nhwc_f32
    return cat16


class ResidualDenseBlock(nn.Module):
    """One RDB (reference model.py:64-106): conv1..4 (C+32k -> 32) + LeakyReLU, conv5 (C+128 -> C), out = conv5 * 0.2 + x.
    forward() runs the five convolutions through the tensor-core kernel on an in-place concat buffer."""

    def __init__(self, channels: int, growth_channels: int) -> None:
        super().__init__()
        self.channels, self.growth_channels = channels, growth_channels
        for k in range(5):
            setattr(self, f"conv{k + 1}",
                    _conv(channels + growth_channels * k, growth_channels if k < 4 else channels))
        # reference model.py:100-106: kaiming_normal * 0.1, zero bias, in module order
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
                m.weight.data *= 0.1
                nn.init.constant_(m.bias, 0)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if (self.channels, self.growth_channels) != (64, 32):
            raise _lib.ResrError("the native dense block implements channels=64, growth_channels=32 (the RRDBNet configuration)")
        _check_block_input(x, 64)
        with torch.no_grad():
            xf = x.detach().float().permute(0, 2, 3, 1).contiguous()   # fp32 NHWC residual (model.py:88 identity)
            out = _rdb_native(self, _to_cat16(xf), xf)
            return out.permute(0, 3, 1, 2).contiguous()


class ResidualResidualDenseBlock(nn.Module):
    """One RRDB (reference model.py:109-132): out = rdb3(rdb2(rdb1(x))) * 0.2 + x, 15 tensor-core convolutions."""

    def __init__(self, channels: int, growth_channels: int) -> None:
        super().__init__()
        self.rdb1 = ResidualDenseBlock(channels, growth_channels)
        self.rdb2 = ResidualDenseBlock(channels, growth_channels)
        self.rdb3 = ResidualDenseBlock(channels, growth_channels)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        _check_block_input(x, 64)
        with torch.no_grad():
            xf = x.detach().float().permute(0, 2, 3, 1).contiguous()
            cats = [_to_cat16(xf), torch.zeros_like(_to_cat16(xf)), None]
            cats[2] = torch.zeros_like(cats[1])
            o1 = _rdb_native(self.rdb1, cats[0], xf, out16=cats[1])                       # model.py:124-126
            o2 = _rdb_native(self.rdb2, cats[1], o1, out16=cats[2])
            out = _rdb_native(self.rdb3, cats[2], o2, ep_mode=2, res2=xf)                 # model.py:127-130
            return out.permute(0, 3, 1, 2).contiguous()


class Generator(nn.Module):
    """RRDBNet x4 (23 RRDB, nf=64, gc=32). Reference: model.py:206-275."""

    def __init__(self, in_channels: int, out_channels: int, upscale_factor: int) -> None:
        super().__init__()
        if (in_channels, out_channels, upscale_factor) != (3, 3, 4):
            # the reference also supports x2/x1 through PixelUnshuffle (model.py:209-217); out of scope (DESIGN.md)
            raise ValueError("resr_b200.Generator implements the x4 RGB configuration Generator(3, 3, 4) only")
        self.conv1 = _conv(in_channels, 64)
        self.trunk = nn.Sequential(*[ResidualResidualDenseBlock(64, 32) for _ in range(23)])
        self.conv2 = _conv(64, 64)
        self.upsampling1 = nn.Sequential(_conv(64, 64), nn.LeakyReLU(0.2, True))
        self.upsampling2 = nn.Sequential(_conv(64, 64), nn.LeakyReLU(0.2, True))
        self.conv3 = nn.Sequential(_conv(64, 64), nn.LeakyReLU(0.2, True))
        self.conv4 = _conv(64, out_channels)
        self._handle = None
        self._handle_device = None
        self._packed_version = None
        self._flat = None
        self._workspace = None
        self._static_weights = False
        self._precision = "fp16"
        self._fwd_generation = 0   # bumped by every training-mode forward (autograd.py ties a backward to its forward)

    # ------------------------------------------------------------------ native plumbing
    def _device(self):
        return next(self.parameters()).device

    def _native(self):
        """The library handle of the device the parameters live on (one handle per device, SURVEY §8b); recreated after
        `.to(other_device)`."""
        dev = self._device()
        if not dev.type == "cuda":
            raise _lib.ResrError("resr_b200.Generator runs on a CUDA (sm_100a) device only; move it with .cuda() / .to(device)")
        if self._handle is not None and self._handle_device != dev:
            with torch.cuda.device(self._handle_device):
                torch.cuda.synchronize()
                _lib.lib().resr_generator_destroy(self._handle)
            self._handle, self._packed_version, self._workspace = None, None, None
            if hasattr(self, "_train_ws"):
                del self._train_ws
        if self._handle is None:
            h = ctypes.c_void_p()
            with torch.cuda.device(dev):
                _lib.check(_lib.lib().resr_generator_create(ctypes.byref(h), 3, 3, 4))
                _lib.check(_lib.lib().resr_generator_set_precision(h, _PRECISIONS[self._precision]))
            self._handle, self._handle_device = h, dev
        return self._handle

    def set_precision(self, precision: str):
        """Recipe of the forward and of the training path: "fp16" (default: fp16 tensor-core operands, the trunk's residual
        stream is the fp16 conv input; training keeps fp16 activations + bf16 gradients and takes its weight gradients
        from a bf16 copy of each layer's input) or "bf16" (BASELINE.json north_star: bf16 operands and activations + fp32
        masters of the residual stream; training keeps bf16 activations and gradients and takes its weight gradients
        straight from the NHWC buffers, faster per step). Neither has a shape rule. Both run at the same tensor-core
        rate; fp16 is ~2-3x closer to the fp32 reference."""
        if precision not in _PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_PRECISIONS)}")
        if precision != self._precision:
            self._precision = precision
            if self._handle is not None:
                with torch.cuda.device(self._handle_device):
                    torch.cuda.synchronize()
                    _lib.check(_lib.lib().resr_generator_set_precision(self._handle, _PRECISIONS[precision]))
            self._packed_version = None
        return self

    @property
    def precision(self) -> str:
        return self._precision

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None:
            try:
                with torch.cuda.device(self._handle_device):
                    _lib.lib().resr_generator_destroy(h)
            except Exception:
                pass

    def _param_version(self):
        """Identity of the weights the packed tensor-core tiles were built from. `_version` alone misses `param.data = t`
        (EMA.apply_shadow / restore, reference model.py:51-61), `load_state_dict(assign=True)` and dtype round trips, so
        the storage pointer, dtype and device of every parameter are part of the key."""
        return tuple((p._version, p.data_ptr(), p.dtype) for p in self.parameters()) + (self._device(),)

    def assume_static_weights(self, flag: bool = True):
        """Serving loops with frozen weights: skip the per-call walk over the 702 parameters (pack once, then trust
        the caller). `invalidate()` forces a repack."""
        self._static_weights = bool(flag)
        return self

    def invalidate(self):
        self._packed_version = None

    def flat_parameters(self) -> torch.Tensor:
        """All parameters in state_dict order as one contiguous fp32 device vector (layout of resr_generator_tensor_span)."""
        ps = [p.detach().reshape(-1).float() for p in self.parameters()]
        flat = torch.cat(ps)
        assert flat.numel() == _lib.lib().resr_generator_num_params()
        return flat

    def _ensure_packed(self):
        if self._static_weights and self._packed_version is not None:
            return
        ver = self._param_version()
        if self._packed_version != ver:
            master = getattr(self, "_flat_master", None)
            first = next(self.parameters())
            if master is not None and first.data_ptr() == master.data_ptr() and first.device == master.device:
                self._flat = master  # parameters are views of one flat vector (optim.FlatAdamEMA): nothing to gather
            else:
                self._flat = self.flat_parameters()
            dev = self._device()
            h = self._native()
            with torch.cuda.device(dev):
                _lib.check(_lib.lib().resr_generator_load_params(h, _lib.ptr(self._flat), _lib.stream_ptr(dev)))
            self._packed_version = ver

    def _get_workspace(self, n: int, h: int, w: int, device, extra: int = 0) -> torch.Tensor:
        need = _lib.lib().resr_generator_workspace_bytes_for(self._native(), n, h, w) + extra
        return self._workspace_of(need, device)

    def _workspace_of(self, need: int, device) -> torch.Tensor:
        ws = self._workspace
        if ws is None or ws.numel() < need + 1024 or ws.device != device:
            ws = torch.empty(need + 1024, dtype=torch.uint8, device=device)
            self._workspace = ws
        return ws

    @staticmethod
    def _aligned(ws: torch.Tensor):
        base = ws.data_ptr()
        off = (-base) % 1024
        return ctypes.c_void_p(base + off), ws.numel() - off

    # ------------------------------------------------------------------ reference API
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._forward_impl(x)

    def _forward_impl(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 4 or x.size(1) != 3:
            raise ValueError(f"expected [N, 3, H, W] input, got {tuple(x.shape)}")
        if not x.is_cuda:
            raise _lib.ResrError("resr_b200.Generator runs on a CUDA (sm_100a) device only; there is no CPU path")
        if x.device != self._device():
            raise _lib.ResrError(f"input on {x.device} but the generator lives on {self._device()}")
        if torch.is_grad_enabled():
            if x.requires_grad:
                # the reference feeds a detached LR batch (train_realesrnet.py:377-384); the conv1 data gradient is not built
                raise _lib.ResrError("resr_b200.Generator does not produce a gradient w.r.t. its input: detach() the LR batch")
            if any(p.requires_grad for p in self.parameters()):
                from . import autograd  # training path (SURVEY §8 row a5)
                return autograd.generator_apply(self, x)
        return self.infer(x)

    @torch.no_grad()
    def infer(self, x: torch.Tensor) -> torch.Tensor:
        n, _, h, w = x.shape
        xc = x.detach().contiguous(memory_format=torch.contiguous_format).float()
        self._ensure_packed()
        y = torch.empty((n, 3, 4 * h, 4 * w), dtype=torch.float32, device=x.device)
        ws = self._get_workspace(n, h, w, x.device)
        wp, wbytes = self._aligned(ws)
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().resr_generator_forward(self._native(), _lib.ptr(xc), _lib.ptr(y), n, h, w, wp, wbytes,
                                                         _lib.stream_ptr(x.device)))
        return y

    @torch.no_grad()
    def infer_u8(self, x_u8: torch.Tensor) -> torch.Tensor:
        """Image in, image out: x_u8 is an NHWC uint8 RGB batch [N, H, W, 3] on the device (what cv2.imread + cvtColor
        hold); returns the NHWC uint8 SR batch [N, 4H, 4W, 3]. `image / 255` + image_to_tensor (inference.py:40-46) is fused
        into the first layout kernel and tensor_to_image (inference.py:56, imgproc.py:1594) into the last convolution: the
        result equals tensor_to_image(self(image_to_tensor(x / 255))) bit for bit."""
        if x_u8.dim() != 4 or x_u8.size(3) != 3 or x_u8.dtype != torch.uint8:
            raise ValueError(f"expected a uint8 [N, H, W, 3] batch, got {tuple(x_u8.shape)} {x_u8.dtype}")
        if not x_u8.is_cuda:
            raise _lib.ResrError("resr_b200.Generator runs on a CUDA (sm_100a) device only; there is no CPU path")
        n, h, w, _ = x_u8.shape
        xc = x_u8.contiguous()
        self._ensure_packed()
        y = torch.empty((n, 4 * h, 4 * w, 3), dtype=torch.uint8, device=x_u8.device)
        ws = self._get_workspace(n, h, w, x_u8.device)
        wp, wbytes = self._aligned(ws)
        with torch.cuda.device(x_u8.device):
            _lib.check(_lib.lib().resr_generator_forward_u8(self._native(), _lib.ptr(xc), _lib.ptr(y), n, h, w, wp, wbytes,
                                                            _lib.stream_ptr(x_u8.device)))
        return y

    @torch.no_grad()
    def infer_u8_host(self, x_host: torch.Tensor, y_host: torch.Tensor = None, device=None) -> torch.Tensor:
        """infer_u8 with HOST uint8 tensors (pinned recommended): H2D + forward + D2H inside the C ABI; 3 bytes per LR pixel
        in, 48 bytes per LR pixel out (the fp32 host call moves 12 and 192)."""
        device = device or self._device()
        n, h, w, _ = x_host.shape
        if x_host.dtype != torch.uint8 or x_host.size(3) != 3:
            raise ValueError("expected a uint8 [N, H, W, 3] host batch")
        xc = x_host.contiguous()
        if y_host is None:
            y_host = torch.empty((n, 4 * h, 4 * w, 3), dtype=torch.uint8, pin_memory=True)
        self._ensure_packed()
        extra = xc.numel() * 17 + 4096
        ws = self._get_workspace(n, h, w, device, extra)
        wp, wbytes = self._aligned(ws)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().resr_generator_forward_u8_host(self._native(), _lib.ptr(xc), _lib.ptr(y_host), n, h, w, wp, wbytes,
                                                                 _lib.stream_ptr(device)))
        return y_host

    @torch.no_grad()
    def infer_host(self, x_host: torch.Tensor, y_host: torch.Tensor = None, device=None) -> torch.Tensor:
        """End-to-end call with HOST tensors (pinned recommended): H2D + forward + D2H inside the C ABI."""
        device = device or next(self.parameters()).device
        n, _, h, w = x_host.shape
        xc = x_host.contiguous().float()
        if y_host is None:
            y_host = torch.empty((n, 3, 4 * h, 4 * w), dtype=torch.float32, pin_memory=True)
        self._ensure_packed()
        extra = xc.numel() * 4 * 17 + 4096
        ws = self._get_workspace(n, h, w, device, extra)
        wp, wbytes = self._aligned(ws)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().resr_generator_forward_host(self._native(), _lib.ptr(xc), _lib.ptr(y_host), n, h, w,
                                                              wp, wbytes, _lib.stream_ptr(device)))
        return y_host


    @torch.no_grad()
    def infer_host_async(self, x_host: torch.Tensor, y_host: torch.Tensor, device=None) -> torch.Tensor:
        """Pipelined serving call: queues H2D + forward + D2H and returns; copies of neighbouring calls overlap this call's
        compute (two staging slots inside the workspace). `x_host` / `y_host` must be pinned fp32 tensors that stay alive
        and untouched until `host_sync()` (or two further calls) — alternate between two `y_host` buffers."""
        device = device or next(self.parameters()).device
        n, _, h, w = x_host.shape
        if not (x_host.is_pinned() and y_host.is_pinned()) or x_host.dtype != torch.float32 or not x_host.is_contiguous():
            raise _lib.ResrError("infer_host_async needs pinned contiguous fp32 host tensors")
        self._ensure_packed()
        extra = 2 * (x_host.numel() * 4 * 17 + 4096)
        cur = self._workspace
        if cur is not None and (cur.device != device or
                                cur.numel() < _lib.lib().resr_generator_workspace_bytes_for(self._native(), n, h, w) + extra + 1024):
            self.host_sync()  # queued copies still use the workspace that is about to be replaced
            torch.cuda.synchronize(device)
        ws = self._get_workspace(n, h, w, device, extra)
        wp, wbytes = self._aligned(ws)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().resr_generator_forward_host_async(self._native(), _lib.ptr(x_host), _lib.ptr(y_host), n, h,
                                                                    w, wp, wbytes, _lib.stream_ptr(device)))
        return y_host

    def host_sync(self):
        _lib.check(_lib.lib().resr_generator_host_sync(self._native()))

    # ------------------------------------------------------------------ lists of differently sized images
    @torch.no_grad()
    def infer_many(self, images, max_pixels: int = CANVAS_MAX_PIXELS):
        """SR of a list of differently sized images ([1, 3, h, w] or [3, h, w] fp32 CUDA tensors), returned in input order
        with infer()'s shape per image ([1, 3, 4h, 4w] or [3, 4h, 4w]). The loops of the reference's test.py, validate()
        and inference.py over a folder run one image per forward; here consecutive images are packed into canvases of at
        most `max_pixels` LR pixels (an image larger than that runs alone) and each canvas is one forward
        (resr_generator_forward_many). Every result is its image's own forward, up to fp32 summation order."""
        xs = []
        for x in images:
            if x.dim() not in (3, 4) or x.size(-3) != 3 or (x.dim() == 4 and x.size(0) != 1):
                raise ValueError(f"expected a [1, 3, H, W] or [3, H, W] image, got {tuple(x.shape)}")
            self._check_device(x)
            xs.append(x.detach().float().contiguous())
        ys = [torch.empty(x.shape[:-2] + (4 * x.size(-2), 4 * x.size(-1)), dtype=torch.float32, device=x.device) for x in xs]
        self._run_many(xs, ys, [tuple(x.shape[-2:]) for x in xs], max_pixels, "resr_generator_forward_many")
        return ys

    @torch.no_grad()
    def infer_u8_many(self, images_u8, max_pixels: int = CANVAS_MAX_PIXELS):
        """infer_u8 for a list of differently sized uint8 [h, w, 3] CUDA images: a list of [4h, 4w, 3] uint8 results in
        input order, each equal to infer_u8 of its image up to fp32 summation order (packing as in infer_many)."""
        xs = []
        for x in images_u8:
            if x.dim() != 3 or x.size(2) != 3 or x.dtype != torch.uint8:
                raise ValueError(f"expected a uint8 [H, W, 3] image, got {tuple(x.shape)} {x.dtype}")
            self._check_device(x)
            xs.append(x.contiguous())
        ys = [torch.empty((4 * x.size(0), 4 * x.size(1), 3), dtype=torch.uint8, device=x.device) for x in xs]
        self._run_many(xs, ys, [tuple(x.shape[:2]) for x in xs], max_pixels, "resr_generator_forward_many_u8")
        return ys

    def _check_device(self, x):
        if not x.is_cuda:
            raise _lib.ResrError("resr_b200.Generator runs on a CUDA (sm_100a) device only; there is no CPU path")
        if x.device != self._device():
            raise _lib.ResrError(f"input on {x.device} but the generator lives on {self._device()}")

    def _run_many(self, xs, ys, sizes, max_pixels, fn):
        if not xs:
            return
        self._ensure_packed()
        h = self._native()
        dev = xs[0].device
        call = getattr(_lib.lib(), fn)
        with torch.cuda.device(dev):
            for idx in canvas_groups(sizes, max_pixels):
                n = len(idx)
                hs = (ctypes.c_int * n)(*[sizes[i][0] for i in idx])
                ws_ = (ctypes.c_int * n)(*[sizes[i][1] for i in idx])
                need = _lib.lib().resr_generator_forward_many_workspace_bytes(h, hs, ws_, n)
                if need == 0:
                    raise _lib.ResrError(f"no canvas for these {n} images: {_lib.lib().resr_last_error().decode()}")
                wp, wbytes = self._aligned(self._workspace_of(need, dev))
                xp = (ctypes.c_void_p * n)(*[xs[i].data_ptr() for i in idx])
                yp = (ctypes.c_void_p * n)(*[ys[i].data_ptr() for i in idx])
                _lib.check(call(h, xp, yp, hs, ws_, n, wp, wbytes, _lib.stream_ptr(dev)))


# ----------------------------------------------------------------------------------------------------------------------
# Large-image inference by spatial tiles with a receptive-field halo (BASELINE.json configs[4]; new functionality around
# the unchanged reference API: inference.py:52-53 runs one whole-image forward). Tile indexing is integer arithmetic.


def plan_tiles(h: int, w: int, tile_h: int, tile_w: int, halo: int):
    """Covers an h x w LR image with interior rectangles of at most tile_h x tile_w. Returns a list of
    (y0, y1, x0, x1, wy0, wy1, wx0, wx1): interior [y0,y1) x [x0,x1) and the input window = interior grown by `halo`,
    clamped at the image border (where the convolutions' zero padding applies instead of neighbour data)."""
    tiles = []
    for y0 in range(0, h, tile_h):
        y1 = min(y0 + tile_h, h)
        for x0 in range(0, w, tile_w):
            x1 = min(x0 + tile_w, w)
            tiles.append((y0, y1, x0, x1, max(y0 - halo, 0), min(y1 + halo, h), max(x0 - halo, 0), min(x1 + halo, w)))
    return tiles


@torch.no_grad()
def infer_tiled(gen: "Generator", x: torch.Tensor, tile_h: int = 512, tile_w: int = 1024, halo: int = 16, rank: int = 0,
                world: int = 1, out: torch.Tensor = None):
    """x: [1, 3, H, W] CUDA LR image. Tiles are dealt round-robin to `world` ranks (no collective: every rank computes
    its own tiles from the shared input); this rank's interiors are written into `out` ([1, 3, 4H, 4W], allocated if
    None) and also returned as [(y0, x0, tensor)] for a host-side gather."""
    assert x.dim() == 4 and x.size(0) == 1 and x.size(1) == 3
    _, _, h, w = x.shape
    s = 4
    if out is None:
        out = torch.zeros((1, 3, s * h, s * w), dtype=torch.float32, device=x.device)
    mine = []
    for i, (y0, y1, x0, x1, wy0, wy1, wx0, wx1) in enumerate(plan_tiles(h, w, tile_h, tile_w, halo)):
        if i % world != rank:
            continue
        win = x[:, :, wy0:wy1, wx0:wx1].contiguous()
        sr = gen.infer(win)
        oy, ox = s * (y0 - wy0), s * (x0 - wx0)
        piece = sr[:, :, oy:oy + s * (y1 - y0), ox:ox + s * (x1 - x0)]
        out[:, :, s * y0:s * y1, s * x0:s * x1] = piece
        mine.append((s * y0, s * x0, piece))
    return out, mine


# ----------------------------------------------------------------------------------------------------------------------
# Several GPUs from one process: one Generator replica per device and one host thread per replica for the length of a
# call. The work is dealt out, never recomputed differently: every band and every canvas is the forward one GPU runs.


def default_band_rows(h: int, w: int, replicas: int, max_pixels: int = CANVAS_MAX_PIXELS) -> int:
    """Interior LR rows per full-width band of MultiDeviceInference.infer_large: at least two bands per replica whenever
    h >= 2 * replicas (a replica uploads band k + 1 while band k computes), and at most `max_pixels` LR pixels per band
    interior (the forward's workspace grows with the band, about 8 KB per LR pixel)."""
    return max(1, min(h // (2 * replicas), max_pixels // w))


def deal_groups(sizes, replicas: int, max_pixels: int = CANVAS_MAX_PIXELS):
    """The canvases of a list of (h, w) LR sizes (canvas_groups: the canvases Generator.infer_many runs) dealt to
    `replicas`: largest canvas (in LR pixels) first, onto the replica with the least work so far; ties go to the earlier
    canvas and the lower replica. Returns (groups, dealt): dealt[r] lists the indices into `groups` replica r runs."""
    groups = canvas_groups(sizes, max_pixels)
    work = [sum(sizes[i][0] * sizes[i][1] for i in g) for g in groups]
    load, dealt = [0] * replicas, [[] for _ in range(replicas)]
    for k in sorted(range(len(groups)), key=lambda k: (-work[k], k)):
        r = min(range(replicas), key=lambda r: (load[r], r))
        dealt[r].append(k)
        load[r] += work[k]
    return groups, dealt


class MultiDeviceInference:
    """Inference of one Generator on several GPUs from one process: a large image as full-width halo bands
    (infer_large / infer_u8_large) or a list of images as packed canvases (infer_many / infer_u8_many), dealt to one
    replica of `gen` per entry of `devices` (default: every visible CUDA device). Entries may repeat: [0, 0] runs two
    replicas on one GPU. Inputs are host tensors (pinned or not) or CUDA tensors on any device; results are written to
    page-locked host memory.

    Every replica is an ordinary Generator on its device with gen's precision recipe and static weights. Each call
    compares gen's weights with the ones the replicas hold and reloads them when they changed (an optimizer step,
    EMA.apply_shadow); when gen.assume_static_weights() is set that walk is skipped, and invalidate() forces a reload.
    A call runs one host thread per replica, each with its device current and on the replica's own streams (compute,
    upload, download), and joins them all before it returns. ctypes releases the GIL around every library call, so the
    launches to different GPUs are enqueued in parallel. If a replica fails, every thread is still joined, then the
    first error is raised naming the replica's device; the contents of the output are unspecified in that case.

    `last_enqueue` holds, per replica of the last call, (device, bands or canvases, host seconds spent enqueuing them)."""

    def __init__(self, gen: Generator, devices=None):
        if not isinstance(gen, Generator):
            raise ValueError(f"expected a resr_b200 Generator, got {type(gen).__name__}")
        if devices is not None:
            devices = [torch.device("cuda", d) if isinstance(d, int) else torch.device(d) for d in devices]
            if not devices or any(d.type != "cuda" or d.index is None for d in devices):
                raise ValueError(f"devices must be a non-empty list of CUDA device indices, got {devices}")
        self.gen = gen
        self.devices = devices
        self._replicas = None
        self._streams = None
        self._loaded = None
        self.last_enqueue = None

    def invalidate(self):
        """Reload the replicas' weights from gen on the next call (for a gen with assume_static_weights set)."""
        self._loaded = None

    # ------------------------------------------------------------------ large images
    @torch.no_grad()
    def infer_large(self, x: torch.Tensor, out: torch.Tensor = None, band_rows: int = None, halo: int = 16) -> torch.Tensor:
        """SR of one fp32 [1, 3, H, W] image into `out`, a page-locked host tensor [1, 3, 4H, 4W] (allocated if None;
        callers that loop pass their own: pinning 805 MB costs more than the forward of a 2048^2 image).

        The image is cut into full-width bands plan_tiles(H, W, band_rows, W, halo) (band_rows: default_band_rows),
        dealt round-robin to the replicas in infer_tiled's order. Per band: one upload of the window rows per channel
        plane, the replica's infer(), and one download per channel plane of the interior rows straight into `out`.

        The result is torch.equal to infer_tiled(gen, x, band_rows, W, halo)[0] on one GPU: every band is the same
        forward at the same shape with the same kernels. That holds across devices of one GPU model, because a forward's
        plan depends only on the shape, the SM count and the pair policy. Against the whole-image forward the error is
        infer_tiled's (DESIGN §6)."""
        if x.dim() != 4 or x.size(0) != 1 or x.size(1) != 3 or x.dtype != torch.float32:
            raise ValueError(f"expected a float32 [1, 3, H, W] image, got {tuple(x.shape)} {x.dtype}")
        return self._large(x, out, band_rows, halo, u8=False)

    @torch.no_grad()
    def infer_u8_large(self, img: torch.Tensor, out: torch.Tensor = None, band_rows: int = None, halo: int = 16) -> torch.Tensor:
        """infer_large for a uint8 [H, W, 3] image (what cv2.imread + cvtColor hold) into a page-locked uint8
        [4H, 4W, 3] host tensor: per band one upload of the window rows, infer_u8(), one download of the interior rows.
        Equal to assembling Generator.infer_u8 of the same bands on one GPU."""
        if img.dim() != 3 or img.size(2) != 3 or img.dtype != torch.uint8:
            raise ValueError(f"expected a uint8 [H, W, 3] image, got {tuple(img.shape)} {img.dtype}")
        return self._large(img, out, band_rows, halo, u8=True)

    def _large(self, x, out, band_rows, halo, u8):
        h, w = (x.size(0), x.size(1)) if u8 else (x.size(2), x.size(3))
        if h == 0 or w == 0:
            raise ValueError(f"empty image {tuple(x.shape)}")
        if band_rows is not None and band_rows < 1 or halo < 0:
            raise ValueError(f"band_rows must be >= 1 and halo >= 0, got {band_rows} and {halo}")
        shape = (4 * h, 4 * w, 3) if u8 else (1, 3, 4 * h, 4 * w)
        if out is not None and (tuple(out.shape) != shape or out.dtype != x.dtype or out.is_cuda or not out.is_contiguous()):
            raise ValueError(f"out must be a contiguous {x.dtype} host tensor of shape {shape}, got {tuple(out.shape)} "
                             f"{out.dtype} on {out.device}")
        self._check_devices()
        if out is not None and not out.is_pinned():
            raise ValueError("out must be page-locked host memory (tensor.pin_memory())")
        self._prepare()
        if out is None:
            out = torch.empty(shape, dtype=x.dtype, pin_memory=True)
        nrep = len(self._replicas)
        bands = plan_tiles(h, w, band_rows or default_band_rows(h, w, nrep), w, halo)
        x = x.detach().contiguous()
        if x.is_cuda:
            torch.cuda.current_stream(x.device).synchronize()   # the caller's work on x is done before the copies
        self._run(lambda rep, streams, mine: _run_bands(rep, streams, mine, x, out, u8), [bands[r::nrep] for r in range(nrep)])
        return out

    # ------------------------------------------------------------------ lists of differently sized images
    @torch.no_grad()
    def infer_many(self, images, max_pixels: int = CANVAS_MAX_PIXELS):
        """Generator.infer_many on several GPUs: floating-point [1, 3, h, w] or [3, h, w] images, host or CUDA, in; one
        page-locked fp32 host tensor per image ([1, 3, 4h, 4w] or [3, 4h, 4w]) out, in input order. The canvases are
        canvas_groups(...) of the list, dealt by deal_groups, so each result is torch.equal to the matching element of
        gen.infer_many(images, max_pixels) on one GPU."""
        for x in images:
            if x.dim() not in (3, 4) or x.size(-3) != 3 or (x.dim() == 4 and x.size(0) != 1) or not x.is_floating_point():
                raise ValueError(f"expected a floating-point [1, 3, H, W] or [3, H, W] image, got {tuple(x.shape)} {x.dtype}")
        return self._many(list(images), [tuple(x.shape[-2:]) for x in images], max_pixels, u8=False)

    @torch.no_grad()
    def infer_u8_many(self, images_u8, max_pixels: int = CANVAS_MAX_PIXELS):
        """infer_many for uint8 [h, w, 3] images: page-locked uint8 [4h, 4w, 3] results in input order, each torch.equal
        to the matching element of gen.infer_u8_many(images_u8, max_pixels) on one GPU."""
        for x in images_u8:
            if x.dim() != 3 or x.size(2) != 3 or x.dtype != torch.uint8:
                raise ValueError(f"expected a uint8 [H, W, 3] image, got {tuple(x.shape)} {x.dtype}")
        return self._many(list(images_u8), [tuple(x.shape[:2]) for x in images_u8], max_pixels, u8=True)

    def _many(self, xs, sizes, max_pixels, u8):
        if not xs:
            raise ValueError("empty image list")
        if any(hh == 0 or ww == 0 for hh, ww in sizes):
            raise ValueError(f"empty image among {sizes}")
        if max_pixels < 1:
            raise ValueError(f"max_pixels must be >= 1, got {max_pixels}")
        self._check_devices()
        self._prepare()
        outs = [torch.empty((4 * x.size(0), 4 * x.size(1), 3) if u8 else x.shape[:-2] + (4 * x.size(-2), 4 * x.size(-1)),
                            dtype=torch.uint8 if u8 else torch.float32, pin_memory=True) for x in xs]
        for dev in {x.device for x in xs if x.is_cuda}:
            torch.cuda.current_stream(dev).synchronize()   # the caller's work on the inputs is done before the copies
        groups, dealt = deal_groups(sizes, len(self._replicas), max_pixels)
        self._run(lambda rep, streams, mine: _run_canvases(rep, streams, mine, xs, outs, max_pixels, u8),
                  [[groups[k] for k in d] for d in dealt])
        return outs

    # ------------------------------------------------------------------ replicas and threads
    def _check_devices(self):
        if not torch.cuda.is_available():
            raise _lib.ResrError("MultiDeviceInference needs CUDA (sm_100a) devices; none is visible")
        count = torch.cuda.device_count()
        if self.devices is None:
            self.devices = [torch.device("cuda", i) for i in range(count)]
        for d in self.devices:
            if d.index >= count:
                raise _lib.ResrError(f"{d} is not visible ({count} CUDA device(s))")

    def _prepare(self):
        """Builds the replicas once and brings their weights up to date with gen's."""
        gen = self.gen
        _lib.lib()   # loaded here, not by racing worker threads
        if self._replicas is None:
            self._replicas = [self._replica(d) for d in self.devices]
            self._streams = [tuple(torch.cuda.Stream(d) for _ in range(3)) for d in self.devices]
        if self._loaded is not None and gen._static_weights and self._loaded[1] == gen.precision:
            return
        ver = (gen._param_version(), gen.precision)
        if ver != self._loaded:
            flat = gen.flat_parameters()
            for rep, d in zip(self._replicas, self.devices):
                rep.set_precision(gen.precision)
                with torch.cuda.device(d):
                    rep._flat_master.copy_(flat)
                rep.invalidate()
            for d in set(self.devices):
                torch.cuda.synchronize(d)   # the workers pack from these vectors on their own streams
            self._loaded = ver

    @staticmethod
    def _replica(dev) -> Generator:
        with torch.device("meta"):
            rep = Generator(3, 3, 4)   # on meta: no initialisation, no draw from the global RNG
        rep = rep.to_empty(device=dev).eval().requires_grad_(False)
        flat = torch.empty(_lib.lib().resr_generator_num_params(), dtype=torch.float32, device=dev)
        off = 0
        for p in rep.parameters():
            p.data = flat[off:off + p.numel()].view_as(p)
            off += p.numel()
        rep._flat_master = flat   # the replica packs straight from this vector (Generator._ensure_packed)
        return rep.assume_static_weights(True)

    def _run(self, job, work):
        """job(replica, (compute, upload, download) streams, items) on one thread per replica with work; all joined."""
        n = len(self._replicas)
        errors, spent = [None] * n, [0.0] * n

        def worker(r):
            streams = self._streams[r]
            try:
                with torch.cuda.device(self.devices[r]), torch.cuda.stream(streams[0]):
                    try:
                        t0 = time.perf_counter()
                        job(self._replicas[r], streams, work[r])
                        spent[r] = time.perf_counter() - t0
                    finally:
                        for s in streams:
                            s.synchronize()
            except BaseException as e:   # noqa: B036 -- handed to the calling thread
                errors[r] = e

        threads = [threading.Thread(target=worker, args=(r,), name=f"resr-replica-{r}") for r in range(n) if work[r]]
        try:
            for t in threads:
                t.start()
        finally:
            for t in threads:
                if t.ident is not None:
                    t.join()
        self.last_enqueue = [(self.devices[r], len(work[r]), spent[r]) for r in range(n)]
        for r, e in enumerate(errors):
            if e is not None:
                raise _lib.ResrError(f"replica {r} on {self.devices[r]} failed: {type(e).__name__}: {e}") from e


def _run_bands(rep, streams, bands, x, out, u8):
    """One replica's bands: upload band k + 1 (upload stream) while band k computes (compute stream) and band k - 1
    downloads (download stream). Two window slots; events order each slot's reuse."""
    s, up, down = streams
    w = x.size(1) if u8 else x.size(3)
    most = max(b[5] - b[4] for b in bands) * 3 * w
    slots = [torch.empty(most, dtype=x.dtype, device=s.device) for _ in range(2)]
    landed, read = [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)]
    for k, (y0, y1, _, _, wy0, wy1, _, _) in enumerate(bands):
        i, rows = k % 2, wy1 - wy0
        if k >= 2:
            up.wait_event(read[i])   # the forward of band k - 2 has read this slot
        with torch.cuda.stream(up):
            if u8:
                win = slots[i][:rows * w * 3].view(1, rows, w, 3)
                win[0].copy_(x[wy0:wy1], non_blocking=True)
            else:
                win = slots[i][:3 * rows * w].view(1, 3, rows, w)
                for c in range(3):
                    win[0, c].copy_(x[0, c, wy0:wy1], non_blocking=True)
            landed[i].record(up)
        s.wait_event(landed[i])
        y = rep.infer_u8(win) if u8 else rep.infer(win)
        read[i].record(s)
        down.wait_event(read[i])
        oy, n = 4 * (y0 - wy0), 4 * (y1 - y0)
        with torch.cuda.stream(down):
            if u8:
                out[4 * y0:4 * y1].copy_(y[0, oy:oy + n], non_blocking=True)
            else:
                for c in range(3):
                    out[0, c, 4 * y0:4 * y1].copy_(y[0, c, oy:oy + n], non_blocking=True)
        y.record_stream(down)   # the next band's output must not take this memory before the download has read it


def _run_canvases(rep, streams, groups, xs, outs, max_pixels, u8):
    """One replica's canvases: inputs to the device on the compute stream, results downloaded on the download stream
    while the next canvas computes."""
    s, _, down = streams
    for idx in groups:
        src = [xs[i].to(s.device, non_blocking=True) for i in idx]
        # one canvas: the group fits max_pixels (or is one image), so infer_many regroups it into itself
        ys = rep.infer_u8_many(src, max_pixels) if u8 else rep.infer_many(src, max_pixels)
        down.wait_stream(s)
        with torch.cuda.stream(down):
            for i, y in zip(idx, ys):
                outs[i].copy_(y, non_blocking=True)
        for y in ys:
            y.record_stream(down)


# ----------------------------------------------------------------------------------------------------------------------
# VGG19 content loss of the RealESRGAN generator step (reference ContentLoss, model.py:278-335): forward and d/d sr in
# libresr.so (C ABI resr_vgg_*, include/resr.h).

VGG19_CONV_FEATURES = (0, 2, 5, 7, 10, 12, 14, 16, 19, 21, 23, 25, 28, 30, 32, 34)
_VGG19_CHANNELS = ((3, 64), (64, 64), (64, 128), (128, 128), (128, 256), (256, 256), (256, 256), (256, 256), (256, 512),
                   (512, 512), (512, 512), (512, 512), (512, 512), (512, 512), (512, 512), (512, 512))
_VGG19_POOLS_BEFORE = (0, 0, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4)
VGG19_CHECKPOINT = "vgg19-dcbb9e9d.pth"   # torchvision's ImageNet weights (models.vgg19(True), reference model.py:296)


def parse_vgg19_nodes(nodes):
    """Node names ("features.<i>") -> features indices, in the caller's order. Only the convolution outputs of
    vgg19().features are supported; anything else raises ValueError naming the supported nodes."""
    if isinstance(nodes, str) or len(nodes) == 0:
        raise ValueError("feature_model_extractor_nodes must be a non-empty list of node names")
    out = []
    for name in nodes:
        idx = None
        if isinstance(name, str) and name.startswith("features."):
            tail = name[len("features."):]
            if tail.isdigit() and str(int(tail)) == tail:
                idx = int(tail)
        if idx not in VGG19_CONV_FEATURES:
            supported = ", ".join(f"features.{i}" for i in VGG19_CONV_FEATURES)
            raise ValueError(f"unsupported content-loss node {name!r}: the supported nodes are {supported}")
        if idx in out:
            raise ValueError(f"content-loss node {name!r} is listed twice")
        out.append(idx)
    return out


def _vgg19_min_size(features):
    """Smallest H (and W) that leaves one pixel at the deepest of `features` (2x2 / stride 2 floor pooling)."""
    return 1 << _VGG19_POOLS_BEFORE[VGG19_CONV_FEATURES.index(max(features))]


class _ContentLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sr, gt, mod):
        n, _, h, w = sr.shape
        src, gtc = sr.detach().contiguous().float(), gt.detach().contiguous().float()
        mod._ensure_packed()
        losses = torch.empty(len(mod.nodes), dtype=torch.float32, device=sr.device)
        wp, wbytes = mod._workspace(n, h, w, sr.device)
        with torch.cuda.device(sr.device):
            _lib.check(_lib.lib().resr_vgg_forward(mod._native(), _lib.ptr(src), _lib.ptr(gtc), _lib.ptr(losses), n, h, w, wp,
                                                   wbytes, _lib.stream_ptr(sr.device)))
        # the saved activations live in the module's single workspace: stamp this forward (as Generator does)
        mod._fwd_generation += 1
        ctx.mod, ctx.shape, ctx.generation, ctx.packed_version = mod, (n, h, w), mod._fwd_generation, mod._packed_version
        return losses

    @staticmethod
    def backward(ctx, grad_losses):
        mod = ctx.mod
        n, h, w = ctx.shape
        if mod._fwd_generation != ctx.generation:
            raise _lib.ResrError(
                "backward of a stale forward: another forward of this ContentLoss ran in between and overwrote the saved "
                "activations (one shared workspace per module). Call backward() before the next forward.")
        if mod._packed_version != ctx.packed_version:
            raise _lib.ResrError("the VGG weights were repacked between forward and backward (parameters changed)")
        g = grad_losses.detach().contiguous().float()
        grad_sr = torch.empty((n, 3, h, w), dtype=torch.float32, device=g.device)
        wp, wbytes = mod._workspace(n, h, w, g.device)
        with torch.cuda.device(g.device):
            _lib.check(_lib.lib().resr_vgg_backward(mod._native(), _lib.ptr(g), _lib.ptr(grad_sr), n, h, w, wp, wbytes,
                                                    _lib.stream_ptr(g.device)))
        return grad_sr, None, None


class ContentLoss(nn.Module):
    """VGG19 content loss (reference model.py:278-335). `forward(sr, gt)` returns the 1-D tensor of the per-node L1 losses
    (mean), in node order; the caller weights and sums them. Semantics are those of torchvision:
    `create_feature_extractor(vgg19, nodes)` on `Normalize(mean, std)` inputs, so a node other than the deepest is the
    conv output after the in-place ReLU that follows it, and the deepest node is the raw conv output. The gradient flows
    to `sr` only; the VGG weights are frozen.

    `vgg`: a torchvision vgg19 module or its state_dict; None loads `vgg19-dcbb9e9d.pth` from
    `torch.hub.get_dir()/checkpoints` if that file exists and raises FileNotFoundError otherwise (nothing is downloaded).
    The 16 convolutions are held as `features.<i>` nn.Conv2d modules, so torchvision's state_dict keys load unchanged."""

    def __init__(self, feature_model_extractor_nodes, feature_model_normalize_mean, feature_model_normalize_std, vgg=None):
        super().__init__()
        self.nodes = list(feature_model_extractor_nodes)
        self.features_idx = parse_vgg19_nodes(self.nodes)
        self.mean = [float(v) for v in feature_model_normalize_mean]
        self.std = [float(v) for v in feature_model_normalize_std]
        if len(self.mean) != 3 or len(self.std) != 3:
            raise ValueError("feature_model_normalize_mean / _std need 3 values (RGB)")
        if any(s == 0 or s != s for s in self.std):
            raise ValueError("feature_model_normalize_std must be non-zero")
        self.features = nn.ModuleDict({str(i): nn.Conv2d(ci, co, 3, 1, 1) for i, (ci, co) in zip(VGG19_CONV_FEATURES, _VGG19_CHANNELS)})
        if vgg is None:
            import os
            path = os.path.join(torch.hub.get_dir(), "checkpoints", VGG19_CHECKPOINT)
            if not os.path.isfile(path):
                raise FileNotFoundError(
                    f"ContentLoss(vgg=None) loads the torchvision VGG19 weights from {path}, which does not exist; place "
                    f"{VGG19_CHECKPOINT} there or pass vgg= (a torchvision vgg19 module or its state_dict). Nothing is downloaded.")
            vgg = torch.load(path, map_location="cpu", weights_only=True)
        sd = vgg.state_dict() if isinstance(vgg, nn.Module) else vgg
        self.load_state_dict({k: v for k, v in sd.items() if k.startswith("features.")})
        for p in self.parameters():
            p.requires_grad_(False)   # reference model.py:301-303: the feature extractor is frozen
        self._handle = None
        self._handle_device = None
        self._packed_version = None
        self._ws = None
        self._fwd_generation = 0

    def _device(self):
        return next(self.parameters()).device

    def _native(self):
        dev = self._device()
        if dev.type != "cuda":
            raise _lib.ResrError("resr_b200.ContentLoss runs on a CUDA (sm_100a) device only; move it with .cuda() / .to(device)")
        if self._handle is not None and self._handle_device != dev:
            self._release()
        if self._handle is None:
            h = ctypes.c_void_p()
            feats = (ctypes.c_int * len(self.features_idx))(*self.features_idx)
            _lib.check(_lib.lib().resr_vgg_create(ctypes.byref(h), feats, len(self.features_idx), (ctypes.c_float * 3)(*self.mean),
                                                  (ctypes.c_float * 3)(*self.std)))
            self._handle, self._handle_device = h, dev
        return self._handle

    def _release(self):
        with torch.cuda.device(self._handle_device):
            torch.cuda.synchronize()
            _lib.lib().resr_vgg_destroy(self._handle)
        self._handle, self._packed_version, self._ws = None, None, None

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None:
            try:
                with torch.cuda.device(self._handle_device):
                    _lib.lib().resr_vgg_destroy(h)
            except Exception:
                pass

    def _param_version(self):
        return tuple((p._version, p.data_ptr(), p.dtype) for p in self.parameters()) + (self._device(),)

    def _ensure_packed(self):
        ver = self._param_version()
        if self._packed_version != ver:
            flat = torch.cat([p.detach().reshape(-1).float() for p in self.parameters()])
            assert flat.numel() == _lib.lib().resr_vgg_num_params()
            dev = self._device()
            h = self._native()
            with torch.cuda.device(dev):
                _lib.check(_lib.lib().resr_vgg_load_params(h, _lib.ptr(flat), _lib.stream_ptr(dev)))
                torch.cuda.current_stream(dev).synchronize()   # `flat` is a temporary
            self._packed_version = ver

    def _workspace(self, n, h, w, device):
        need = _lib.lib().resr_vgg_workspace_bytes(self._native(), n, h, w)
        if need == 0:
            raise ValueError(_lib.lib().resr_last_error().decode())
        if self._ws is None or self._ws.numel() < need + 1024 or self._ws.device != device:
            self._ws = torch.empty(need + 1024, dtype=torch.uint8, device=device)
        return Generator._aligned(self._ws)

    def forward(self, sr: torch.Tensor, gt: torch.Tensor) -> torch.Tensor:
        if sr.dim() != 4 or sr.size(1) != 3 or sr.shape != gt.shape:
            raise ValueError(f"expected sr and gt of one [N, 3, H, W] shape, got {tuple(sr.shape)} and {tuple(gt.shape)}")
        if not (sr.is_cuda and gt.is_cuda):
            raise _lib.ResrError("resr_b200.ContentLoss runs on a CUDA (sm_100a) device only; there is no CPU path")
        if sr.device != self._device() or gt.device != self._device():
            raise _lib.ResrError(f"inputs on {sr.device} / {gt.device} but the loss lives on {self._device()}")
        m = _vgg19_min_size(self.features_idx)
        if sr.size(2) < m or sr.size(3) < m:
            raise ValueError(f"{sr.size(2)} x {sr.size(3)} leaves no pixel at features.{max(self.features_idx)}: "
                             f"H and W must be at least {m}")
        return _ContentLossFn.apply(sr, gt, self)
