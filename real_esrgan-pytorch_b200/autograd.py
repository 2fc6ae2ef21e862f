"""Training path of the generator mirror: forward that keeps activations, fused L1 loss and the full backward pass,
all inside libresr.so (resr_generator_forward_train / _backward_l1 / _backward, include/resr.h).

Replaces, for the generator, `sr = model(lr); loss = L1(sr, hr); loss.backward()` of the reference training loop
(train_realesrnet.py:383-388). Gradients arrive as ONE flat fp32 vector in state_dict order (the layout a DDP
all-reduce or a fused optimizer wants) and are scattered into `param.grad`.
"""
import ctypes

import torch

from . import _lib


def _train_workspace(gen, n, h, w, device):
    need = _lib.lib().resr_generator_train_workspace_bytes(n, h, w)
    ws = getattr(gen, "_train_ws", None)
    if ws is None or ws.numel() < need + 1024 or ws.device != device:
        ws = torch.empty(need + 1024, dtype=torch.uint8, device=device)
        gen._train_ws = ws
    base = ws.data_ptr()
    off = (-base) % 1024
    return ctypes.c_void_p(base + off), ws.numel() - off


def _scatter_grads(gen, flat: torch.Tensor, accumulate: bool = True):
    pos = 0
    for p in gen.parameters():
        n = p.numel()
        g = flat[pos:pos + n].view_as(p)
        if p.requires_grad:
            if p.grad is None or not accumulate:
                p.grad = g.clone()
            else:
                p.grad.add_(g)
        pos += n


class _GeneratorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gen, *params):
        n, _, h, w = x.shape
        xc = x.detach().contiguous().float()
        gen._ensure_packed()
        y = torch.empty((n, 3, 4 * h, 4 * w), dtype=torch.float32, device=x.device)
        wp, wbytes = _train_workspace(gen, n, h, w, x.device)
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().resr_generator_forward_train(gen._native(), _lib.ptr(xc), _lib.ptr(y), n, h, w, wp, wbytes,
                                                               _lib.stream_ptr(x.device)))
        # The saved activations live in the generator's single training workspace: stamp this forward so that the
        # matching backward can tell whether a later forward (or a weight repack) has overwritten them.
        gen._fwd_generation += 1
        ctx.gen = gen
        ctx.shape = (n, h, w)
        ctx.generation = gen._fwd_generation
        ctx.packed_version = gen._packed_version
        return y

    @staticmethod
    def backward(ctx, dy):
        gen = ctx.gen
        n, h, w = ctx.shape
        if ctx.needs_input_grad[0]:
            raise _lib.ResrError("resr_b200.Generator does not produce a gradient w.r.t. its input: detach() the LR batch")
        if gen._fwd_generation != ctx.generation:
            raise _lib.ResrError(
                "backward of a stale forward: another training-mode forward of this Generator ran in between and "
                "overwrote the saved activations (one shared workspace per Generator). Call backward() before the next "
                "forward, or run the second forward under torch.no_grad().")
        if gen._packed_version is not ctx.packed_version and gen._packed_version != ctx.packed_version:
            raise _lib.ResrError("the weights were repacked between forward and backward (parameters changed)")
        dyc = dy.detach().contiguous().float()
        flat = torch.empty(_lib.lib().resr_generator_num_params(), dtype=torch.float32, device=dy.device)
        wp, wbytes = _train_workspace(gen, n, h, w, dy.device)
        with torch.cuda.device(dy.device):
            _lib.check(_lib.lib().resr_generator_backward(gen._native(), _lib.ptr(dyc), _lib.ptr(flat), n, h, w, wp, wbytes,
                                                          _lib.stream_ptr(dy.device)))
        grads, pos = [], 0
        for p in gen.parameters():
            grads.append(flat[pos:pos + p.numel()].view_as(p) if p.requires_grad else None)
            pos += p.numel()
        return (None, None) + tuple(grads)  # no gradient w.r.t. the LR input (the degradation output is detached)


def generator_apply(gen, x):
    return _GeneratorFn.apply(x, gen, *list(gen.parameters()))


def l1_loss_backward(gen, lr: torch.Tensor, hr: torch.Tensor, accumulate: bool = False):
    """Fused training step core: sr = G(lr); loss = mean|sr - hr|; d loss / d params. Returns (loss, sr, flat_grads);
    flat_grads (fp32, state_dict order) is also scattered into param.grad."""
    n, _, h, w = lr.shape
    dev = lr.device
    xc = lr.detach().contiguous().float()
    hrc = hr.detach().contiguous().float()
    gen._ensure_packed()
    sr = torch.empty((n, 3, 4 * h, 4 * w), dtype=torch.float32, device=dev)
    flat = torch.empty(_lib.lib().resr_generator_num_params(), dtype=torch.float32, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    wp, wbytes = _train_workspace(gen, n, h, w, dev)
    lib = _lib.lib()
    gen._fwd_generation += 1  # invalidates any autograd graph still holding activations in this workspace
    with torch.cuda.device(dev):
        _lib.check(lib.resr_generator_forward_train(gen._native(), _lib.ptr(xc), _lib.ptr(sr), n, h, w, wp, wbytes, _lib.stream_ptr(dev)))
        _lib.check(lib.resr_generator_backward_l1(gen._native(), _lib.ptr(hrc), _lib.ptr(flat), _lib.ptr(loss), n, h, w, wp, wbytes,
                                                  _lib.stream_ptr(dev)))
    _scatter_grads(gen, flat, accumulate)
    return loss, sr, flat


class TrainStep:
    """Persistent-buffer training-step core for a fixed (N, H, W): `step(lr, hr)` copies the batch into static device
    buffers and runs forward + L1 + backward as ONE CUDA-graph replay (C ABI resr_generator_train_step_l1).
    Gradients land in `self.flat` (fp32, state_dict order); with a process group they are averaged over ranks with a
    single NCCL all-reduce (data parallel, reference has none: SURVEY.md §2.1) before being scattered to param.grad."""

    def __init__(self, gen, n: int, h: int, w: int, device=None, process_group=None, world_size: int = 1):
        self.gen, self.shape = gen, (n, h, w)
        dev = device or next(gen.parameters()).device
        self.lr = torch.zeros((n, 3, h, w), dtype=torch.float32, device=dev)
        self.hr = torch.zeros((n, 3, 4 * h, 4 * w), dtype=torch.float32, device=dev)
        self.sr = torch.empty_like(self.hr)
        self.flat = torch.zeros(_lib.lib().resr_generator_num_params(), dtype=torch.float32, device=dev)
        self.loss = torch.zeros((), dtype=torch.float32, device=dev)
        self.group, self.world = process_group, world_size
        # CUDA graphs cannot be captured on the legacy default stream: the step runs on its own stream, ordered
        # against the caller's current stream on both sides
        self.stream = torch.cuda.Stream(device=dev)
        # data parallel: the flat gradient vector is all-reduced in 4 buckets on a communication stream, each as soon as
        # the backward has finished it (C ABI resr_generator_grad_buckets / resr_generator_wait_grad_bucket)
        self.comm = torch.cuda.Stream(device=dev) if world_size > 1 else None
        offs = (ctypes.c_size_t * 5)()
        self.nbuckets = _lib.lib().resr_generator_grad_buckets(offs, 5)
        self.bucket_offsets = [int(o) for o in offs]
        self.overlap = True

    def step(self, lr: torch.Tensor = None, hr: torch.Tensor = None, scatter: bool = True):
        n, h, w = self.shape
        gen = self.gen
        cur = torch.cuda.current_stream(self.lr.device)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            if lr is not None:
                self.lr.copy_(lr, non_blocking=True)
            if hr is not None:
                self.hr.copy_(hr, non_blocking=True)
            gen._ensure_packed()
            gen._fwd_generation += 1
            wp, wbytes = _train_workspace(gen, n, h, w, self.lr.device)
            with torch.cuda.device(self.lr.device):
                _lib.check(_lib.lib().resr_generator_train_step_l1(
                    gen._native(), _lib.ptr(self.lr), _lib.ptr(self.hr), _lib.ptr(self.sr), _lib.ptr(self.flat), _lib.ptr(self.loss), n, h,
                    w, wp, wbytes, _lib.stream_ptr(self.lr.device)))
            if self.world > 1:
                if self.overlap and self.nbuckets == 4:
                    self._allreduce_buckets()
                else:
                    allreduce_mean_(self.flat, self.group, self.world)
        cur.wait_stream(self.stream)
        if scatter:
            _scatter_grads(gen, self.flat, accumulate=False)
        return self.loss, self.sr, self.flat

    def _allreduce_buckets(self):
        """Gradient all-reduce overlapped with the backward (SURVEY.md §8e): the communication stream waits for each
        bucket's completion event inside the running step (tail and trunk.22-17 first), reduces that slice of the flat
        vector over NCCL while the rest of the backward is still executing, and the step's stream joins at the end."""
        import torch.distributed as dist
        dev = self.lr.device
        with torch.cuda.device(dev):
            for k in (3, 2, 1, 0):
                if k == 0:
                    self.comm.wait_stream(self.stream)     # the front of the vector completes with the step itself
                else:
                    _lib.check(_lib.lib().resr_generator_wait_grad_bucket(self.gen._native(), k, ctypes.c_void_p(self.comm.cuda_stream)))
                a, b = self.bucket_offsets[k], self.bucket_offsets[k + 1]
                with torch.cuda.stream(self.comm):
                    sl = self.flat[a:b]
                    dist.all_reduce(sl, op=dist.ReduceOp.SUM, group=self.group)
                    sl.div_(self.world)
        self.stream.wait_stream(self.comm)

    @property
    def is_graph(self) -> bool:
        return bool(_lib.lib().resr_generator_step_is_graph(self.gen._native()))


def allreduce_mean_(flat: torch.Tensor, group=None, world_size: int = None):
    """The one collective of data-parallel training: sum the flat gradient vector over ranks (NCCL over NVLink on the
    GPU box, gloo in the CPU tests) and divide by the world size."""
    import torch.distributed as dist
    world_size = world_size or dist.get_world_size(group)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.div_(world_size)
    return flat
