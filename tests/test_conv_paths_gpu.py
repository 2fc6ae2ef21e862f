"""Every launch configuration of the tcgen05 3x3 convolution kernels (csrc/conv3x3_tc.cu: one CTA, csrc/conv3x3_pair.cu:
CTA pairs; shared epilogue in csrc/conv3x3_common.cuh) against a float64 reference of the same operation, at the shapes
where the configuration changes or goes ragged.

Each case names the configuration it means to reach; resr_conv3x3_plan (host only, the function resr_conv3x3 plans
through) must report exactly that configuration under the case's policy, so a changed threshold fails loudly instead
of moving a case off its path. Every case then runs under pair policies 0, 1 and 2 (each distinct plan once).
test_conv_args_cpu.py::test_every_configuration_has_a_case checks on the CPU that the table reaches every value of
each axis the planner can produce.

Operands are random values rounded to the 16-bit operand format, so every product is exact in fp32. The reference is
F.conv2d in float64 of the same operands (on the GPU, where TF32 does not apply to doubles), followed by the epilogue
arithmetic in float64. Tolerance per element, S = conv2d(|x|, |w|) + |b| carried through the epilogue with the
residual magnitudes added:

  * The accumulator is fp32. A 64-channel chunk is 4 K16 steps, times 3 dx times 3 dy taps: at most 36 MMA steps per
    chunk, 108 for cin = 192 and 180 for the largest cin a kernel accepts (320), plus the bias the accumulator starts
    from and a handful of epilogue roundings (0.2 v, + r, fma). Each rounds to at most 2^-24 of a partial sum whose
    magnitude is at most S, so |got - ref| <= 190 * 2^-24 * S < 2^-16 * S.
  * 16-bit outputs add half an ulp of the output format at the reference value; fp16 saturates at 65504.
  * out_u8 is exact, except where 255 * ref lies within the fp32 bound of an integer.
  * Canvas (vmask) pixels outside the images must be exactly 0 in every output.

The bound is tight enough to see one lost product: dropping a single (channel, tap) term at one pixel changes the sum
by S / (9 cin) on average, 38x the bound at cin = 192 (test_conv_args_cpu.py::test_bound_catches_one_dropped_product).

Every output lives in a region pre-filled with NaN and framed by sentinels: NHWC outputs have sentinel channels
before choff and after the channels written, and sentinel pixels before and after the tensor; NCHW and u8 outputs
have sentinel elements before and after. Every output element must be written and no sentinel may change. The inputs
(channels past cin filled with NaN, which the tensor map must not read), residuals (NaN outside the channels read)
and mask16 must be unchanged after the call, except for the in-place RRDB buffer."""
import ctypes
import json
import math
import os
import zlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

P = 0x1000                   # dummy device pointer for host-only planning; never dereferenced
GUARD_PIX = 64               # sentinel pixels before / after an NHWC output
GUARD = 4096                 # sentinel elements before / after an NCHW / u8 output
SENT32 = -12345.5
SENT16 = -1152.0             # exact in fp16 and bf16
SENT8 = 0xA5
C02 = float(np.float32(0.2))  # the kernels scale by the fp32 constant 0.2f
F16_MAX = 65504.0
BOUND = 2.0 ** -16
RING = {(0, 32): 16, (0, 16): 16, (1, 64): 6, (1, 32): 14, (1, 16): 14}   # (pair, nout) -> accumulator ring positions


def _L():
    import resr_b200
    return resr_b200._lib


# ============================================================================================== the table
def C(cid, want, n=1, h=5, w=128, cin=64, cout=32, **kw):
    """One case: the convolution, its epilogue and outputs, and `want`, the configuration tag resr_conv3x3_plan must
    report under `policy` (default 2: CTA pairs wherever two column groups exist)."""
    c = dict(id=cid, want=want, n=n, h=h, w=w, cin=cin, cout=cout, c_total=None, fmt=1, mode=-1, ep=0, res=None,
             res2_scale=0.0, lrelu=0, clamp01=0, o16=None, up2=0, outf=None, nchw=0, raw=0, u8=0, mask16=0, o16scale=0.0,
             nores=0, noutf=0, no16=0, fixed=0, vmask=None, reverse=0, inplace=0, big=0, lap=0, policy=2)
    for k, v in kw.items():
        assert k in c, k
        c[k] = v
    if c["c_total"] is None:
        c["c_total"] = max(64, -(-cin // 64) * 64)
    if c["inplace"]:   # the RRDB output overwrites its res2 input: the trunk's 16-bit residual stream
        c["o16"] = (c["res"], cout + 64, 0)
    if c["o16"] is None and c["outf"] is None and not (c["nchw"] or c["raw"] or c["u8"]):
        if cout % 32 == 0:
            c["outf"] = (cout, 0)
        else:
            c["nchw"] = 1
    return c


W_LIST = [1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 130, 255, 257, 383]
_BN = {8: 16, 16: 8, 32: 4, 64: 2}

CASES = (
    # ---- lane split and ragged edges: BN 16 / 8 / 4 / 2 / 1, last segments of 1, 2, 127 pixels, odd ncg under pairs
    [C(f"w{w}", f"pair32 bn{_BN.get(w, 1)} m{1 if w in _BN else 0} k4 e2x2", n=3, w=w, fmt=w & 1)
     for w in W_LIST if w not in (8, 16, 32)]
    + [C("w16", "single32 bn8 m1 k4 e2x1", n=3, w=16, fmt=0),        # N < BN: one column group
       C("w32", "single32 bn4 m1 k4 e2x1", n=3, w=32)]
    + [C("w8-n3", "single32 bn16 m1 k4 e2x1", n=3, w=8),          # N < BN: one column group
       C("w8-n33", "pair32 bn16 m1 k4 e2x2", n=33, w=8),          # N not a multiple of BN, odd ncg (3)
       C("w16-n9", "pair32 bn8 m1 k4 e2x2", n=9, w=16, fmt=0),
       C("w32-n6", "pair32 bn4 m1 k4 e2x2", n=6, w=32),
       C("w64-n5", "pair32 bn2 m1 k4 e2x2", n=5, w=64, fmt=0),
       C("w200-mode1", "pair32 bn1 m1 k4 e2x2", n=1, w=200, mode=1),
       C("w383-mode1", "pair32 bn1 m1 k4 e2x2", n=1, w=383, mode=1, fmt=0)]
    # ---- image height
    + [C(f"h{h}", "pair32 bn1 m0 k4 e2x2", n=2, h=h, fmt=h & 1) for h in (1, 2, 3, 5, 7)]
    # ---- K tail: every tail length, c_total past cin (NaN there), the largest cin of each kernel
    + [C(f"cin{ci}", f"pair32 bn2 m1 k{4 if ci % 64 in (0,) or ci % 64 > 32 else (2 if ci % 64 > 16 else 1)} e2x2",
         n=4, h=6, w=64, cin=ci, fmt=ci & 1) for ci in (3, 8, 16, 17, 32, 33, 40, 63, 64, 65, 96, 128, 160, 192)]
    + [C("cin40-ctotal192", "pair32 bn1 m0 k4 e2x2", n=2, h=4, cin=40, c_total=192),
       C("cin3-mode0", "pair32 bn1 m0 k1 e2x2", n=2, h=6, cin=3, fmt=0),
       C("cin17-mode1", "pair32 bn1 m1 k2 e2x2", n=2, h=6, cin=17, mode=1),
       C("cin64-ctotal192", "pair32 bn1 m0 k4 e2x2", n=2, h=4, cin=64, c_total=192),
       C("cinmax-single32", "single32 bn1 m0 k4 e1x1", n=2, h=6, cin=256, policy=0),
       C("cinmax-single32-o16", "single32 bn1 m0 k4 e1x1", n=2, h=6, cin=320, outf=None, o16=(1, 32, 0), policy=0),
       C("cinmax-single16", "single16 bn1 m0 k4 e1x1", n=2, h=6, cin=640, cout=3, policy=0),
       C("cinmax-pair32", "pair32 bn1 m0 k4 e1x1", n=2, h=6, cin=576, fmt=0),
       C("cinmax-pair64", "pair64 bn1 m0 k4 e1x1", n=2, h=6, cin=256, cout=64),
       C("cinmax-pair16", "pair16 bn1 m0 k4 e1x1", n=2, h=6, cin=1344, cout=3)]
    # ---- output width: NOUT 16 (NCHW only), 32, 64; odd slice counts
    + [C(f"cout{co}", f"pair16 bn1 m0 k4 e3x2", n=2, cout=co) for co in (1, 3, 16)]
    + [C("cout32", "pair32 bn1 m0 k4 e2x2", n=2, cout=32),
       C("cout64", "pair64 bn1 m0 k4 e2x2", n=2, cout=64),
       C("cout96", "pair32 bn1 m0 k4 e2x2", n=2, cout=96, fmt=0),
       C("cout128", "pair64 bn1 m0 k4 e2x2", n=2, cout=128),
       C("cout192", "pair64 bn1 m0 k4 e2x1", n=2, cout=192, cin=192, fmt=0),
       C("cout64-n192", "pair64 bn2 m1 k4 e2x2", n=192, h=3, w=64, cout=64),
       C("cout128-n192", "pair64 bn4 m1 k4 e2x2", n=192, h=2, w=32, cout=128, fmt=0)]
    # ---- NOUT x BN of both kernels
    + [C(f"nout16-bn{bn}", f"pair16 bn{bn} m{0 if bn == 1 else 1} k4 e3x2", n=2 * bn + 1, w=128 // bn, cout=3,
         fmt=bn & 1) for bn in (1, 2, 4, 8, 16)]
    + [C(f"nout64-bn{bn}", f"pair64 bn{bn} m{0 if bn == 1 else 1} k4 e2x2", n=2 * bn + 1, w=128 // bn, cout=64,
         fmt=bn & 1) for bn in (1, 2, 4, 8, 16)]
    # ---- accumulator ring laps (a CTA's strip at least twice the ring on the device's SM count)
    + [C("lap-single32", "single32 bn1 m0 k4 e2x1", h=4800, w=100, lap=1),
       C("lap-single16", "single16 bn1 m0 k4 e3x1", h=4800, w=100, cout=3, lap=1, fmt=0),
       C("lap-single32-groups", "single32 bn1 m0 k4 e2x1", n=64, h=75, w=128, lap=1, policy=0),
       C("lap-pair64", "pair64 bn1 m0 k4 e2x2", h=1480, w=256, cout=64, lap=1),
       C("lap-pair64-rev", "pair64 bn1 m0 k4 e2x2", h=1480, w=256, cout=64, lap=1, reverse=1, fmt=0),
       C("lap-pair32", "pair32 bn1 m0 k4 e2x2", h=2400, w=256, lap=1),
       C("lap-pair16", "pair16 bn1 m0 k4 e3x2", h=2400, w=256, cout=3, lap=1, reverse=1),
       C("lap-pair32-groups", "pair32 bn1 m0 k4 e2x2", n=80, h=75, w=128, lap=1, fmt=0)]
    # ---- pair traversal, odd ncg included
    + [C(f"rev{r}-nout{no}-ncg{k}", f"pair{no} bn1 m0 k4 e{3 if no == 16 else 2}x2", n=k, h=9, reverse=r,
         cout={64: 64, 32: 96, 16: 3}[no], fmt=r) for r in (0, 1) for no in (64, 32, 16) for k in (2, 3)]
    # ---- epilogue modes with fp32 and 16-bit residuals
    + [C(f"ep{e}-res{rn}", f"pair64 bn1 m0 k4 e{2 if rn == 'f32' else 3}x2", n=2, h=7, cout=64, ep=e, res=r,
         outf=(64, 0) if r == "f32" else None, o16=None if r == "f32" else (r, 64, 0), fmt=1 if r == "f32" else r)
       for e in (1, 2, 3) for r, rn in (("f32", "f32"), (0, "f16"), (1, "bf16"))]
    + [C("ep0", "pair64 bn1 m0 k4 e2x2", n=2, h=7, cout=64),
       C("ep4-res1-res2", "pair64 bn1 m0 k4 e2x2", n=2, h=7, cout=64, ep=4, res="f32", res2_scale=-0.75),
       C("ep4-res2-only", "pair32 bn1 m0 k4 e2x2", n=2, h=7, cout=96, ep=4, res="f32-res2", res2_scale=2.5),
       C("ep3-nchw", "pair32 bn1 m0 k4 e3x2", n=2, h=7, cout=32, ep=3, res="f32", outf=None, nchw=1),
       C("rrdb-inplace-f16", "pair64 bn1 m0 k4 e3x2", n=2, h=7, cout=64, ep=2, res=0, inplace=1, fmt=0),
       C("rrdb-inplace-bf16", "pair64 bn1 m0 k4 e3x2", n=2, h=7, cout=64, ep=2, res=1, inplace=1),
       C("rrdb-inplace-rows", "pair64 bn1 m0 k4 e3x2", n=2, h=300, cout=64, ep=2, res=0, inplace=1, fmt=0),
       C("rrdb-inplace-rows-single", "single32 bn1 m0 k4 e3x1", n=1, h=300, cout=64, ep=2, res=1, inplace=1)]
    # ---- activation, clamp, 16-bit and fp32 stores at offsets, up2, NCHW / raw / u8
    + [C("lrelu", "pair32 bn1 m0 k4 e2x2", n=2, cout=96, lrelu=1),
       C("clamp01", "pair64 bn1 m0 k4 e2x2", n=2, cout=64, clamp01=1),
       C("o16-f16-choff", "pair64 bn1 m0 k4 e3x2", n=2, cout=64, o16=(0, 192, 72), fmt=0),
       C("o16-bf16-choff", "pair32 bn1 m0 k4 e3x2", n=2, cout=32, o16=(1, 200, 96)),
       C("o16-f16-up2-bn4", "pair64 bn4 m1 k4 e3x2", n=9, h=4, w=32, cout=64, o16=(0, 128, 64), up2=1),
       C("o16-bf16-up2-bn1", "pair32 bn1 m0 k4 e3x2", n=2, h=4, w=130, cout=32, o16=(1, 64, 8), up2=1),
       C("outf-choff", "pair64 bn1 m0 k4 e2x2", n=2, cout=64, outf=(100, 36)),
       C("outf-o16", "pair64 bn2 m1 k4 e2x1", n=3, w=64, cout=64, outf=(128, 32), o16=(1, 64, 0)),
       C("nchw-raw-u8-rgb", "pair16 bn1 m0 k4 e3x2", n=2, h=6, cout=3, nchw=1, raw=1, u8=1, clamp01=1),
       C("nchw-raw-u8-w32", "pair32 bn4 m1 k4 e3x2", n=5, h=6, w=32, cout=32, nchw=1, raw=1, u8=1, clamp01=1, fmt=0),
       C("u8-only", "pair16 bn2 m1 k4 e3x2", n=5, w=64, cout=3, u8=1, clamp01=1),
       C("mask16-f16", "pair64 bn1 m0 k4 e3x2", n=2, cout=64, o16=(0, 64, 0), mask16=1, fmt=0),
       C("mask16-bf16-scale", "pair32 bn1 m0 k4 e3x2", n=2, cout=96, o16=(1, 96, 0), mask16=1, o16scale=-3.0),
       C("o16scale-outf", "pair64 bn1 m0 k4 e2x1", n=2, cout=64, outf=(64, 0), o16=(1, 64, 0), o16scale=0.125),
       C("f16-saturate", "pair32 bn1 m0 k4 e3x2", n=2, cout=32, o16=(0, 32, 0), big=1, fmt=0),
       C("f16-saturate-single", "single32 bn1 m0 k4 e3x1", n=1, cout=64, o16=(0, 64, 0), big=1, fmt=0)]
    # ---- per-slice flags (the training step's data-gradient launches)
    + [C(f"slices-{k}-nout{no}", f"pair{no} bn1 m0 k4 e2x{1 if no == 64 else 2}", n=2, h=6, cout=co, ep=1, res="f32",
         outf=(co, 0), o16=(1, co + 32, 32), **{k: m})
       for no, co in ((64, 128), (32, 96)) for k, m in (("nores", 0b010), ("noutf", 0b101), ("no16", 0b011))]
    + [C(f"slice-fixed-nout{no}", f"pair{no} bn1 m0 k4 e3x2", n=2, h=6, cout=co, o16=(0, 64, 16), fixed=1,
         no16=(1 << (co // 32)) - 1 - (1 << 1), fmt=0) for no, co in ((64, 128), (32, 96))]
    # ---- packed canvas (MASKED instantiations)
    + [C(f"vmask-s{s}-nout{no}", f"pair{no} bn1 m0 k4 e{3 if no == 16 else 2}x2", h=24, w=256,
         cout={64: 64, 32: 32, 16: 3}[no], vmask=s, lrelu=1, fmt=s & 1, **({"nchw": 1, "u8": 1, "clamp01": 1} if no == 16 else {}))
       for no in (64, 32, 16) for s in (0, 1, 2)]
    + [C("vmask-single32", "single32 bn1 m0 k4 e3x1", h=40, w=96, cout=64, vmask=1, outf=None, o16=(1, 64, 0),
         ep=3, res=1),
       C("vmask-single16", "single16 bn1 m0 k4 e3x1", h=40, w=100, cout=3, vmask=2, nchw=1, raw=1, u8=1, clamp01=1)]
    # ---- epilogue stage counts of both kernels (the largest-cin rows above take e1x1)
    + [C("epi-single32-e3x1", "single32 bn1 m0 k4 e3x1", n=1, h=9, cout=32, outf=None, o16=(1, 32, 0)),
       C("epi-single32-e2x1", "single32 bn1 m0 k4 e2x1", n=2, h=9, cin=192, outf=(32, 0), o16=(0, 32, 0), policy=0),
       C("epi-pair64-e3x1", "pair64 bn1 m0 k4 e3x1", n=2, h=9, cin=192, cout=64, outf=None, o16=(1, 64, 0)),
       C("epi-pair64-e1x1-o16", "pair64 bn1 m0 k4 e1x1", n=2, h=9, cin=320, cout=64, outf=None, o16=(1, 64, 0), fmt=0),
       C("epi-pair64-e2x1", "pair64 bn1 m0 k4 e2x1", n=2, h=9, cin=128, cout=64, outf=(64, 0), o16=(1, 64, 0)),
       C("epi-pair64-e1x1-both", "pair64 bn1 m0 k4 e1x1", n=2, h=9, cin=256, cout=64, outf=(64, 0), o16=(1, 64, 0)),
       C("epi-pair32-e2x1", "pair32 bn1 m0 k4 e2x1", n=2, h=9, cin=256, cout=32, fmt=0),
       C("epi-pair32-e3x1", "pair32 bn1 m0 k4 e3x1", n=2, h=9, cin=320, cout=32, outf=None, o16=(0, 32, 0)),
       C("epi-pair16-e3x1", "pair16 bn1 m0 k4 e3x1", n=2, h=9, cin=896, cout=3)]
)


def tag(plan):
    return (f"{'pair' if plan.pair else 'single'}{plan.nout} bn{plan.bn} m{plan.mode} k{plan.tail_ksteps} "
            f"e{plan.nepi}x{plan.epi_bufs}")


# ============================================================================================== descriptor and plan
def desc(c, ptr=None):
    """resr_conv_desc of case `c`; `ptr(name)` gives the device pointer of each buffer (None: dummies for planning)."""
    L = _L()
    p = ptr or (lambda name: P)
    d = L.ConvDesc()
    d.in16 = p("in16")
    d.n, d.h, d.w, d.c_total, d.cin, d.cout = c["n"], c["h"], c["w"], c["c_total"], c["cin"], c["cout"]
    d.fmt_in, d.mode = c["fmt"], c["mode"]
    d.weight, d.bias = p("weight"), p("bias")
    d.ep_mode, d.lrelu, d.clamp01 = c["ep"], c["lrelu"], c["clamp01"]
    if c["o16"] is not None:
        f, cs, co = c["o16"]
        d.out16, d.out16_fmt, d.out16_cstride, d.out16_choff, d.out16_up2 = p("out16"), f, cs, co, c["up2"]
    if c["outf"] is not None:
        d.outf, d.outf_cstride, d.outf_choff = p("outf"), c["outf"][0], c["outf"][1]
    lay = res_layout(c)
    if lay:
        d.res_cstride, d.res_choff = lay["cs"], lay["choff"]
        if lay["res1"]:
            d.res1 = p("res1")
        if lay["res2"]:
            d.res2, d.res2_cstride = p("res2"), lay["cs2"]
        d.res16, d.res16_fmt = (0, 0) if lay["f32"] else (1, c["res"])
        d.res2_scale = c["res2_scale"]
    if c["nchw"]:
        d.out_nchw = p("out_nchw")
    if c["raw"]:
        d.out_nchw_raw = p("out_nchw_raw")
    if c["u8"]:
        d.out_u8 = p("out_u8")
    if c["nchw"] or c["raw"] or c["u8"]:
        d.out_nchw_c = c["cout"]
    d.reverse = c["reverse"]
    if c["vmask"] is not None:
        d.vmask, d.vmask_words, d.vmask_shift = p("vmask"), vmask_words(c), c["vmask"]
    if c["mask16"]:
        d.mask16, d.mask16_cstride, d.mask16_choff = p("mask16"), c["cout"] + 16, 8
    d.out16_scale = c["o16scale"]
    d.slice_nores_mask, d.slice_noutf_mask, d.slice_no16_mask = c["nores"], c["noutf"], c["no16"]
    d.out16_slice_fixed = c["fixed"]
    return d


def res_layout(c):
    """Residual buffers of case `c`: channels [choff, choff + cout) of cs-channel (res1) / cs2-channel (res2) tensors."""
    r, ep = c["res"], c["ep"]
    if r is None:
        return None
    f32 = r in ("f32", "f32-res2")
    if c["inplace"]:
        cs, choff = c["cout"] + 64, 0    # the trunk's layout: the RRDB input at channels [0, 64) of the concat buffer
        return dict(f32=False, cs=cs, choff=choff, cs2=cs, res1=True, res2=True)
    return dict(f32=f32, cs=c["cout"] + 40, choff=24 if f32 else 32, cs2=c["cout"] + 48,
                res1=r != "f32-res2" and ep in (1, 2, 3, 4), res2=ep in (2, 4))


def vmask_words(c):
    return -(-(-(-c["w"] // (1 << c["vmask"]))) // 32)


def plan_of(d, sms, policy):
    L = _L()
    lib = L.lib()
    prev = lib.resr_set_conv_pair_policy(policy)
    try:
        pl = L.ConvPlan()
        rc = lib.resr_conv3x3_plan(ctypes.byref(d), sms, ctypes.byref(pl))
    finally:
        lib.resr_set_conv_pair_policy(prev)
    return pl if rc == 0 else None


def cta_accumulators(units, clusters, h):
    """Virtual accumulators (output rows plus two halo rows per strip) each CTA / pair drains, as the kernels split
    their (column group, row) range into strips."""
    out = []
    for i in range(clusters):
        g0, g1 = units * i // clusters, units * (i + 1) // clusters
        g, acc = g0, 0
        while g < g1:
            ya = g % h
            yb = min(h, ya + (g1 - g))
            acc += min(yb, h - 1) - max(ya - 1, 0) + 3
            g += yb - ya
        out.append(acc)
    return out


def laps(plan, h):
    """The strip of every CTA is at least twice the accumulator ring."""
    return min(cta_accumulators(plan.units, plan.clusters, h)) >= 2 * RING[(plan.pair, plan.nout)]


# ============================================================================================== GPU run
def _half_ulp(x, fmt):
    """Half an ulp of the 16-bit format `fmt` at |x| (float64 tensor)."""
    _, e = torch.frexp(x.abs().clamp_min(1e-300))
    e = e.to(torch.float64) - 1
    if fmt == 0:
        return torch.exp2(torch.clamp(e, min=-14) - 11)
    return torch.exp2(torch.clamp(e, min=-126) - 8)


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else (t.view(torch.int32) if t.element_size() == 4 else t)


class NHWCOut:
    """An NHWC output [n, h, w, cs] framed by sentinel pixels, its written channels NaN (or `init`), the rest sentinel."""

    def __init__(self, n, h, w, cs, chans, dtype, init=None):
        sent = SENT32 if dtype == torch.float32 else SENT16
        pix = n * h * w
        self.buf = torch.full(((pix + 2 * GUARD_PIX) * cs,), sent, dtype=dtype, device="cuda")
        self.t = self.buf[GUARD_PIX * cs:(GUARD_PIX + pix) * cs].view(n, h, w, cs)
        self.chans = torch.tensor(chans, dtype=torch.long, device="cuda")
        self.t[..., self.chans] = float("nan") if init is None else init
        self.before = self.buf.clone()
        self.written = torch.zeros(self.buf.numel(), dtype=torch.bool, device="cuda")
        self.written.view(-1)[GUARD_PIX * cs:(GUARD_PIX + pix) * cs].view(n, h, w, cs)[..., self.chans] = True

    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        torch.cuda.synchronize()
        keep = ~self.written
        assert torch.equal(_bits(self.buf)[keep], _bits(self.before)[keep]), f"{what}: a store outside the output's channels"
        got = self.t[..., self.chans].double()
        assert bool(torch.isfinite(got).all()), f"{what}: output elements left unwritten"
        return got


class FlatOut:
    """A NaN-filled (u8: 0xA5-filled) NCHW / NHWC-u8 output framed by GUARD sentinel elements."""

    def __init__(self, shape, dtype):
        n = int(np.prod(shape))
        sent = SENT8 if dtype == torch.uint8 else SENT32
        self.buf = torch.full((n + 2 * GUARD,), sent, dtype=dtype, device="cuda")
        self.t = self.buf[GUARD:GUARD + n].view(shape)
        if dtype != torch.uint8:
            self.t.fill_(float("nan"))
        self.before = self.buf.clone()
        self.n = n

    def ptr(self):
        return self.t.data_ptr()

    def check(self, what):
        torch.cuda.synchronize()
        assert torch.equal(self.buf[:GUARD], self.before[:GUARD]), f"{what}: store before the output"
        assert torch.equal(self.buf[GUARD + self.n:], self.before[GUARD + self.n:]), f"{what}: store past the output"
        if self.t.dtype != torch.uint8:
            assert bool(torch.isfinite(self.t).all()), f"{what}: output elements left unwritten"
        return self.t.double()


def _slices_on(c, off_mask):
    return [s for s in range(-(-c["cout"] // 32)) if not (off_mask >> s) & 1]


def _run_case(c, policy, report):
    L = _L()
    torch.cuda.synchronize()
    g = torch.Generator().manual_seed(zlib.crc32(c["id"].encode()))
    n, h, w, cin, cout, ct = c["n"], c["h"], c["w"], c["cin"], c["cout"], c["c_total"]
    dt = torch.bfloat16 if c["fmt"] else torch.float16
    dev = "cuda"
    # operands rounded to the operand format; channels the map must not read hold NaN
    x = torch.randn(n, h, w, cin, generator=g).to(dt)
    x16 = torch.full((n, h, w, ct), float("nan"), dtype=dt)
    x16[..., :cin] = x
    x16 = x16.to(dev)
    wscale = (0.25 if c["u8"] or c["clamp01"] else 1.0) / math.sqrt(9 * cin)
    wt = (torch.randn(cout, cin, 3, 3, generator=g) * wscale).to(dt).float().to(dev)
    b = (torch.randn(cout, generator=g) * 0.5).to(dev)
    if c["u8"] or c["clamp01"]:
        b += 0.5
    if c["big"]:   # fp16 outputs far beyond 65504 of both signs: the store must saturate
        b = torch.where(torch.arange(cout, device=dev) % 2 == 0, 9e4, -2e5).float() + b
    bufs = {"in16": x16, "weight": wt, "bias": b}
    inputs = [x16]

    lay = res_layout(c)
    r1 = r2 = None
    if lay:
        rdt = torch.float32 if lay["f32"] else (torch.bfloat16 if c["res"] == 1 else torch.float16)
        sl = slice(lay["choff"], lay["choff"] + cout)
        if lay["res1"]:
            t = torch.full((n, h, w, lay["cs"]), float("nan"), dtype=rdt)
            t[..., sl] = torch.randn(n, h, w, cout, generator=g).to(rdt)
            bufs["res1"] = t.to(dev)
            inputs.append(bufs["res1"])
            r1 = bufs["res1"][..., sl].double()
        if lay["res2"]:
            r2v = torch.randn(n, h, w, cout, generator=g).to(rdt)
            if c["inplace"]:
                out16 = NHWCOut(n, h, w, lay["cs2"], list(range(lay["choff"], lay["choff"] + cout)), rdt,
                                init=r2v.to(dev))
                bufs["res2"] = out16.t
            else:
                t = torch.full((n, h, w, lay["cs2"]), float("nan"), dtype=rdt)
                t[..., sl] = r2v
                bufs["res2"] = t.to(dev)
                inputs.append(bufs["res2"])
            r2 = r2v.double().to(dev)

    # outputs
    lsl = -(-cout // 32)
    outs = {}
    if c["o16"] is not None:
        f, cs, co = c["o16"]
        odt = torch.bfloat16 if f else torch.float16
        on = _slices_on(c, c["no16"])
        chans = sorted({co + (0 if c["fixed"] else 32 * s) + k for s in on for k in range(32)})
        hh, ww = (2 * h, 2 * w) if c["up2"] else (h, w)
        if c["inplace"]:
            outs["out16"] = out16
        else:
            outs["out16"] = NHWCOut(n, hh, ww, cs, chans, odt)
        bufs["out16"] = outs["out16"].t
    if c["outf"] is not None:
        cs, co = c["outf"]
        chans = [co + 32 * s + k for s in _slices_on(c, c["noutf"]) for k in range(32)]
        outs["outf"] = NHWCOut(n, h, w, cs, chans, torch.float32)
        bufs["outf"] = outs["outf"].t
    for k in ("nchw", "raw"):
        if c[k]:
            outs[k] = FlatOut((n, cout, h, w), torch.float32)
            bufs["out_nchw" if k == "nchw" else "out_nchw_raw"] = outs[k].t
    if c["u8"]:
        outs["u8"] = FlatOut((n, h, w, cout), torch.uint8)
        bufs["out_u8"] = outs["u8"].t
    inside = torch.ones(h, w, dtype=torch.float64, device=dev)
    if c["vmask"] is not None:
        s = c["vmask"]
        hl, wl, words = -(-h // (1 << s)), -(-w // (1 << s)), vmask_words(c)
        bits = torch.rand(hl, words * 32, generator=g) < 0.7
        bits[:, wl:] = False
        packed = np.packbits(bits.numpy(), axis=1, bitorder="little")   # bit x of a row is bit x % 32 of word x / 32
        bufs["vmask"] = torch.from_numpy(np.ascontiguousarray(packed).view(np.int32)).to(dev)
        inside = bits[:, :wl].repeat_interleave(1 << s, 0).repeat_interleave(1 << s, 1)[:h, :w].double().to(dev)
        inputs.append(bufs["vmask"])
    act = None
    if c["mask16"]:
        f = c["o16"][0]
        mdt = torch.bfloat16 if f else torch.float16
        m = torch.randn(n, h, w, cout, generator=g)
        sel = torch.randint(0, 4, m.shape, generator=g)
        m = torch.where(sel == 0, torch.zeros_like(m), torch.where(sel == 1, -torch.zeros_like(m), m))
        t = torch.full((n, h, w, cout + 16), float("nan"), dtype=mdt)
        t[..., 8:8 + cout] = m.to(mdt)
        bufs["mask16"] = t.to(dev)
        inputs.append(bufs["mask16"])
        mb = t[..., 8:8 + cout].view(torch.int16).int() & 0xFFFF
        act = (((mb & 0x8000) == 0) & ((mb & 0x7FFF) != 0)).to(dev)   # strictly positive: -0 and +0 are not
    snap = [t.clone() for t in inputs]

    d = desc(c, ptr=lambda name: bufs[name].data_ptr())
    prev = L.lib().resr_set_conv_pair_policy(policy)
    try:
        L.check(L.lib().resr_conv3x3(ctypes.byref(d), L.stream_ptr()))
    finally:
        L.lib().resr_set_conv_pair_policy(prev)
    torch.cuda.synchronize()
    for a, bb in zip(inputs, snap):
        assert torch.equal(_bits(a), _bits(bb)), f"{c['id']}: an input was modified"

    # ---- float64 reference
    import torch.nn.functional as F
    x64 = x.to(dev).double().permute(0, 3, 1, 2)
    w64, b64 = wt.double(), b.double()
    v = F.conv2d(x64, w64, b64, padding=1).permute(0, 2, 3, 1)
    S = F.conv2d(x64.abs(), w64.abs(), b64.abs(), padding=1).permute(0, 2, 3, 1)
    ch = torch.arange(cout, device=dev)
    ep = c["ep"]
    if r1 is not None:
        use1 = ((c["nores"] >> (ch // 32)) & 1) == 0
        if ep in (3, 4):
            v = torch.where(use1, v + r1, v)
            S = torch.where(use1, S + r1.abs(), S)
        else:
            v = torch.where(use1, C02 * v + r1, v)
            S = torch.where(use1, C02 * S + r1.abs(), S)
    if ep == 2:
        v, S = C02 * v + r2, C02 * S + r2.abs()
    if ep == 4:
        v, S = v + c["res2_scale"] * r2, S + abs(c["res2_scale"]) * r2.abs()
    if c["lrelu"]:
        v = torch.maximum(v, C02 * v)
    ins = inside.view(1, h, w, 1)
    v, S = v * ins, S * ins
    raw = v
    if c["clamp01"]:
        v = v.clamp(0, 1)
    tol = BOUND * S
    errs = []

    def close(got, ref, tol_, what):
        err = (got - ref).abs()
        bad = ~(err <= tol_)
        assert not bool(bad.any()), (f"{c['id']} policy {policy} {what}: {int(bad.sum())} elements off, worst "
                                     f"|err| {err.max().item():.3e} at tolerance {tol_.flatten()[err.flatten().argmax()].item():.3e}")
        return err

    def ratio(err, s):
        errs.append((err / s.clamp_min(1e-300)).max().item())

    if "outf" in outs:
        got = outs["outf"].check(c["id"] + " outf")
        on = [32 * s + k for s in _slices_on(c, c["noutf"]) for k in range(32)]
        ratio(close(got, v[..., on], tol[..., on], "outf"), S[..., on])
    if "out16" in outs:
        f = c["o16"][0]
        got = outs["out16"].check(c["id"] + " out16")
        ref, tol16 = v, tol
        if act is not None:
            ref = torch.where(act, ref, C02 * ref)
        if c["o16scale"]:
            ref, tol16 = ref * c["o16scale"], tol16 * abs(c["o16scale"])
        if f == 0:
            ref = ref.clamp(-F16_MAX, F16_MAX)
        on = _slices_on(c, c["no16"])
        if c["fixed"]:
            assert len(on) == 1
            idx = [32 * on[0] + k for k in range(32)]
        else:
            idx = [32 * s + k for s in on for k in range(32)]
        ref, tol16 = ref[..., idx], tol16[..., idx]
        if c["up2"]:
            got = got.view(n, h, 2, w, 2, len(idx)).permute(0, 1, 3, 2, 4, 5)
            ref, tol16 = ref[:, :, :, None, None, :], tol16[:, :, :, None, None, :]
        close(got, ref, tol16 + _half_ulp(ref.abs() + tol16, f), "out16")
        if c["big"]:
            assert bool((got.abs() <= F16_MAX).all()) and bool((got.abs() == F16_MAX).any()), "fp16 store did not saturate"
    if "nchw" in outs:
        got = outs["nchw"].check(c["id"] + " out_nchw").permute(0, 2, 3, 1)
        ratio(close(got, v, tol, "out_nchw"), S)
    if "raw" in outs:
        got = outs["raw"].check(c["id"] + " out_nchw_raw").permute(0, 2, 3, 1)
        ratio(close(got, raw, tol, "out_nchw_raw"), S)
    if "u8" in outs:
        got = outs["u8"].check(c["id"] + " out_u8")
        # the kernel truncates fl(255 v') for a v' within tol of the reference: exact unless an integer lies within
        # e of 255 ref, and then either neighbour of that integer boundary
        t = 255.0 * v
        e = 255.0 * tol + 2.0 ** -14
        ok = (got >= torch.floor(t - e).clamp(0, 255)) & (got <= torch.floor(t + e).clamp(0, 255))
        bad = [(tuple(i), got[tuple(i)].item(), t[tuple(i)].item(), 255.0 * tol[tuple(i)].item())
               for i in (~ok).nonzero()[:4].tolist()]
        assert bool(ok.all()), f"{c['id']} policy {policy} out_u8: {int((~ok).sum())} values off (index, got, 255 ref, 255 tol): {bad}"
    # canvas: every output of an invalid pixel is exactly 0
    if c["vmask"] is not None:
        outside = inside == 0
        for k, o in outs.items():
            t = o.t.double() if k != "out16" or not c["up2"] else None
            if t is None:
                continue
            if k in ("nchw", "raw"):
                t = t.permute(0, 2, 3, 1)
            if k in ("out16", "outf"):
                t = t[..., o.chans]
            assert bool((t[:, outside] == 0).all()), f"{c['id']} {k}: a masked-out pixel is not 0"
    if report and errs:
        with open(report, "a") as fh:
            fh.write(json.dumps({"id": c["id"], "policy": policy, "plan": tag(plan_of(d, _sms(), policy)),
                                 "max_err_over_S": max(errs)}) + "\n")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_conv_path(c):
    sms = _sms()
    d = desc(c)
    plan = plan_of(d, sms, c["policy"])
    assert plan is not None, f"{c['id']}: rejected by the planner ({_L().lib().resr_last_error()})"
    assert tag(plan) == c["want"], f"{c['id']}: planned as {tag(plan)}, the case means {c['want']}"
    if c["lap"]:
        assert laps(plan, c["h"]), f"{c['id']}: no accumulator ring lap at {sms} SMs ({cta_accumulators(plan.units, plan.clusters, c['h'])[:4]})"
    report = os.environ.get("RESR_CONV_PATHS_REPORT")
    seen = set()
    for policy in (0, 1, 2):
        pl = plan_of(d, sms, policy)
        if pl is None:      # e.g. a cin only the pair kernel's halved weights fit: the single kernel rejects it
            continue
        key = (tag(pl), pl.nslices, pl.nstages, pl.units, pl.clusters)
        if key in seen:
            continue
        seen.add(key)
        _run_case(c, policy, report)
