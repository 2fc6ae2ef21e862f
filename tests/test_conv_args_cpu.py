"""CPU: the planner of the tcgen05 3x3 convolution (resr_conv3x3_plan, host only) and the argument checks of resr_conv3x3.

Every rejected descriptor must return RESR_E_INVALID from both entry points before any device work: the pointers are
dummies that are never dereferenced, and a check that let a call through to a launch would fail here with RESR_E_CUDA
(no device) instead. resr_conv3x3 is only called with a descriptor the planner has already rejected, so that on a
machine with a GPU no dummy pointer can reach a kernel.

test_every_configuration_has_a_case evaluates the planner over the case table of test_conv_paths_gpu.py and requires
every value of each configuration axis the planner can produce (found by sweeping it over shapes, channel counts and
outputs) to appear in some case."""
import ctypes
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_conv_paths_gpu as paths  # noqa: E402

INVALID = 1
SMS = 148  # B200
C = paths.C


@pytest.fixture(scope="module")
def lib():
    import resr_b200
    return resr_b200._lib.lib()


def _plan(d, policy=2, sms=SMS):
    return paths.plan_of(d, sms, policy)


BASE = dict(n=2, h=8, w=64, cin=64, cout=64, outf=(64, 0), o16=(1, 64, 0))


def _bad(**kw):
    """The base case with the fields of `kw` overridden (case keys), plus raw descriptor fields under `raw`."""
    raw = kw.pop("raw", {})
    c = C("bad", "", **{**BASE, **kw})
    d = paths.desc(c)
    for k, v in raw.items():
        setattr(d, k, v)
    return d


REJECTED = {
    "n0": _bad(n=0), "h-1": _bad(h=-1), "w0": _bad(w=0), "cout0": _bad(cout=0, outf=None, o16=None, nchw=1),
    "cin0": _bad(raw={"cin": 0}), "cin-5": _bad(raw={"cin": -5}),
    "ctotal-not-8": _bad(c_total=68), "cin>ctotal": _bad(cin=72, c_total=64),
    "ctotal<round64(cin)": _bad(cin=65, c_total=72),
    "fmt_in2": _bad(fmt=2), "mode2": _bad(mode=2), "mode-2": _bad(mode=-2),
    "ep5": _bad(ep=5), "ep-1": _bad(ep=-1),
    "ep1-no-res1": _bad(ep=1), "ep2-no-res2": _bad(ep=2, res="f32", raw={"res2": None}),
    "ep2-no-res1": _bad(ep=2, res="f32", raw={"res1": None}), "ep3-no-res1": _bad(ep=3),
    "ep4-no-res2": _bad(ep=4, res="f32", raw={"res2": None}), "ep4-res16": _bad(ep=4, res=1),
    "res16-2": _bad(ep=1, res=1, raw={"res16": 2}), "res16_fmt2": _bad(ep=1, res=1, raw={"res16_fmt": 2}),
    # cout % 32 != 0 with an NHWC output: the stores write whole 32-channel slices
    "cout48-out16": _bad(cout=48, outf=None, o16=(1, 192, 0)), "cout48-outf": _bad(cout=48, outf=(192, 0), o16=None),
    "cout3-out16": _bad(cout=3, outf=None, o16=(1, 64, 0)), "cout3-outf": _bad(cout=3, outf=(64, 0), o16=None),
    "cout3-res1": _bad(cout=3, outf=None, o16=None, nchw=1, ep=3, res="f32"),
    "out16-choff+cout>cstride": _bad(o16=(1, 64, 8)), "outf-choff+cout>cstride": _bad(outf=(64, 4)),
    "out16-choff<0": _bad(o16=(1, 128, -8)), "outf-choff<0": _bad(outf=(128, -4)),
    "out16-cstride%8": _bad(o16=(1, 68, 0)), "outf-cstride%4": _bad(outf=(66, 0)),
    "out16_fmt2": _bad(o16=(2, 64, 0)), "up2-2": _bad(up2=2),
    "slice-fixed-past-cstride": _bad(o16=(1, 64, 40), fixed=1),
    "out_nchw_c!=cout": _bad(outf=None, o16=None, nchw=1, raw={"out_nchw_c": 3}),
    "out_u8_c!=cout": _bad(cout=3, outf=None, o16=None, u8=1, raw={"out_nchw_c": 4}),
    "raw_c!=cout": _bad(cout=3, outf=None, o16=None, raw={"out_nchw_raw": paths.P, "out_nchw_c": 0}),
    "res1-fp32-choff%4": _bad(ep=1, res="f32", raw={"res_choff": 2}),
    "res1-16bit-choff%8": _bad(ep=1, res=1, raw={"res_choff": 4}),
    "res1-fp32-cstride%4": _bad(ep=1, res="f32", raw={"res_cstride": 102}),
    "res1-past-cstride": _bad(ep=1, res="f32", raw={"res_choff": 48}),
    "res2-past-cstride": _bad(ep=2, res="f32", raw={"res2_cstride": 64}),
    "res2-cstride%4": _bad(ep=4, res="f32-res2", raw={"res2_cstride": 118}),
    "mask16-choff%8": _bad(mask16=1, raw={"mask16_choff": 4}),
    "mask16-past-cstride": _bad(mask16=1, raw={"mask16_cstride": 64}),
    "vmask-words": _bad(w=200, vmask=0, raw={"vmask_words": 6}),
    "vmask-shift": _bad(vmask=0, raw={"vmask_shift": -1}),
    "null-in16": _bad(raw={"in16": None}), "null-weight": _bad(raw={"weight": None}),
}


@pytest.mark.parametrize("name", sorted(REJECTED))
def test_conv3x3_rejects(lib, name):
    d = REJECTED[name]
    pl = paths._L().ConvPlan()
    assert lib.resr_conv3x3_plan(ctypes.byref(d), SMS, ctypes.byref(pl)) == INVALID, name
    assert lib.resr_conv3x3(ctypes.byref(d), None) == INVALID, name


def test_base_descriptor_is_accepted(lib):
    """The descriptor every rejection above perturbs is itself valid (so each rejection is the perturbed field's)."""
    assert _plan(_bad()) is not None
    assert _plan(_bad(ep=2, res="f32")) is not None and _plan(_bad(mask16=1)) is not None
    assert _plan(_bad(w=200, vmask=0)) is not None and _plan(_bad(cout=48, outf=None, o16=None, nchw=1)) is not None
    pl = paths._L().ConvPlan()
    assert lib.resr_conv3x3_plan(ctypes.byref(_bad()), 0, ctypes.byref(pl)) == INVALID   # no SMs
    assert lib.resr_conv3x3_plan(ctypes.byref(_bad()), SMS, None) == INVALID


@pytest.mark.parametrize("c", [c for c in paths.CASES if c["id"].startswith("cinmax")], ids=lambda c: c["id"])
def test_largest_cin_is_the_planners_limit(lib, c):
    """The largest-cin cases sit exactly at the limit: one input channel more does not fit in shared memory and is
    rejected with RESR_E_INVALID before any device work."""
    assert _plan(paths.desc(c), c["policy"]) is not None
    more = dict(c, cin=c["cin"] + 1, c_total=c["c_total"] + 64)
    d = paths.desc(more)
    assert _plan(d, c["policy"]) is None
    prev = lib.resr_set_conv_pair_policy(c["policy"])
    try:
        assert lib.resr_conv3x3(ctypes.byref(d), None) == INVALID
    finally:
        lib.resr_set_conv_pair_policy(prev)


def test_plan_follows_the_pair_policy_and_the_grid_formula(lib):
    d = paths.desc(C("p", "", n=3, h=40, w=128, cout=64))
    single, pair = _plan(d, 0), _plan(d, 2)
    assert (single.pair, single.nout, single.nslices) == (0, 32, 2)
    assert (pair.pair, pair.nout, pair.nslices) == (1, 64, 1)
    assert single.units == 3 * 40 and pair.units == 2 * 40   # (column group, row) / (column-group pair, row)
    assert single.clusters == min(SMS // 2, -(-120 // 4)) and pair.clusters == min(SMS // 2, -(-80 // 4))
    assert _plan(d, 1).pair == 0                              # policy 1: 80 pair rows are too few to pay off
    assert lib.resr_set_conv_pair_policy(-1) == lib.resr_set_conv_pair_policy(-1)   # planning left the policy alone
    m = _plan(paths.desc(C("m", "", h=20, w=256, vmask=1)), 2)
    assert m.masked == 1 and (m.ncg, m.nxs, m.bw, m.bn) == (2, 2, 128, 1)


# ============================================================================================== coverage
def _axes(plan, c):
    k = "pair" if plan.pair else "single"
    out = {("kernel", k, plan.nout, plan.bn), ("mode", k, plan.mode), ("tail", k, plan.tail_ksteps),
           ("epi", k, plan.nout, plan.nepi, plan.epi_bufs)}
    if plan.pair:
        out.add(("reverse", plan.nout, c["reverse"]))
    if plan.masked:
        out.add(("masked", k, plan.nout))
    if c["h"] > 1 and paths.laps(plan, c["h"]):
        out.add(("lap", k, plan.nout))
    return out


def _reachable():
    """Every axis value the planner produces, from sweeps over the inputs it decides on."""
    want = set()

    def add(c, policies=(0, 2)):
        for p in policies:
            pl = _plan(paths.desc(c), p)
            if pl is not None:
                k = "pair" if pl.pair else "single"
                want.update({("kernel", k, pl.nout, pl.bn), ("mode", k, pl.mode), ("tail", k, pl.tail_ksteps),
                             ("epi", k, pl.nout, pl.nepi, pl.epi_bufs), ("masked", k, pl.nout), ("lap", k, pl.nout)})
                if pl.pair:
                    want.update({("reverse", pl.nout, 0), ("reverse", pl.nout, 1)})

    for cout in (3, 32, 64, 96):
        for w in (1, 8, 16, 32, 64, 128, 200):
            bn = 128 // w if w in (8, 16, 32, 64) else 1
            for mode in (-1, 0, 1):
                add(C("s", "", n=2 * bn + 1, w=w, cout=cout, mode=mode))
        for cin in range(1, 129):
            add(C("s", "", n=2, cin=cin, cout=cout))
        outs = [dict(nchw=1)] if cout % 32 else [dict(outf=(cout, 0)), dict(o16=(1, cout, 0)),
                                                  dict(outf=(cout, 0), o16=(1, cout, 0))]
        for o in outs:
            for k in range(1, 40):
                add(C("s", "", n=2, cin=64 * k, cout=cout, **o))
    return want


def test_every_configuration_has_a_case():
    seen = set()
    for c in paths.CASES:
        d = paths.desc(c)
        for policy in (0, 1, 2):
            pl = _plan(d, policy)
            if pl is not None:
                seen |= _axes(pl, c)
    missing = _reachable() - seen
    assert not missing, sorted(missing)


def test_case_ids_are_unique():
    ids = [c["id"] for c in paths.CASES]
    assert len(ids) == len(set(ids))


def test_bound_catches_one_dropped_product():
    """The 2^-16 S tolerance of test_conv_paths_gpu.py is tight enough to see a single lost (channel, tap) product at
    one pixel: at cin = 192 the term is on average S / (9 cin), ~38x the bound, and nearly every one exceeds it."""
    g = torch.Generator().manual_seed(5)
    cin, cout = 192, 8
    x = torch.randn(1, cin, 6, 6, generator=g).bfloat16().double()
    w = (torch.randn(cout, cin, 3, 3, generator=g) / (9 * cin) ** 0.5).bfloat16().double()
    b = torch.randn(cout, generator=g).double() * 0.5
    S = torch.nn.functional.conv2d(x.abs(), w.abs(), b.abs(), padding=1)[0, :, 3, 3]   # an interior pixel
    terms = (x[0, :, 2:5, 2:5][None] * w).abs()                                         # [cout, cin, 3, 3]
    ratio = terms / (paths.BOUND * S[:, None, None, None])
    assert ratio.mean().item() > 30
    assert (ratio > 1).double().mean().item() > 0.9
