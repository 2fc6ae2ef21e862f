"""CPU: libresr.so loads, exports exactly the symbols include/resr.h declares, and refuses to compute without a GPU
(no CPU fallback). Also host-side logic that needs no device."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "resr.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(resr_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported_and_bound():
    import resr_b200
    L = resr_b200._lib
    lib = L.lib()
    declared = _declared()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/resr.h but not exported by libresr.so"
    assert sorted(L.SIGNATURES) == declared, "ctypes SIGNATURES and include/resr.h disagree"


def test_ctypes_argument_counts_and_kinds_match_the_header():
    """Every prototype of include/resr.h against the ctypes signature table: same number of parameters, pointers bound as
    pointers, integers / floats / size_t as such (ctypes would pass a wrong list silently)."""
    import resr_b200
    L = resr_b200._lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "resr.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    protos = dict(re.findall(r"\b(resr_[a-z0-9_]+)\s*\(([^;{}]*?)\)\s*;", hdr, flags=re.S))
    checked = 0
    for name, (res, args) in L.SIGNATURES.items():
        params = [a.strip() for a in protos[name].replace("\n", " ").split(",")]
        if params == ["void"] or params == [""]:
            params = []
        assert len(params) == len(args), f"{name}: header has {len(params)} parameters, ctypes binds {len(args)}"
        for decl, ct in zip(params, args):
            is_ptr_h = "*" in decl
            is_ptr_c = ct in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(ct, "contents") or getattr(ct, "_type_", None) not in (
                "i", "f", "d", "l", "q", "L", "Q", "I")
            if is_ptr_h:
                assert is_ptr_c, f"{name}: '{decl}' is a pointer in the header, bound as {ct}"
            else:
                assert not (ct in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(ct, "contents")), f"{name}: '{decl}' bound as a pointer"
                if decl.startswith(("float", "double")):
                    assert ct in (ctypes.c_float, ctypes.c_double), f"{name}: '{decl}' bound as {ct}"
                    assert (ct is ctypes.c_double) == decl.startswith("double"), f"{name}: '{decl}' bound as {ct}"
                elif decl.startswith("size_t"):
                    assert ct is ctypes.c_size_t, f"{name}: '{decl}' bound as {ct}"
                elif decl.startswith(("unsigned long long", "long long")):
                    assert ctypes.sizeof(ct) == 8, f"{name}: '{decl}' bound as {ct}"
                else:
                    assert ct is ctypes.c_int, f"{name}: '{decl}' bound as {ct}"
            checked += 1
    assert checked > 250


def test_abi_constants():
    import resr_b200
    lib = resr_b200._lib.lib()
    assert lib.resr_version() >= 1
    assert lib.resr_generator_num_params() == 16697987
    assert lib.resr_generator_num_tensors() == 702
    off, cnt = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.resr_generator_tensor_span(0, ctypes.byref(off), ctypes.byref(cnt)) == 0
    assert (off.value, cnt.value) == (0, 64 * 3 * 9)
    assert lib.resr_generator_tensor_span(701, ctypes.byref(off), ctypes.byref(cnt)) == 0
    assert off.value + cnt.value == 16697987 and cnt.value == 3
    assert lib.resr_generator_tensor_span(702, ctypes.byref(off), ctypes.byref(cnt)) != 0
    # cfg3 workspace: fp16 input + 3 concat buffers (192 ch) + fp32 skip copy + 2x / 4x tail activations
    px = 64 * 128 * 128
    assert lib.resr_generator_workspace_bytes(64, 128, 128) == px * (64 * 2 + 3 * 192 * 2 + 64 * 4 + 4 * 64 * 2 + 3 * 16 * 64 * 2)
    assert lib.resr_generator_workspace_bytes(0, 1, 1) == 0


def test_tensor_spans_follow_state_dict_order():
    import resr_b200
    lib = resr_b200._lib.lib()
    g = resr_b200.model.Generator(3, 3, 4)
    off, cnt = ctypes.c_size_t(), ctypes.c_size_t()
    pos = 0
    for i, (name, p) in enumerate(g.named_parameters()):
        assert lib.resr_generator_tensor_span(i, ctypes.byref(off), ctypes.byref(cnt)) == 0
        assert (off.value, cnt.value) == (pos, p.numel()), name
        pos += p.numel()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    import resr_b200
    L = resr_b200._lib
    h = ctypes.c_void_p()
    rc = L.lib().resr_generator_create(ctypes.byref(h), 3, 3, 4)
    assert rc == 2, "without a CUDA device creation must fail with RESR_E_CUDA"
    assert b"CUDA" in L.lib().resr_last_error() or b"device" in L.lib().resr_last_error()
    g = resr_b200.model.Generator(3, 3, 4)
    with pytest.raises(L.ResrError):
        g(torch.rand(1, 3, 8, 8))
    with pytest.raises(L.ResrError):
        resr_b200.imgproc.filter2d_torch(torch.rand(1, 3, 32, 32), torch.ones(1, 3, 3) / 9)


def test_generator_mirror_matches_reference_layout():
    import resr_b200
    from oracle import generator as og
    torch.manual_seed(3)
    g = resr_b200.model.Generator(3, 3, 4)
    sd = og.random_state_dict(3)
    msd = g.state_dict()
    assert list(msd.keys()) == list(sd.keys())
    assert all(torch.equal(msd[k], sd[k]) for k in sd)  # same init, same RNG consumption order as the reference
    with pytest.raises(ValueError):
        resr_b200.model.Generator(3, 3, 2)
    with pytest.raises(ValueError):
        resr_b200.imgproc.filter2d_torch(torch.rand(1, 3, 8, 8), torch.ones(1, 4, 4))


def test_invalid_arguments_are_rejected():
    import resr_b200
    L = resr_b200._lib
    h = ctypes.c_void_p()
    assert L.lib().resr_generator_create(ctypes.byref(h), 3, 3, 2) == 1  # RESR_E_INVALID before touching the device
    assert b"Generator(3, 3, 4)" in L.lib().resr_last_error()
    assert L.lib().resr_filter2d(None, None, None, 1, 3, 8, 8, 3, 1, None) == 1


def test_tile_plan_is_an_exact_integer_cover():
    import numpy as np
    import resr_b200
    for (h, w, th, tw, halo) in [(2048, 2048, 512, 1024, 16), (72, 200, 32, 128, 16), (100, 100, 64, 64, 8)]:
        cover = np.zeros((h, w), np.int32)
        for (y0, y1, x0, x1, wy0, wy1, wx0, wx1) in resr_b200.model.plan_tiles(h, w, th, tw, halo):
            cover[y0:y1, x0:x1] += 1
            assert wy0 == max(y0 - halo, 0) and wy1 == min(y1 + halo, h) and wx0 == max(x0 - halo, 0) and wx1 == min(x1 + halo, w)
        assert (cover == 1).all()
    assert len(resr_b200.model.plan_tiles(2048, 2048, 512, 1024, 16)) == 8


def test_pod_plan_layout_matches_the_header(tmp_path):
    """ctypes mirrors of the POD structs in include/resr.h have the C compiler's size and field offsets."""
    import shutil
    import subprocess
    import resr_b200
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    L = resr_b200._lib
    src = tmp_path / "sz.c"
    src.write_text('''#include <stdio.h>
#include <stddef.h>
#include "resr.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(resr_degrade_plan), sizeof(resr_resize_spec),
           sizeof(resr_noise_spec), offsetof(resr_degrade_plan, noise1), offsetof(resr_degrade_plan, rng_state),
           sizeof(resr_conv_desc), sizeof(resr_kernel_params), offsetof(resr_conv_desc, out16_scale),
           offsetof(resr_conv_desc, out16_slice_fixed), sizeof(resr_conv_plan), offsetof(resr_conv_plan, units));
    return 0;
}
''')
    exe = tmp_path / "sz"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    subprocess.run(["gcc", "-I", inc, str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [ctypes.sizeof(L.DegradePlan), ctypes.sizeof(L.ResizeSpec), ctypes.sizeof(L.NoiseSpec), L.DegradePlan.noise1.offset,
            L.DegradePlan.rng_state.offset, ctypes.sizeof(L.ConvDesc), ctypes.sizeof(L.KernelParams),
            L.ConvDesc.out16_scale.offset, L.ConvDesc.out16_slice_fixed.offset, ctypes.sizeof(L.ConvPlan),
            L.ConvPlan.units.offset]
    assert got == want


def test_patch_reference_rebinds_the_three_names_without_touching_call_sites():
    """compat.patch_reference: `model`, `imgproc`, `F` of a reference-script namespace point at the mirrors; F keeps
    every torch.nn.functional attribute and only reroutes the interpolate calls the degradation block makes."""
    import types
    import torch.nn.functional as F
    import resr_b200
    ns = types.SimpleNamespace(model=object(), imgproc=object(), F=F, np=None)
    assert resr_b200.patch_reference(ns) == ["model", "imgproc", "F"]
    assert ns.model is resr_b200.model and ns.imgproc is resr_b200.imgproc
    assert ns.F.leaky_relu is F.leaky_relu and ns.F.l1_loss is F.l1_loss
    x = torch.rand(1, 3, 8, 10)
    for kw in (dict(scale_factor=2, mode="nearest"), dict(size=(5, 7), mode="bicubic"), dict(scale_factor=0.5, mode="area")):
        assert torch.equal(ns.F.interpolate(x, **kw), F.interpolate(x, **kw))  # CPU tensors fall through to torch
    d = {"F": F, "imgproc": 1}
    assert resr_b200.patch_reference(d) == ["imgproc", "F"] and "model" not in d


def test_param_version_key_sees_data_swaps():
    """ADVICE r01: the repack key must change when `param.data` is re-pointed (which does not bump `_version`)."""
    import resr_b200
    g = resr_b200.model.Generator(3, 3, 4)
    v0 = g._param_version()
    p = list(g.parameters())[10]
    old = p.data
    p.data = old.clone()
    v1 = g._param_version()
    assert v1 != v0
    p.data = old
    assert g._param_version() == v0
    with torch.no_grad():
        p.mul_(1.0)
    assert g._param_version() != v0


def test_gradient_bucket_offsets_follow_state_dict_order():
    """resr_generator_grad_buckets (host-only): the flat gradient vector is cut at trunk.5 / trunk.11 / trunk.17."""
    import ctypes
    import resr_b200
    g = resr_b200.model.Generator(3, 3, 4)
    offs = (ctypes.c_size_t * 5)()
    assert resr_b200._lib.lib().resr_generator_grad_buckets(offs, 5) == 4
    pos, want = 0, {}
    for k, v in g.state_dict().items():
        if k in ("trunk.5.rdb1.conv1.weight", "trunk.11.rdb1.conv1.weight", "trunk.17.rdb1.conv1.weight"):
            want[k] = pos
        pos += v.numel()
    assert [int(o) for o in offs] == [0, want["trunk.5.rdb1.conv1.weight"], want["trunk.11.rdb1.conv1.weight"],
                                      want["trunk.17.rdb1.conv1.weight"], pos]
    assert resr_b200._lib.lib().resr_niqe_num_blocks(200, 304, 4, 96) == 6 and resr_b200._lib.lib().resr_niqe_num_blocks(90, 200, 0, 96) == 0
