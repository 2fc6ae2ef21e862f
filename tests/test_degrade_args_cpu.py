"""CPU: every degradation entry point of the C ABI rejects bad arguments on the host, before it touches the device.

Each call below must return RESR_E_INVALID (or RESR_E_NOMEM for a short workspace) without a GPU. The pointers are
dummies that are never dereferenced, so a check that let a call through to a launch would fail here with RESR_E_CUDA
(no device) instead of RESR_E_INVALID."""
import pytest

INVALID, NOMEM = 1, 3
P = 0x1000  # non-null dummy device pointer; never reached by a rejected call
BIG = 1 << 40  # workspace bytes large enough for any shape below


@pytest.fixture(scope="module")
def lib():
    import resr_b200
    return resr_b200._lib.lib()


@pytest.mark.parametrize("b, c, h, w, k, kb", [
    (1, 3, 32, 32, 4, 1),      # even k: "Wrong kernel size." (imgproc.py:1106)
    (1, 3, 32, 32, 0, 1),
    (1, 3, 32, 32, -3, 1),
    (1, 3, 100, 100, 65, 1),   # k > 63
    (1, 3, 10, 32, 21, 1),     # k / 2 >= h
    (1, 3, 32, 10, 21, 1),     # k / 2 >= w
    (1, 3, 0, 32, 1, 1),
    (0, 3, 32, 32, 3, 1),      # b <= 0
    (-1, 3, 32, 32, 3, 1),
    (2, 0, 32, 32, 3, 1),      # c <= 0
    (2, -3, 32, 32, 3, 2),
    (2, 3, 32, 32, 3, 3),      # kernel batch neither 1 nor b
])
def test_filter2d_rejects(lib, b, c, h, w, k, kb):
    assert lib.resr_filter2d(P, P, P, b, c, h, w, k, kb, None) == INVALID


@pytest.mark.parametrize("b, c, h, w, radius", [
    (1, 3, 512, 512, 130),     # 131 taps > 129
    (1, 3, 512, 512, 200),
    (1, 3, 25, 64, 50),        # 51 taps: reflect padding 25 needs h, w > 25
    (1, 3, 64, 25, 50),
    (1, 3, 3, 64, 7),
    (0, 3, 64, 64, 50),
    (1, 0, 64, 64, 50),
])
def test_usm_rejects(lib, b, c, h, w, radius):
    assert lib.resr_usm_sharp(P, P, b, c, h, w, radius, 0, 0.5, 10.0, P, BIG, None) == INVALID
    assert lib.resr_usm_sharp_backward(P, P, P, b, c, h, w, radius, 0, 0.5, 10.0, P, BIG, None) == INVALID


def test_usm_short_workspace(lib):
    need = lib.resr_usm_workspace_bytes(2, 3, 64, 64)
    assert need == 2 * 3 * 64 * 64 * 4 * 3
    assert lib.resr_usm_sharp(P, P, 2, 3, 64, 64, 50, 0, 0.5, 10.0, P, need - 1, None) == NOMEM
    need_b = lib.resr_usm_backward_workspace_bytes(2, 3, 64, 64)
    assert lib.resr_usm_sharp_backward(P, P, P, 2, 3, 64, 64, 50, 0, 0.5, 10.0, P, need_b - 1, None) == NOMEM
    assert lib.resr_usm_sharp(P, P, 2, 3, 64, 64, 50, 0, 0.5, 10.0, None, BIG, None) == INVALID


@pytest.mark.parametrize("planes, hi, wi, ho, wo, mode", [
    (3, 32, 32, 16, 16, 3),    # bad mode
    (3, 32, 32, 16, 16, -1),
    (3, 32, 32, 0, 16, 1),     # h_out / w_out <= 0
    (3, 32, 32, 16, -2, 2),
    (3, 0, 32, 16, 16, 0),     # h_in / w_in / planes <= 0
    (3, 32, 0, 16, 16, 1),
    (3, -4, 32, 16, 16, 2),
    (0, 32, 32, 16, 16, 1),
    (-3, 32, 32, 16, 16, 0),
])
def test_resize_rejects(lib, planes, hi, wi, ho, wo, mode):
    assert lib.resr_resize(P, P, planes, hi, wi, ho, wo, mode, 0.0, 0.0, None) == INVALID


@pytest.mark.parametrize("dumps", [(P, 0, 0), (0, P, 0), (0, 0, P), (P, P, 0), (P, 0, P), (0, P, P)])
def test_jpeg_rejects_partial_coefficient_dumps(lib, dumps):
    assert lib.resr_jpeg(P, P, P, P, 1, 16, 16, 0, *dumps, None) == INVALID


@pytest.mark.parametrize("b, h, w", [(0, 16, 16), (-1, 16, 16), (1, 0, 16), (1, 16, 0), (2, -8, 16), (2, 16, -8)])
def test_jpeg_rejects_empty_images(lib, b, h, w):
    assert lib.resr_jpeg(P, P, P, P, b, h, w, 0, None, None, None, None) == INVALID
    assert lib.resr_jpeg(P, P, P, P, b, h, w, 1, P, P, P, None) == INVALID


@pytest.mark.parametrize("planes, hi, wi, top, left, ho, wo", [
    (3, 32, 32, -1, 0, 8, 8),      # window out of range
    (3, 32, 32, 0, -1, 8, 8),
    (3, 32, 32, 25, 0, 8, 8),
    (3, 32, 32, 0, 25, 8, 8),
    (3, 32, 32, 0, 0, 33, 32),
    (3, 32, 32, 0, 0, 0, 8),       # h_out / w_out <= 0
    (3, 32, 32, 0, 0, 8, 0),
    (3, 32, 32, 4, 4, -2, 8),
    (0, 32, 32, 0, 0, 8, 8),       # planes <= 0
])
def test_crop_rejects(lib, planes, hi, wi, top, left, ho, wo):
    for round_to_u8 in (0, 1):
        assert lib.resr_crop(P, P, planes, hi, wi, top, left, ho, wo, round_to_u8, None) == INVALID


def test_null_pointers_are_rejected(lib):
    assert lib.resr_filter2d(P, None, P, 1, 3, 32, 32, 3, 1, None) == INVALID
    assert lib.resr_resize(None, P, 3, 32, 32, 16, 16, 1, 0.0, 0.0, None) == INVALID
    assert lib.resr_jpeg(P, P, None, P, 1, 16, 16, 0, None, None, None, None) == INVALID
    assert lib.resr_crop(P, None, 3, 32, 32, 0, 0, 8, 8, 0, None) == INVALID
