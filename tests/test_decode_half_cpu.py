"""Argument checks of the 16-bit head modes of yolo_b200_decode_compact_ex (YOLO_B200_VARIANT_F16 / _BF16).  They return
before any CUDA call, so they run without a GPU.  The device pointers below are never dereferenced."""

import pytest

from pytorch_yolo_b200 import _lib

E_RANGE, E_ALIGN, E_UNSUPPORTED = -2, -3, -5
F16, BF16 = _lib.VARIANT_F16, _lib.VARIANT_BF16


def call(variant, head=0x10000):
    lib = _lib.load()
    arr = (_lib.Scale * 1)()
    s = arr[0]
    s.head, s.ny, s.nx, s.na, s.row_off, s.stride = head, 8, 8, 1, 0, 8.0
    fake = 0x20000                                  # 16-byte aligned, never touched
    return lib.yolo_b200_decode_compact_ex(arr, 1, 1, 1, 64, 0.3, 2.0, fake, fake + 0x1000, 64, fake + 0x2000,
                                           fake + 0x2000 + 4, variant, None)


def test_bits_match_the_header():
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "yolo_b200.h")).read()
    bits = dict(re.findall(r"#define (YOLO_B200_VARIANT_\w+) (0x[0-9a-f]+)", header))
    assert int(bits["YOLO_B200_VARIANT_F16"], 16) == F16
    assert int(bits["YOLO_B200_VARIANT_BF16"], 16) == BF16
    assert int(bits["YOLO_B200_VARIANT_ACCUMULATE"], 16) == _lib.VARIANT_ACCUMULATE


@pytest.mark.parametrize("variant", [0, 1, 4])
def test_both_bits_is_a_range_error(variant):
    assert call(variant | F16 | BF16) == E_RANGE
    assert call(variant | F16 | BF16 | _lib.VARIANT_ACCUMULATE) == E_RANGE


@pytest.mark.parametrize("bit", [F16, BF16])
@pytest.mark.parametrize("variant", [2, 3])
def test_tma_variants_are_unsupported(bit, variant):
    assert call(variant | bit) == E_UNSUPPORTED
    assert call(variant | bit | _lib.VARIANT_ACCUMULATE) == E_UNSUPPORTED


@pytest.mark.parametrize("bit", [F16, BF16])
@pytest.mark.parametrize("variant", [0, 1, 4])
def test_odd_head_address_is_an_alignment_error(bit, variant):
    assert call(variant | bit, head=0x10001) == E_ALIGN


def test_fp32_still_needs_four_byte_alignment():
    assert call(0, head=0x10002) == E_ALIGN


def test_unknown_variant_is_still_a_range_error():
    assert call(5 | F16) == E_RANGE
    assert call(0x800) == E_RANGE
