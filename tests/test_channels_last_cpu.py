"""channels_last (NHWC) heads and feature maps without a GPU: the flag values, every argument check of the NHWC modes of
yolo_b200_decode_compact_ex and yolo_b200_head_decode_compact (they return before any CUDA call; the device pointers below
are never dereferenced), the geometry yolo_b200_head_supported_ex accepts for NHWC feature maps, and the layout test of
ops.is_channels_last on CPU tensors."""
import ctypes as C
import os
import re

import pytest
import torch

from pytorch_yolo_b200 import _lib, ops

E_RANGE, E_ALIGN, E_UNSUPPORTED = -2, -3, -5
NHWC, HEAD_NHWC = _lib.VARIANT_NHWC, _lib.HEAD_NHWC
ANCHORS = [(10, 13), (16, 30), (33, 23)]
FEATURE_BITS = [0, _lib.HEAD_F16, _lib.HEAD_BF16]


def decode_call(variant, head=0x10000):
    lib = _lib.load()
    arr = (_lib.Scale * 1)()
    s = arr[0]
    s.head, s.ny, s.nx, s.na, s.row_off, s.stride = head, 8, 8, 1, 0, 8.0
    fake = 0x20000                                  # 16-byte aligned, never touched
    return lib.yolo_b200_decode_compact_ex(arr, 1, 1, 1, 64, 0.3, 2.0, fake, fake + 0x1000, 64, fake + 0x2000,
                                           fake + 0x2000 + 4, variant, None)


def head_call(flags, c_in=64, ny=8, nx=8, pitch=0, x=0x10000, weight=0x20000):
    lib = _lib.load()
    arr = (_lib.Head * 1)()
    bias = (C.c_float * 255)()
    h = arr[0]
    h.x, h.weight, h.bias_host, h.head_out = x, weight, bias, None
    h.c_in, h.x_row_pitch, h.negative_slope = c_in, pitch, 0.1
    s = h.scale
    s.ny, s.nx, s.na, s.row_off, s.stride = ny, nx, 3, 0, 8.0
    fake = 0x40000
    return lib.yolo_b200_head_decode_compact(arr, 1, 1, 80, 3 * ny * nx, 0.3, 2.0, fake, fake + 0x1000, 64, fake + 0x2000,
                                             fake + 0x2000 + 4, flags, None)


def supported(c_in, ny, nx, flags, pitch=0, nc=80, na=3):
    return _lib.load().yolo_b200_head_supported_ex(c_in, ny, nx, pitch, na, nc, flags)


def test_bits_match_the_header():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "yolo_b200.h")).read()
    variant = {k: int(v, 0) for k, v in re.findall(r"#define (YOLO_B200_VARIANT_\w+)\s+(0x[0-9a-fA-F]+)", header)}
    head = {k: int(v, 0) for k, v in re.findall(r"#define (YOLO_B200_HEAD_\w+)\s+(0x[0-9a-fA-F]+|\d+)", header)}
    assert variant["YOLO_B200_VARIANT_NHWC"] == NHWC == 0x1000
    assert head["YOLO_B200_HEAD_NHWC"] == HEAD_NHWC == 0x40
    assert not any(v & NHWC for k, v in variant.items() if k != "YOLO_B200_VARIANT_NHWC")
    assert not any(v & HEAD_NHWC for k, v in head.items() if k != "YOLO_B200_HEAD_NHWC")
    assert re.search(r"#define YOLO_B200_ABI_VERSION 3\b", header)


# ------------------------------------------------------------------------------------------ decode
@pytest.mark.parametrize("variant", [1, 2, 3, 4])
@pytest.mark.parametrize("extra", [0, _lib.VARIANT_F16, _lib.VARIANT_BF16, _lib.VARIANT_ACCUMULATE])
def test_decode_nhwc_with_an_nchw_variant_is_unsupported(variant, extra):
    assert decode_call(variant | NHWC | extra) == E_UNSUPPORTED


def test_decode_nhwc_keeps_the_other_refusals():
    assert decode_call(NHWC | _lib.VARIANT_F16 | _lib.VARIANT_BF16) == E_RANGE
    assert decode_call(5 | NHWC) == E_RANGE
    assert decode_call(NHWC, head=0x10002) == E_ALIGN                       # fp32 needs 4-byte alignment
    assert decode_call(NHWC | _lib.VARIANT_F16, head=0x10001) == E_ALIGN     # 16-bit needs 2-byte alignment


# ------------------------------------------------------------------------------------------ fused head
@pytest.mark.parametrize("bits", FEATURE_BITS)
def test_head_nhwc_with_cta_pair_is_unsupported(bits):
    assert head_call(HEAD_NHWC | _lib.HEAD_CTA_PAIR | bits) == E_UNSUPPORTED
    assert supported(256, 76, 76, HEAD_NHWC | _lib.HEAD_CTA_PAIR | bits) == 0


@pytest.mark.parametrize("bits", FEATURE_BITS)
def test_head_nhwc_with_a_pitch_is_unsupported(bits):
    assert head_call(HEAD_NHWC | bits, ny=19, nx=19, pitch=368) == E_UNSUPPORTED
    assert head_call(HEAD_NHWC | bits, pitch=64) == E_UNSUPPORTED
    assert supported(256, 19, 19, HEAD_NHWC | bits, pitch=368) == 0


@pytest.mark.parametrize("bits", FEATURE_BITS)
def test_head_nhwc_misaligned_x_is_an_alignment_error(bits):
    for x in (0x10008, 0x10004, 0x10002):
        assert head_call(HEAD_NHWC | bits, x=x) == E_ALIGN
    assert head_call(HEAD_NHWC | bits, ny=19, nx=19, x=0x10008) == E_ALIGN


def test_head_nhwc_other_refusals():
    assert head_call(HEAD_NHWC | _lib.HEAD_F16 | _lib.HEAD_BF16) == E_RANGE
    assert head_call(HEAD_NHWC | _lib.HEAD_F16 | _lib.HEAD_FP32X3) == E_UNSUPPORTED
    assert head_call(HEAD_NHWC | _lib.HEAD_FP32X3 | _lib.HEAD_CTA_PAIR) == E_RANGE
    assert head_call(HEAD_NHWC | _lib.HEAD_F16, c_in=96) == E_UNSUPPORTED
    assert head_call(HEAD_NHWC, c_in=48) == E_UNSUPPORTED


@pytest.mark.parametrize("bits", FEATURE_BITS)
def test_head_nhwc_supports_every_plane(bits):
    c_in = 64
    for ny, nx in ((76, 76), (38, 38), (26, 26), (19, 19), (13, 13), (15, 14), (7, 9), (1, 1), (1, 3)):
        assert supported(c_in, ny, nx, HEAD_NHWC | bits) == 1, (ny, nx)
    if bits:                                                # the odd 16-bit planes the NCHW kernel cannot read in place
        assert supported(c_in, 19, 19, bits) == 0 and supported(c_in, 13, 13, bits) == 0
    else:
        assert supported(c_in, 19, 19, HEAD_NHWC | _lib.HEAD_FP32X3) == 1    # the three-pass mode without a padded copy
        assert supported(c_in, 19, 19, _lib.HEAD_FP32X3) == 0


@pytest.mark.parametrize("bits", FEATURE_BITS)
def test_head_nhwc_keeps_the_cin_anchor_and_class_rules(bits):
    f = HEAD_NHWC | bits
    step = 32 if bits == 0 else 64
    assert supported(step, 76, 76, f) == 1 and supported(4 * step, 19, 19, f) == 1
    assert supported(step + 16, 76, 76, f) == 0 and supported(step // 2, 76, 76, f) == 0
    assert supported(256, 76, 76, f, nc=81) == 0
    assert supported(256, 76, 76, f, na=2) == 0
    assert supported(256, 76, 76, f, nc=37) == 1
    assert supported(256, 76, 76, f, nc=1) == 1


def test_head_supported_takes_a_memory_format():
    spec = ops.scale_spec(ANCHORS, 19, 19, 608)
    for dt in (torch.float16, torch.bfloat16):
        assert not ops.head_supported(256, spec, 80, dtype=dt)
        assert ops.head_supported(256, spec, 80, dtype=dt, memory_format=torch.channels_last)
    assert ops.head_supported(256, spec, 80, fp32x3=True, memory_format=torch.channels_last)
    assert not ops.head_supported(256, spec, 80, row_pitch=364, memory_format=torch.channels_last)
    with pytest.raises(ValueError):
        ops.head_supported(256, spec, 80, memory_format=torch.preserve_format)


# ------------------------------------------------------------------------------------------ the layout helper
def test_is_channels_last():
    x = torch.randn(2, 255, 13, 13)
    assert not ops.is_channels_last(x)
    assert ops.is_channels_last(x.to(memory_format=torch.channels_last))
    assert ops.is_channels_last(x.to(torch.float16).to(memory_format=torch.channels_last))
    # both layouts at once: NCHW to every kernel
    assert not ops.is_channels_last(torch.randn(2, 255, 1, 1).to(memory_format=torch.channels_last))
    assert not ops.is_channels_last(torch.randn(2, 1, 13, 13).to(memory_format=torch.channels_last))
    # a non-dense view of channels_last memory, and a permuted tensor that is neither layout
    assert not ops.is_channels_last(x.to(memory_format=torch.channels_last)[:, :, ::2])
    assert not ops.is_channels_last(x.to(memory_format=torch.channels_last)[:, :128])
    assert not ops.is_channels_last(x.permute(0, 1, 3, 2))
    assert not ops.is_channels_last(torch.randn(2, 255, 13))
