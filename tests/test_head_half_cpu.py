"""The fp16 / bf16 fused head (YOLO_B200_HEAD_F16 / _BF16) without a GPU: flag values, every argument check of
yolo_b200_head_decode_compact for the 16-bit modes (they return before any CUDA call; the device pointers below are never
dereferenced), the geometry yolo_b200_head_supported_ex accepts, and the host-side fold to 16-bit operands."""
import ctypes as C
import os
import re

import pytest
import torch
from torch import nn

from pytorch_yolo_b200 import _lib, ops

E_RANGE, E_ALIGN, E_UNSUPPORTED = -2, -3, -5
F16, BF16 = _lib.HEAD_F16, _lib.HEAD_BF16
ANCHORS = [(10, 13), (16, 30), (33, 23)]


def call(flags, c_in=64, ny=8, nx=8, pitch=0, x=0x10000, weight=0x20000):
    lib = _lib.load()
    arr = (_lib.Head * 1)()
    bias = (C.c_float * 255)()
    h = arr[0]
    h.x, h.weight, h.bias_host, h.head_out = x, weight, bias, None
    h.c_in, h.x_row_pitch, h.negative_slope = c_in, pitch, 0.1
    s = h.scale
    s.ny, s.nx, s.na, s.row_off, s.stride = ny, nx, 3, 0, 8.0
    fake = 0x40000                                   # 16-byte aligned, never touched
    return lib.yolo_b200_head_decode_compact(arr, 1, 1, 80, 3 * ny * nx, 0.3, 2.0, fake, fake + 0x1000, 64, fake + 0x2000,
                                             fake + 0x2000 + 4, flags, None)


def supported(c_in, ny, nx, flags, pitch=0, nc=80):
    return _lib.load().yolo_b200_head_supported_ex(c_in, ny, nx, pitch, 3, nc, flags)


def test_bits_match_the_header():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "yolo_b200.h")).read()
    bits = {k: int(v, 0) for k, v in re.findall(r"#define (YOLO_B200_HEAD_\w+)\s+(0x[0-9a-fA-F]+|\d+)", header)}
    assert bits["YOLO_B200_HEAD_F16"] == F16 == 0x10
    assert bits["YOLO_B200_HEAD_BF16"] == BF16 == 0x20
    assert bits["YOLO_B200_HEAD_CTA_PAIR"] == _lib.HEAD_CTA_PAIR
    assert bits["YOLO_B200_HEAD_FP32X3"] == _lib.HEAD_FP32X3
    assert not any(v & (F16 | BF16) for k, v in bits.items() if k not in ("YOLO_B200_HEAD_F16", "YOLO_B200_HEAD_BF16"))
    assert ops.FEATURE_DTYPE_FLAGS == {torch.float32: 0, torch.float16: F16, torch.bfloat16: BF16}


def test_both_bits_is_a_range_error():
    assert call(F16 | BF16) == E_RANGE
    assert call(F16 | BF16 | _lib.HEAD_ACCUMULATE) == E_RANGE
    assert supported(64, 8, 8, F16 | BF16) == 0


@pytest.mark.parametrize("bit", [F16, BF16])
@pytest.mark.parametrize("mode", [_lib.HEAD_FP32X3, _lib.HEAD_CTA_PAIR])
def test_three_pass_and_cta_pair_are_unsupported(bit, mode):
    assert call(bit | mode) == E_UNSUPPORTED
    assert supported(256, 76, 76, bit | mode) == 0


@pytest.mark.parametrize("bit", [F16, BF16])
def test_geometry_errors_are_unsupported(bit):
    assert call(bit, c_in=96) == E_UNSUPPORTED                     # c_in % 64
    assert call(bit, c_in=32) == E_UNSUPPORTED
    assert call(bit, ny=13, nx=13) == E_UNSUPPORTED                # odd plane, not padded
    assert call(bit, ny=19, nx=19, pitch=364) == E_UNSUPPORTED     # a pitch of 4 elements is 8 bytes
    assert call(bit, ny=19, nx=19, pitch=360) == E_UNSUPPORTED     # pitch below the plane


@pytest.mark.parametrize("bit", [F16, BF16])
def test_misaligned_operands_are_alignment_errors(bit):
    assert call(bit, x=0x10008) == E_ALIGN
    assert call(bit, weight=0x20002) == E_ALIGN
    assert call(bit, ny=19, nx=19, pitch=368, x=0x10004) == E_ALIGN


@pytest.mark.parametrize("bit", [F16, BF16])
def test_supported_planes(bit):
    # plane % 8 == 0: tensor maps; even planes: the loader warps (8-byte copies at plane % 4 == 0, else 4-byte copies);
    # odd planes: only with a padded pitch that is a multiple of 8 elements
    for g, want in ((76, 1), (52, 1), (38, 1), (26, 1), (19, 0), (13, 0)):
        assert supported(256, g, g, bit) == want, g
    assert supported(256, 15, 14, bit) == 1                         # 210 = 2 mod 8
    assert supported(256, 19, 19, bit, pitch=ops.padded_pitch(ops.scale_spec(ANCHORS, 19, 19, 608), torch.float16)) == 1
    assert supported(256, 13, 13, bit, pitch=176) == 1
    assert supported(256, 13, 13, bit, pitch=172) == 0
    assert supported(64, 76, 76, bit) == 1
    assert supported(96, 76, 76, bit) == 0
    assert supported(96, 76, 76, 0) == 1                            # fp32 takes c_in % 32
    assert supported(256, 19, 19, 0) == 1                           # ... and reads odd fp32 planes in place
    assert supported(256, 76, 76, bit, nc=37) == 1                  # run-time class loop
    assert supported(256, 76, 76, bit, nc=81) == 0


def test_padded_pitch():
    pitch = lambda g, dt: ops.padded_pitch(ops.scale_spec(ANCHORS, g, g, 608), dt)
    for dt in (torch.float16, torch.bfloat16):
        assert [pitch(g, dt) for g in (76, 38, 26, 19, 13)] == [5776, 1448, 680, 368, 176]
    assert [pitch(g, torch.float32) for g in (76, 38, 26, 19, 13)] == [5776, 1444, 676, 364, 172]


def conv_block(c_in, n_out, seed):
    g = torch.Generator().manual_seed(seed)
    blk = nn.Sequential(nn.Conv2d(c_in, n_out, 1, bias=False), nn.BatchNorm2d(n_out), nn.LeakyReLU(0.1))
    with torch.no_grad():
        blk[0].weight.copy_(torch.randn(n_out, c_in, 1, 1, generator=g))
        blk[1].weight.copy_(torch.rand(n_out, generator=g) + 0.5)
        blk[1].bias.copy_(torch.randn(n_out, generator=g))
        blk[1].running_mean.copy_(torch.randn(n_out, generator=g))
        blk[1].running_var.copy_(torch.rand(n_out, generator=g) + 0.5)
    return blk.eval()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_fold_head_rounds_fp64_to_fp32_then_to_dtype(dtype):
    blk = conv_block(64, 255, seed=1)
    hw32 = ops.fold_head(blk, "cpu")
    hw = ops.fold_head(blk, "cpu", dtype=dtype)
    assert hw.dtype == dtype and hw.weight.shape == (256, 64) and hw32.dtype == torch.float32
    assert torch.equal(hw.weight, hw32.weight.to(dtype))
    assert bool((hw.weight[255:] == 0).all())
    assert torch.equal(hw.bias, hw32.bias) and hw.bias.dtype == torch.float32
    assert hw.negative_slope == hw32.negative_slope == pytest.approx(0.1)
    # the fold itself is fp64: the fp32 rounding of the fp64 product, not a product of rounded factors
    bn = blk[1]
    g = bn.weight.double() / torch.sqrt(bn.running_var.double() + bn.eps)
    want = (blk[0].weight.double().reshape(255, 64) * g[:, None]).float().to(dtype)
    assert torch.equal(hw.weight[:255], want)


def test_fold_head_refuses_fp16_overflow():
    conv = nn.Conv2d(64, 255, 1)
    with torch.no_grad():
        conv.weight.normal_()
        conv.weight[7, 3] = 7.0e4                                   # beyond 65504
    with pytest.raises(ValueError, match="range"):
        ops.fold_head(conv, "cpu", dtype=torch.float16)
    hw = ops.fold_head(conv, "cpu", dtype=torch.bfloat16)           # bf16 has fp32's exponent range
    assert bool(torch.isfinite(hw.weight).all())


def test_fold_head_refuses_fp32x3_with_16_bit():
    conv = nn.Conv2d(64, 255, 1)
    for dt in (torch.float16, torch.bfloat16):
        with pytest.raises(ValueError, match="fp32x3"):
            ops.fold_head(conv, "cpu", fp32x3=True, dtype=dt)
    with pytest.raises(TypeError):
        ops.fold_head(conv, "cpu", dtype=torch.float64)
