"""GPU: the fused head kernel on fp16 and bf16 feature maps (YOLO_B200_HEAD_F16 / _BF16, csrc/head.cu).

The 16-bit kernel shares the epilogue of the fp32 one and differs in its main loop: tcgen05.mma kind::f16 over 64-channel
k-blocks, X staged in the plain SWIZZLE_128B layout by TMA (planes with a 16-byte pitch), by the loader warps with 8- or
4-byte copies (even planes), or from the 16-bit padded copy (odd planes).  Three bars:
  * head values against an fp64 contraction of exactly the operands the tensor core multiplies (the 16-bit feature map and
    the 16-bit folded weights: their products are exact), then fp32 bias and activation -- first, on small shapes, so that
    a layout or descriptor slip shows up as wrong values rather than as a candidate mismatch;
  * candidates and detections bit-exact against decode_compact + NMS fed the fp32 head tensor the same kernel wrote;
  * at model level, the same against ``detect`` on the kernel's head tensors, and loosely against the model's own 16-bit
    convolution.
"""
import pytest
import torch
from torch import nn

from pytorch_yolo_b200 import ops, synth
from pytorch_yolo_b200.detect import PipelinedDetector, detect
from pytorch_yolo_b200.head import FusedHeadModel, HeadDetector, head_forward
from tests.test_gpu_head import MiniYolo, conv_block
from tests.test_gpu_head_steady import (assert_same_candidates, assert_same_detections, deal_tiles, heaviest_first,
                                        longest_run, row_offsets, sm_count, sorted_candidates)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ANCHORS = [(10, 13), (16, 30), (33, 23)]
NMS = 0.5
DTYPES = [torch.float16, torch.bfloat16]
DT_IDS = ["fp16", "bf16"]


def feature(batch, c_in, ny, nx, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(batch, c_in, ny, nx, generator=g, device=DEV).to(dtype)


def as_kernel_input(x):
    """What HeadDetector hands the kernel: odd 16-bit planes through the padded copy, everything else as it is."""
    return ops.pad_feature(x) if (x.shape[-1] * x.shape[-2]) % 2 else x


# ------------------------------------------------------------------------------------------------------------------
# Head values
def check_head_values(got, x, hw):
    """``got`` (B, n_out, ny, nx), the fp32 head tensor the kernel wrote for the 16-bit feature map ``x``, against the fp64
    contraction of the same 16-bit operands, per element:

        |got - ref| <= 4e-6 S + 1e-6,   S = sum_c |w| |x|.

    The products of two fp16 / bf16 values are exact in fp32 and in fp64, so what remains is the kernel's fp32
    accumulation: c_in / 16 instructions, each adding one rounded partial sum of magnitude <= S, i.e. at most
    (c_in / 16) 2^-24 S = 3.8e-6 S at c_in = 1024 if every step rounded the whole sum the wrong way (typical errors are
    far smaller: the largest err / S is printed).  1e-6 covers the fp32 bias addition and LeakyReLU product (2^-24 of
    values below 10).  A wrong layout or descriptor gives O(S) errors.

    Zeros (or any constant) in the accumulator would be off by |W x|; the test asserts that for at least 90 % of the
    elements |W x| exceeds 50 times the bar, so that the comparison cannot pass on an empty accumulator."""
    batch, n = got.shape[:2]
    plane = got.shape[2] * got.shape[3]
    wd = hw.weight[:n].double()
    wa = wd.abs()
    bias = hw.bias.to(got.device).double()[None, :, None]
    step = max(1, (1 << 27) // (n * plane))
    worst, far, total = 0.0, 0, 0
    for i in range(0, batch, step):
        xd = x[i:i + step].flatten(2).double()
        acc = torch.matmul(wd, xd)
        ref = acc + bias
        if hw.negative_slope != 1.0:
            ref = torch.maximum(ref, ref * hw.negative_slope)
        s = torch.matmul(wa, xd.abs())
        err = (got[i:i + step].flatten(2).double() - ref).abs()
        bar = 4e-6 * s + 1e-6
        worst = max(worst, float((err / s).max()))
        far += int((acc.abs() > 50 * bar).sum())
        total += acc.numel()
        excess = err - bar
        if not bool((excess <= 0).all()):
            flat = int(torch.nan_to_num(excess, nan=float("inf")).flatten().argmax())
            b, o, p = flat // (n * plane), (flat // plane) % n, flat % plane
            pytest.fail(f"head value off: image {i + b}, channel {o}, position {p} (tile {p // 128}): got "
                        f"{float(got[i + b].flatten(1)[o, p])}, fp64 {float(ref[b, o, p])}, S {float(s[b, o, p]):.4g}")
    assert far >= 0.9 * total, f"only {far} of {total} products exceed 50x the bar: the check would not see an empty accumulator"
    return worst


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("batch,c_in,ny,nx,path", [
    (2, 64, 8, 8, "one tile, 64 positions"),
    (2, 64, 8, 16, "one tile, 128 positions"),
    (3, 128, 10, 20, "ragged last tile, 2-D boxes"),
    (1, 256, 76, 76, "3-D box + ragged tile"),
    (2, 512, 38, 38, "loader warps, 8-byte copies"),
    (2, 256, 26, 26, "loader warps, 8-byte copies"),
    (2, 64, 15, 14, "loader warps, 4-byte copies"),
    (2, 1024, 19, 19, "padded copy"),
    (2, 512, 13, 13, "padded copy"),
], ids=lambda v: v if isinstance(v, str) else None)
def test_head_values_against_fp64(dtype, batch, c_in, ny, nx, path):
    spec = ops.scale_spec(ANCHORS, ny, nx, 16 * max(ny, nx))
    blk = conv_block(c_in, 255, seed=c_in + ny).to(DEV)
    x = feature(batch, c_in, ny, nx, dtype, seed=ny * nx)
    xin = as_kernel_input(x)
    assert ops.head_supported(c_in, spec, 80, xin.shape[2] if xin.dim() == 3 else 0, dtype=dtype)
    hw = ops.fold_head(blk, DEV, dtype=dtype)
    got = head_forward(xin, hw, spec, 80)
    worst = check_head_values(got, x, hw)
    print(f"{path}: largest err / S {worst:.3e}")
    # folded from the module by head_forward itself: the same operands, the same values
    assert torch.equal(head_forward(xin, blk, spec, 80).view(torch.int32), got.view(torch.int32))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_pad_feature_16_bit(dtype):
    x = feature(3, 64, 13, 13, dtype, seed=7)
    p = ops.pad_feature(x)
    assert p.dtype == dtype and p.shape == (3, 64, 176)
    assert torch.equal(p[..., :169].view(torch.int16), x.flatten(2).view(torch.int16))
    assert bool((p[..., 169:].view(torch.int16) == 0).all())
    out = torch.full_like(p, 5.0)
    assert ops.pad_feature(x, out=out) is out and torch.equal(out.view(torch.int16), p.view(torch.int16))
    with pytest.raises(ValueError):
        ops.pad_feature(x, out=torch.empty(3, 64, 176, device=DEV))                # fp32 out for a 16-bit map


# ------------------------------------------------------------------------------------------------------------------
# Candidates
def fused_candidates(feats, hws, specs, nc, conf, head_outs=None, cap=None):
    offs, rows = row_offsets(specs)
    buf = ops.Buffers(DEV, feats[0].shape[0], cap or rows, nc)
    ops.head_decode_compact(feats, hws, specs, offs, rows, nc, conf, buf, head_outs=head_outs)
    return buf


def unfused_candidates(heads, specs, nc, conf, cap=None):
    buf = ops.Buffers(DEV, heads[0].shape[0], cap or sum(s.rows for s in specs), nc)
    ops.decode_compact(heads, specs, nc, conf, buf)
    return buf


def head_tensors(feats, hws, specs):
    return [torch.full((f.shape[0], hw.n_out, s.ny, s.nx), float("nan"), device=DEV) for f, hw, s in zip(feats, hws, specs)]


def spp_scales(nc, batch, dtype, seed, cins=(1024, 512, 256)):
    w = synth.WORKLOADS["spp-608"]
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    heads = [conv_block(c, 3 * (nc + 5), seed + i).to(DEV) for i, c in enumerate(cins)]
    feats = [feature(batch, c, s.ny, s.nx, dtype, seed + 10 + i) for i, (c, s) in enumerate(zip(cins, specs))]
    return specs, heads, feats


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("conf", [0.3, 0.001])
def test_candidates_bit_exact_against_decode_compact_on_own_head_tensor(dtype, conf):
    """spp-608 grids, batch 2, all three scales in one launch: 19x19 padded (TMA), 38x38 loader-filled, 76x76 TMA."""
    nc = 80
    specs, heads, feats = spp_scales(nc, 2, dtype, seed=60)
    hws = [ops.fold_head(m, DEV, dtype=dtype) for m in heads]
    xs = [as_kernel_input(x) for x in feats]
    hts = head_tensors(feats, hws, specs)
    with_head = sorted_candidates(fused_candidates(xs, hws, specs, nc, conf, head_outs=hts))
    for h, x, hw in zip(hts, feats, hws):
        check_head_values(h, x, hw)
    want = sorted_candidates(unfused_candidates(hts, specs, nc, conf))
    assert int(want[0].sum()) > 0
    assert_same_candidates(with_head, want, "head_out instantiation vs decode_compact")
    assert_same_candidates(sorted_candidates(fused_candidates(xs, hws, specs, nc, conf)), want,
                           "production instantiation vs decode_compact")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_overflowing_cap_is_reported_with_the_same_counts(dtype):
    nc, conf, cap = 80, 0.001, 64
    specs, heads, feats = spp_scales(nc, 2, dtype, seed=70)
    hws = [ops.fold_head(m, DEV, dtype=dtype) for m in heads]
    xs = [as_kernel_input(x) for x in feats]
    hts = head_tensors(feats, hws, specs)
    fused_candidates(xs, hws, specs, nc, conf, head_outs=hts)
    got_cnt, _, got_ovf = ops.read_counts(fused_candidates(xs, hws, specs, nc, conf, cap=cap))
    want_cnt, _, want_ovf = ops.read_counts(unfused_candidates(hts, specs, nc, conf, cap=cap))
    assert got_ovf == want_ovf == 1
    assert bool((want_cnt > cap).all()) and torch.equal(got_cnt, want_cnt)


# ------------------------------------------------------------------------------------------------------------------
# Steady state at the benchmark's head shapes
def geometry16(feats, specs):
    """(c_in, plane, manual) per scale as the host derives them for 16-bit maps: ``manual`` = no 16-byte row pitch
    (pitch % 8 != 0), so the loader warps fill those tiles (head.cu, S.manual)."""
    out = []
    for x, s in zip(feats, specs):
        plane = s.ny * s.nx
        pitch = x.shape[2] if x.dim() == 3 else plane
        out.append((x.shape[1], plane, pitch % 8 != 0))
    return out


def switches(deal):
    """(loader -> TMA, TMA -> loader): the most tiles of one kind a CTA runs right before a tile of the other kind."""
    best = [0, 0]
    for seq in deal:
        run, prev = 0, None
        for *_, m in seq:
            if prev is not None and m != prev:
                best[0 if prev else 1] = max(best[0 if prev else 1], run)
                run = 0
            run += 1
            prev = m
    return tuple(best)


def check_steady(heads, specs, feats, nc, dtype, conf=0.3):
    hws = [ops.fold_head(m, DEV, dtype=dtype) for m in heads]
    xs = [as_kernel_input(x) for x in feats]
    hts = head_tensors(feats, hws, specs)
    with_head = sorted_candidates(fused_candidates(xs, hws, specs, nc, conf, head_outs=hts))
    worst = [check_head_values(h, x, hw) for h, x, hw in zip(hts, feats, hws)]
    print(f"largest err / S per scale: {', '.join(f'{r:.3e}' for r in worst)}")
    want = sorted_candidates(unfused_candidates(hts, specs, nc, conf))
    assert int(want[0].sum()) > 0
    assert_same_candidates(with_head, want, "head_out instantiation vs decode_compact")
    assert_same_candidates(sorted_candidates(fused_candidates(xs, hws, specs, nc, conf)), want,
                           "production instantiation vs decode_compact")
    want_det = detect(hts, specs, nc, conf, NMS, return_rows=True)
    det = HeadDetector(heads, specs, nc, feats[0].shape[0], DEV, conf_thres=conf, nms_thres=NMS, feature_dtype=dtype)
    assert det.fused == [True] * len(specs)
    assert [p is not None for p in det.padded] == [(s.ny * s.nx) % 2 == 1 for s in specs]
    assert assert_same_detections(det.run(feats, return_rows=True, clone=True), want_det) > 0


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_spp608_batch64(dtype):
    """spp-608, batch 64, ConvBlock heads: 19x19 (c_in 1024) padded and TMA-filled, dealt first; 38x38 (512) loader-filled;
    76x76 (256) TMA-filled: every CTA recycles its accumulator stages and runs loader tiles followed by TMA tiles."""
    nc, batch = 80, 64
    specs, heads, feats = spp_scales(nc, batch, dtype, seed=80, cins=tuple(synth.WORKLOADS["spp-608"]["head_cin"]))
    xs = [as_kernel_input(x) for x in feats]
    geo = geometry16(xs, specs)
    assert [g[2] for g in geo] == [False, True, False] and heaviest_first(geo) == [0, 1, 2]
    deal = deal_tiles(geo, batch, sm_count())
    assert longest_run(deal) >= 20, "no CTA runs many tiles"
    loader_to_tma, tma_to_loader = switches(deal)
    assert loader_to_tma >= 4 and tma_to_loader >= 1, (loader_to_tma, tma_to_loader)
    check_steady(heads, specs, feats, nc, dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_tiny416_batch1024(dtype):
    """tiny-416, batch 1024, the synthetic plain-convolution heads: 13x13 (c_in 512) padded and TMA-filled, dealt first,
    then 26x26 (256) loader-filled with 8-byte copies: every CTA runs ~14 TMA tiles, then ~40 loader tiles -- the order in
    which the loader warps skip ahead of the ring before their first tile."""
    batch = 1024
    w = synth.WORKLOADS["tiny-416"]
    nc = w["nc"]
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    feats32, convs = synth.synth_head_convs("tiny-416", batch, device=DEV)
    feats = [f.to(dtype) for f in feats32]
    del feats32
    xs = [as_kernel_input(x) for x in feats]
    geo = geometry16(xs, specs)
    assert [g[2] for g in geo] == [True, False] and heaviest_first(geo) == [1, 0]     # scales listed 26x26, 13x13
    deal = deal_tiles(geo, batch, sm_count())
    assert longest_run(deal) >= 50
    assert switches(deal)[1] >= 10, switches(deal)
    check_steady(convs, specs, feats, nc, dtype)


# ------------------------------------------------------------------------------------------------------------------
# Model level
def mini_yolo():
    torch.manual_seed(3)
    model = MiniYolo().to(DEV).eval()
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.2)
                m.running_var.uniform_(0.5, 1.5)
        model.branch2[1].bias[4::85] -= 3.0
    return model


def fallback_head(module, x, dtype):
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        return module(x)


@pytest.mark.parametrize("mode", ["half", "autocast-bf16"])
def test_fused_head_model(mode):
    """MiniYolo (tests/test_gpu_head.py): its 13x13 ConvBlock head (c_in 64) runs on the 16-bit kernel through the padded
    copy, its 26x26 plain head (c_in 32, not a multiple of 64) through the module's own convolution + decode_compact."""
    model = mini_yolo()
    x = torch.rand(2, 3, 52, 52, device=DEV)
    if mode == "half":
        model, x, dtype, ctx = model.half(), x.half(), torch.float16, torch.no_grad
    else:
        dtype = torch.bfloat16
        ctx = lambda: torch.autocast("cuda", dtype=dtype)                     # noqa: E731
    with ctx():
        fused = FusedHeadModel(model, x, conf_thres=0.25, nms_thres=0.5)
        det = fused.detector
        assert det.feature_dtype == dtype and det.fused == [True, False]
        assert det.padded[0] is not None and det.padded[0].dtype == dtype and det.padded[1] is None
        got, got_rows = fused(x, return_rows=True)
        feats = fused.features(x)
        heads = [model.branch1[1], model.branch2[1]]
        assert all(f.dtype == dtype for f in feats)
        # bit-exact against detect on the kernel's head tensor and the fallback's (16-bit, decoded as its fp32 upcast)
        hts = [head_forward(ops.pad_feature(feats[0]), heads[0], fused.specs[0], 80),
               fallback_head(heads[1], feats[1], dtype).float()]
        want, want_rows = detect(hts, fused.specs, 80, 0.25, 0.5, return_rows=True)
        assert assert_same_detections((got, got_rows), (want, want_rows)) > 0
        # against the model's own heads: scores move by the different summation, which reorders near-equal overlapping
        # boxes of a random-init model; most kept anchors must still coincide (the fp32 test's rule).  fp16: the model's
        # own 16-bit heads.  bf16: its head modules in fp32 on the same bf16 feature maps -- the model's own bf16 head
        # tensor is rounded to 8 mantissa bits (logits of magnitude 4-8 move by up to 2^-6), which on this model flips 8
        # of 14 kept rows, while the fused kernel keeps fp32 head values.
        with torch.no_grad():
            if dtype == torch.float16:
                own = [h.float() for h in model._forward_encoder(x)]
            else:
                with torch.autocast("cuda", enabled=False):
                    own = [m(f.float()) for m, f in zip(heads, feats)]
        ref, ref_rows = detect(own, fused.specs, 80, 0.25, 0.5, return_rows=True)
    for gr, rr in zip(got_rows, ref_rows):
        a = set() if gr is None else set(gr.tolist())
        b = set() if rr is None else set(rr.tolist())
        assert len(a ^ b) <= max(4, len(b) // 5), (len(a), len(b), len(a ^ b))
    assert isinstance(model.branch1[1], nn.Sequential) and isinstance(model.branch2[1], nn.Conv2d)


def spp_small(dtype, batch, seed):
    specs, heads, feats = spp_scales(80, batch, dtype, seed, cins=(256, 128, 64))
    return specs, heads, feats


def want_detections(heads, specs, feats, dtype, conf):
    hts = [head_forward(as_kernel_input(x), m, s, 80) for x, m, s in zip(feats, heads, specs)]
    return detect(hts, specs, 80, conf, NMS, return_rows=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_head_detector_graph_refilled_in_place(dtype):
    specs, heads, feats1 = spp_small(dtype, 4, seed=90)
    feats2 = [feature(*f.shape, dtype, seed=100 + i) for i, f in enumerate(feats1)]
    det = HeadDetector(heads, specs, 80, 4, DEV, conf_thres=0.3, nms_thres=NMS, use_graph=True, feature_dtype=dtype)
    assert det.fused == [True] * 3 and det.padded[0] is not None
    static = [torch.empty_like(f) for f in feats1]
    for src in (feats1, feats2, feats1):
        for s_, f in zip(static, src):
            s_.copy_(f)
        want = want_detections(heads, specs, src, dtype, 0.3)
        assert assert_same_detections(det.run(static, return_rows=True, clone=True), want) > 0


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_pipelined_detector_with_head_factory(dtype):
    specs, heads, feats = spp_small(dtype, 4, seed=110)
    pd = PipelinedDetector(specs, 80, 4, DEV, depth=2, factory=lambda lane: HeadDetector(
        heads, specs, 80, 4, DEV, conf_thres=0.3, nms_thres=NMS, use_graph=True, feature_dtype=dtype))
    ticket = pd.submit(feats)
    got = pd.collect(ticket, return_rows=True, clone=True)
    pd.drain()
    assert assert_same_detections(got, want_detections(heads, specs, feats, dtype, 0.3)) > 0


# ------------------------------------------------------------------------------------------------------------------
# Errors: each raises before anything is enqueued
@pytest.fixture
def problem():
    spec = ops.scale_spec(ANCHORS, 16, 16, 256)
    blk = conv_block(64, 255, seed=1).to(DEV)
    buf = ops.Buffers(DEV, 2, spec.rows, 80)
    buf.meta.fill_(7)
    return spec, blk, buf


def assert_untouched(buf):
    torch.cuda.synchronize()
    assert bool((buf.meta == 7).all())


def test_mixed_feature_dtypes_raise(problem):
    spec, blk, buf = problem
    xs = [feature(2, 64, 16, 16, torch.float16, 1), feature(2, 64, 16, 16, torch.bfloat16, 2)]
    hws = [ops.fold_head(blk, DEV, dtype=torch.float16), ops.fold_head(blk, DEV, dtype=torch.bfloat16)]
    with pytest.raises(ValueError, match="share a dtype"):
        ops.head_decode_compact(xs, hws, [spec, spec], [0, 0], spec.rows, 80, 0.3, buf)
    with pytest.raises(ValueError, match="folded to"):
        ops.head_decode_compact(xs[:1], [ops.fold_head(blk, DEV)], [spec], [0], spec.rows, 80, 0.3, buf)
    with pytest.raises(TypeError):
        ops.head_decode_compact([xs[0].double()], hws[:1], [spec], [0], spec.rows, 80, 0.3, buf)
    assert_untouched(buf)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_dtype_mismatch_at_run_raises(problem, dtype):
    spec, blk, _ = problem
    det = HeadDetector([blk], [spec], 80, 2, DEV, conf_thres=0.3, feature_dtype=dtype)
    det.buf.meta.fill_(7)
    other = torch.bfloat16 if dtype == torch.float16 else torch.float16
    for wrong in (other, torch.float32):
        with pytest.raises(TypeError, match=f"{wrong}.*{dtype}"):
            det.run([feature(2, 64, 16, 16, wrong, 3)])
    assert_untouched(det.buf)


def test_fp32x3_with_16_bit_raises(problem):
    spec, blk, _ = problem
    with pytest.raises(ValueError, match="fp32x3"):
        HeadDetector([blk], [spec], 80, 2, DEV, precision="fp32x3", feature_dtype=torch.float16)
    with pytest.raises(ValueError, match="fp32x3"):
        ops.fold_head(blk, DEV, fp32x3=True, dtype=torch.bfloat16)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_cta_pair_and_odd_plane_are_refused(problem, dtype):
    spec, blk, buf = problem
    hw = ops.fold_head(blk, DEV, dtype=dtype)
    x = feature(2, 64, 16, 16, dtype, 4)
    with pytest.raises(ops.YoloB200Error, match="not covered"):
        ops.head_decode_compact([x], [hw], [spec], [0], spec.rows, 80, 0.3, buf, cta_pair=True)
    odd = ops.scale_spec(ANCHORS, 13, 13, 208)
    buf13 = ops.Buffers(DEV, 2, odd.rows, 80)
    buf13.meta.fill_(7)
    with pytest.raises(ops.YoloB200Error, match="not covered"):
        ops.head_decode_compact([feature(2, 64, 13, 13, dtype, 5)], [hw], [odd], [0], odd.rows, 80, 0.3, buf13)
    assert_untouched(buf)
    assert_untouched(buf13)
