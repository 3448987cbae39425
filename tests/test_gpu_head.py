"""GPU parity tests of the fused head kernel (csrc/head.cu, SURVEY.md section 8f-3) through the C ABI.

Two bars, both written here:
  * the convolution itself: TF32 tensor-core products (operands truncated to 10 mantissa bits, fp32 accumulation).
    Against an fp64 product of the truncated operands the error is fp32 accumulation noise (<= 3e-5 absolute at
    these magnitudes); against the reference's fp32 convolution it is the TF32 rounding, bounded by
    2^-9 * sum_c |w||x| per element;
  * everything after the accumulator: BIT-EXACT against decode_compact + NMS fed with the head tensor the same
    kernel wrote (same candidates, same kept rows, same order).
"""
import pytest
import torch
from torch import nn

from pytorch_yolo_b200 import _lib, ops
from pytorch_yolo_b200 import YOLOLayer, non_max_suppression
from pytorch_yolo_b200.head import FusedHeadModel, HeadDetector, head_forward, split_head

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ANCHORS = [(10, 13), (16, 30), (33, 23)]


def tf32_trunc(t):
    return (t.contiguous().view(torch.int32) & ~0x1fff).view(torch.float32)


def conv_block(c_in, n_out, seed):
    """The reference's ConvBlock(c_in, n_out, size=1) (models/yolo_base.py:19-44) with non-trivial BatchNorm statistics."""
    g = torch.Generator().manual_seed(seed)
    blk = nn.Sequential(nn.Conv2d(c_in, n_out, 1, bias=False), nn.BatchNorm2d(n_out), nn.LeakyReLU(0.1, inplace=True))
    with torch.no_grad():
        blk[0].weight.copy_(torch.randn(n_out, c_in, 1, 1, generator=g) * (2.0 / c_in ** 0.5))
        blk[1].weight.copy_(torch.rand(n_out, generator=g) + 0.5)
        blk[1].bias.copy_(torch.randn(n_out, generator=g))
        blk[1].running_mean.copy_(torch.randn(n_out, generator=g) * 0.3)
        blk[1].running_var.copy_(torch.rand(n_out, generator=g) + 0.5)
    return blk.eval()


def plain_conv(c_in, n_out, nc, seed):
    """A plain 1x1 head (models/yolov3_tiny.py:38,42) whose output follows SYNTH-A for unit-variance features."""
    g = torch.Generator().manual_seed(seed)
    std = torch.tensor(([1.0, 1.0, 0.5, 0.5, 3.0] + [2.0] * nc) * (n_out // (nc + 5)))
    mean = torch.tensor(([0.0, 0.0, 0.0, 0.0, -4.0] + [-2.0] * nc) * (n_out // (nc + 5)))
    conv = nn.Conv2d(c_in, n_out, 1, bias=True)
    with torch.no_grad():
        conv.weight.copy_((torch.randn(n_out, c_in, generator=g) * (std[:, None] / c_in ** 0.5)).view(n_out, c_in, 1, 1))
        conv.bias.copy_(mean)
    return conv.eval()


@pytest.mark.parametrize("batch,c_in,ny,nx,nc", [(2, 64, 16, 20, 80), (3, 256, 38, 38, 80), (2, 96, 12, 12, 20),
                                                 (1, 32, 8, 8, 1), (2, 128, 10, 26, 80),
                                                 (2, 64, 16, 20, 37), (2, 96, 12, 12, 5), (1, 32, 8, 8, 2)])   # run-time class loop
def test_head_convolution_tf32(batch, c_in, ny, nx, nc):
    spec = ops.scale_spec(ANCHORS, ny, nx, 16 * max(ny, nx))
    n_out = 3 * (nc + 5)
    blk = conv_block(c_in, n_out, seed=c_in + nc)
    x = torch.randn(batch, c_in, ny, nx, generator=torch.Generator().manual_seed(1)).to(DEV)
    got = head_forward(x, blk, spec, nc)
    hw = ops.fold_head(blk, DEV)
    w, b = hw.weight[:n_out], hw.bias.to(DEV)
    # (a) exactness of the data path: fp64 product of the TF32-truncated operands
    y = torch.einsum("oc,bcp->bop", tf32_trunc(w).double(), tf32_trunc(x).double().flatten(2)) + b.double()[None, :, None]
    y = torch.maximum(y, y * 0.1).view_as(got)
    assert float((got.double() - y).abs().max()) <= 3e-5
    # (b) against the reference module in fp32 (CPU: no TF32 there): the TF32 operand rounding, 2 * 2^-11 per product
    with torch.no_grad():
        want = blk(x.cpu()).to(DEV)
    bound = 2.0 ** -9 * torch.einsum("oc,bcp->bop", w.abs(), x.abs().flatten(2)).view_as(got) + 1e-5
    assert bool(((got - want).abs() <= bound).all())


@pytest.mark.parametrize("batch,c_in,ny,nx,nc,conf", [(4, 64, 16, 20, 80, 0.3), (2, 256, 76, 76, 80, 0.1), (2, 128, 12, 12, 20, 0.01),
                                                      (2, 32, 8, 8, 1, 0.2), (3, 64, 6, 6, 80, 0.001),
                                                      (3, 64, 16, 20, 37, 0.1), (2, 128, 12, 12, 5, 0.05), (2, 32, 24, 24, 2, 0.1),
                                                      (2, 64, 10, 10, 64, 0.05)])            # the last four: run-time class loop
@pytest.mark.parametrize("cta_pair", [False, True])
def test_fused_candidates_equal_decode_compact_on_own_head_tensor(batch, c_in, ny, nx, nc, conf, cta_pair):
    spec = ops.scale_spec(ANCHORS, ny, nx, 8 * max(ny, nx))
    n_out = 3 * (nc + 5)
    conv = plain_conv(c_in, n_out, nc, seed=7)
    with torch.no_grad():
        # two saturated class logits per anchor, the second one larger: the first arg-max must be taken in sigmoid
        # space where both are exactly 1.0 (SURVEY.md section 7 hard part; rescan path of the kernel)
        if nc > 20:
            conv.bias[20::nc + 5] += 30.0              # classes 15 and 16
            conv.bias[21::nc + 5] += 31.0
    x = torch.randn(batch, c_in, ny, nx, generator=torch.Generator().manual_seed(2)).to(DEV)
    x[0, :, 0, 0] = float("nan")                         # a poisoned position must drop out of both paths alike
    x[-1, 3, -1, -1] = float("inf")
    hw = ops.fold_head(conv, DEV)
    buf = ops.Buffers(DEV, batch, spec.rows, nc)
    ho = torch.empty(batch, n_out, ny, nx, device=DEV)
    if cta_pair and nc != 80:
        pytest.skip("the CTA-pair kernel is instantiated for 3 anchors x 80 classes")
    ops.head_decode_compact([x], [hw], [spec], [0], spec.rows, nc, conf, buf, head_outs=[ho], cta_pair=cta_pair)
    cand_f, _, ovf = ops.read_counts(buf)
    cand_f = cand_f.clone()
    assert ovf == 0
    box_f, meta_f = buf.cand_box.clone().view(batch, -1, 4), buf.cand_meta.clone().view(batch, -1, 4)
    ops.decode_compact([ho], [spec], nc, conf, buf)
    cand_d, _, _ = ops.read_counts(buf)
    assert torch.equal(cand_f, cand_d)
    assert int(cand_f.sum()) > 0
    box_d, meta_d = buf.cand_box.view(batch, -1, 4), buf.cand_meta.view(batch, -1, 4)
    for b in range(batch):
        k = int(cand_f[b])
        of, od = meta_f[b, :k, 3].argsort(), meta_d[b, :k, 3].argsort()
        assert torch.equal(meta_f[b, :k][of], meta_d[b, :k][od])                      # score, cls_conf, class, row: bit-exact
        assert torch.equal(box_f[b, :k][of].view(torch.int32), box_d[b, :k][od].view(torch.int32))
    if nc > 20:                                          # the saturated pair resolved to the FIRST index
        assert bool((meta_f[0, :int(cand_f[0]), 2] == 15).all())


def spp_like(batch, seed=5):
    """Three scales shaped like YOLOv3-SPP at 608 divided by 4 in channels: 19x19 (not fusable), 38x38, 76x76."""
    specs = [ops.scale_spec(a, g, g, 608) for a, g in zip(
        [[(116, 90), (156, 198), (373, 326)], [(30, 61), (62, 45), (59, 119)], [(10, 13), (16, 30), (33, 23)]], (19, 38, 76))]
    heads = [plain_conv(c, 255, 80, seed + i).to(DEV) for i, c in enumerate((256, 128, 64))]
    g = torch.Generator().manual_seed(seed)
    feats = [torch.randn(batch, c, s.ny, s.nx, generator=g).to(DEV) for c, s in zip((256, 128, 64), specs)]
    return specs, heads, feats


def test_head_detector_mixed_scales_bit_exact_against_unfused_on_same_heads():
    batch, nc = 3, 80
    specs, heads, feats = spp_like(batch)
    det = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5, unaligned="unfused")
    assert det.fused == [False, True, True]              # 19x19 planes are not a multiple of 4 floats
    got, got_rows = det.run(feats, return_rows=True, clone=True)
    # the unfused path on the same head tensors: scale 0 from the module, scales 1, 2 as the fused kernel computes them
    with torch.no_grad():
        hts = [heads[0](feats[0])] + [head_forward(feats[k], heads[k], specs[k], nc) for k in (1, 2)]
    from pytorch_yolo_b200.detect import detect
    want, want_rows = detect(hts, specs, nc, 0.3, 0.5, return_rows=True)
    assert sum(d is not None for d in want) == batch
    for g, w, gr, wr in zip(got, want, got_rows, want_rows):
        assert torch.equal(g.view(torch.int32), w.view(torch.int32))
        assert torch.equal(gr, wr)


def test_head_detector_padded_19x19_all_scales_fused():
    """19x19 through the plane-padded copy: all three scales on the tensor-core kernel, bit-exact against the unfused path
    fed with the head tensors the kernel writes (the padded path must produce the same head values as an aligned one)."""
    batch, nc = 3, 80
    specs, heads, feats = spp_like(batch, seed=9)
    det = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5, unaligned="pad")
    assert det.fused == [True, True, True] and det.padded[0] is not None and det.padded[0].shape == (batch, 256, 364)
    got, got_rows = det.run(feats, return_rows=True, clone=True)
    # the same detector as a captured CUDA graph, replayed twice on the same input tensors
    det_g = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5, use_graph=True, unaligned="pad")
    for _ in range(2):
        gg, gg_rows = det_g.run(feats, return_rows=True, clone=True)
        for a_, b_, ar, br in zip(gg, got, gg_rows, got_rows):
            assert torch.equal(a_.view(torch.int32), b_.view(torch.int32)) and torch.equal(ar, br)
    hts = [head_forward(ops.pad_feature(feats[0]), heads[0], specs[0], nc)] + [head_forward(feats[k], heads[k], specs[k], nc) for k in (1, 2)]
    # the padded 19x19 head tensor is a TF32 convolution of the same data
    import copy
    with torch.no_grad():
        ref0 = copy.deepcopy(heads[0]).cpu()(feats[0].cpu()).to(DEV)
    assert float((hts[0] - ref0).abs().max()) < 0.05
    xp = ops.pad_feature(feats[0])
    assert torch.equal(xp[:, :, :361], feats[0].flatten(2)) and bool((xp[:, :, 361:] == 0).all())
    from pytorch_yolo_b200.detect import detect
    want, want_rows = detect(hts, specs, nc, 0.3, 0.5, return_rows=True)
    for g, w, gr, wr in zip(got, want, got_rows, want_rows):
        assert torch.equal(g.view(torch.int32), w.view(torch.int32))
        assert torch.equal(gr, wr)


@pytest.mark.parametrize("c_in,ny,nx,batch", [(256, 19, 19, 3), (512, 13, 13, 5), (96, 19, 19, 2), (1024, 19, 19, 2),
                                              (64, 13, 11, 2), (32, 5, 5, 2), (128, 21, 21, 2)])
def test_unaligned_planes_read_in_place_by_the_loader_warps(c_in, ny, nx, batch):
    """19x19 / 13x13 planes without the padded copy: two warps of the kernel fill the X stages with 4-byte asynchronous
    copies in TMA's swizzled layout.  The head tensor is BIT-IDENTICAL to the one the same kernel computes from the padded
    copy (same products, same accumulation order), and so are the candidates; the convolution is checked against the fp64
    product as well."""
    nc = 80
    spec = ops.scale_spec(ANCHORS, ny, nx, 32 * max(ny, nx))
    assert (ny * nx) % 4 and ops.head_supported(c_in, spec, nc) and not ops.head_supported(c_in, spec, nc, fp32x3=True)
    conv = plain_conv(c_in, 255, nc, seed=c_in + ny)
    x = torch.randn(batch, c_in, ny, nx, generator=torch.Generator().manual_seed(4)).to(DEV)
    x[0, :, 0, 0] = float("nan")
    hw = ops.fold_head(conv, DEV)
    outs, cands = [], []
    for feat in (x, ops.pad_feature(x)):
        ho = torch.full((batch, 255, ny, nx), float("nan"), device=DEV)
        buf = ops.Buffers(DEV, batch, spec.rows, nc)
        ops.head_decode_compact([feat], [hw], [spec], [0], spec.rows, nc, 0.2, buf, head_outs=[ho])
        cnt, _, ovf = ops.read_counts(buf)
        assert ovf == 0
        k = cnt.clone()
        meta = buf.cand_meta.view(batch, -1, 4)
        box = buf.cand_box.view(batch, -1, 4)
        rows = [sorted(zip(meta[i, :int(k[i]), 3].tolist(), meta[i, :int(k[i]), 0].tolist(),
                           box[i, :int(k[i])].view(torch.int32).tolist())) for i in range(batch)]
        outs.append(ho)
        cands.append((k, rows))
    assert torch.equal(outs[0][1:].view(torch.int32), outs[1][1:].view(torch.int32))           # image 0 holds the NaN position
    assert torch.equal(torch.isnan(outs[0][0]), torch.isnan(outs[1][0]))
    assert torch.equal(cands[0][0], cands[1][0]) and cands[0][1] == cands[1][1] and int(cands[0][0].sum()) > 0
    w, b = hw.weight[:255], hw.bias.to(DEV)
    y = torch.einsum("oc,bcp->bop", tf32_trunc(w).double(), tf32_trunc(x[1:]).double().flatten(2)) + b.double()[None, :, None]
    assert float((outs[0][1:].double() - y.view_as(outs[0][1:])).abs().max()) <= 3e-5 * max(1.0, (c_in / 256) ** 0.5)


def test_head_detector_reads_unaligned_scale_in_place():
    batch, nc = 3, 80
    specs, heads, feats = spp_like(batch, seed=9)
    det = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5, use_graph=True)
    assert det.fused == [True, True, True] and det.padded == [None, None, None]
    assert det.kernels_per_step == 4                       # fused head + 3 NMS kernels: no pad copy, no cuDNN
    pad = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5, unaligned="pad")
    for _ in range(2):
        got, got_rows = det.run(feats, return_rows=True, clone=True)
        want, want_rows = pad.run(feats, return_rows=True, clone=True)
        for g, w_, gr, wr in zip(got, want, got_rows, want_rows):
            assert torch.equal(g.view(torch.int32), w_.view(torch.int32)) and torch.equal(gr, wr)
    x3 = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5, precision="fp32x3")
    assert x3.fused == [True, True, True] and x3.padded[0] is not None      # the three-pass mode still pads 19x19


def test_head_detector_close_to_fp32_modules():
    """Against the reference modules run in fp32 (no TF32): same detections except where a score sits within the TF32
    error of the confidence threshold or two scores swap order; the kept sets must overlap almost entirely."""
    batch, nc = 2, 80
    specs, heads, feats = spp_like(batch, seed=11)
    det = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=0.3, nms_thres=0.5)
    _, got_rows = det.run(feats, return_rows=True, clone=True)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            hts = [m(x) for m, x in zip(heads, feats)]
    finally:
        torch.backends.cudnn.allow_tf32 = old
    from pytorch_yolo_b200.detect import detect
    _, want_rows = detect(hts, specs, nc, 0.3, 0.5, return_rows=True)
    for gr, wr in zip(got_rows, want_rows):
        a, b = set(gr.tolist()), set(wr.tolist())
        assert len(a ^ b) <= max(2, len(b) // 50), (len(a), len(b), len(a ^ b))


def test_convblock_branch_split_and_leaky_head():
    """A reference-style branch (3x3 ConvBlock, then the 1x1 ConvBlock head with BatchNorm + LeakyReLU) split by split_head."""
    nc, batch = 80, 2
    branch = nn.Sequential(nn.Sequential(nn.Conv2d(16, 64, 3, padding=1, bias=False), nn.BatchNorm2d(64), nn.LeakyReLU(0.1)),
                           conv_block(64, 255, seed=3)).to(DEV).eval()
    trunk, head = split_head(branch)
    spec = ops.scale_spec(ANCHORS, 20, 20, 160)
    x = torch.randn(batch, 16, 20, 20, generator=torch.Generator().manual_seed(4)).to(DEV)
    with torch.no_grad():
        feat = trunk(x)
    det = HeadDetector([head], [spec], nc, batch, DEV, conf_thres=0.2, nms_thres=0.5)
    assert det.fused == [True]
    got = det.run([feat], clone=True)
    from pytorch_yolo_b200.detect import detect
    want = detect([head_forward(feat, head, spec, nc)], [spec], nc, 0.2, 0.5)
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if g is not None:
            assert torch.equal(g.view(torch.int32), w.view(torch.int32))


def test_fused_head_overflow_is_reported_not_silent():
    batch, nc = 2, 80
    spec = ops.scale_spec(ANCHORS, 16, 16, 128)
    conv = plain_conv(64, 255, nc, seed=1)
    with torch.no_grad():
        conv.bias[4::85] += 12.0                           # nearly every anchor passes
    x = torch.randn(batch, 64, 16, 16, generator=torch.Generator().manual_seed(8)).to(DEV)
    hw = ops.fold_head(conv, DEV)
    buf = ops.Buffers(DEV, batch, 50, nc)                  # capacity 50 per image, far below the ~700 that pass
    ops.head_decode_compact([x], [hw], [spec], [0], spec.rows, nc, 0.3, buf)
    cand, _, ovf = ops.read_counts(buf)
    assert ovf == 1 and bool((cand > 50).all())            # counts keep counting, the excess is dropped, the flag is set
    det = HeadDetector([conv], [spec], nc, batch, DEV, 0.3, 0.5, cap=50)
    with pytest.raises(ops.YoloB200Error, match="capacity"):
        det.run([x])


def test_fused_head_in_a_cuda_graph_on_a_side_stream():
    """The C ABI promises stream order and graph capture: pad + fused head + NMS captured once, replayed on new data."""
    batch, nc = 2, 80
    specs, heads, feats = spp_like(batch, seed=21)
    hws = [ops.fold_head(h, DEV) for h in heads]
    rows = sum(s.rows for s in specs)
    offs = [0, specs[0].rows, specs[0].rows + specs[1].rows]
    buf = ops.Buffers(DEV, batch, rows, nc)
    out, out_row = buf.new_outputs()
    static = [f.clone() for f in feats]
    xp = torch.zeros(batch, 256, 364, device=DEV)

    def enqueue():
        ops.pad_feature(static[0], out=xp)
        ops.head_decode_compact([xp, static[1], static[2]], hws, specs, offs, rows, nc, 0.3, buf)
        ops.nms(buf, 0.5, out, out_row)

    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        enqueue()                                          # warm-up outside the capture
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            enqueue()
        for trial in range(2):
            new = [torch.randn(f.shape, generator=torch.Generator().manual_seed(100 + trial)).to(DEV) for f in feats]
            for s_, n_ in zip(static, new):
                s_.copy_(n_)
            g.replay()
            side.synchronize()
            kept_g = buf.meta[batch + 1:].clone()
            got = out.clone()
            enqueue()                                      # the same data, eagerly
            side.synchronize()
            assert torch.equal(kept_g, buf.meta[batch + 1:]) and int(kept_g.sum()) > 0
            for b in range(batch):
                n = int(kept_g[b])
                assert torch.equal(got[b, :n].view(torch.int32), out[b, :n].view(torch.int32))
    torch.cuda.current_stream(DEV).wait_stream(side)


def test_head_abi_argument_checks(lib):
    assert lib.yolo_b200_head_supported(256, 76, 76, 0, 3, 80) == 1
    assert lib.yolo_b200_head_supported(256, 19, 19, 0, 3, 80) == 1   # 361 positions: no 16-byte pitch, read by the loader warps
    assert lib.yolo_b200_head_supported_ex(256, 19, 19, 0, 3, 80, _lib.HEAD_FP32X3) == 0   # ... which the three-pass mode lacks
    assert lib.yolo_b200_head_supported(256, 19, 19, 362, 3, 80) == 0 # an explicit pitch must be a multiple of 4 floats
    assert lib.yolo_b200_head_supported(256, 19, 19, 364, 3, 80) == 1 # ... unless the planes are padded
    assert lib.yolo_b200_head_supported(256, 19, 19, 360, 3, 80) == 0 # pitch smaller than the plane
    assert lib.yolo_b200_head_supported(100, 76, 76, 0, 3, 80) == 0   # c_in not a multiple of 32
    assert lib.yolo_b200_head_supported(256, 76, 76, 0, 3, 7) == 1    # any class count with 3 * (5 + nc) <= 256
    assert lib.yolo_b200_head_supported(256, 76, 76, 0, 3, 81) == 0   # 258 output channels
    assert lib.yolo_b200_head_supported(256, 76, 76, 0, 2, 80) == 0   # epilogue warps are laid out for 3 anchors
    spec = ops.scale_spec(ANCHORS, 19, 19, 608)
    hw = ops.fold_head(plain_conv(64, 255, 80, 1), DEV, fp32x3=True)   # the three-pass mode cannot read 19x19 planes in place
    x = torch.randn(1, 64, 19, 19, device=DEV)
    buf = ops.Buffers(DEV, 1, spec.rows, 80)
    buf.meta.fill_(7)
    with pytest.raises(ops.YoloB200Error, match="not covered"):
        ops.head_decode_compact([x], [hw], [spec], [0], spec.rows, 80, 0.3, buf)
    torch.cuda.synchronize()
    assert bool((buf.meta == 7).all())                                 # E_UNSUPPORTED: nothing was launched or zeroed
    assert _lib.E_UNSUPPORTED == -5


class MiniYolo(nn.Module):
    """A stand-in with the structure of the reference models (models/yolov3_tiny.py:67-100): ``_forward_encoder`` returns
    the head tensors, ``yolo_layers`` the YOLOLayers; one ConvBlock head (BatchNorm + LeakyReLU) and one plain Conv2d head."""

    def __init__(self, nc=80):
        super().__init__()
        def block(ci, co, k, s=1):
            return nn.Sequential(nn.Conv2d(ci, co, k, s, (k - 1) // 2, bias=False), nn.BatchNorm2d(co), nn.LeakyReLU(0.1, inplace=True))
        self.stem = block(3, 32, 3, 2)
        self.down = block(32, 64, 3, 2)
        self.branch1 = nn.Sequential(block(64, 64, 3), block(64, 3 * (nc + 5), 1))                 # coarse scale, ConvBlock head
        self.up = nn.Upsample(scale_factor=2)
        self.branch2 = nn.Sequential(block(96, 32, 3), nn.Conv2d(32, 3 * (nc + 5), 1))              # fine scale, plain head
        anchors = [[(81, 82), (135, 169), (344, 319)], [(10, 14), (23, 27), (37, 58)]]
        self.yolo1, self.yolo2 = YOLOLayer(anchors[0], nc, anchors), YOLOLayer(anchors[1], nc, anchors)

    @property
    def yolo_layers(self):
        return self.yolo1, self.yolo2

    def _forward_encoder(self, x):
        a = self.stem(x)
        b = self.down(a)
        return self.branch1(b), self.branch2(torch.cat([self.up(b), a], 1))

    def forward(self, x):
        img_size = max(x.shape[-2:])
        outs = [y(h, img_size) for y, h in zip(self.yolo_layers, self._forward_encoder(x))]
        io, p = list(zip(*outs))
        return torch.cat(io, 1), p


def test_fused_head_model_wraps_a_reference_style_model():
    torch.manual_seed(3)
    model = MiniYolo().to(DEV).eval()
    with torch.no_grad():
        for m in model.modules():                      # non-trivial BatchNorm statistics, objectness biased down
            if isinstance(m, nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.2)
                m.running_var.uniform_(0.5, 1.5)
        model.branch2[1].bias[4::85] -= 3.0
    x = torch.rand(2, 3, 52, 52, device=DEV)           # 13x13 (read in place by the loader warps) and 26x26 grids
    fused = FusedHeadModel(model, x, conf_thres=0.25, nms_thres=0.5)
    assert fused.detector.fused == [True, True] and fused.detector.padded == [None, None]
    got, got_rows = fused(x, return_rows=True)
    assert isinstance(model.branch1[1], nn.Sequential) and isinstance(model.branch2[1], nn.Conv2d)   # heads restored
    # bit-exact against the unfused kernels on the head tensors the tensor-core kernel produces
    feats = fused.features(x)
    hts = [head_forward(f if p is None else ops.pad_feature(f), m, s, 80)
           for f, p, m, s in zip(feats, fused.detector.padded, [model.branch1[1], model.branch2[1]], fused.specs)]
    from pytorch_yolo_b200.detect import detect
    want, want_rows = detect(hts, fused.specs, 80, 0.25, 0.5, return_rows=True)
    assert sum(0 if d is None else len(d) for d in want) > 0
    for g, w, gr, wr in zip(got, want, got_rows, want_rows):
        assert (g is None) == (w is None)
        if g is not None:
            assert torch.equal(g.view(torch.int32), w.view(torch.int32)) and torch.equal(gr, wr)
    # sanity against the model's own forward + non_max_suppression (cuDNN convolution, a different TF32 summation): scores move
    # by ~1e-3, which reorders near-equal overlapping boxes of a random-init model; most kept anchors must still coincide
    with torch.no_grad():
        ref, ref_rows = non_max_suppression(model(x)[0], 0.25, 0.5, return_rows=True)
    for gr, rr in zip(got_rows, ref_rows):
        a = set() if gr is None else set(gr.tolist())
        b = set() if rr is None else set(rr.tolist())
        assert len(a ^ b) <= max(4, len(b) // 5), (len(a), len(b), len(a ^ b))


# ------------------------------------------------------------------------------------------------------------------
# fp32-accurate mode: three TF32 passes over split operands (YOLO_B200_HEAD_FP32X3).  The bar here is the ORACLE
# (oracle/yolo_oracle.py: the reference's op sequence in fp32 on the CPU), not the repo's own kernels.
@pytest.mark.parametrize("batch,c_in,ny,nx,nc,kind", [(2, 64, 16, 20, 80, "block"), (2, 256, 38, 38, 80, "block"),
                                                      (1, 1024, 19, 19, 80, "block"), (2, 512, 12, 12, 80, "plain"),
                                                      (2, 96, 12, 12, 20, "block"), (1, 32, 8, 8, 1, "plain"),
                                                      (2, 64, 16, 20, 37, "block")])
def test_head_convolution_fp32x3_matches_oracle(batch, c_in, ny, nx, nc, kind):
    from oracle import yolo_oracle
    spec = ops.scale_spec(ANCHORS, ny, nx, 16 * max(ny, nx))
    n_out = 3 * (nc + 5)
    mod = conv_block(c_in, n_out, seed=c_in + nc) if kind == "block" else plain_conv(c_in, n_out, nc, seed=3)
    x = torch.randn(batch, c_in, ny, nx, generator=torch.Generator().manual_seed(1))
    xd = x.to(DEV)
    if ny * nx % 4:                                       # 19x19: through the padded copy, like HeadDetector does
        xd = ops.pad_feature(xd)
    got = head_forward(xd, mod, spec, nc, fp32x3=True).cpu()
    if kind == "block":
        bn = mod[1]
        want = yolo_oracle.head_conv(x, mod[0].weight.detach(), None, 0.1,
                                     (bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var, bn.eps))
    else:
        want = yolo_oracle.head_conv(x, mod.weight.detach(), mod.bias.detach())
    # the north_star's tolerance for floating point, 1e-5 relative; the absolute term covers cancellation in the sum of
    # c_in products (both sides accumulate in fp32, in different orders): 2e-6 of sum |w||x| is ~16 ulp of the largest term
    hw = ops.fold_head(mod, "cpu")
    mag = torch.einsum("oc,bcp->bop", hw.weight[:n_out].abs(), x.abs().flatten(2)).view_as(want)
    err = (got - want).abs()
    assert bool((err <= 1e-5 * want.abs() + 2e-6 * mag + 1e-7).all()), float((err / (want.abs() + 1e-3)).max())
    # and the one-pass TF32 kernel is two to three orders of magnitude further away on the same input
    tf = head_forward(xd, mod, spec, nc).cpu()
    assert float((tf - want).abs().max()) > 30 * float(err.max())


def test_head_detector_fp32x3_matches_oracle_detections():
    """feature maps -> detections in the three-pass mode against the oracle's fp32 convolution + decode + NMS: identical
    kept anchor rows and classes, boxes and scores within 1e-5, except for candidates whose score sits within 1e-5
    (relative) of the confidence threshold on either side."""
    from oracle import yolo_oracle
    batch, nc, conf, nms = 2, 80, 0.3, 0.5
    specs, heads, feats = spp_like(batch, seed=11)
    det = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=conf, nms_thres=nms, precision="fp32x3")
    got, got_rows = det.run(feats, return_rows=True, clone=True)
    hts = []
    for m, x in zip(heads, feats):
        if isinstance(m, nn.Conv2d):
            hts.append(yolo_oracle.head_conv(x.cpu(), m.weight.detach().cpu(), m.bias.detach().cpu()))
        else:
            bn = m[1]
            hts.append(yolo_oracle.head_conv(x.cpu(), m[0].weight.detach().cpu(), None, 0.1,
                                             (bn.weight.detach().cpu(), bn.bias.detach().cpu(), bn.running_mean.cpu(),
                                              bn.running_var.cpu(), bn.eps)))
    anchors = [s.anchors for s in specs]
    img = int(round(specs[0].stride * max(specs[0].ny, specs[0].nx)))
    pred = yolo_oracle.decode_heads(hts, anchors, nc, img)
    want, want_rows = yolo_oracle.non_max_suppression_indexed(pred, conf, nms)
    assert assert_fp32x3_detections_match_oracle(got, got_rows, want, want_rows) > 50


def assert_fp32x3_detections_match_oracle(got, got_rows, want, want_rows, score_rtol=3e-5):
    """The three-pass mode's detections against the oracle's on fp32 head tensors: kept anchor rows as sets up to one in
    200, classes equal, scores within ``score_rtol`` relative, boxes within 1e-5 (1e-3 in an image with a one-sided
    detection).  Returns the number of detections the oracle kept."""
    n_total = 0
    for g, gr, o, orow in zip(got, got_rows, want, want_rows):
        gset, oset = set(gr.cpu().tolist()), set(orow.tolist())
        n_total += len(oset)
        assert len(gset ^ oset) <= max(1, len(oset) // 200), (len(gset), len(oset), sorted(gset ^ oset)[:8])
        common = sorted(gset & oset)
        gi = {r: i for i, r in enumerate(gr.cpu().tolist())}
        oi = {r: i for i, r in enumerate(orow.tolist())}
        gsel = g.cpu()[[gi[r] for r in common]]
        osel = o[[oi[r] for r in common]]
        assert torch.equal(gsel[:, 6], osel[:, 6])                                   # class
        # score, class confidence: the kernel's logits t are within ~2e-6 * sum |w||x| of fp64 (the tensor core's fp32
        # accumulation over three passes; the oracle's CPU convolution is closer), which moves sigmoid(t) by
        # (1 - sigmoid(t)) * dt relative: 3e-5 covers that for the spp_like heads (c_in <= 256); 1e-5 is the bar on
        # identical head tensors (test_gpu_parity.py)
        torch.testing.assert_close(gsel[:, 4:6], osel[:, 4:6], rtol=score_rtol, atol=1e-7)
        # boxes: a MERGE box averages its cluster, so a member that differs between the two sides moves it; compare the
        # rows whose clusters cannot have changed (no one-sided detection in the image) strictly, the others loosely
        tol = 1e-5 if gset == oset else 1e-3
        torch.testing.assert_close(gsel[:, :4], osel[:, :4], rtol=tol, atol=tol * 600)
    return n_total
