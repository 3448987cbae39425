"""GPU: the fused head kernel (csrc/head.cu) in its steady state, at the batch sizes the benchmark times.

The kernel is persistent: one CTA per SM takes 128-position tiles round-robin, and its correctness over many tiles rests on
bookkeeping that a small batch never exercises -- the recycling of the two TMEM accumulator stages (a CTA's third tile
waits for the epilogue to drain stage 0), the per-stage parity of the loader warps' barrier when a CTA mixes loader-filled
tiles (19x19, 13x13 planes) with TMA-filled ones, the three-pass mode's converter warps over several tiles, and the CTA
pair's accumulator handshake through the leader.  A slip there shows up only at production batch sizes, as an epilogue
that reads a stale or half-written accumulator in late tiles.  Every test here

  * first checks, with a restatement of the tile dealing, that its shape reaches the state it exists to test (on the
    device's own SM count), so that a change to the dealing or a smaller GPU fails loudly instead of passing vacuously;
  * compares the head values the kernel writes with an fp64 product (of the TF32-truncated operands for the one-pass
    kernel) per element, at a bar relative to S = sum_c |w| |x|: a stale or corrupted accumulator is off by O(S);
  * compares the production instantiation (no head tensor written) with decode_compact + NMS fed the head tensor,
    bit for bit.

Candidates and detections of the last images of a batch are the ones dealt in the last rounds of every CTA: whatever is
checked on a subset of the images is checked on the last ones.
"""
import pytest
import torch

from pytorch_yolo_b200 import ops, synth
from pytorch_yolo_b200.detect import detect
from pytorch_yolo_b200.head import HeadDetector
from tests.test_gpu_head import assert_fp32x3_detections_match_oracle, conv_block, tf32_trunc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CONF, NMS = 0.3, 0.5


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------------------------
# Tile dealing, restated from the host and kernel code
def scale_geometry(feats, specs):
    """(c_in, plane, manual) per scale, in call order, as the host code derives them: ``manual`` = the X rows have no
    16-byte pitch (no tensor map: the kernel's loader warps fill those tiles, head.cu:1056-1058)."""
    out = []
    for x, s in zip(feats, specs):
        plane = s.ny * s.nx
        pitch = x.shape[2] if x.dim() == 3 else plane          # (B, C, pitch) = planes padded by ops.pad_feature
        out.append((x.shape[1], plane, pitch % 4 != 0))
    return out


def heaviest_first(scales):
    """The launch order of the scales: the host's swap sort on c_in, descending (head.cu:1046-1048)."""
    order = list(range(len(scales)))
    for i in range(len(order)):
        for j in range(i + 1, len(order)):
            if scales[order[j]][0] > scales[order[i]][0]:
                order[i], order[j] = order[j], order[i]
    return order


def deal_tiles(scales, batch, sms):
    """Per CTA of the single-CTA kernel, the ordered list of ``(scale, image, tile, manual)`` it works through.

    head.cu:1040-1126: the scales are sorted heaviest ``c_in`` first (:1046-1048), scale k covers global tiles
    ``first_tile .. first_tile + batch * tiles_per_img`` with ``tiles_per_img = ceil(plane / 128)``, image-major
    (:1085-1087), and the grid is ``min(tiles, SMs)`` (:1125).  In the kernel, CTA ``c`` takes tiles ``c, c + grid, ...``
    (:477, :515, :567, :633) and locates each one (:457-466).  ``scale`` indexes ``scales`` (call order)."""
    firsts, n_tiles = [], 0
    for k in heaviest_first(scales):
        tpi = -(-scales[k][1] // 128)
        firsts.append((n_tiles, k, tpi))
        n_tiles += batch * tpi
    grid = min(n_tiles, sms)
    deal = []
    for c in range(grid):
        seq = []
        for t in range(c, n_tiles, grid):
            first, k, tpi = [f for f in firsts if f[0] <= t][-1]
            img, tile = divmod(t - first, tpi)
            seq.append((k, img, tile, scales[k][2]))
        deal.append(seq)
    return deal


def deal_pair_tiles(scales, batch, sms):
    """The CTA-pair kernel: one launch per scale, in the same heaviest-first order (head.cu:1110-1116), on
    ``2 * min(pairs, SMs // 2)`` CTAs; pair ``p`` takes the scale's 256-position tiles ``p, p + n_pairs, ...`` with
    ``tiles_per_img = ceil(plane / 256)`` (:730-732, :776, :802, :829).  Returns, per launch, per pair, the ordered list of
    ``(scale, image, tile)``."""
    launches = []
    for k in heaviest_first(scales):
        tpi = -(-scales[k][1] // 256)
        n_tiles = batch * tpi
        n_pairs = min(n_tiles, sms // 2)
        launches.append([[(k,) + divmod(t, tpi) for t in range(p, n_tiles, n_pairs)] for p in range(n_pairs)])
    return launches


def longest_run(deal):
    return max(len(seq) for seq in deal)


def loader_tiles_before_tma(deal):
    """The most loader-filled tiles a CTA runs before a TMA-filled tile that follows them (0: no CTA switches)."""
    best = 0
    for seq in deal:
        manual = [m for *_, m in seq]
        if False in manual and True in manual[:manual.index(False)]:
            best = max(best, manual.index(False))
    return best


# ------------------------------------------------------------------------------------------------------------------
# References
def check_head_values(got, x, hw, fp32x3=False):
    """``got`` (B, n_out, ny, nx), the head tensor the kernel wrote for feature map ``x`` (B, c_in, ny, nx), against an
    fp64 product on the device, per element:
      * one pass (TF32): the fp64 product of the TF32-truncated operands, |got - ref| <= 2e-6 S + 1e-6;
      * three passes: the fp64 product of the fp32 operands, |got - ref| <= 1e-5 |ref| + 2e-6 S + 1e-7 (the bar of
        test_head_convolution_fp32x3_matches_oracle);
    with S = sum_c |w| |x| over the same operands, then bias and activation in fp64.  Returns the largest err / S."""
    batch, n = got.shape[:2]
    plane = got.shape[2] * got.shape[3]
    w = hw.weight[:n] if fp32x3 else tf32_trunc(hw.weight[:n])
    wd = w.double()
    wa = wd.abs()
    bias = hw.bias.to(got.device).double()[None, :, None]
    step = max(1, (1 << 27) // (n * plane))                  # images per chunk: 1 GB per fp64 intermediate
    worst = 0.0
    for i in range(0, batch, step):
        xs = x[i:i + step].flatten(2)
        xd = (xs if fp32x3 else tf32_trunc(xs)).double()
        ref = torch.matmul(wd, xd) + bias
        if hw.negative_slope != 1.0:
            ref = torch.maximum(ref, ref * hw.negative_slope)
        s = torch.matmul(wa, xd.abs())
        err = (got[i:i + step].flatten(2).double() - ref).abs()
        bar = (1e-5 * ref.abs() + 2e-6 * s + 1e-7) if fp32x3 else (2e-6 * s + 1e-6)
        ratio = float((err / s).max())
        worst = max(worst, ratio)
        excess = err - bar
        if not bool((excess <= 0).all()):                    # NaN fails too
            flat = int(torch.nan_to_num(excess, nan=float("inf")).flatten().argmax())
            b, o, p = flat // (n * plane), (flat // plane) % n, flat % plane
            pytest.fail(f"head value off: image {i + b}, channel {o}, position {p} (tile {p // 128}): got "
                        f"{float(got[i + b].flatten(1)[o, p])}, fp64 {float(ref[b, o, p])}, S {float(s[b, o, p]):.4g}; "
                        f"largest err / S in images {i}..{i + len(xs) - 1}: {ratio:.3e}")
    return worst


def sorted_candidates(buf):
    """(counts, meta, int32 view of box) of the candidates in ``buf``, ordered by (image, anchor row); asserts that the
    overflow flag is clear (it also carries the watchdog code 0x100 + role of a pipeline wait that timed out)."""
    cnt, _, ovf = ops.read_counts(buf)
    assert ovf == 0, f"overflow flag {ovf:#x}"
    cnt = cnt.clone()
    c = cnt.to(buf.device, torch.int64)
    live = (torch.arange(buf.cap, device=buf.device)[None, :] < c[:, None]).flatten()
    n = buf.batch * buf.cap
    meta, box = buf.cand_meta[:n][live], buf.cand_box[:n][live]
    key = torch.repeat_interleave(torch.arange(buf.batch, device=buf.device), c) * (1 << 32) + meta[:, 3].long()
    assert key.unique().numel() == key.numel()              # one candidate per anchor at most
    order = key.argsort()
    return cnt, meta[order], box[order].view(torch.int32)


def assert_same_candidates(got, want, what):
    assert torch.equal(got[0], want[0]), f"{what}: candidate counts differ in images " \
        f"{(got[0] != want[0]).nonzero().flatten().tolist()[:8]}"
    assert torch.equal(got[1], want[1]), f"{what}: score / class confidence / class / row differ"
    assert torch.equal(got[2], want[2]), f"{what}: boxes differ"


def row_offsets(specs):
    offs, o = [], 0
    for s in specs:
        offs.append(o)
        o += s.rows
    return offs, o


def fused_candidates(feats, hws, specs, nc, head_outs=None, cta_pair=False):
    """One launch of the fused kernel over all scales; head_outs given = the instantiation that writes the head tensor."""
    offs, rows = row_offsets(specs)
    buf = ops.Buffers(DEV, feats[0].shape[0], rows, nc)
    ops.head_decode_compact(feats, hws, specs, offs, rows, nc, CONF, buf, head_outs=head_outs, cta_pair=cta_pair)
    return sorted_candidates(buf)


def unfused_candidates(heads, specs, nc):
    buf = ops.Buffers(DEV, heads[0].shape[0], sum(s.rows for s in specs), nc)
    ops.decode_compact(heads, specs, nc, CONF, buf)
    return sorted_candidates(buf)


def assert_same_detections(got, want):
    """(dets, rows) pairs of ragged lists: bit for bit, image by image.  Returns the number of detections."""
    assert len(got[0]) == len(want[0])
    n = 0
    for i, (g, w, gr, wr) in enumerate(zip(got[0], want[0], got[1], want[1])):
        assert (g is None) == (w is None), f"image {i}"
        if g is not None:
            assert torch.equal(g.view(torch.int32), w.view(torch.int32)) and torch.equal(gr, wr), f"image {i}"
            n += len(g)
    return n


def head_tensors(feats, hws, specs):
    return [torch.full((f.shape[0], hw.n_out, s.ny, s.nx), float("nan"), device=DEV) for f, hw, s in zip(feats, hws, specs)]


def spp608_specs():
    w = synth.WORKLOADS["spp-608"]
    return [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]


def spp608_convblocks(nc, seed):
    """ConvBlock heads (1x1 conv + BatchNorm + LeakyReLU(0.1)) with the reference SPP model's input channels."""
    return [conv_block(c, 3 * (nc + 5), seed + i).to(DEV) for i, c in enumerate(synth.WORKLOADS["spp-608"]["head_cin"])]


def device_feats(specs, cins, batch, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(batch, c, s.ny, s.nx, generator=g, device=DEV) for c, s in zip(cins, specs)]


def check_one_pass(heads, specs, feats, nc):
    """The one-pass kernel on all scales in one launch: head values against fp64, and the candidates and detections of both
    instantiations against the unfused path on the head tensor.  Returns the folded weights and the detections of the
    unfused path, so that a caller can compare further runs with them."""
    hws = [ops.fold_head(m, DEV) for m in heads]
    hts = head_tensors(feats, hws, specs)
    with_head = fused_candidates(feats, hws, specs, nc, head_outs=hts)
    worst = [check_head_values(h, x, hw) for h, x, hw in zip(hts, feats, hws)]
    print(f"largest err / S per scale: {', '.join(f'{r:.3e}' for r in worst)}")
    want = unfused_candidates(hts, specs, nc)
    assert int(want[0].sum()) > 0
    assert_same_candidates(with_head, want, "head_out instantiation vs decode_compact")
    assert_same_candidates(fused_candidates(feats, hws, specs, nc), want, "production instantiation vs decode_compact")
    want_det = detect(hts, specs, nc, CONF, NMS, return_rows=True)
    det = HeadDetector(heads, specs, nc, feats[0].shape[0], DEV, conf_thres=CONF, nms_thres=NMS)
    assert det.fused == [True] * len(specs) and det.padded == [None] * len(specs)
    assert assert_same_detections(det.run(feats, return_rows=True, clone=True), want_det) > 0
    return hws, want_det


# ------------------------------------------------------------------------------------------------------------------
def test_spp608_batch64_convblock_heads_and_graph_replays():
    """The benchmark's headline head shape: spp-608, batch 64, ConvBlock heads (the LeakyReLU instantiation), 19x19 read
    in place by the loader warps.  Then a captured CUDA graph replayed on two feature sets copied into the same tensors."""
    nc, batch = 80, 64
    specs = spp608_specs()
    heads = spp608_convblocks(nc, seed=31)
    cins = synth.WORKLOADS["spp-608"]["head_cin"]
    feats = device_feats(specs, cins, batch, seed=32)
    deal = deal_tiles(scale_geometry(feats, specs), batch, sm_count())
    assert longest_run(deal) >= 3, "no CTA recycles an accumulator stage"
    assert loader_tiles_before_tma(deal) >= 2, "no CTA runs two loader-filled tiles and then a TMA tile"
    hws, want1 = check_one_pass(heads, specs, feats, nc)

    feats2 = device_feats(specs, cins, batch, seed=33)
    hts2 = head_tensors(feats2, hws, specs)
    fused_candidates(feats2, hws, specs, nc, head_outs=hts2)
    want2 = detect(hts2, specs, nc, CONF, NMS, return_rows=True)
    static = [torch.empty_like(f) for f in feats]
    det = HeadDetector(heads, specs, nc, batch, DEV, conf_thres=CONF, nms_thres=NMS, use_graph=True)
    for src, want in ((feats, want1), (feats2, want2)):
        for s_, f in zip(static, src):
            s_.copy_(f)
        assert assert_same_detections(det.run(static, return_rows=True, clone=True), want) > 0


def test_tiny416_batch1024_loader_then_tma_tiles():
    """The benchmark's second head shape: tiny-416, batch 1024, its synthetic plain-convolution heads and inputs.  13x13 at
    c_in 512 is loader-filled and dealt first, 26x26 is TMA-filled: every CTA runs about 14 loader tiles, then TMA tiles."""
    batch = 1024
    w = synth.WORKLOADS["tiny-416"]
    nc = w["nc"]
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    feats, convs = synth.synth_head_convs("tiny-416", batch, device=DEV)
    deal = deal_tiles(scale_geometry(feats, specs), batch, sm_count())
    assert longest_run(deal) >= 50
    assert loader_tiles_before_tma(deal) >= 14, "no CTA runs a long stretch of loader-filled tiles before TMA tiles"
    check_one_pass(convs, specs, feats, nc)


@pytest.mark.parametrize("nc", [20, 37], ids=["voc20", "runtime37"])
def test_spp608_class_counts(nc):
    """spp-608 grids and channels, batch 32, ConvBlock heads, at other class counts: 20 classes has its own
    instantiation (80 accumulator columns per stage); 37 runs the run-time class loop over full 256-column stages, so its
    two stages fill the whole 512-column TMEM allocation (head.cu:959-962)."""
    batch = 32
    runtime_loop = nc not in (1, 20, 80)
    assert runtime_loop == (nc == 37)
    specs = spp608_specs()
    heads = spp608_convblocks(nc, seed=41)
    feats = device_feats(specs, synth.WORKLOADS["spp-608"]["head_cin"], batch, seed=42)
    deal = deal_tiles(scale_geometry(feats, specs), batch, sm_count())
    assert longest_run(deal) >= 3, "no CTA recycles an accumulator stage"
    check_one_pass(heads, specs, feats, nc)


def test_spp608_batch16_fp32x3():
    """The three-pass (fp32-accurate) mode at spp-608, batch 16, on the benchmark's synthetic heads: 19x19 through the
    padded copy as in HeadDetector, 976 tiles, up to 7 per CTA through two accumulator stages and the converter warps."""
    from oracle import yolo_oracle
    batch = 16
    w = synth.WORKLOADS["spp-608"]
    nc = w["nc"]
    specs = spp608_specs()
    feats, convs = synth.synth_head_convs("spp-608", batch, device=DEV)
    xs = [ops.pad_feature(x) if (s.ny * s.nx) % 4 else x for x, s in zip(feats, specs)]
    deal = deal_tiles(scale_geometry(xs, specs), batch, sm_count())
    assert longest_run(deal) >= 3, "no CTA recycles an accumulator stage"
    hws = [ops.fold_head(m, DEV, fp32x3=True) for m in convs]
    hts = head_tensors(feats, hws, specs)
    got = fused_candidates(xs, hws, specs, nc, head_outs=hts)
    worst = [check_head_values(h, x, hw, fp32x3=True) for h, x, hw in zip(hts, feats, hws)]
    print(f"largest err / S per scale: {', '.join(f'{r:.3e}' for r in worst)}")
    want = unfused_candidates(hts, specs, nc)
    assert int(want[0].sum()) > 0
    assert_same_candidates(got, want, "fp32x3 kernel vs decode_compact on its own head tensor")

    det = HeadDetector(convs, specs, nc, batch, DEV, conf_thres=CONF, nms_thres=NMS, precision="fp32x3")
    assert det.fused == [True] * 3 and det.padded[0] is not None
    dets, rows = det.run(feats, return_rows=True, clone=True)
    ref = [yolo_oracle.head_conv(x[-2:].cpu(), m.weight.detach().cpu(), m.bias.detach().cpu()) for x, m in zip(feats, convs)]
    pred = yolo_oracle.decode_heads(ref, [s.anchors for s in specs], nc, w["img_size"])
    want_det, want_rows = yolo_oracle.non_max_suppression_indexed(pred, CONF, NMS)
    # The logits differ from the oracle's mostly by the kernel's accumulation error, ~2e-6 S at most (checked per element
    # above; the oracle's CPU convolution is closer to fp64).  For unit-variance features S = sum_c |w| |x| grows as
    # sqrt(c_in): at c_in = 1024 it is twice that of the c_in <= 256 heads the oracle test's 3e-5 on scores was set on.
    score_rtol = 3e-5 * (max(w["head_cin"]) / 256) ** 0.5
    assert assert_fp32x3_detections_match_oracle(dets[-2:], rows[-2:], want_det, want_rows, score_rtol) > 50


def test_cta_pair_spp608_batch16():
    """The CTA-pair kernel on the spp-608 38x38 and 76x76 scales (c_in 512, 256), batch 16: about five pair tiles per pair
    on 76x76, so the leader's accumulator stages are recycled on the peer's remote arrivals."""
    nc, batch = 80, 16
    specs = spp608_specs()[1:]
    cins = synth.WORKLOADS["spp-608"]["head_cin"][1:]
    heads = [conv_block(c, 255, seed=51 + i).to(DEV) for i, c in enumerate(cins)]
    feats = device_feats(specs, cins, batch, seed=52)
    launches = deal_pair_tiles(scale_geometry(feats, specs), batch, sm_count())
    assert max(longest_run(pairs) for pairs in launches) >= 3, "no pair recycles an accumulator stage"
    hws = [ops.fold_head(m, DEV) for m in heads]
    hts = head_tensors(feats, hws, specs)
    got = fused_candidates(feats, hws, specs, nc, head_outs=hts, cta_pair=True)
    worst = [check_head_values(h, x, hw) for h, x, hw in zip(hts, feats, hws)]
    print(f"largest err / S per scale: {', '.join(f'{r:.3e}' for r in worst)}")
    want = unfused_candidates(hts, specs, nc)
    assert int(want[0].sum()) > 0
    assert_same_candidates(got, want, "pair kernel vs decode_compact on its own head tensor")
    assert_same_candidates(fused_candidates(feats, hws, specs, nc, cta_pair=True), want,
                           "pair kernel, production instantiation, vs decode_compact")
    single = head_tensors(feats, hws, specs)
    fused_candidates(feats, hws, specs, nc, head_outs=single)
    for k, (p, s) in enumerate(zip(hts, single)):
        diff = p.view(torch.int32) != s.view(torch.int32)
        assert not bool(diff.any()), f"scale {k}: {int(diff.sum())} of {diff.numel()} head values differ between the " \
            f"pair and the single-CTA kernel, max |diff| {float((p - s).abs().max()):.3e}"
