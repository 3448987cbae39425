"""decode_compact on fp16 and bf16 heads.  The contract: 16-bit heads give exactly the candidates of the same call on their
fp32 upcast ``[h.float() for h in heads]`` -- meta and box records bit-equal after sorting by anchor row, equal counts and
overflow flag -- because the kernel converts each value to fp32 as it loads it and runs the fp32 code from there.  Every
result of the fused path (detect, Detector, PipelinedDetector, EvalPipeline) follows from that and is checked here too."""
import pytest
import torch

from oracle import yolo_oracle
from pytorch_yolo_b200 import YOLOLayer, detect_layers, ops, synth
from pytorch_yolo_b200.detect import Detector, PipelinedDetector, detect
from tests.test_gpu_decode_gated import SHAPES, candidates, random_heads, single_scale, workload_specs
from tests.test_gpu_parity import _explain_one_sided, make_layers

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16]
VARIANTS = ("auto", "ldg", "ldg_dense")


def bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int32)


def assert_same_candidates(got, want, what):
    imgs, counts, ovf = got
    want_imgs, want_counts, want_ovf = want
    assert torch.equal(counts, want_counts), what
    assert ovf == want_ovf, what
    for (ma, ba), (mb, bb) in zip(imgs, want_imgs):
        assert torch.equal(ma, mb) and torch.equal(bits(ba), bits(bb)), what


def assert_same_as_upcast(h16, specs, nc, conf, variants=VARIANTS, **kw):
    """Every variant on the 16-bit heads against the same variant on their fp32 upcast; returns the upcast's counts."""
    up = [h.float() for h in h16]
    counts = None
    for v in variants:
        want = candidates(up, specs, nc, conf, v, **kw)
        assert_same_candidates(candidates(h16, specs, nc, conf, v, **kw), want, v)
        counts = want[1]
    return counts


def assert_same_dets(got, want):
    """Ragged results (dets, rows) bit-equal, image by image."""
    (gd, gr), (wd, wr) = got, want
    assert len(gd) == len(wd)
    for a, b, ra, rb in zip(gd, wd, gr, wr):
        assert (a is None) == (b is None)
        if a is not None:
            assert torch.equal(bits(a.cpu()), bits(b.cpu())) and torch.equal(ra.cpu(), rb.cpu())


# ------------------------------------------------------------------------------------------ 1. workloads
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("workload,batch", SHAPES)
@pytest.mark.parametrize("kind", ["A", "B"])
@pytest.mark.parametrize("conf", [0.001, 0.3, 0.9])
def test_workloads_equal_upcast(dtype, workload, batch, kind, conf):
    specs, w = workload_specs(workload)
    h16 = [h.to(DEV).to(dtype) for h in synth.synth_heads(workload, batch, kind, seed=17)]
    counts = assert_same_as_upcast(h16, specs, w["nc"], conf)
    if conf <= 0.3:
        assert int(counts.sum()) > 0


# ------------------------------------------------------------------------------------------ 2. every 16-bit value
def all_values(dtype, shift=0):
    """The 65536 bit patterns of the dtype as a 256 x 256 plane (rolled by `shift` positions)."""
    b = (torch.arange(65536, dtype=torch.int32) - 32768).to(torch.int16)
    return torch.roll(b, shift).view(dtype).view(256, 256)


def plane_heads(dtype, nc=80):
    h = torch.full((1, 5 + nc, 256, 256), -10.0)
    h[0, 0:4] = 0.0
    h[0, 4] = 10.0
    h[0, 5 + 17] = 30.0                                        # sigma(max class) = 1.0
    return h.to(dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("conf", [0.001, 0.3, 0.9])
def test_every_value_as_objectness(dtype, conf):
    h = plane_heads(dtype)
    h[0, 4] = all_values(dtype)
    counts = assert_same_as_upcast([h.to(DEV)], single_scale(256, 256, 1, 80), 80, conf)
    assert 0 < int(counts[0]) < 65536


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("channels", [(2, 3), (0, 1)], ids=["wh", "xy"])
def test_every_value_as_box_logit(dtype, channels):
    """NaN, +-inf, subnormals, -0, the largest finite values (exp overflows: not emitted) in w / h, then in x / y; the
    second channel runs through the same values shifted, so that they meet many different partners."""
    h = plane_heads(dtype)
    h[0, channels[0]] = all_values(dtype)
    h[0, channels[1]] = all_values(dtype, shift=12345)
    counts = assert_same_as_upcast([h.to(DEV)], single_scale(256, 256, 1, 80), 80, 0.3)
    assert 0 < int(counts[0]) < 65536


# ------------------------------------------------------------------------------------------ 3. geometry and alignment
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("ny,nx", [(64, 64), (63, 65), (19, 19)])
@pytest.mark.parametrize("conf", [0.05, 0.3])
def test_plane_shapes(dtype, ny, nx, conf):
    specs = single_scale(ny, nx, 3, 80)
    h16 = [h.to(DEV).to(dtype) for h in random_heads(specs, 80, 3, seed=ny * nx, obj_mean=-3.0)]
    assert int(assert_same_as_upcast(h16, specs, 80, conf).sum()) > 0


@pytest.mark.parametrize("dtype", DTYPES)
def test_head_at_odd_element_offset(dtype):
    """A view one element into a larger buffer: 2-byte aligned only, so the 64 x 64 plane takes the scalar loads."""
    specs = single_scale(64, 64, 3, 80)
    src = random_heads(specs, 80, 2, seed=3, obj_mean=-3.0)[0].to(dtype)
    buf = torch.empty(src.numel() + 1, dtype=dtype, device=DEV)
    h = buf[1:].view(src.shape)
    h.copy_(src.to(DEV))
    assert h.is_contiguous() and h.data_ptr() % 4 == 2
    assert int(assert_same_as_upcast([h], specs, 80, 0.3).sum()) > 0


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("pattern", ["one_per_warp", "one_per_sector", "alternate_lanes", "every_lane"])
def test_sparsity_patterns(dtype, pattern):
    """The lane layouts of the gated kernel on the 64 x 64 plane (units of 4 positions, one 8-byte load per plane)."""
    ny = nx = 64
    nc, na, batch, vec = 80, 3, 2, 4
    specs = single_scale(ny, nx, na, nc)
    g = torch.Generator().manual_seed(11)
    h = torch.empty(batch, na, 5 + nc, ny * nx)
    h[:, :, 0:2].normal_(0.0, 0.5, generator=g)
    h[:, :, 2:4] = 0.0
    h[:, :, 5:].normal_(-2.0, 2.0, generator=g)
    h[:, :, 5 + 7] = 8.0
    pos = torch.arange(ny * nx)
    lane = (torch.arange(batch * na).view(batch, na, 1) * (ny * nx // vec) + pos // vec) % 32
    on = {"one_per_warp": lane == 13, "one_per_sector": (lane % 8) == 5, "alternate_lanes": (lane % 2) == 0,
          "every_lane": torch.ones_like(lane, dtype=torch.bool)}[pattern]
    if pattern != "every_lane":
        on = on & ((pos % vec) == (pos // 97) % vec)
    h[:, :, 4] = torch.where(on, torch.tensor(4.0), torch.tensor(-20.0))
    counts = assert_same_as_upcast([h.view(batch, -1, ny, nx).to(dtype).to(DEV)], specs, nc, 0.3)
    assert counts.tolist() == on.view(batch, -1).sum(1).tolist()


# ------------------------------------------------------------------------------------------ 4. modes
@pytest.mark.parametrize("dtype", DTYPES)
def test_accumulate_split(dtype):
    specs, w = workload_specs("tiny-416")
    h16 = [h.to(DEV).to(dtype) for h in synth.synth_heads("tiny-416", 5, "B", seed=23)]
    acc = assert_same_as_upcast(h16, specs, w["nc"], 0.3, split=1)
    for v in VARIANTS:
        assert_same_candidates(candidates(h16, specs, w["nc"], 0.3, v, split=1), candidates(h16, specs, w["nc"], 0.3, v), v)
    assert int(acc.sum()) > 0


@pytest.mark.parametrize("dtype", DTYPES)
def test_overflowing_cap(dtype):
    specs, w = workload_specs("mini-160")
    h16 = [h.to(DEV).to(dtype) for h in synth.synth_heads("mini-160", 3, "B", seed=29)]
    up = [h.float() for h in h16]
    full_imgs, full_counts, _ = candidates(up, specs, w["nc"], 0.05, "ldg_dense")
    cap = 16
    assert int(full_counts.min()) > cap
    for v in VARIANTS:
        imgs, counts, ovf = candidates(h16, specs, w["nc"], 0.05, v, cap=cap)
        assert ovf == 1 and torch.equal(counts, full_counts), v
        for (m, b), (fm, fb) in zip(imgs, full_imgs):
            assert len(m) == cap
            idx = torch.searchsorted(fm[:, 3].contiguous(), m[:, 3].contiguous())
            assert torch.equal(fm[idx], m) and torch.equal(bits(fb[idx]), bits(b)), v


# ------------------------------------------------------------------------------------------ 5. end to end
@pytest.mark.parametrize("dtype", DTYPES)
def test_detect_and_detect_layers(dtype):
    specs, w = workload_specs("spp-608")
    h16 = [h.to(DEV).to(dtype) for h in synth.synth_heads("spp-608", 3, "B", seed=31)]
    up = [h.float() for h in h16]
    want = detect(up, specs, w["nc"], 0.3, 0.5, return_rows=True)
    assert any(d is not None for d in want[0])
    assert_same_dets(detect(h16, specs, w["nc"], 0.3, 0.5, return_rows=True), want)
    layers, _ = make_layers("spp-608")
    assert_same_dets(detect_layers(layers, h16, w["img_size"], 0.3, 0.5, return_rows=True),
                     detect_layers(layers, up, w["img_size"], 0.3, 0.5, return_rows=True))


@pytest.mark.parametrize("dtype", DTYPES)
def test_detector_graph_refilled_in_place(dtype):
    specs, w = workload_specs("tiny-416")
    batch = 4
    det16 = Detector(specs, w["nc"], batch, DEV, 0.3, 0.5, use_graph=True)
    det32 = Detector(specs, w["nc"], batch, DEV, 0.3, 0.5, use_graph=True)
    static = [torch.empty(h.shape, dtype=dtype, device=DEV) for h in synth.synth_heads("tiny-416", batch, "B", seed=0)]
    static32 = [torch.empty(h.shape, device=DEV) for h in static]
    for step in range(3):
        for s, s32, h in zip(static, static32, synth.synth_heads("tiny-416", batch, "B", seed=40 + step)):
            s.copy_(h.to(DEV).to(dtype))
            s32.copy_(s.float())
        want = det32.run(static32, return_rows=True, clone=True)
        assert any(d is not None for d in want[0])
        assert_same_dets(det16.run(static, return_rows=True), want)


def test_detector_rebinds_when_only_the_dtype_changes():
    """An fp16 tensor at the address of the fp32 tensor the graph was captured for must not replay the fp32 kernel."""
    specs, w = workload_specs("tiny-416")
    heads = synth.synth_heads("tiny-416", 2, "B", seed=50)
    det = Detector(specs, w["nc"], 2, DEV, 0.3, 0.5, use_graph=True)
    storage = [h.to(DEV) for h in heads]
    det.run(storage)
    h16 = [s.view(-1).view(torch.float16)[:s.numel()].view(s.shape) for s in storage]
    assert [a.data_ptr() for a in h16] == [b.data_ptr() for b in storage]
    for a, h in zip(h16, synth.synth_heads("tiny-416", 2, "B", seed=51)):
        a.copy_(h.half())
    want = Detector(specs, w["nc"], 2, DEV, 0.3, 0.5, use_graph=False).run([a.float() for a in h16], return_rows=True,
                                                                           clone=True)
    assert any(d is not None for d in want[0])
    assert_same_dets(det.run(h16, return_rows=True), want)


@pytest.mark.parametrize("dtype", DTYPES)
def test_pipelined_submit_and_submit_host(dtype):
    specs, w = workload_specs("spp-608")
    batch = 2
    sets = [[h.to(dtype) for h in synth.synth_heads("spp-608", batch, "B", seed=60 + k)] for k in range(3)]
    p16 = PipelinedDetector(specs, w["nc"], batch, DEV, 0.3, 0.5, depth=2)
    p32 = PipelinedDetector(specs, w["nc"], batch, DEV, 0.3, 0.5, depth=2)
    dev_sets = [[h.to(DEV) for h in s] for s in sets]
    up_sets = [[h.float() for h in s] for s in dev_sets]
    tickets = [(p16.submit(s), p32.submit(u)) for s, u in zip(dev_sets, up_sets)]
    for t16, t32 in tickets:
        want = p32.collect(t32, return_rows=True, clone=True)
        assert any(d is not None for d in want[0])
        assert_same_dets(p16.collect(t16, return_rows=True, clone=True), want)
    host = [[h.pin_memory() for h in s] for s in sets]
    assert host[0][0].dtype == dtype and host[0][0].is_pinned()
    tickets = [(p16.submit_host(s), p32.submit(u)) for s, u in zip(host, up_sets)]
    for t16, t32 in tickets:
        assert_same_dets(p16.collect(t16, return_rows=True, clone=True), p32.collect(t32, return_rows=True, clone=True))


class _HalfStub:
    """A model for EvalPipeline whose backbone returns 16-bit heads (as a ``.half()`` or autocast model does), looked up
    by the batch id stored in the image tensor."""

    def __init__(self, workload, heads_per_batch):
        w = synth.WORKLOADS[workload]
        self.yolo_layers = [YOLOLayer(a, w["nc"], w["anchors"]).eval() for a in w["anchors"]]
        self.heads = heads_per_batch

    def _forward_encoder(self, x):
        return tuple(self.heads[int(x[0, 0, 0, 0].item())])


@pytest.mark.parametrize("dtype", DTYPES)
def test_eval_pipeline(dtype):
    from pytorch_yolo_b200.pipeline import EvalPipeline
    wl, batch = "tiny-416", 3
    w = synth.WORKLOADS[wl]
    h16 = [[h.to(DEV).to(dtype) for h in synth.synth_heads(wl, batch, "B", seed=70 + k)] for k in range(3)]
    up = [[h.float() for h in hs] for hs in h16]
    size = w["img_size"]

    def batches():
        for k in range(3):
            yield (torch.full((batch, 3, size, size), float(k)), [f"{k}_{i}.jpg" for i in range(batch)],
                   [(480, 640)] * batch)

    got = EvalPipeline(_HalfStub(wl, h16), DEV, 0.3, 0.5, depth=2).run(batches())
    want = EvalPipeline(_HalfStub(wl, up), DEV, 0.3, 0.5, depth=2).run(batches())
    assert want and got == want


# ------------------------------------------------------------------------------------------ 6. against the oracle
@pytest.mark.parametrize("workload,batch", [("tiny-416", 4), ("spp-608", 2)])
def test_fp16_matches_oracle_on_upcast(workload, batch):
    """detect_layers on fp16 heads against the CPU oracle on h16.float(), by the procedure of
    test_fused_matches_oracle_end_to_end (same tolerances, same checked explanations for one-sided detections)."""
    conf, nms_thres = 0.3, 0.5
    layers, w = make_layers(workload)
    h16 = [h.half() for h in synth.synth_heads(workload, batch, "B", seed=61)]
    got, rows = detect_layers(layers, [h.to(DEV) for h in h16], w["img_size"], conf, nms_thres, return_rows=True)
    pred = yolo_oracle.decode_heads([h.float() for h in h16], w["anchors"], w["nc"], w["img_size"])
    want, wrows = yolo_oracle.non_max_suppression_indexed(pred.clone(), conf, nms_thres, write_back=False)
    excluded = total = boxes_checked = 0
    for i, (g, r, o, orow) in enumerate(zip(got, rows, want, wrows)):
        gm = {int(k): v for k, v in zip(r.cpu().tolist(), g.cpu())} if g is not None else {}
        om = {int(k): v for k, v in zip(orow.tolist(), o)} if o is not None else {}
        total += len(om)
        one_sided = set(gm) ^ set(om)
        cand = {}
        if one_sided:
            crow, cdet = yolo_oracle.select_candidates(pred[i].clone(), conf * (1 - 1e-4), write_back=False)
            cand = {int(a): d for a, d in zip(crow.tolist(), cdet)}
        touched_classes = set()
        for k in sorted(one_sided):
            why = _explain_one_sided(k, cand, one_sided, conf, nms_thres)
            assert why is not None, (f"image {i} anchor row {k}: detection on the {'GPU' if k in gm else 'oracle'} side only "
                                     f"with no borderline explanation: {gm.get(k, om.get(k)).tolist()}")
            excluded += 1
            touched_classes.add(float(cand[k][6]))
        for k in set(gm) & set(om):
            assert float(gm[k][6]) == float(om[k][6])
            torch.testing.assert_close(gm[k][4:6], om[k][4:6], rtol=1e-5, atol=1e-12)
            if float(gm[k][6]) not in touched_classes:
                torch.testing.assert_close(gm[k][:4], om[k][:4], rtol=1e-5, atol=1e-4)
                boxes_checked += 1
    assert total > 0
    assert boxes_checked > 0.9 * total
    assert excluded <= max(2, total // 200), f"{excluded} of {total} detections differ between GPU and oracle"


# ------------------------------------------------------------------------------------------ 7. errors
def test_mixed_dtypes_raise_value_error():
    specs, w = workload_specs("tiny-416")
    heads = [h.to(DEV) for h in synth.synth_heads("tiny-416", 1, "B", seed=1)]
    buf = ops.Buffers(DEV, 1, sum(s.rows for s in specs), w["nc"])
    for mixed in ([heads[0].half(), heads[1]], [heads[0].half(), heads[1].bfloat16()]):
        with pytest.raises(ValueError, match="share a dtype"):
            ops.decode_compact(mixed, specs, w["nc"], 0.3, buf)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("variant", ["tma", "tma2d"])
def test_tma_variants_refuse_16_bit_heads(dtype, variant):
    specs, w = workload_specs("tiny-416")
    h16 = [h.to(DEV).to(dtype) for h in synth.synth_heads("tiny-416", 2, "B", seed=1)]
    buf = ops.Buffers(DEV, 2, sum(s.rows for s in specs), w["nc"])
    buf.meta.fill_(7)
    with pytest.raises(ops.YoloB200Error):
        ops.decode_compact(h16, specs, w["nc"], 0.3, buf, variant=variant)
    assert buf.meta.tolist() == [7] * buf.meta.numel()               # nothing was enqueued, not even the counter reset


def test_other_dtypes_and_other_entry_points_raise_type_error():
    from pytorch_yolo_b200 import non_max_suppression
    specs, w = workload_specs("tiny-416")
    heads = [h.to(DEV) for h in synth.synth_heads("tiny-416", 1, "B", seed=1)]
    buf = ops.Buffers(DEV, 1, sum(s.rows for s in specs), w["nc"])
    with pytest.raises(TypeError, match="expected float32 or float16 or bfloat16, got torch.float64"):
        ops.decode_compact([h.double() for h in heads], specs, w["nc"], 0.3, buf)
    h16 = [h.half() for h in heads]
    with pytest.raises(TypeError, match="expected float32, got torch.float16"):
        ops.decode_dense(h16, specs, w["nc"])
    layer = YOLOLayer(w["anchors"][0], w["nc"], w["anchors"]).eval()
    with pytest.raises(TypeError, match="expected float32"):
        layer(h16[0], w["img_size"])
    pred = torch.zeros(1, 10, 5 + w["nc"], dtype=torch.float16, device=DEV)
    with pytest.raises(TypeError, match="expected float32"):
        non_max_suppression(pred, 0.3, 0.5)
    with pytest.raises(TypeError, match="expected float32"):
        ops.compact_from_dense(pred, 0.3, buf)
