"""decode_compact on channels_last heads (YOLO_B200_VARIANT_NHWC, decode_compact_nhwc_kernel).  The contract: heads whose
memory is channels_last give exactly the candidates of the same call on their NCHW copies ``[h.contiguous() for h in
heads]`` -- meta and box records bit-equal after sorting by (image, anchor row), equal counts and overflow flag -- at every
dtype.  Every result built on it (detect, Detector, PipelinedDetector, EvalPipeline) follows and is checked here too."""
import ctypes as C

import pytest
import torch

from pytorch_yolo_b200 import YOLOLayer, _lib, detect_layers, ops, synth
from pytorch_yolo_b200.detect import Detector, PipelinedDetector, detect
from tests.test_gpu_decode_gated import SHAPES, candidates, random_heads, single_scale, workload_specs
from tests.test_gpu_decode_half import assert_same_candidates, assert_same_dets
from tests.test_gpu_parity import make_layers

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
DT_IDS = ["fp32", "fp16", "bf16"]
CL = torch.channels_last


def nhwc(heads):
    out = [h.contiguous(memory_format=CL) for h in heads]
    assert all(ops.is_channels_last(h) for h in out)
    return out


def assert_same_as_nchw(cl_heads, specs, nc, conf, **kw):
    """decode_compact on the channels_last heads against the same call on their NCHW copies; returns the counts."""
    want = candidates([h.contiguous() for h in cl_heads], specs, nc, conf, "auto", **kw)
    assert_same_candidates(candidates(cl_heads, specs, nc, conf, "auto", **kw), want, "channels_last vs NCHW copy")
    return want[1]


def peak_extra_bytes(fn):
    """Bytes the caching allocator hands out beyond what is allocated now while ``fn`` runs: 0 when the heads are read in
    place, the size of the NCHW copies when they are copied first."""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


# ------------------------------------------------------------------------------------------ 1. workloads
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("workload,batch", SHAPES)
@pytest.mark.parametrize("kind", ["A", "B"])
@pytest.mark.parametrize("conf", [0.001, 0.3, 0.9])
def test_workloads_equal_nchw(dtype, workload, batch, kind, conf):
    specs, w = workload_specs(workload)
    heads = nhwc([h.to(DEV).to(dtype) for h in synth.synth_heads(workload, batch, kind, seed=17)])
    counts = assert_same_as_nchw(heads, specs, w["nc"], conf)
    if conf <= 0.3:
        assert int(counts.sum()) > 0


def test_channels_last_heads_are_read_in_place():
    specs, w = workload_specs("spp-608")
    heads = nhwc([h.to(DEV) for h in synth.synth_heads("spp-608", 2, "B", seed=3)])
    buf = ops.Buffers(DEV, 2, sum(s.rows for s in specs), w["nc"])
    assert peak_extra_bytes(lambda: ops.decode_compact(heads, specs, w["nc"], 0.3, buf)) == 0
    copies = sum(h.numel() * h.element_size() for h in heads)
    assert peak_extra_bytes(lambda: ops.decode_compact(heads, specs, w["nc"], 0.3, buf, variant="ldg")) >= copies


# ------------------------------------------------------------------------------------------ 2. geometry
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("ny,nx", [(19, 19), (13, 13), (10, 23), (1, 7), (1, 1)])
@pytest.mark.parametrize("na", [1, 3, 8])
def test_grids_and_anchor_counts(dtype, ny, nx, na):
    spec = ops.scale_spec([(10.0 + 3 * a, 13.0 + 5 * a) for a in range(na)], ny, nx, 32 * max(ny, nx))
    h = random_heads([spec], 80, 5, seed=ny * nx + na, obj_mean=-2.0)[0].to(DEV).to(dtype)
    cl = h.contiguous(memory_format=CL)
    counts = assert_same_as_nchw([cl], [spec], 80, 0.05)
    assert int(counts.sum()) > 0


def rows_tile(nc, esize):
    """Rows per tile the host picks for decode_compact_nhwc_kernel (decode.cu)."""
    r = 128
    while r > 16 // esize and 2 * r * (nc + 5) * esize > 200 * 1024:
        r //= 2
    return r


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("nc", [1, 2, 195, 196, 395, 396, 795, 796, 1595, 1596, 3195, 3196, 4096])
def test_class_counts_across_every_tile_size_many_tiles_per_cta(dtype, nc):
    """Class counts on both sides of every change of the rows per tile, each with enough rows that every CTA of the
    persistent grid runs at least three tiles (both ring stages refilled)."""
    esize = 4 if dtype == torch.float32 else 2
    r = rows_tile(nc, esize)
    smem = 2 * r * (nc + 5) * esize
    grid = torch.cuda.get_device_properties(0).multi_processor_count * max(1, (220 * 1024) // (smem + 1024))
    spec = ops.scale_spec([(10.0, 13.0), (16.0, 30.0), (33.0, 23.0)], 16, 16, 512)
    batch = -(-(3 * grid * r + r // 2) // spec.rows)             # and a tail tile
    h = random_heads([spec], nc, batch, seed=nc, obj_mean=-3.0)[0].to(DEV).to(dtype)
    counts = assert_same_as_nchw([h.contiguous(memory_format=CL)], [spec], nc, 0.3)
    assert int(counts.sum()) > 0


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_head_at_an_unaligned_storage_offset(dtype):
    """channels_last memory one element into a buffer: not 16-byte aligned, so every tile takes the plain copy."""
    specs, w = workload_specs("tiny-416")
    src = [h.to(dtype) for h in synth.synth_heads("tiny-416", 3, "B", seed=5)]
    heads = []
    for h in src:
        b, c, ny, nx = h.shape
        store = torch.empty(h.numel() + 1, dtype=dtype, device=DEV)
        v = store[1:].view(b, ny, nx, c).permute(0, 3, 1, 2)
        v.copy_(h.to(DEV))
        assert ops.is_channels_last(v) and v.data_ptr() % 16 != 0
        heads.append(v)
    assert int(assert_same_as_nchw(heads, specs, w["nc"], 0.3).sum()) > 0


# ------------------------------------------------------------------------------------------ 3. values
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_nan_inf_and_near_ties(dtype):
    """NaN and +-inf sprinkled over every channel, and anchors whose two largest class logits ({20, 25}) have the same
    fp32 sigmoid, which sends them to rescan_classes over the row in shared memory."""
    specs, w = workload_specs("mini-160")
    g = torch.Generator().manual_seed(5)
    heads = synth.synth_heads("mini-160", 4, "B", seed=3)
    for h in heads:
        u = torch.rand(h.shape, generator=g)
        h[u < 0.01] = float("nan")
        h[(u >= 0.01) & (u < 0.02)] = float("inf")
        h[(u >= 0.02) & (u < 0.03)] = float("-inf")
        v = h.view(h.shape[0], 3, 85, h.shape[2], h.shape[3])
        v[:, :, 4, ::3, ::2] = 6.0
        v[:, :, 5 + 10, ::3, ::2] = 20.0
        v[:, :, 5 + 40, ::3, ::2] = 25.0
        v[:, :, 0:4, ::3, ::2] = 0.0
    cl = nhwc([h.to(DEV).to(dtype) for h in heads])
    assert int(assert_same_as_nchw(cl, specs, 80, 0.05).sum()) > 0
    # the rescan picks class 10 (sigma(20) == sigma(25) == 1.0 in fp32): the first arg-max of the decoded tensor
    imgs, counts, _ = candidates(cl, specs, 80, 0.05, "auto")
    assert any(bool((m[:, 2] == 10).any()) for m, _ in imgs)


# ------------------------------------------------------------------------------------------ 4. modes
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_accumulate_split_and_overflowing_cap(dtype):
    specs, w = workload_specs("tiny-416")
    cl = nhwc([h.to(DEV).to(dtype) for h in synth.synth_heads("tiny-416", 5, "B", seed=23)])
    acc = assert_same_as_nchw(cl, specs, w["nc"], 0.3, split=1)
    assert_same_candidates(candidates(cl, specs, w["nc"], 0.3, "auto", split=1), candidates(cl, specs, w["nc"], 0.3, "auto"),
                           "split vs whole")
    assert int(acc.sum()) > 0
    specs, w = workload_specs("mini-160")
    cl = nhwc([h.to(DEV).to(dtype) for h in synth.synth_heads("mini-160", 3, "B", seed=29)])
    full_imgs, full_counts, _ = candidates([h.contiguous() for h in cl], specs, w["nc"], 0.05, "ldg_dense")
    cap = 16
    assert int(full_counts.min()) > cap
    imgs, counts, ovf = candidates(cl, specs, w["nc"], 0.05, "auto", cap=cap)
    assert ovf == 1 and torch.equal(counts, full_counts)
    for (m, b), (fm, fb) in zip(imgs, full_imgs):
        assert len(m) == cap
        idx = torch.searchsorted(fm[:, 3].contiguous(), m[:, 3].contiguous())
        assert torch.equal(fm[idx], m) and torch.equal(fb[idx].view(torch.int32), b.view(torch.int32))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_mixed_layouts_and_explicit_variants_copy_to_nchw(dtype):
    specs, w = workload_specs("tiny-416")
    heads = [h.to(DEV).to(dtype) for h in synth.synth_heads("tiny-416", 4, "B", seed=31)]
    want = candidates(heads, specs, w["nc"], 0.3, "auto")
    assert int(want[1].sum()) > 0
    mixed = [heads[0].contiguous(memory_format=CL), heads[1]]
    assert_same_candidates(candidates(mixed, specs, w["nc"], 0.3, "auto"), want, "mixed layouts")
    for v in ("ldg", "ldg_dense"):
        assert_same_candidates(candidates(nhwc(heads), specs, w["nc"], 0.3, v), want, v)
    buf = ops.Buffers(DEV, 4, sum(s.rows for s in specs), w["nc"])
    assert peak_extra_bytes(lambda: ops.decode_compact(mixed, specs, w["nc"], 0.3, buf)) >= mixed[0].numel() * mixed[0].element_size()


# ------------------------------------------------------------------------------------------ 5. end to end
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_detect_and_detect_layers(dtype):
    specs, w = workload_specs("spp-608")
    heads = [h.to(DEV).to(dtype) for h in synth.synth_heads("spp-608", 3, "B", seed=31)]
    cl = nhwc(heads)
    want = detect(heads, specs, w["nc"], 0.3, 0.5, return_rows=True)
    assert any(d is not None for d in want[0])
    assert_same_dets(detect(cl, specs, w["nc"], 0.3, 0.5, return_rows=True), want)
    if dtype == torch.float32:
        layers, _ = make_layers("spp-608")
        assert_same_dets(detect_layers(layers, cl, w["img_size"], 0.3, 0.5, return_rows=True),
                         detect_layers(layers, heads, w["img_size"], 0.3, 0.5, return_rows=True))


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("use_graph", [False, True], ids=["eager", "graph"])
def test_detector_refilled_in_place(dtype, use_graph):
    specs, w = workload_specs("tiny-416")
    batch = 4
    det = Detector(specs, w["nc"], batch, DEV, 0.3, 0.5, use_graph=use_graph)
    ref = Detector(specs, w["nc"], batch, DEV, 0.3, 0.5, use_graph=False)
    static = [torch.empty(h.shape, dtype=dtype, device=DEV, memory_format=CL)
              for h in synth.synth_heads("tiny-416", batch, "B", seed=0)]
    for step in range(3):
        for s, h in zip(static, synth.synth_heads("tiny-416", batch, "B", seed=40 + step)):
            s.copy_(h.to(DEV).to(dtype))
        want = ref.run([s.contiguous() for s in static], return_rows=True, clone=True)
        assert any(d is not None for d in want[0])
        assert_same_dets(det.run(static, return_rows=True), want)


@pytest.mark.parametrize("direction", ["nchw_then_channels_last", "channels_last_then_nchw"])
def test_detector_rebinds_when_only_the_layout_changes(direction):
    """A channels_last tensor at the address of the NCHW tensor the graph was captured for (or the reverse) must not
    replay the graph of the other layout."""
    specs, w = workload_specs("tiny-416")
    det = Detector(specs, w["nc"], 2, DEV, 0.3, 0.5, use_graph=True)
    first = [h.to(DEV) for h in synth.synth_heads("tiny-416", 2, "B", seed=50)]
    if direction == "channels_last_then_nchw":
        first = nhwc(first)
    det.run(first)
    # the same storage, viewed in the other layout, filled with new values in that layout
    if direction == "nchw_then_channels_last":
        other = [s.view(s.shape[0], s.shape[2], s.shape[3], s.shape[1]).permute(0, 3, 1, 2) for s in first]
    else:
        other = [torch.as_strided(s, s.shape, (s.shape[1] * s.shape[2] * s.shape[3], s.shape[2] * s.shape[3], s.shape[3], 1))
                 for s in first]
    assert [a.data_ptr() for a in other] == [b.data_ptr() for b in first]
    assert [ops.is_channels_last(a) for a in other] == [direction == "nchw_then_channels_last"] * len(other)
    new = [h.to(DEV) for h in synth.synth_heads("tiny-416", 2, "B", seed=51)]
    for a, h in zip(other, new):
        a.copy_(h)
    want = Detector(specs, w["nc"], 2, DEV, 0.3, 0.5, use_graph=False).run(new, return_rows=True, clone=True)
    assert any(d is not None for d in want[0])
    assert_same_dets(det.run(other, return_rows=True), want)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_pipelined_submit_and_submit_host(dtype):
    specs, w = workload_specs("spp-608")
    batch = 2
    sets = [[h.to(dtype) for h in synth.synth_heads("spp-608", batch, "B", seed=60 + k)] for k in range(3)]
    pcl = PipelinedDetector(specs, w["nc"], batch, DEV, 0.3, 0.5, depth=2)
    ref = PipelinedDetector(specs, w["nc"], batch, DEV, 0.3, 0.5, depth=2)
    dev_sets = [[h.to(DEV) for h in s] for s in sets]
    tickets = [(pcl.submit(nhwc(s)), ref.submit(s)) for s in dev_sets]
    for t, r in tickets:
        want = ref.collect(r, return_rows=True, clone=True)
        assert any(d is not None for d in want[0])
        assert_same_dets(pcl.collect(t, return_rows=True, clone=True), want)
    host = [[h.contiguous(memory_format=CL).pin_memory() for h in s] for s in sets]
    assert host[0][0].is_pinned() and ops.is_channels_last(host[0][0])
    tickets = [(pcl.submit_host(s), ref.submit(d)) for s, d in zip(host, dev_sets)]
    for t, r in tickets:
        assert_same_dets(pcl.collect(t, return_rows=True, clone=True), ref.collect(r, return_rows=True, clone=True))
    assert all(ops.is_channels_last(d) for d in pcl._staging[0])


class _Stub:
    """A model for EvalPipeline whose backbone returns the given heads, looked up by the batch id in the image tensor."""

    def __init__(self, workload, heads_per_batch):
        w = synth.WORKLOADS[workload]
        self.yolo_layers = [YOLOLayer(a, w["nc"], w["anchors"]).eval() for a in w["anchors"]]
        self.heads = heads_per_batch

    def _forward_encoder(self, x):
        return tuple(self.heads[int(x[0, 0, 0, 0].item())])


def test_eval_pipeline_over_a_channels_last_backbone():
    from pytorch_yolo_b200.pipeline import EvalPipeline
    wl, batch = "tiny-416", 3
    w = synth.WORKLOADS[wl]
    heads = [[h.to(DEV) for h in synth.synth_heads(wl, batch, "B", seed=70 + k)] for k in range(3)]
    size = w["img_size"]

    def batches():
        for k in range(3):
            yield (torch.full((batch, 3, size, size), float(k)), [f"{k}_{i}.jpg" for i in range(batch)],
                   [(480, 640)] * batch)

    got = EvalPipeline(_Stub(wl, [nhwc(hs) for hs in heads]), DEV, 0.3, 0.5, depth=2).run(batches())
    want = EvalPipeline(_Stub(wl, heads), DEV, 0.3, 0.5, depth=2).run(batches())
    assert want and got == want


# ------------------------------------------------------------------------------------------ 6. buffers
def test_nhwc_kernel_stays_inside_its_buffers():
    """Candidate records and counters carved out of one arena with 4 KB canary zones on both sides (the head too): after
    the NHWC call the canaries are intact and the results equal those of ordinary allocations."""
    lib = _lib.load()
    specs, w = workload_specs("mini-160")
    batch, conf, nc = 3, 0.02, w["nc"]
    heads = nhwc([h.to(DEV) for h in synth.synth_heads("mini-160", batch, "B", seed=123)])
    rows = sum(s.rows for s in specs)
    sizes = {"cand_box": batch * rows * 16, "cand_meta": batch * rows * 16, "meta": (batch + 1) * 4}
    sizes.update({f"head{k}": h.numel() * 4 for k, h in enumerate(heads)})
    guard = 4096
    offs, o = {}, guard
    for k, v in sizes.items():
        offs[k] = o
        o += (v + 255) // 256 * 256 + guard
    arena = torch.full((o,), 0xA5, dtype=torch.uint8, device=DEV)
    base = arena.data_ptr()
    arr = (_lib.Scale * len(heads))()
    row_off = 0
    for k, (s_, sp, h) in enumerate(zip(arr, specs, heads)):
        arena[offs[f"head{k}"]:offs[f"head{k}"] + sizes[f"head{k}"]].view(torch.float32).copy_(h.permute(0, 2, 3, 1).flatten())
        s_.head, s_.ny, s_.nx, s_.na, s_.row_off, s_.stride = base + offs[f"head{k}"], sp.ny, sp.nx, sp.na, row_off, sp.stride
        for a, (aw, ah) in enumerate(sp.anchor_vec.tolist()):
            s_.anchor_vec[a][0], s_.anchor_vec[a][1] = aw, ah
        row_off += sp.rows
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    meta = base + offs["meta"]
    _lib.check(lib.yolo_b200_decode_compact_ex(arr, len(heads), batch, nc, rows, conf, 2.0, base + offs["cand_box"],
                                               base + offs["cand_meta"], rows, meta, meta + 4 * batch, _lib.VARIANT_NHWC,
                                               stream), "decode_compact_ex")
    torch.cuda.synchronize()
    host = arena.cpu()
    prev_end = 0
    for start, end in sorted((offs[k], offs[k] + sizes[k]) for k in sizes) + [(o, o)]:
        assert bool((host[prev_end:start] == 0xA5).all()), f"canary before offset {start} was overwritten"
        prev_end = end
    counts = arena[offs["meta"]:offs["meta"] + 4 * batch].view(torch.int32).cpu()
    assert int(arena[offs["meta"] + 4 * batch:offs["meta"] + 4 * batch + 4].view(torch.int32).item()) == 0
    want_imgs, want_counts, _ = candidates([h.contiguous() for h in heads], specs, nc, conf, "auto")
    assert torch.equal(counts, want_counts) and int(counts.sum()) > 0
    cm = arena[offs["cand_meta"]:offs["cand_meta"] + sizes["cand_meta"]].view(torch.int32).view(batch, rows, 4).cpu()
    cb = arena[offs["cand_box"]:offs["cand_box"] + sizes["cand_box"]].view(torch.float32).view(batch, rows, 4).cpu()
    for b, (wm, wb) in enumerate(want_imgs):
        m, bx = cm[b, :int(counts[b])], cb[b, :int(counts[b])]
        order = torch.argsort(m[:, 3])
        assert torch.equal(m[order], wm) and torch.equal(bx[order].view(torch.int32), wb.view(torch.int32))
