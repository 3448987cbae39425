"""The gated decode_compact kernel ("auto" / "ldg": objectness first, box and class planes only where it can pass) against
the dense kernels that read every plane ("ldg_dense", "tma2d").  Candidates are compared after sorting by anchor row
(compaction order is not deterministic): meta, box, counts and the overflow flag must be bit-equal.

The LDG CTA covers 128 units of 4 positions (planes that are a multiple of 4 floats) or of 1 position (19x19, 13x13,
odd test planes): the shapes below end in partial CTAs, and the sparsity patterns are laid out on those lane groups."""
import math

import numpy as np
import pytest
import torch

from pytorch_yolo_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GATED = ("auto", "ldg")
DENSE = ("ldg_dense", "tma2d")


def workload_specs(workload):
    w = synth.WORKLOADS[workload]
    return [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])], w


def candidates(heads, specs, nc, conf, variant, cap=None, split=None):
    """Per image (meta, box) sorted by anchor row, the counts and the overflow flag.  ``split``: decode scales [0, split)
    and then the rest into the same buffers, both in accumulate mode."""
    batch = heads[0].shape[0]
    rows = sum(s.rows for s in specs)
    buf = ops.Buffers(DEV, batch, cap or rows, nc)
    if split is None:
        ops.decode_compact(heads, specs, nc, conf, buf, variant=variant)
    else:
        offs = np.cumsum([0] + [s.rows for s in specs]).tolist()
        buf.meta.zero_()                                   # accumulate mode leaves the counters to the caller
        ops.decode_compact(heads[:split], specs[:split], nc, conf, buf, variant=variant, row_offs=offs[:split],
                           rows_per_img=rows, accumulate=True)
        ops.decode_compact(heads[split:], specs[split:], nc, conf, buf, variant=variant, row_offs=offs[split:len(specs)],
                           rows_per_img=rows, accumulate=True)
    counts, _, overflow = ops.read_counts(buf)
    counts = counts.clone()
    per_img = []
    for b in range(batch):
        n = min(int(counts[b]), buf.cap)
        meta = buf.cand_meta[b * buf.cap:b * buf.cap + n].cpu()
        box = buf.cand_box[b * buf.cap:b * buf.cap + n].cpu()
        order = torch.argsort(meta[:, 3])
        per_img.append((meta[order], box[order]))
    return per_img, counts, overflow


def assert_variants_equal(heads, specs, nc, conf, **kw):
    got = {v: candidates(heads, specs, nc, conf, v, **kw) for v in GATED + DENSE}
    want_imgs, want_counts, want_ovf = got["ldg_dense"]
    for v in GATED + DENSE:
        imgs, counts, ovf = got[v]
        assert torch.equal(counts, want_counts), v
        assert ovf == want_ovf, v
        for (ma, ba), (mb, bb) in zip(imgs, want_imgs):
            assert torch.equal(ma, mb) and torch.equal(ba, bb), v
    return want_counts, want_ovf


def random_heads(specs, nc, batch, seed, obj_mean=-7.0):
    """SYNTH-A-like logits for any class count."""
    g = torch.Generator().manual_seed(seed)
    heads = []
    for s in specs:
        h = torch.empty(batch, s.na, 5 + nc, s.ny, s.nx)
        h[:, :, 0:4].normal_(0.0, 0.5, generator=g)
        h[:, :, 4].normal_(obj_mean, 3.0, generator=g)
        h[:, :, 5:].normal_(-2.0, 2.0, generator=g)
        heads.append(h.view(batch, -1, s.ny, s.nx))
    return heads


SHAPES = [("mini-96", 3), ("mini-96", 37), ("mini-160", 5), ("tiny-416", 7), ("spp-608", 5), ("spp-1024", 2)]


@pytest.mark.parametrize("workload,batch", SHAPES)
@pytest.mark.parametrize("kind", ["A", "B"])
@pytest.mark.parametrize("conf", [0.001, 0.05, 0.3, 0.9])
def test_gated_equals_dense_on_workloads(workload, batch, kind, conf):
    specs, w = workload_specs(workload)
    heads = [h.to(DEV) for h in synth.synth_heads(workload, batch, kind, seed=17)]
    counts, _ = assert_variants_equal(heads, specs, w["nc"], conf)
    if conf <= 0.3:
        assert int(counts.sum()) > 0


def single_scale(ny, nx, na, nc):
    return [ops.scale_spec([(10.0, 13.0), (16.0, 30.0), (33.0, 23.0)][:na], ny, nx, 64 * max(ny, nx))]


@pytest.mark.parametrize("ny,nx", [(64, 64), (63, 65)])
@pytest.mark.parametrize("conf", [0.05, 0.3, 0.9])
def test_gate_boundary(ny, nx, conf):
    """4096 consecutive fp32 objectness logits around logit(conf), one class logit at 30 so that sigma(max) is 1.0: where
    the gate, the cheap test and the final test meet."""
    nc = 80
    specs = single_scale(ny, nx, 1, nc)
    h = torch.full((1, 5 + nc, ny, nx), -10.0)
    h[0, 0:4] = 0.0
    h[0, 5 + 17] = 30.0
    centre = torch.tensor([math.log(conf / (1 - conf))], dtype=torch.float32).view(torch.int32)
    bits = centre + torch.arange(-2048, 2048, dtype=torch.int32)[: ny * nx]
    h[0, 4] = bits.view(torch.float32).view(ny, nx)
    counts, _ = assert_variants_equal([h.to(DEV)], specs, nc, conf)
    assert 0 < int(counts[0]) < ny * nx


def test_nan_and_inf():
    """NaN / -inf objectness, NaN box and class logits of passing and of gated-off anchors, +inf class logits, and the
    {20, 25} sigmoid collapse that sends an anchor to the rescan."""
    specs, w = workload_specs("mini-96")
    heads = [torch.full_like(h, -9.0) for h in synth.synth_heads("mini-96", 2, "A", seed=1)]
    nan, inf = float("nan"), float("inf")
    for k, h in enumerate(heads):
        v = h.view(2, 3, 85, specs[k].ny, specs[k].nx)
        v[:, :, 0:4] = 0.0
        g = specs[k].ny
        v[0, 0, 4, 0, 0] = nan                                                     # NaN objectness
        v[0, 0, 4, 0, 1] = -inf                                                    # -inf objectness
        v[0, 1, 4, 0, 0] = 6.0; v[0, 1, 5 + 1, 0, 0] = 5.0; v[0, 1, 0, 0, 0] = nan  # NaN box, passing anchor
        v[0, 1, 1, 0, 1] = nan; v[0, 1, 5 + 3, 0, 1] = nan                         # NaN box / class, gated-off anchor
        v[0, 2, 4, 1, 0] = 6.0; v[0, 2, 5 + 1, 1, 0] = 5.0; v[0, 2, 5 + 4, 1, 0] = nan  # NaN class, passing anchor
        v[0, 2, 4, g - 1, 0] = 6.0; v[0, 2, 5 + 2, g - 1, 0] = 5.0                 # an ordinary candidate
        v[1, 0, 4, 1, 1] = 6.0; v[1, 0, 5 + 9, 1, 1] = inf                         # +inf class logit
        v[1, 1, 4, 2, 2] = 6.0; v[1, 1, 5 + 10, 2, 2] = 20.0; v[1, 1, 5 + 40, 2, 2] = 25.0   # rescan: class 10
        v[1, 2, 4, g - 1, g - 1] = 6.0; v[1, 2, 5 + 2, g - 1, g - 1] = 5.0         # an ordinary candidate
    dev_heads = [h.to(DEV) for h in heads]
    counts, _ = assert_variants_equal(dev_heads, specs, 80, 0.3)
    assert counts.tolist() == [3 * 1, 3 * 3]                                        # per scale: 1 in image 0, 3 in image 1
    # and sprinkled over realistic heads
    g = torch.Generator().manual_seed(5)
    heads = synth.synth_heads("mini-160", 4, "B", seed=3)
    for h in heads:
        u = torch.rand(h.shape, generator=g)
        h[u < 0.01] = nan
        h[(u >= 0.01) & (u < 0.02)] = inf
        h[(u >= 0.02) & (u < 0.03)] = -inf
    specs, _ = workload_specs("mini-160")
    assert_variants_equal([h.to(DEV) for h in heads], specs, 80, 0.05)


# lanes of one warp hold 32 units of 4 positions (64 x 64 plane) or of 1 position (63 x 65 plane)
PATTERNS = ["one_per_warp", "one_per_sector", "alternate_lanes", "every_lane"]


@pytest.mark.parametrize("ny,nx", [(64, 64), (63, 65)])
@pytest.mark.parametrize("pattern", PATTERNS)
def test_sparsity_patterns(ny, nx, pattern):
    nc, na, batch = 80, 3, 2
    specs = single_scale(ny, nx, na, nc)
    vec = 4 if (ny * nx) % 4 == 0 else 1
    g = torch.Generator().manual_seed(11)
    h = torch.empty(batch, na, 5 + nc, ny * nx)
    h[:, :, 0:2].normal_(0.0, 0.5, generator=g)
    h[:, :, 2:4] = 0.0                                                  # every passing anchor's box is large enough
    h[:, :, 5:].normal_(-2.0, 2.0, generator=g)
    h[:, :, 5 + 7] = 8.0
    pos = torch.arange(ny * nx)
    unit = torch.arange(batch * na).view(batch, na, 1) * (ny * nx // vec) + pos // vec   # units run on across slabs
    lane = unit % 32
    on = {"one_per_warp": lane == 13, "one_per_sector": (lane % 8) == 5, "alternate_lanes": (lane % 2) == 0,
          "every_lane": torch.ones_like(lane, dtype=torch.bool)}[pattern]
    if pattern != "every_lane":
        on = on & ((pos % vec) == (pos // 97) % vec)                  # one position of each passing unit
    h[:, :, 4] = torch.where(on, torch.tensor(4.0), torch.tensor(-20.0))
    heads = [h.view(batch, -1, ny, nx).to(DEV)]
    counts, _ = assert_variants_equal(heads, specs, nc, 0.3)
    assert counts.tolist() == on.view(batch, -1).sum(1).tolist()


@pytest.mark.parametrize("nc", [1, 20, 37, 80])
@pytest.mark.parametrize("conf", [0.05, 0.3])
def test_class_counts(nc, conf):
    w = synth.WORKLOADS["mini-160"]
    specs = [ops.scale_spec(a, gr, gr, w["img_size"]) for a, gr in zip(w["anchors"], w["grids"])]
    heads = [h.to(DEV) for h in random_heads(specs, nc, 6, seed=nc)]
    counts, _ = assert_variants_equal(heads, specs, nc, conf)
    assert int(counts.sum()) > 0


def test_accumulate_mode():
    """Scale 0 first, the others appended (what the fused head's fallback does for scales it cannot take)."""
    specs, w = workload_specs("tiny-416")
    heads = [h.to(DEV) for h in synth.synth_heads("tiny-416", 5, "B", seed=23)]
    acc, _ = assert_variants_equal(heads, specs, w["nc"], 0.3, split=1)
    whole, _ = assert_variants_equal(heads, specs, w["nc"], 0.3)
    assert torch.equal(acc, whole)


def test_overflowing_cap():
    """Counts and the overflow flag are those of the dense kernel; the stored candidates are some of its candidates."""
    specs, w = workload_specs("mini-160")
    heads = [h.to(DEV) for h in synth.synth_heads("mini-160", 3, "B", seed=29)]
    full_imgs, full_counts, _ = candidates(heads, specs, w["nc"], 0.05, "ldg_dense")
    cap = 16
    assert int(full_counts.min()) > cap
    for v in GATED + DENSE:
        imgs, counts, ovf = candidates(heads, specs, w["nc"], 0.05, v, cap=cap)
        assert ovf == 1 and torch.equal(counts, full_counts), v
        for (m, b), (fm, fb) in zip(imgs, full_imgs):
            assert len(m) == cap
            idx = torch.searchsorted(fm[:, 3].contiguous(), m[:, 3].contiguous())
            assert torch.equal(fm[idx], m) and torch.equal(fb[idx], b), v
