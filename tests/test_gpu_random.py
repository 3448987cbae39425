"""GPU: randomised sweeps against the oracle -- shapes (non-square grids, odd planes, 1..8 anchors), class counts,
thresholds, heavy score ties, segment sizes around the 32 / 100 / 128 boundaries."""
import random

import pytest
import torch

from oracle import yolo_oracle
from pytorch_yolo_b200 import YOLOLayer, decode_layers, detect_layers, non_max_suppression, synth
from tests.helpers import assert_dets_equal, prediction_with_class_sizes

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("seed", range(24))
def test_nms_random_configs_bit_exact(seed):
    rng = random.Random(1000 + seed)
    batch = rng.choice([1, 1, 2, 3, 5])
    n = rng.choice([1, 2, 7, 33, 100, 129, 500, 1500, 3000])
    nc = rng.choice([1, 2, 3, 5, 20, 80, 200])
    ties = rng.choice([0, 0, 2, 4, 16])
    conf = rng.choice([0.0, 0.001, 0.05, 0.2, 0.5])
    nms = rng.choice([0.0, 0.1, 0.45, 0.5, 0.7, 0.95])
    pred_cpu = synth.synth_prediction(batch, n, nc=nc, seed=seed, tie_levels=ties)
    if seed % 5 == 0:                                   # sprinkle non-finite values: those rows must drop
        idx = torch.randint(0, n, (max(1, n // 20),))
        pred_cpu[0, idx, rng.randrange(0, 5 + nc)] = rng.choice([float("nan"), float("inf"), float("-inf")])
    pred = pred_cpu.clone().to(DEV)
    got, rows = non_max_suppression(pred, conf, nms, return_rows=True)
    want, wrows = yolo_oracle.non_max_suppression_indexed(pred_cpu, conf, nms)
    assert_dets_equal(got, want, box_rtol=1e-5, what=f"seed {seed} B{batch} N{n} nc{nc} ties{ties} conf{conf} nms{nms}")
    for r, wr in zip(rows, wrows):
        assert (r is None) == (wr is None)
        if r is not None:
            assert torch.equal(r.cpu().long(), wr)
    assert torch.equal(torch.nan_to_num(pred[..., 4].cpu(), nan=-7.0), torch.nan_to_num(pred_cpu[..., 4], nan=-7.0))


@pytest.mark.parametrize("seed", range(12))
def test_decode_random_shapes(seed):
    """Non-square grids (stride uses max(nx, ny), yolo_layer.py:102), odd and aligned planes, 1..8 anchors per scale,
    1..3 scales, several class counts; dense decode within 1e-5 of the oracle and fused == dense bit for bit."""
    rng = random.Random(2000 + seed)
    nc = rng.choice([1, 2, 4, 20, 80, 91])
    n_scales = rng.choice([1, 2, 3])
    img = rng.choice([96, 160, 224, 320])
    batch = rng.choice([1, 2, 3, 7])
    g = torch.Generator().manual_seed(seed)
    layers, heads, anchors_all = [], [], []
    for _ in range(n_scales):
        na = rng.choice([1, 2, 3, 3, 5, 8])
        anchors = tuple((float(rng.randint(4, 120)), float(rng.randint(4, 120))) for _ in range(na))
        anchors_all.append(anchors)
    for anchors in anchors_all:
        ny, nx = rng.choice([(3, 5), (4, 4), (7, 9), (8, 12), (13, 13), (10, 6), (16, 16), (1, 1), (2, 20)])
        h = torch.randn(batch, len(anchors) * (5 + nc), ny, nx, generator=g)
        h[:, 4::5 + nc] += 1.0                              # objectness up a bit so that something passes
        heads.append(h)
        layers.append(YOLOLayer(anchors, nc, anchors_all).eval())
    dev_heads = [h.to(DEV) for h in heads]
    pred, _ = decode_layers(layers, dev_heads, img)
    want = yolo_oracle.decode_heads(heads, anchors_all, nc, img)
    torch.testing.assert_close(pred.cpu(), want, rtol=1e-5, atol=1e-30)
    conf = rng.choice([0.05, 0.2, 0.4])
    fused, frows = detect_layers(layers, dev_heads, img, conf, 0.5, return_rows=True)
    dense, drows = non_max_suppression(pred, conf, 0.5, return_rows=True)
    for f, fr, d, dr in zip(fused, frows, dense, drows):
        assert (f is None) == (d is None)
        if f is not None:
            assert torch.equal(f, d) and torch.equal(fr, dr)


def test_max_per_class_boundaries():
    """Classes holding exactly 31/32/33 and 99/100/101/128/129/300 candidates (warp path vs CTA path vs cap)."""
    for n_in_class in (31, 32, 33, 99, 100, 101, 128, 129, 300):
        g = torch.Generator().manual_seed(n_in_class)
        n = n_in_class + 5
        pred = torch.zeros(1, n, 8)
        pred[0, :, 0:2] = 200 + 60 * torch.randn(n, 2, generator=g)
        pred[0, :, 2:4] = 30 + 20 * torch.rand(n, 2, generator=g)
        pred[0, :, 4] = 0.5 + 0.5 * torch.rand(n, generator=g)
        pred[0, :n_in_class, 5] = 0.9                     # class 0 holds n_in_class boxes
        pred[0, n_in_class:, 6] = 0.8                     # class 1 holds 5
        want, wrows = yolo_oracle.non_max_suppression_indexed(pred.clone(), 0.1, 0.5)
        got, rows = non_max_suppression(pred.clone().to(DEV), 0.1, 0.5, return_rows=True)
        assert_dets_equal(got, want, box_rtol=1e-5, what=f"{n_in_class} in class")
        assert torch.equal(rows[0].cpu().long(), wrows[0])


@pytest.mark.parametrize("nc,grids,batch", [(80, ((19, 19), (38, 38), (76, 76)), 3),     # spp-608: unaligned + aligned planes
                                            (80, ((26, 26), (13, 13)), 5),               # tiny-416
                                            (1, ((16, 16), (8, 12)), 2),                 # 6 floats per row (even pitch)
                                            (20, ((32, 40),), 4),                        # 1280-position planes: 10 full tiles
                                            (130, ((12, 12), (24, 20)), 2),              # 135 rows: 2 input stages + 1 output tile
                                            (80, ((10, 6), (2, 20), (1, 1)), 2)])        # planes smaller than one tile
def test_dense_decode_tma_equals_ldg(nc, grids, batch):
    """The TMA variant of the dense decode (tensor-map tile loads, bulk stores) writes the same bits as the LDG variant,
    including the floats before / after the 16-byte aligned body of every tile and rows next to the tensor's end."""
    from pytorch_yolo_b200 import ops
    g = torch.Generator().manual_seed(nc * 1000 + batch)
    anchors = ((10.0, 13.0), (16.0, 30.0), (33.0, 23.0))
    img = 32 * max(max(ny, nx) for ny, nx in grids)
    heads = [torch.randn(batch, 3 * (5 + nc), ny, nx, generator=g).to(DEV) for ny, nx in grids]
    specs = [ops.scale_spec(anchors, ny, nx, img) for ny, nx in grids]
    rows = sum(s.rows for s in specs)
    outs = {}
    for variant in ("ldg", "tma"):
        buf = torch.full((batch * rows * (5 + nc) + 64,), float("nan"), device=DEV)      # canary behind the tensor
        out = buf[:batch * rows * (5 + nc)].view(batch, rows, 5 + nc)
        ops.decode_dense(heads, specs, nc, out=out, variant=variant)
        torch.cuda.synchronize()
        assert torch.isnan(buf[batch * rows * (5 + nc):]).all()
        outs[variant] = out
    assert not torch.isnan(outs["tma"]).any()
    assert torch.equal(outs["ldg"], outs["tma"])


def test_packed_groups_mixed_class_sizes():
    """The segment stage's two work lists in one call: empty, single-box, small (packed several to a warp, runs that end
    at 8-class block borders, exactly 32 lanes), 33..64, 65..128 and capped (> 100) classes interleaved -- bit-exact
    against the oracle, rows included."""
    nc = 21
    sizes = [
        [0, 1, 2, 5, 32, 33, 1, 7, 64, 3, 100, 2, 0, 31, 9, 9, 9, 6, 140, 2, 30],
        [3] * 21,
        [16, 16, 16, 16, 1, 0, 17, 15, 2, 2, 2, 2, 2, 2, 2, 2, 8, 8, 8, 8, 65],
        [0] * 20 + [2],
    ]
    pred_cpu = prediction_with_class_sizes(sizes, nc, seed=11)
    want, wrows = yolo_oracle.non_max_suppression_indexed(pred_cpu.clone(), 0.05, 0.45)
    got, rows = non_max_suppression(pred_cpu.clone().to(DEV), 0.05, 0.45, return_rows=True)
    assert_dets_equal(got, want, box_rtol=1e-5, what="mixed class sizes")
    for r, wr in zip(rows, wrows):
        assert torch.equal(r.cpu().long(), wr)


@pytest.mark.parametrize("mpc", [5, 16, 31, 32, 40])
def test_small_max_per_class_turns_packing_off(mpc, monkeypatch):
    """max_per_class below 32 would cut small segments, so packing is off and every class goes through the one-segment
    paths; 32 and 40 pack.  All against the oracle with the same cap (utils.py:247-250 hard-codes 100)."""
    from pytorch_yolo_b200 import ops
    nc = 12
    sizes = [[0, 1, 2, 4, 6, 20, 31, 32, 33, 50, 3, 3], [7] * 12]
    pred_cpu = prediction_with_class_sizes(sizes, nc, seed=mpc)
    monkeypatch.setattr(yolo_oracle, "MAX_PER_CLASS", mpc)
    want, wrows = yolo_oracle.non_max_suppression_indexed(pred_cpu.clone(), 0.05, 0.5)
    pred = pred_cpu.clone().to(DEV)
    buf = ops.Buffers(DEV, pred.shape[0], pred.shape[1], nc, max_per_class=mpc)
    ops.compact_from_dense(pred, 0.05, buf)
    out, out_row = buf.new_outputs()
    ops.nms(buf, 0.5, out, out_row)
    _, kept, overflow = ops.read_counts(buf)
    assert overflow == 0
    got, rows = ops.ragged(out, out_row, kept, with_rows=True)
    assert_dets_equal(got, want, box_rtol=1e-5, what=f"max_per_class {mpc}")
    for r, wr in zip(rows, wrows):
        assert torch.equal(r.cpu().long(), wr)


@pytest.mark.parametrize("n,nc", [(3000, 80), (4096, 50), (2049, 30)])
def test_small_image_finalize_beyond_the_register_sort(n, nc):
    """Images with a small capacity (<= 4096 rows) use 128-thread finalize CTAs whose register sort takes 2048 staged rows;
    more rows go through the generic network over the shared-memory key area.  Every class stays under 100 boxes here, so
    every candidate is staged."""
    pred_cpu = synth.synth_prediction(2, n, nc=nc, seed=n + nc)
    want, wrows = yolo_oracle.non_max_suppression_indexed(pred_cpu.clone(), 0.0, 0.6)
    got, rows = non_max_suppression(pred_cpu.clone().to(DEV), 0.0, 0.6, return_rows=True)
    assert_dets_equal(got, want, box_rtol=1e-5, what=f"N{n} nc{nc}")
    for r, wr in zip(rows, wrows):
        assert torch.equal(r.cpu().long(), wr)
