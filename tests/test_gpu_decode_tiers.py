"""GPU: the decode kernels (csrc/decode.cu) at every tile geometry the class count selects, with CTAs that run many tiles.

Four decode-side kernels size their shared-memory tiles from no = 5 + nc, and the host code picks one geometry from it:

  kernel                                          geometry from no                       class counts
  decode_compact_tma_kernel ("tma", "tma2d")      tp = 256 / 128 / 64 / 32 positions    1-95 / 96-195 / 196-395 / 396-795;
                                                                                         "tma" refused from 796, "tma2d"
                                                                                         (no <= 256) from 252
  decode_dense_tma_kernel ("tma", part of "auto") ring (stages_in, bufs_out) =          1-85 / 86-107 / 108-145; refused
                                                  (3,2) / (2,2) / (2,1)                 from 146 (the LDG kernel runs)
  decode_dense_kernel ("ldg", the rest of "auto") one 128-position tile of no rows      up to 434; every dense decode is
                                                                                         refused from 435
  compact_from_dense_kernel                       rows_tile = 128 / 64 / 32 / 16 / 8 / 4 1-195 / 196-395 / 396-795 /
                                                                                         796-1595 / 1596-3195 / 3196-4096

The functions below restate that choice and each kernel's grid.  Every case checks the restatement against the launches the
profiler records (kernel, grid, shared memory) and asserts that every kernel with a shared-memory ring runs at least three
tiles per CTA, so that each stage's mbarrier phase flips more than once, so a change to the selection fails loudly instead
of quietly testing something else.  Each case combines a 16-byte aligned scale with a 13x13 or 19x19 one (the stages that
decode_compact_tma_kernel's consumers fill themselves, the LDG launch that follows dense decode's TMA kernel), and:

1. decode_dense ("ldg", "tma", "auto") against oracle.decode_heads within rtol 1e-5; "ldg", "tma" and "auto" bit-identical;
   NaN canary floats behind the output intact.  From 435 classes no dense decode takes the head: the dense tensor is
   assembled from calls on class slices (the five box / objectness channels plus at most 434 classes each); every column
   depends on its own channel only, so it holds the bits one call would write.
2. decode_compact, every variant the library accepts, emits exactly the candidates the dense tensor defines
   (helpers.expected_candidates), bit for bit; fp16 and bf16 heads on the LDG variants emit those of their fp32 upcast.
3. compact_from_dense at a 16-byte aligned base (TMA bulk copies) and at a 4-byte offset (every tile copied by the threads)
   emits the same candidates and writes fl(obj * max_cls) into column 4.
4. For one case per compact_from_dense tier and per tp: NMS on those candidates against the oracle on the same dense tensor
   (kept rows, order, score, class confidence and class bit-exact, boxes within rtol 1e-5).
5. Above each limit the refused variant raises and leaves its outputs untouched; from 435 classes the dense drop-in path
   (YOLOLayer.forward, decode_layers) raises while detect_layers still runs.
"""
import json

import numpy as np
import pytest
import torch

from oracle import yolo_oracle
from pytorch_yolo_b200 import YOLOLayer, decode_layers, detect_layers, non_max_suppression, ops
from tests.helpers import assert_dets_equal, assert_same_candidates, expected_candidates, read_candidates
from tests.test_gpu_decode_numerics import KSLACK, class_logits, near_tie_logits

GPU = pytest.mark.gpu
DEV = "cuda:0"
IMG = 416
CONF, NMS_THR = 0.3, 0.5
CANARY = 0x7FC0DEAD               # a NaN payload no kernel writes
SENTINEL = -0x2D2D2D2E
ANCHORS3 = [(10.0, 13.0), (16.0, 30.0), (33.0, 23.0)]
ANCHORS8 = [(10.0, 13.0), (16.0, 30.0), (33.0, 23.0), (30.0, 61.0), (62.0, 45.0), (59.0, 119.0), (116.0, 90.0),
            (156.0, 198.0)]
F32 = 4


# ------------------------------------------------------------------------------------------------------------------
# The selection, restated from the host code of csrc/decode.cu
TC_STAGES, TC_RING = 2, 200 * 1024        # tma_tile_positions (decode.cu:975-979): kTcStages, ring budget
TMA_BOX_ROWS = 256                        # "tma2d": a tensor-map box is at most 256 rows (decode.cu:1048)
DD_POS = 128                              # kDdPos: positions per dense decode tile
DT_BUDGET = 226 * 1024                    # dense TMA ring budget (decode.cu:1106-1111)
DD_LDG_LIMIT = 220 * 1024                 # LDG dense tile limit (decode.cu:1115)
CF_ROWS, CF_STAGES, CF_RING = 128, 2, 200 * 1024      # compact_from_dense rows_tile loop (decode.cu:1160)
CF_SM, CF_CTA_RESERVE = 220 * 1024, 1024              # its CTAs per SM (decode.cu:1177-1178)
UNROLLS = (16, 40)                        # YB_DC_UNROLL / YB_DC_UNROLL1: class planes per scan_classes batch


def compact_tp(no):
    """Positions per tile of decode_compact_tma_kernel: the largest of 256..32 whose 2-stage ring fits; 0 = refused."""
    for tp in (256, 128, 64, 32):
        if TC_STAGES * no * tp * F32 <= TC_RING:
            return tp
    return 0


def dense_ring(no):
    """(stages_in, bufs_out) of decode_dense_tma_kernel, or None when only the LDG kernel runs."""
    tile = DD_POS * no * F32
    if no <= TMA_BOX_ROWS:
        for ring, slack in (((3, 2), 32), ((2, 2), 32), ((2, 1), 16)):
            if sum(ring) * tile + slack <= DT_BUDGET:
                return ring
    return None


def dense_tma_smem(no, ring):
    tile = DD_POS * no * F32
    return ring[0] * tile + ring[1] * (tile + 16)


def dense_ldg_smem(no):
    return DD_POS * no * F32 + 16


def cfd_rows_tile(no):
    rt = CF_ROWS
    while rt > 4 and CF_STAGES * rt * no * F32 > CF_RING:
        rt //= 2
    return rt


def aligned(scale):
    _, ny, nx = scale
    return ny * nx % 4 == 0


def tiers(nc):
    """The geometry each kernel takes at nc classes (None / 0 / False: the variant is refused)."""
    no = nc + 5
    tp = compact_tp(no)
    return {"tp": tp, "tma2d": bool(tp) and no <= TMA_BOX_ROWS, "ring": dense_ring(no),
            "dense_ldg": dense_ldg_smem(no) <= DD_LDG_LIMIT, "rows_tile": cfd_rows_tile(no)}


def restate(scales, nc, batch, sms):
    """{kernel: (tiles, grid, dynamic shared memory)} of the ring kernels one case runs.  Both TMA kernels launch
    min(tiles, SMs) CTAs (decode.cu:1066, 1127); the dense one tiles only the aligned scales."""
    no = nc + 5
    geo = {}
    tp = compact_tp(no)
    if tp:
        tiles = sum(batch * len(a) * -(-ny * nx // tp) for a, ny, nx in scales)
        geo["decode_compact_tma_kernel"] = (tiles, min(tiles, sms), TC_STAGES * no * tp * F32)
    ring = dense_ring(no)
    if ring and any(aligned(s) for s in scales):
        tiles = sum(batch * len(a) * -(-ny * nx // DD_POS) for a, ny, nx in scales if aligned((a, ny, nx)))
        geo["decode_dense_tma_kernel"] = (tiles, min(tiles, sms), dense_tma_smem(no, ring))
    rt = cfd_rows_tile(no)
    smem = CF_STAGES * rt * no * F32
    per_sm = max(1, CF_SM // (smem + CF_CTA_RESERVE))
    rows = batch * sum(len(a) * ny * nx for a, ny, nx in scales)
    tiles = -(-rows // rt)
    geo["compact_from_dense_kernel"] = (tiles, min(sms * per_sm, tiles), smem)
    return geo


def case_batch(scales, nc, sms):
    """The smallest batch at which every ring kernel runs >= 3 tiles per CTA."""
    batch = 1
    while any(tiles < 3 * grid for tiles, grid, _ in restate(scales, nc, batch, sms).values()):
        batch += 1
    return batch


def head_bytes(scales, nc, batch):
    return batch * sum(len(a) * (nc + 5) * ny * nx for a, ny, nx in scales) * F32


# ------------------------------------------------------------------------------------------------------------------
# Cases: both sides of every boundary of the table, a 16-byte aligned 32x40 scale with a 13x13 or a 19x19 one (either
# order in the row layout)
BOUNDARY_NC = [85, 86, 95, 96, 107, 108, 145, 146, 195, 196, 251, 252, 395, 396, 434, 435, 795, 796, 1595, 1596, 3195,
               3196, 4096]
# NMS runs on one case per compact_from_dense tier and per tp (checked by test_cases_cover_every_tier)
NMS_NC = {95, 195, 395, 795, 1595, 3195, 4096}
FOUR_SCALES = [(ANCHORS3, 24, 32), (ANCHORS8, 13, 13), (ANCHORS3, 8, 8), (ANCHORS3, 1, 1)]


def case_scales(nc):
    if BOUNDARY_NC.index(nc) % 2 == 0:
        return [(ANCHORS3, 32, 40), (ANCHORS3, 13, 13)]
    return [(ANCHORS3, 19, 19), (ANCHORS3, 32, 40)]


def test_cases_cover_every_tier():
    """The parametrisation reaches both sides of every boundary of the selection, stays under 100 MB of heads, and the NMS
    cases cover every compact_from_dense tier and every tp (restatement only: no GPU needed)."""
    for lo in range(1, 4096):
        if tiers(lo) != tiers(lo + 1):                           # a boundary of the selection
            assert lo in BOUNDARY_NC and lo + 1 in BOUNDARY_NC, (lo, tiers(lo), tiers(lo + 1))
    assert 4096 in BOUNDARY_NC
    nms = {(tiers(nc)["tp"], tiers(nc)["rows_tile"]) for nc in NMS_NC}
    assert {tp for tp, _ in nms} == {256, 128, 64, 32, 0}
    assert {rt for _, rt in nms} == {128, 64, 32, 16, 8, 4}
    for nc in BOUNDARY_NC:
        scales = case_scales(nc)
        assert sorted(aligned(s) for s in scales) == [False, True]
        assert head_bytes(scales, nc, case_batch(scales, nc, 148)) < 100e6, nc
    for nc in (80, 396):
        assert head_bytes(FOUR_SCALES, nc, case_batch(FOUR_SCALES, nc, 148)) < 100e6, nc


# ------------------------------------------------------------------------------------------------------------------
# Inputs
def special_classes(nc):
    """Classes a wrong scan would miss: the last one, the tail after the last full batch of 16 (aligned planes) and 40
    (other planes) class planes, and the pairs on either side of a batch boundary (the last full one and one inside)."""
    s = {"last": [nc - 1]}
    for u in UNROLLS:
        full = nc // u * u
        if full < nc:
            s[f"tail{u}"] = list(range(full, nc))
        for edge in {full, u * max(1, nc // u // 2)}:
            if 0 < edge < nc:
                s[f"edge{u}@{edge}"] = [edge - 1, edge]
    return s


TIE_COLS = 6


def make_heads(scales, nc, batch, seed):
    """Seeded fp32 heads.  Objectness makes a few percent of the anchors pass CONF; one winning class logit per anchor,
    40 % of them in the special classes; 3 % of the anchors carry a near-tie pattern (near_tie_logits: ulp-apart logits,
    duplicates, +inf, NaN in a non-max class, sigma collapsing to 1.0) over TIE_COLS special classes."""
    rng = np.random.default_rng(seed)
    pool = np.unique(np.concatenate([[0]] + [np.asarray(v) for v in special_classes(nc).values()]))
    heads = []
    for anchors, ny, nx in scales:
        plane, na = ny * nx, len(anchors)
        n = batch * na * plane
        rows = np.empty((n, 5 + nc), np.float32)
        rows[:, 0:2] = rng.normal(0.0, 0.5, (n, 2))
        rows[:, 2:4] = rng.normal(0.0, 0.3, (n, 2))
        rows[:, 4] = rng.normal(-4.0, 2.5, n)
        rows[:, 5:] = rng.random((n, nc), dtype=np.float32) * np.float32(6.0) - np.float32(9.0)
        win = rng.integers(0, nc, n)
        sp = rng.random(n) < 0.4
        win[sp] = rng.choice(pool, int(sp.sum()))
        rows[np.arange(n), 5 + win] = rng.uniform(-2.0, 6.0, n)
        tie = np.nonzero(rng.random(n) < 0.03)[0]
        rows[tie, 4] = rng.uniform(1.0, 6.0, tie.size)
        for r, logits in zip(tie, near_tie_logits(rng, tie.size, TIE_COLS)):
            rows[r, 5 + np.sort(rng.choice(pool, TIE_COLS, replace=False))] = logits
        h = torch.from_numpy(rows).view(batch, na, plane, 5 + nc).permute(0, 1, 3, 2).reshape(batch, -1, ny, nx)
        heads.append(h.contiguous())
    return heads


def assert_reach(dense, heads, specs, nc, emit, cls, what):
    """Candidates reach every special class set, and some take the rescan (sigma of the second largest logit within
    kSlack of sigma of the largest: finish_anchor's test)."""
    for name, cs in special_classes(nc).items():
        assert np.isin(cls[emit], cs).any(), f"{what}: no candidate in class set {name}"
    logits = class_logits(heads, specs, nc)[emit]
    s = dense.cpu().numpy()[..., 5:][emit]
    with np.errstate(invalid="ignore"):
        raw = np.argmax(np.where(np.isnan(logits), -np.inf, logits), -1)
        k2 = np.argmax(np.where(np.arange(nc) == raw[:, None], -np.inf, logits), -1)
    sm = np.take_along_axis(s, raw[:, None], -1)[:, 0]
    sm2 = np.take_along_axis(s, k2[:, None], -1)[:, 0]
    rescan = sm2 * np.float32(KSLACK) >= sm
    print(f"{what}: {int(emit.sum())} candidates, {int(rescan.sum())} take the rescan, "
          f"{int((rescan & (cls[emit] != raw)).sum())} of them pick another class than the raw-logit arg-max")
    assert int(rescan.sum()) >= 10, what
    assert int(emit.sum()) >= 20 * dense.shape[0], what


# ------------------------------------------------------------------------------------------------------------------
# Launches as the profiler records them
def launches(prof, tmp_path):
    """[(kernel base name, grid x, static + dynamic shared memory)] of the decode-side kernels in a profiled region."""
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    out = []
    for e in events:
        if e.get("cat") != "kernel":
            continue
        base = e["name"].split("(")[0].split("::")[-1].split("<")[0]
        if base in ("decode_compact_tma_kernel", "decode_dense_tma_kernel", "decode_dense_kernel",
                    "compact_from_dense_kernel"):
            out.append((base, e["args"]["grid"][0], e["args"]["shared memory"]))
    return out


def assert_launches(seen, geo, no, ldg_dense_calls, what):
    """Every ring kernel launched with the restated grid and shared memory (the static part is at most 256 bytes), and
    >= 3 tiles per CTA; the dense LDG kernel with one tile of no rows."""
    for kernel, (tiles, grid, smem) in geo.items():
        got = [(g, s) for k, g, s in seen if k == kernel]
        assert got, f"{what}: {kernel} never ran"
        for g, s in got:
            assert g == grid and smem <= s < smem + 256, f"{what}: {kernel} grid {g} smem {s}, restated {grid} / {smem}"
        assert tiles >= 3 * grid, f"{what}: {kernel} runs {tiles} tiles on {grid} CTAs"
        print(f"{what}: {kernel} {tiles} tiles on {grid} CTAs ({tiles / grid:.1f} per CTA), {smem} B shared memory")
    ldg = [s for k, _, s in seen if k == "decode_dense_kernel"]
    assert len(ldg) == ldg_dense_calls, (what, ldg)
    if ldg_dense_calls and dense_ldg_smem(no) <= DD_LDG_LIMIT:
        assert all(dense_ldg_smem(no) <= s < dense_ldg_smem(no) + 256 for s in ldg), (what, ldg)


# ------------------------------------------------------------------------------------------------------------------
# Calls
def canary_out(shape):
    """(flat buffer filled with CANARY, contiguous view of `shape` at its start): 64 canary floats follow the view."""
    n = int(np.prod(shape))
    flat = torch.full((n + 64,), CANARY, dtype=torch.int32, device=DEV).view(torch.float32)
    return flat, flat[:n].view(shape)


def dense_call(heads, specs, nc, variant):
    flat, out = canary_out((heads[0].shape[0], sum(s.rows for s in specs), nc + 5))
    ops.decode_dense(heads, specs, nc, out=out, variant=variant)
    assert bool((flat[out.numel():].view(torch.int32) == CANARY).all()), f"decode_dense {variant}: canary overwritten"
    return out


def class_slice(h, spec, nc, c0, c1):
    """Head h restricted to the box / objectness channels and classes [c0, c1)."""
    b = h.shape[0]
    ch = torch.cat([torch.arange(5), 5 + torch.arange(c0, c1)]).to(h.device)
    return h.view(b, spec.na, nc + 5, spec.ny, spec.nx)[:, :, ch].reshape(b, -1, spec.ny, spec.nx).contiguous()


def dense_decode(heads, specs, nc, variant):
    """decode_dense of the whole head, or above 434 classes the columns of calls on class slices of at most 434."""
    if nc <= 434:
        return dense_call(heads, specs, nc, variant)
    n = -(-nc // 434)
    edges = [nc * k // n for k in range(n + 1)]                 # slices of > 1 class: one class would set column 5 := 1
    parts = []
    for c0, c1 in zip(edges, edges[1:]):
        part = dense_call([class_slice(h, s, nc, c0, c1) for h, s in zip(heads, specs)], specs, c1 - c0, variant)
        if parts:
            assert torch.equal(part[..., :5].view(torch.int32), parts[0][..., :5].view(torch.int32))
            part = part[..., 5:]
        parts.append(part)
    return torch.cat(parts, 2)


def cfd_run(dense, buf, offset):
    """compact_from_dense with write-back on a copy of dense at `offset` floats into a buffer; returns the copy."""
    flat = torch.empty(dense.numel() + 4, device=DEV)
    pred = flat[offset:offset + dense.numel()].view(dense.shape)
    assert pred.data_ptr() % 16 == 4 * offset
    pred.copy_(dense)
    ops.compact_from_dense(pred, CONF, buf, write_back=True)
    return pred


def assert_write_back(pred, dense, what):
    d = dense.cpu().numpy()
    with np.errstate(invalid="ignore", over="ignore"):
        want = d[..., 4] * np.max(d[..., 5:], -1)
    got = pred.cpu().numpy()
    same = (got[..., 4].view(np.int32) == want.view(np.int32)) | (np.isnan(got[..., 4]) & np.isnan(want))
    assert same.all(), f"{what}: column 4 differs from fl(obj * max_cls) in {int((~same).sum())} rows"
    got[..., 4] = d[..., 4]
    assert np.array_equal(got.view(np.int32), d.view(np.int32)), f"{what}: columns other than 4 changed"


def assert_nms_oracle(buf, dense, what):
    out, out_row = buf.new_outputs()
    ops.nms(buf, NMS_THR, out, out_row)
    kept = ops.read_counts(buf)[1].clone()
    got, rows = ops.ragged(out, out_row, kept, with_rows=True)
    want, wrows = yolo_oracle.non_max_suppression_indexed(dense.cpu(), CONF, NMS_THR)
    assert sum(w is not None for w in want) == dense.shape[0], what
    assert_dets_equal(got, want, box_rtol=1e-5, what=what)
    for i, (r, wr) in enumerate(zip(rows, wrows)):
        assert (r is None) == (wr is None) and (r is None or torch.equal(r.cpu().long(), wr)), f"{what} image {i}: rows"


def compact_refusal_wrote(heads, specs, nc, buf, variant):
    """decode_compact `variant` must raise; returns whether it wrote count / overflow anyway."""
    buf.meta.fill_(SENTINEL)
    with pytest.raises(ops.YoloB200Error):
        ops.decode_compact(heads, specs, nc, CONF, buf, variant=variant)
    torch.cuda.synchronize()
    return not bool((buf.meta == SENTINEL).all())


def dense_refusal_wrote(heads, specs, nc, variant):
    """decode_dense `variant` must raise; returns whether it wrote its output or the canary behind it anyway."""
    flat, out = canary_out((heads[0].shape[0], sum(s.rows for s in specs), nc + 5))
    with pytest.raises(ops.YoloB200Error):
        ops.decode_dense(heads, specs, nc, out=out, variant=variant)
    torch.cuda.synchronize()
    return not bool((flat.view(torch.int32) == CANARY).all())


# ------------------------------------------------------------------------------------------------------------------
def run_case(scales, nc, seed, with_nms, tmp_path):
    """Checks 1-5 of the module docstring on one case; returns (device heads, specs, device dense tensor)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    batch = case_batch(scales, nc, sms)
    geo = restate(scales, nc, batch, sms)
    tier = tiers(nc)
    no = nc + 5
    what = f"nc {nc} batch {batch} {[f'{ny}x{nx}' for _, ny, nx in scales]}"
    print(f"\n{what}: tp {tier['tp']}, dense ring {tier['ring']}, dense LDG {tier['dense_ldg']}, "
          f"rows_tile {tier['rows_tile']}, {head_bytes(scales, nc, batch) / 1e6:.1f} MB of heads")
    specs = [ops.scale_spec(a, ny, nx, IMG) for a, ny, nx in scales]
    heads = make_heads(scales, nc, batch, seed)
    dev = [h.to(DEV) for h in heads]
    rows = sum(s.rows for s in specs)
    buf = ops.Buffers(DEV, batch, rows, nc)
    dense_variants = ["ldg", "auto"] + (["tma"] if tier["ring"] else [])
    compact_variants = ["auto", "ldg", "ldg_dense"] + (["tma"] if tier["tp"] else []) + \
        (["tma2d"] if tier["tma2d"] else [])

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        # 1. dense decode
        dense = {v: dense_decode(dev, specs, nc, v) for v in dense_variants}
        # 2. fused decode
        got = {}
        for v in compact_variants:
            ops.decode_compact(dev, specs, nc, CONF, buf, variant=v)
            got[v] = read_candidates(buf)
        # 3. compact_from_dense at an aligned base and at a 4-byte offset
        d = dense["ldg"]
        cfd = {}
        for offset in (0, 1):
            buf_c = ops.Buffers(DEV, batch, rows, nc)
            cfd[offset] = (cfd_run(d, buf_c, offset), read_candidates(buf_c), buf_c)
        torch.cuda.synchronize()
    if tier["ring"]:            # "ldg"; "auto" and "tma" run the TMA kernel, then the LDG kernel on the unaligned scales
        n_ldg = 1 + 2 * any(not aligned(s) for s in scales)
    else:                       # "ldg" and "auto", once per class slice
        n_ldg = 2 * -(-nc // 434)
    assert_launches(launches(prof, tmp_path), geo, no, n_ldg, what)

    for v in dense_variants[1:]:
        assert torch.equal(dense[v].view(torch.int32), d.view(torch.int32)), f"{what}: decode_dense {v} != ldg"
    want_dense = yolo_oracle.decode_heads(heads, [a for a, _, _ in scales], nc, IMG)
    torch.testing.assert_close(d.cpu(), want_dense, rtol=1e-5, atol=1e-30, equal_nan=True)

    want, emit, cls = expected_candidates(d, CONF)
    assert_reach(d, heads, specs, nc, emit, cls, what)
    for v in compact_variants:
        assert_same_candidates(got[v], want, f"{what} decode_compact {v}")
    for dt in (torch.float16, torch.bfloat16):
        h16 = [h.to(dt) for h in dev]
        ops.decode_compact([h.float() for h in h16], specs, nc, CONF, buf, variant="ldg")
        ref = read_candidates(buf)
        assert sum(len(m) for m, _ in ref) >= 20 * batch
        for v in ("auto", "ldg", "ldg_dense"):
            ops.decode_compact(h16, specs, nc, CONF, buf, variant=v)
            assert_same_candidates(read_candidates(buf), ref, f"{what} decode_compact {v} {dt}")
    for offset, (pred, cands, _) in cfd.items():
        assert_same_candidates(cands, want, f"{what} compact_from_dense offset {4 * offset} B")
        assert_write_back(pred, d, f"{what} compact_from_dense offset {4 * offset} B")

    # 4. NMS
    if with_nms:
        assert_nms_oracle(cfd[1][2], d, what)

    # 5. refusals
    wrote = [f"decode_compact {v}" for v in ("tma", "tma2d")
             if v not in compact_variants and compact_refusal_wrote(dev, specs, nc, buf, v)]
    wrote += [f"decode_dense {v}" for v in ("ldg", "auto", "tma")
              if v not in dense_variants and dense_refusal_wrote(dev, specs, nc, v)]
    assert not wrote, f"{what}: refused, but wrote their outputs: {wrote}"
    assert ("tma" in compact_variants) == (no <= 800) and ("tma2d" in compact_variants) == (no <= 256)
    assert ("tma" in dense_variants) == (no <= 150) and tier["dense_ldg"] == (no <= 439)
    return dev, specs, d


@GPU
@pytest.mark.parametrize("nc", BOUNDARY_NC)
def test_decode_tier(nc, tmp_path):
    scales = case_scales(nc)
    dev, specs, dense = run_case(scales, nc, seed=nc, with_nms=nc in NMS_NC, tmp_path=tmp_path)
    if nc > 434:
        # the drop-in dense path states the 434-class limit; the fused path has none
        layers = [YOLOLayer(a, nc, [a for a, _, _ in scales]).eval() for a, _, _ in scales]
        with pytest.raises(ops.YoloB200Error):
            layers[0](dev[0], IMG)
        with pytest.raises(ops.YoloB200Error):
            decode_layers(layers, dev, IMG)
        got, rows = detect_layers(layers, dev, IMG, CONF, NMS_THR, return_rows=True)
        want, wrows = non_max_suppression(dense.clone(), CONF, NMS_THR, return_rows=True)
        assert sum(w is not None for w in want) == len(want)
        for g, r, w, wr in zip(got, rows, want, wrows):
            assert (g is None) == (w is None)
            if g is not None:
                assert torch.equal(g.view(torch.int32), w.view(torch.int32)) and torch.equal(r, wr)


@GPU
@pytest.mark.parametrize("nc", [80, 396])
def test_four_scales(nc, tmp_path):
    """Four scales, aligned / unaligned / aligned / unaligned, one with 8 anchors and one a 1x1 grid."""
    run_case(FOUR_SCALES, nc, seed=7 + nc, with_nms=True, tmp_path=tmp_path)


@GPU
def test_fifth_scale_raises():
    scales = FOUR_SCALES + [(ANCHORS3, 8, 8)]
    specs = [ops.scale_spec(a, ny, nx, IMG) for a, ny, nx in scales]
    heads = [torch.zeros(1, len(a) * 85, ny, nx, device=DEV) for a, ny, nx in scales]
    buf = ops.Buffers(DEV, 1, sum(s.rows for s in specs), 80)
    for v in ops.DECODE_VARIANTS:
        with pytest.raises(ValueError):
            ops.decode_compact(heads, specs, 80, CONF, buf, variant=v)
    for v in ops.DENSE_VARIANTS:
        with pytest.raises(ValueError):
            ops.decode_dense(heads, specs, 80, variant=v)
