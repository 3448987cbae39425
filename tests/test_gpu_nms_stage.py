"""GPU: the NMS stage (csrc/nms.cu) where its CTAs take more than one work item, at the benchmark's own residency, in
every finalize sort, and with IoU exactly at the threshold.

The segment kernel's single-warp CTAs work through two lists that the bucket kernel draws up on the device: groups of
small segments (CTAs [0, packed_ctas) stride over them) and bigger segments (one entry per CTA, further entries by
ticket).  Both loops, and the reuse of a CTA's shared memory by its next item, run only when a list is longer than the
grid, which a small call never reaches.  Every test here

  * restates from the candidates' class histograms what the bucket kernel deals (list lengths, grid, finalize sort per
    image), reads the kernel's own counters back from the workspace and checks them against the restatement;
  * asserts that its input reaches the state it exists for (lists several times the grid, every finalize branch, ...),
    so that a change to the dealing fails loudly instead of silently testing something else;
  * compares with the oracle under the repository's bar: kept rows, order, score, class-confidence and class bit-exact,
    boxes within rtol 1e-5 (the oracle's MERGE sum runs in torch's reduction order), and results of the same
    candidates at different residencies bit for bit.
"""
import random
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import yolo_oracle
from pytorch_yolo_b200 import YOLOLayer, _lib, decode_layers, ops, synth
from pytorch_yolo_b200.detect import Detector
from tests.helpers import assert_dets_equal, prediction_with_class_sizes

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# constants of csrc/nms.cu (and common.cuh) the restatement below depends on
GROUP_RUN = 8               # kGroupRun: a group is a run of classes inside one block of this many classes
SMALL_SEG = 32              # kSmallSeg
PACK_SLOT_BITS = 27         # kPackSlotBits
FINAL_SMALL_CAP = 4096      # kFinalSmallCap = kSmallImageRows
FINAL_KPT = 16              # kFinalKpt
DEFAULT_RESIDENCY = 16      # seg_warps_per_sm when the option is 0 (yolo_b200_nms_ex)
PAD_BITS = 0x7FA5A5A5       # a NaN payload the kernels never write: marks result rows that must stay untouched


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------------------------
# The dealing, restated from the host and kernel code
def ws_layout(batch, cap, nc, mpc):
    """(offset of work_count, total bytes) of the NMS workspace: 256-byte aligned blocks in the order of ws_layout
    (nms.cu:1033-1048)."""
    def up(v):
        return (v + 255) & ~255
    stage_cap = min(cap, nc * mpc)
    o = up(batch * cap * 8)                  # bucket_key
    o = up(o + batch * cap * 4)              # bucket_slot
    o = up(o + batch * (nc + 1) * 4)         # seg_off
    o = up(o + batch * (nc + 1) * 4)         # stage_off
    work_count = o
    o = up(o + 16)                           # work_count
    o = up(o + batch * nc * 8)               # group_list
    o = up(o + batch * nc * 16)              # seg_list
    o = up(o + batch * stage_cap * 32)       # stage
    o = up(o + batch * stage_cap * 8)        # final_keys
    return work_count, o


def read_work_count(buf):
    """The four counters of the last call on ``buf``: [0] segment tickets handed out, [1] finalize CTAs counted in by the
    completion stamp (reset by the last one), [2] groups of small segments, [3] entries of the segment list."""
    off, total = ws_layout(buf.batch, buf.cap, buf.nc, buf.mpc)
    assert total == _lib.load().yolo_b200_nms_workspace_bytes(buf.batch, buf.cap, buf.nc, buf.mpc)
    return buf.workspace[off:off + 16].view(torch.int32).tolist()


def class_histograms(buf):
    """(B, nc) class histogram of every image's candidates, as the bucket kernel counts them (nms.cu:183-197)."""
    b, cap, nc = buf.batch, buf.cap, buf.nc
    count = buf.meta[:b].clamp(max=cap).long()
    cls = buf.cand_meta[:b * cap, 2].view(b, cap).long()
    valid = (torch.arange(cap, device=buf.device).view(1, cap) < count.view(b, 1)) & (cls >= 0) & (cls < nc)
    idx = (torch.arange(b, device=buf.device).view(b, 1) * nc + cls)[valid]
    return torch.bincount(idx, minlength=b * nc).view(b, nc).cpu().numpy()


def final_branch(n, ft, smem_keys, key_slots):
    """The sort nms_finalize_body picks for an image that staged n rows (nms.cu:967-992)."""
    if n <= smem_keys:
        for kpt in (2, 4, 8):
            if n <= kpt * ft:
                return f"kpt{kpt}"
        return "kpt16"
    return "shared" if n <= key_slots else "global"


def restate_deal(hist, cap, mpc, residency, sms):
    """What one yolo_b200_nms_ex call deals for these (B, nc) class histograms.

    bucket_by_class_kernel (nms.cu:224-236): inside every block of GROUP_RUN classes, classes of 2..32 boxes are filled
    greedily into groups of at most 32 boxes; classes of fewer than 2 boxes take no work; bigger classes (or every class of
    >= 2 boxes when packing is off) are one entry of the segment list each.  Host (nms.cu:1098-1149): the grid of each
    list, the finalize CTA size and its sort areas."""
    batch, nc = hist.shape
    pack_ok = mpc >= SMALL_SEG and cap <= 1 << PACK_SLOT_BITS and nc <= 0xFFFF
    groups = np.zeros(batch, np.int64)
    segs = np.zeros(batch, np.int64)
    for b in range(batch):
        h = hist[b].tolist()
        if not pack_ok:
            segs[b] = sum(n >= 2 for n in h)
            continue
        for c0 in range(0, nc, GROUP_RUN):
            fill = 0
            for n in h[c0:c0 + GROUP_RUN]:
                if n < 2:
                    continue
                if n > SMALL_SEG:
                    segs[b] += 1
                    continue
                if fill + n > 32:
                    groups[b] += 1
                    fill = 0
                fill += n
            if fill:
                groups[b] += 1
    res = residency if 1 <= residency <= 32 else DEFAULT_RESIDENCY
    seg_ctas = min(batch * nc, sms * res)
    stage_cap = min(cap, nc * mpc)
    ft = 128 if stage_cap <= FINAL_SMALL_CAP else 512
    smem_keys = min(stage_cap, ft * FINAL_KPT)
    kpt = 2
    while kpt * ft < smem_keys:
        kpt *= 2
    key_slots = kpt * ft
    if ft == 128 and key_slots < stage_cap:
        key_slots = (stage_cap + 1) & ~1
    staged = np.minimum(hist, mpc).sum(1)
    return SimpleNamespace(pack_ok=pack_ok, groups=groups, segs=segs, n_groups=int(groups.sum()), n_segs=int(segs.sum()),
                           seg_ctas=seg_ctas, packed_ctas=seg_ctas if pack_ok else 0, ft=ft, staged=staged,
                           branches=[final_branch(int(n), ft, smem_keys, key_slots) for n in staged])


def check_counters(wc, deal, stamped=False):
    """The counters of one call against the restated deal.  Every CTA that processes a segment entry takes one ticket
    after it (nms.cu:818-830) unless the list fits the grid, so [0] counts the entries when tickets run, else stays 0."""
    assert wc[2] == deal.n_groups and wc[3] == deal.n_segs, (wc, deal.n_groups, deal.n_segs)
    assert wc[0] == (wc[3] if wc[3] > deal.seg_ctas else 0), (wc, deal.seg_ctas)
    assert wc[1] == 0, wc              # the last finalize CTA resets it when a stamp is asked for; untouched otherwise


def engaged(wc, deal):
    """The loops of the segment kernel a call ran: ticketed segment entries, groups strided over the packed CTAs."""
    return {name for name, on in (("tickets", wc[3] > deal.seg_ctas), ("stride", wc[2] > deal.packed_ctas)) if on}


# ------------------------------------------------------------------------------------------------------------------
# Calls and comparisons
def load_candidates(pred_cpu, conf, mpc, cap=None):
    """Buffers holding the candidates of a decoded (B, N, 5+nc) prediction (compact_from_dense, as the dense path does)."""
    b, n, no = pred_cpu.shape
    buf = ops.Buffers(DEV, b, n if cap is None else cap, no - 5, max_per_class=mpc)
    ops.compact_from_dense(pred_cpu.to(DEV), conf, buf)
    assert ops.read_counts(buf)[2] == 0, "candidate capacity exceeded"
    return buf


def padded_outputs(batch, out_cap):
    out = torch.full((batch, out_cap, ops.DET_COLS), PAD_BITS, dtype=torch.int32, device=DEV).view(torch.float32)
    return out, torch.full((batch, out_cap), -1, dtype=torch.int32, device=DEV)


def run_nms(buf, thr, residency, out_cap=None, step=None):
    """One call into result buffers filled with the pad pattern; returns (out, out_row, kept counts, counters)."""
    out, out_row = padded_outputs(buf.batch, buf.out_cap if out_cap is None else out_cap)
    ops.nms(buf, thr, out, out_row, step=step, seg_warps_per_sm=residency)
    kept = ops.read_counts(buf)[1].clone()
    return out, out_row, kept, read_work_count(buf)


def assert_same_bits(a, b, what):
    (out_a, row_a, kept_a), (out_b, row_b, kept_b) = a, b
    assert torch.equal(kept_a, kept_b), what
    assert torch.equal(out_a.view(torch.int32), out_b.view(torch.int32)), what
    assert torch.equal(row_a, row_b), what


def assert_oracle(out, out_row, kept, want, wrows, what, images=None):
    """Result rows of ``images`` (default: all) against the oracle's result of those images."""
    got, rows = ops.ragged(out, out_row, kept, with_rows=True)
    if images is not None:
        got, rows = [got[i] for i in images], [rows[i] for i in images]
    assert_dets_equal(got, want, box_rtol=1e-5, what=what)
    for i, (r, wr) in enumerate(zip(rows, wrows)):
        assert (r is None) == (wr is None), f"{what} image {i}"
        if r is not None:
            assert torch.equal(r.cpu().long(), wr), f"{what} image {i}: kept rows differ"


def oracle(pred_cpu, conf, thr, mpc, monkeypatch):
    monkeypatch.setattr(yolo_oracle, "MAX_PER_CLASS", mpc)
    return yolo_oracle.non_max_suppression_indexed(pred_cpu.clone(), conf, thr)


# ------------------------------------------------------------------------------------------------------------------
# 1. Multi-item CTAs: small grids (residency 1 and 2), lists several times longer
def multi_item_sizes(batch, nc, mpc, seed):
    """Per image, class sizes alternating inside every 8-class block between small classes (17..32 boxes: one group
    each) and bigger ones (33..64, 65..128, > 128, and mpc - 1, mpc, mpc + 1, 500), with empty, single and 2..8-box
    classes sprinkled in: every CTA gets quad, pair and small items one after another."""
    rng = random.Random(seed)
    big = [lambda: rng.randint(33, 64), lambda: rng.randint(65, 128), lambda: rng.randint(129, 300),
           lambda: rng.choice([mpc - 1, mpc, mpc + 1, 500])]
    sizes = []
    for b in range(batch):
        row = []
        for c in range(nc):
            r = rng.random()
            if r < 0.04:
                row.append(0)
            elif r < 0.08:
                row.append(1)
            elif r < 0.12:
                row.append(rng.randint(2, 8))
            elif (c + b) % 2:
                row.append(rng.randint(17, 32))
            else:
                row.append(max(2, rng.choice(big)()))
        sizes.append(row)
    return sizes


MULTI_ITEM_BATCH, MULTI_ITEM_NC = 28, 80


@pytest.mark.parametrize("thr", [0.45, 0.0, -0.25])
@pytest.mark.parametrize("mpc", [100, 16, 31, 33, 64, 65, 128])
def test_multi_item_ctas(mpc, thr, monkeypatch):
    """Residency 1 and 2 give 1 / 2 CTAs per SM and list: every segment CTA takes several entries by ticket (quad, pair
    and small segments in turn, reusing its shared memory), every packed CTA strides over several groups (mpc >= 32), and
    with mpc < 32 the small segments come by ticket too.  The result is the same at residency 1, 2, 16 and 32, and the
    oracle's."""
    sizes = multi_item_sizes(MULTI_ITEM_BATCH, MULTI_ITEM_NC, mpc, seed=mpc)
    pred_cpu = prediction_with_class_sizes(sizes, MULTI_ITEM_NC, seed=7 * mpc)
    buf = load_candidates(pred_cpu, 0.05, mpc)
    hist = class_histograms(buf)
    assert (hist == np.array(sizes)).all()
    sms = sm_count()
    results = {}
    for res in (1, 2, 16, 32):
        deal = restate_deal(hist, buf.cap, mpc, res, sms)
        out, out_row, kept, wc = run_nms(buf, thr, res)
        check_counters(wc, deal)
        if res <= 2:                                       # the state this test exists for
            assert deal.n_segs >= 3 * deal.seg_ctas, (res, deal.n_segs, deal.seg_ctas)
            assert deal.pack_ok == (mpc >= 32)
            if deal.pack_ok:
                assert deal.n_groups >= 3 * deal.packed_ctas, (res, deal.n_groups, deal.packed_ctas)
            assert engaged(wc, deal) == ({"tickets", "stride"} if deal.pack_ok else {"tickets"})
        results[res] = (out, out_row, kept)
    for res in (2, 16, 32):
        assert_same_bits(results[res], results[1], f"mpc {mpc} thr {thr}: residency {res} vs 1")
    want, wrows = oracle(pred_cpu, 0.05, thr, mpc, monkeypatch)
    assert_oracle(*results[1], want, wrows, f"mpc {mpc} thr {thr}")


# ------------------------------------------------------------------------------------------------------------------
# 2. The benchmark's configurations at the library's default residency
BENCH_CONFIGS = {                # bench.py's configurations: (workload, batch per GPU, conf); SYNTH-B heads, nms 0.5
    "cfg2": ("spp-608", 64, 0.3),
    "cfg3": ("tiny-416", 1024, 0.3),
    "cfg4": ("spp-608", 64, 0.001),
    "cfg2-b128": ("spp-608", 128, 0.3),     # cfg 2 engages neither loop; at twice its batch the groups outnumber the CTAs
}
# the loops each configuration engages at the default residency on a 148-SM B200: cfg 2 holds 64 x 80 (image, class)
# pairs, few of them over 32 boxes, so it fits both grids of 2368 CTAs; cfg 3's 1024 images deal more groups than the
# packed CTAs; at conf 0.001 (cfg 4) most pairs hold over 32 boxes and take tickets
BENCH_ENGAGED = {"cfg2": set(), "cfg3": {"stride"}, "cfg4": {"tickets"}, "cfg2-b128": {"stride"}}


@pytest.mark.parametrize("cfg", sorted(BENCH_CONFIGS))
def test_benchmark_configs_default_residency(cfg, monkeypatch):
    """SYNTH-B heads of a benchmark configuration, decoded on the GPU, through NMS at residency 0 (the library default the
    benchmark runs): the batch result equals, bit for bit, every image run alone (one image: at most nc CTAs per list, no
    ticket, no stride), the batch at residency 1 and 32, a graph-captured Detector replayed twice, and on the images with
    the most segment entries, groups and staged rows, the oracle."""
    wl, batch, conf = BENCH_CONFIGS[cfg]
    thr = 0.5
    w = synth.WORKLOADS[wl]
    nc = w["nc"]
    layers = [YOLOLayer(a, nc, w["anchors"]).eval() for a in w["anchors"]]
    heads = synth.synth_heads(wl, batch, "B", seed=1234, device=DEV)
    pred, _ = decode_layers(layers, heads, w["img_size"])
    pristine = pred.clone()                          # compact_from_dense writes obj * cls into column 4
    rows = pred.shape[1]
    buf = ops.Buffers(DEV, batch, rows, nc)
    ops.compact_from_dense(pred, conf, buf)
    assert ops.read_counts(buf)[2] == 0
    hist = class_histograms(buf)
    sms = sm_count()
    deal = restate_deal(hist, buf.cap, buf.mpc, 0, sms)
    out, out_row, kept, wc = run_nms(buf, thr, 0)
    check_counters(wc, deal)
    if sms == 148:
        assert engaged(wc, deal) == BENCH_ENGAGED[cfg], (cfg, wc, deal.seg_ctas)
    batch_res = (out, out_row, kept)

    for res in (1, 32):
        o, r, k, wc_r = run_nms(buf, thr, res)
        check_counters(wc_r, restate_deal(hist, buf.cap, buf.mpc, res, sms))
        assert_same_bits((o, r, k), batch_res, f"{cfg}: residency {res} vs default")

    # every image alone, through the same candidates, into a batch-shaped result
    single = ops.Buffers(DEV, 1, buf.cap, nc)
    assert single.out_cap == buf.out_cap
    solo_out, solo_row = padded_outputs(batch, buf.out_cap)
    solo_kept = torch.zeros(batch, dtype=torch.int32, device=DEV)
    cap = buf.cap
    for b in range(batch):
        one = restate_deal(hist[b:b + 1], cap, buf.mpc, 0, sms)
        assert one.n_segs <= one.seg_ctas and one.n_groups <= one.packed_ctas
        single.cand_box[:cap].copy_(buf.cand_box[b * cap:(b + 1) * cap])
        single.cand_meta[:cap].copy_(buf.cand_meta[b * cap:(b + 1) * cap])
        single.meta[0:1].copy_(buf.meta[b:b + 1])
        ops.nms(single, thr, None, None, out_ptrs=(solo_out[b].data_ptr(), solo_row[b].data_ptr(),
                                                   solo_kept[b:b + 1].data_ptr()))
    torch.cuda.synchronize()
    assert_same_bits((solo_out, solo_row, solo_kept.cpu()), batch_res, f"{cfg}: batch vs every image alone")

    # the oracle on the images that load the lists and the finalize most
    picks = sorted({int(np.argmax(deal.segs)), int(np.argmax(deal.groups)), int(np.argmax(deal.staged))})
    sub = pristine[picks].cpu()
    want, wrows = oracle(sub, conf, thr, buf.mpc, monkeypatch)
    assert_oracle(out, out_row, kept, want, wrows, f"{cfg} images {picks}", images=picks)

    # the benchmark's own path: a captured Detector (fused decode, default residency), replayed twice
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    det = Detector(specs, nc, batch, DEV, conf, thr, use_graph=True)
    eager = ops.ragged(out, out_row, kept, with_rows=True)
    for _ in range(2):
        got, got_rows = det.run(heads, return_rows=True, clone=True)
        for i, (g, gr, e, er) in enumerate(zip(got, got_rows, *eager)):
            assert (g is None) == (e is None), f"{cfg} graph image {i}"
            if g is not None:
                assert torch.equal(g, e) and torch.equal(gr, er), f"{cfg} graph image {i}"


# ------------------------------------------------------------------------------------------------------------------
# 3. Every finalize sort, several in one launch
def spread_prediction(staged, nc, mpc, seed):
    """(B, N, 5+nc) prediction in which image b stages exactly staged[b] rows: classes of mpc boxes and one remainder
    class (a class of one box is staged as well), boxes on a lattice so that most are kept, every 16th box a near
    duplicate of the previous one (suppressed and merged)."""
    g = torch.Generator().manual_seed(seed)
    n = max(max(staged), 1)
    pred = torch.zeros(len(staged), n, 5 + nc)
    side = int(np.ceil(np.sqrt(n)))
    for b, s in enumerate(staged):
        if s == 0:
            continue
        assert -(-s // mpc) <= nc
        cls = torch.arange(s) // mpc
        k = torch.arange(s)
        cell = k - (k % 16 == 15).long()                   # every 16th box on the previous box's cell
        xy = 20.0 * torch.stack((cell % side, cell // side), 1).float() + 10.0
        xy += (k % 16 == 15).float().view(s, 1) * 0.5
        pred[b, :s, 0:2] = xy
        pred[b, :s, 2:4] = 12.0 + 2.0 * torch.rand(s, 2, generator=g)
        pred[b, :s, 4] = 0.2 + 0.8 * torch.rand(s, generator=g)
        pred[b, k, 5 + cls] = 0.5 + 0.5 * torch.rand(s, generator=g)
        perm = torch.randperm(n, generator=g)
        pred[b] = pred[b, perm]
    return pred


FINAL_EDGES = {128: [0, 1, 256, 257, 512, 513, 1024, 1025, 2048, 2049, 4096],
               512: [1024, 1025, 2048, 2049, 4096, 4097, 8192, 8193]}
FINAL_BRANCHES = {128: {"kpt2", "kpt4", "kpt8", "kpt16", "shared"}, 512: {"kpt2", "kpt4", "kpt8", "kpt16", "global"}}


@pytest.mark.parametrize("ft", [128, 512])
def test_finalize_branches_mixed_launch(ft, monkeypatch):
    """One launch in which the images stage exactly the counts at every edge of the finalize sorts of one CTA size (128
    threads up to 4096 staged rows per image, else 512): every register sort, the shared-memory network (128) or the
    global key network (512) in the same grid.  Results take several chunks of ``ft`` rows, stored at a destination phase
    that is not 16-byte aligned (out_cap * 7 floats per image is not a multiple of 4); rows past each image's count stay
    untouched."""
    mpc = 100
    staged = FINAL_EDGES[ft]
    nc = -(-max(staged) // mpc) + 1
    pred_cpu = spread_prediction(staged, nc, mpc, seed=ft)
    buf = load_candidates(pred_cpu, 0.05, mpc)
    hist = class_histograms(buf)
    deal = restate_deal(hist, buf.cap, mpc, 32, sm_count())
    assert deal.staged.tolist() == staged and deal.ft == ft
    assert set(deal.branches) == FINAL_BRANCHES[ft], deal.branches
    out_cap = buf.out_cap + 1
    assert (out_cap * ops.DET_COLS) % 4 != 0
    out, out_row, kept, wc = run_nms(buf, 0.5, 32, out_cap=out_cap)
    check_counters(wc, deal)
    k = kept.tolist()
    for b, s in enumerate(staged):
        if s >= 2 * ft:
            assert k[b] > ft, (s, k[b])                  # several output chunks
        assert (out[b, k[b]:].view(torch.int32) == PAD_BITS).all() and (out_row[b, k[b]:] == -1).all(), \
            f"image {b} ({s} staged): rows past its count were written"
    want, wrows = oracle(pred_cpu, 0.05, 0.5, mpc, monkeypatch)
    assert_oracle(out, out_row, kept, want, wrows, f"finalize {ft} threads")


# ------------------------------------------------------------------------------------------------------------------
# 4. IoU at the threshold
def f32(v):
    return np.float32(v)


def f32_steps(v, ks):
    """The float32 values k representable steps from v (v > 0), for every k in ks."""
    return (np.array([v], np.float32).view(np.int32)[0] + np.asarray(ks, np.int32)).view(np.float32)


def step_f32(v, k):
    return f32_steps(v, [k])[0]


def reference_iou(a_xywh, b_xywh):
    """fl(inter / union) of box a (the pivot) against every row of b, xywh float32 (n, 4): the oracle's corners and op
    order (yolo_oracle.centre_to_corner, iou_one_to_many)."""
    a = yolo_oracle.centre_to_corner(torch.from_numpy(np.asarray(a_xywh, np.float32).reshape(1, 4)))[0]
    b = yolo_oracle.centre_to_corner(torch.from_numpy(np.asarray(b_xywh, np.float32).reshape(-1, 4)))
    return yolo_oracle.iou_one_to_many(a, b).numpy()


def kernel_iou_gt(a_xywh, b_xywh, thr, f_hi=1.000001, f_lo=0.999999):
    """iou_gt (nms.cu:97-115) in float32 on the host, with the band factors as parameters: the real ones must agree with
    the reference on every pair, a band narrower than fp32 rounding must not (that is what the pairs are for)."""
    a = yolo_oracle.centre_to_corner(torch.from_numpy(np.asarray(a_xywh, np.float32).reshape(1, 4)))[0].numpy()
    b = yolo_oracle.centre_to_corner(torch.from_numpy(np.asarray(b_xywh, np.float32).reshape(-1, 4))).numpy()
    t = f32(thr)
    ok = t > f32(1e-30)
    hi = t * f32(f_hi) if ok else f32(np.inf)
    lo = t * f32(f_lo) if ok else f32(-np.inf)
    with np.errstate(all="ignore"):
        area_a = (a[2] - a[0]) * (a[3] - a[1]) + f32(1e-16)
        area_b = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
        ix = np.minimum(a[2], b[:, 2]) - np.maximum(a[0], b[:, 0])
        iy = np.minimum(a[3], b[:, 3]) - np.maximum(a[1], b[:, 1])
        inter = np.maximum(ix, f32(0)) * np.maximum(iy, f32(0))
        uni = (area_a + area_b) - inter
        yes = inter > hi * uni
        no = inter < lo * uni
        in_range = (uni.view(np.uint32) - np.uint32(0x00800000)) < np.uint32(0x7E800000)
        return np.where((yes | no) & in_range, yes, inter / uni > t)


def scan(a, b, coord, ks):
    """Box a fixed, box b with coordinate ``coord`` (0..3 = x, y, w, h) moved over consecutive float32 values."""
    b = np.tile(np.asarray(b, np.float32), (len(ks), 1))
    b[:, coord] = f32_steps(b[0, coord], ks)
    return b


def pair_families(t, n_fam=1200, seed=0):
    """(a, b candidates) families whose quotient crosses t within the scanned steps.  t >= 1e-20: b overlaps a side by
    side, at ordinary coordinates and at ~1e19 (union >= 2^127: the range test sends those to the division), b's x centre
    moved around the analytic crossing; each step moves the quotient by ~20 of its ulps, and the random sizes spread the
    steps' phases so that every ulp near t is hit.  Smaller t: b inside a ~1e19 box, b's width moved."""
    rng = np.random.default_rng(seed)
    fams = []
    for i in range(n_fam):
        wa, ha, wb, hb = (float(v) for v in 30.0 + 40.0 * rng.random(4))
        if t > f32(1e-20):
            if i % 2 == 0:
                scale = 1.0
            else:                   # sides 1.22e19..1.29e19: areas below 1.7e38 (2 x area is finite), unions above 2^127
                scale = 1.7e17
                wa, ha, wb, hb = (72.0 + (v - 30.0) / 10.0 for v in (wa, ha, wb, hb))
            wa, ha, wb, hb = (f32(v * scale) for v in (wa, ha, wb, hb))
            base = 300.0 * scale if scale == 1.0 else 0.0
            a = (f32(base), f32(base), wa, ha)
            iy = min(float(ha), float(hb))
            ov = float(t) * (float(wa) * float(ha) + float(wb) * float(hb)) / ((1 + float(t)) * iy)
            xb = f32(base + float(wa) / 2 + float(wb) / 2 - ov)
            fams.append((a, scan(a, (xb, f32(base), wb, hb), 0, np.arange(-6, 7))))
        else:
            a = (f32(0.0), f32(0.0), f32(wa * 1.7e17), f32(ha * 1.7e17))
            area_b = float(t) * float(a[2]) * float(a[3])
            side = np.sqrt(area_b * hb / wb)
            b = (f32(side), f32(side), f32(area_b / side), f32(side))
            fams.append((a, scan(a, b, 2, np.arange(-24, 25))))
    return fams


def near_threshold_pairs(thr, per_target=4):
    """(a, b) xywh pairs whose reference quotient is prev(thr), thr or next(thr), or sits at / one step either side of
    the kernel's band edges fl(thr * (1 +- 1e-6)), from both coordinate scales, plus pairs that the comparison without a
    band (inter against fl(thr * union)) decides wrongly."""
    t = f32(thr)
    targets = [step_f32(t, -1), t, step_f32(t, 1)]
    if t > f32(1e-30):
        for edge in (t * f32(1.000001), t * f32(0.999999)):
            targets += [step_f32(edge, -1), edge, step_f32(edge, 1)]
    found = {(q, big): [] for q in targets for big in (False, True)}
    bandless = []
    for a, bs in pair_families(t):
        q = reference_iou(a, bs)
        big = bool(a[2] > 1e10)
        for i, qi in enumerate(q):
            got = found.get((qi, big))
            if got is not None and len(got) < per_target // 2:
                got.append((np.asarray(a, np.float32), bs[i]))
        if t > f32(1e-30) and len(bandless) < per_target:
            wrong = kernel_iou_gt(a, bs, thr, 1.0, 1.0) != (q > t)
            bandless += [(np.asarray(a, np.float32), bs[i]) for i in np.nonzero(wrong)[0][:1]]
    for q_want in targets:
        assert found[(q_want, False)] or found[(q_want, True)], f"no pair with quotient {q_want!r} for threshold {thr!r}"
    return [p for got in found.values() for p in got] + bandless


def special_pairs(thr):
    """Pairs away from any threshold: disjoint, touching (inter exactly 0) and the smallest positive overlap.  For a
    negative threshold also a pair whose union overflows to inf (q = 0): such a box has IoU 0 with itself, so at a
    threshold >= 0 the reference's loop never ends (utils.py:266-275), and only a negative one is a valid input."""
    a = np.array([100.0, 100.0, 20.0, 20.0], np.float32)
    touch = np.array([120.0, 100.0, 20.0, 20.0], np.float32)           # b.x1 == a.x2
    over = touch.copy()
    over[0] = step_f32(120.0, -1)
    far = np.array([400.0, 400.0, 20.0, 20.0], np.float32)
    pairs = [(a, touch), (a, over), (a, far)]
    if thr < 0:
        pairs.append((np.array([0.0, 0.0, 1.5e19, 1.5e19], np.float32), np.array([1e18, 0.0, 1.5e19, 1.5e19], np.float32)))
    return pairs


def self_iou_terminates(box, thr):
    """The reference removes a kept box only through its IoU with itself (utils.py:271, 275)."""
    return bool(reference_iou(box, box)[0] > f32(thr))


def pair_union(a, b):
    """The union of the IoU of pivot a with b, in the reference's op order (iou_one_to_many)."""
    a, b = (yolo_oracle.centre_to_corner(torch.from_numpy(np.asarray(x, np.float32).reshape(1, 4)))[0] for x in (a, b))
    inter = (torch.min(a[2], b[2]) - torch.max(a[0], b[0])).clamp(0) * (torch.min(a[3], b[3]) - torch.max(a[1], b[1])).clamp(0)
    return float(((a[2] - a[0]) * (a[3] - a[1]) + 1e-16) + (b[2] - b[0]) * (b[3] - b[1]) - inter)


# thresholds at which comparing inter with fl(thr * union), without a band, decides some pair of the families wrongly (at
# 0.5, 0.45 and 0.7 none of them is).  A band of 1 +- 1e-7 is still exact: any hi >= next(thr) and lo <= prev(thr) is.
BANDLESS_SENSITIVE = (0.3, float(step_f32(1e-30, 1)))
IOU_THRESHOLDS = [0.5, 0.45, 0.3, 0.7, 1e-30, float(step_f32(1e-30, -1)), float(step_f32(1e-30, 1)), 0.0, -0.0, -0.5]


def embed_pairs(pairs, size, pos_a, pos_b):
    """(1, N, 5+nc) prediction: pair k is class k, with size - 2 filler boxes (identical, far from the pair: they merge into
    one another and never touch the pair for a threshold >= 0); scores put a at sorted position pos_a, b at pos_b."""
    nc = len(pairs)
    pred = torch.zeros(1, nc * size, 5 + nc, dtype=torch.float64)
    for c, (a, b) in enumerate(pairs):
        ext = float(max(abs(a[0]) + a[2], abs(a[1]) + a[3], abs(b[0]) + b[2], abs(b[1]) + b[3]))
        filler = np.array([4 * ext + 1000.0, 4 * ext + 1000.0, min(float(a[2]), 1e18), min(float(a[3]), 1e18)])
        others = [p for p in range(size) if p not in (pos_a, pos_b)]
        for p, box in [(pos_a, a), (pos_b, b)] + [(p, filler) for p in others]:
            r = c * size + p
            pred[0, r, 0:4] = torch.from_numpy(np.asarray(box, np.float64))
            pred[0, r, 4] = 0.95 - 0.005 * p
            pred[0, r, 5 + c] = 1.0
    return pred.float()


IOU_LAYOUTS = [  # (class size, max_per_class, sorted positions of a and b, segment path)
    (2, 100, 0, 1),      # packed with other classes into one warp
    (2, 16, 0, 1),       # packing off: one class per warp, one box per lane
    (40, 100, 5, 36),    # pair path: a in the low register, b in the high one
    (100, 100, 3, 7),    # quad path, both in the first 32-box block
    (100, 100, 30, 33),  # quad path, across two blocks
]


@pytest.mark.parametrize("thr", IOU_THRESHOLDS)
def test_iou_at_threshold_every_segment_path(thr, monkeypatch):
    """Box pairs whose IoU quotient lies on, or one float32 step either side of, the threshold (and just inside / outside
    the band the kernel decides without dividing) through every segment path: the kept rows equal the oracle's.  A union
    is at least 1e-16 and every compacted box is wider than MIN_WH, so the subnormal side of the range test cannot be
    reached from candidates, and a union that overflows (at a threshold >= 0) would leave the reference's loop without
    end; unions in [2^127, inf), whose product with the band edge may overflow, are reached."""
    pairs = special_pairs(thr)
    t = f32(thr)
    if t > 0:
        near = near_threshold_pairs(thr)
        assert len(near) >= 6, len(near)
        pairs = near + pairs
    for a, b in pairs:                                    # the shortcut's claim, on the host
        assert kernel_iou_gt(a, b, thr)[0] == (reference_iou(a, b)[0] > t)
        assert self_iou_terminates(a, thr) and self_iou_terminates(b, thr)
    if t > f32(1e-20):                                    # unions beyond the range test's bound, decided near thr
        assert any(pair_union(a, b) >= 2.0 ** 127 and reference_iou(a, b)[0] > f32(0) for a, b in pairs)
    if thr in BANDLESS_SENSITIVE:                         # pairs that need the band: without it they are decided wrongly
        bandless = [kernel_iou_gt(a, b, thr, 1.0, 1.0)[0] != (reference_iou(a, b)[0] > t) for a, b in pairs]
        assert any(bandless), "no pair separates the kernel's band from no band at all"
    for size, mpc, pos_a, pos_b in IOU_LAYOUTS:
        pred_cpu = embed_pairs(pairs, size, pos_a, pos_b)
        buf = load_candidates(pred_cpu, 0.0, mpc)
        hist = class_histograms(buf)
        assert (hist == size).all(), "a pair box did not pass the candidate filter"
        deal = restate_deal(hist, buf.cap, mpc, 32, sm_count())
        assert deal.pack_ok == (mpc >= 32) and deal.n_segs == (len(pairs) if size > 32 or mpc < 32 else 0)
        out, out_row, kept, wc = run_nms(buf, thr, 32)
        check_counters(wc, deal)
        want, wrows = oracle(pred_cpu, 0.0, thr, mpc, monkeypatch)
        assert_oracle(out, out_row, kept, want, wrows, f"thr {thr!r} class size {size} mpc {mpc} positions {pos_a},{pos_b}")


# ------------------------------------------------------------------------------------------------------------------
# 5. The completion stamp on one GPU
@pytest.mark.parametrize("batch,n,ft", [(1024, 300, 128), (64, 6000, 512)])
def test_completion_stamp_single_gpu(batch, n, ft):
    """``step = (seq, stamp)``: after k calls seq == stamp == k and the finalize CTAs' counter is back at 0 after every call,
    eagerly and inside a captured graph replayed three times; batch 0 still posts; the results are those of the call
    without a stamp."""
    pred_cpu = synth.synth_prediction(batch, n, nc=80, seed=batch)
    buf = load_candidates(pred_cpu, 0.05, 100)
    deal = restate_deal(class_histograms(buf), buf.cap, 100, 0, sm_count())
    assert deal.ft == ft
    seq = torch.zeros(1, dtype=torch.int32, device=DEV)
    stamp = torch.zeros(1, dtype=torch.int32, device=DEV)
    step = (seq.data_ptr(), stamp.data_ptr())
    plain = run_nms(buf, 0.5, 0)
    check_counters(plain[3], deal)
    calls = 0
    for _ in range(3):
        res = run_nms(buf, 0.5, 0, step=step)
        calls += 1
        assert seq.item() == calls and stamp.item() == calls
        assert res[3][1] == 0
        check_counters(res[3], deal)
        assert_same_bits(res[:3], plain[:3], f"stamped call {calls}")

    out, out_row = padded_outputs(batch, buf.out_cap)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            ops.nms(buf, 0.5, out, out_row, step=step)
    torch.cuda.current_stream().wait_stream(stream)
    torch.cuda.synchronize()
    assert seq.item() == calls                         # capture runs nothing
    for _ in range(3):
        graph.replay()
        calls += 1
        torch.cuda.synchronize()
        assert seq.item() == calls and stamp.item() == calls
        wc = read_work_count(buf)
        assert wc[1] == 0
        check_counters(wc, deal)
        assert_same_bits((out, out_row, ops.read_counts(buf)[1].clone()), plain[:3], f"graph replay {calls}")

    empty = ops.Buffers(DEV, 0, n, 80)                 # a rank without images: nothing to write, the stamp still posts
    sink = torch.zeros(8, dtype=torch.int32, device=DEV)
    ops.nms(empty, 0.5, None, None, out_ptrs=(sink.data_ptr(), sink.data_ptr(), empty.out_count_ptr), step=step)
    calls += 1
    torch.cuda.synchronize()
    assert seq.item() == calls and stamp.item() == calls
