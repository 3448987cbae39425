"""Shared helpers for the test-suite (golden loading, ragged unpacking, comparisons)."""
from __future__ import annotations

import os

import numpy as np
import torch

from pytorch_yolo_b200 import ops

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

NMS_GOLDEN = ["nms_clustered", "nms_ties", "nms_lowconf", "nms_cap100", "nms_edges_50", "nms_edges_49", "nms_empty"]
DECODE_GOLDEN = ["decode_nms_mini-96_B", "decode_nms_mini-160_A"]


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        return {k: z[k] for k in z.files}


def unpack(counts, flat):
    """counts (B,), flat (sum,7) -> list of tensors | None, like the reference's return value."""
    out, o = [], 0
    for c in counts.tolist():
        out.append(None if c == 0 else torch.from_numpy(np.ascontiguousarray(flat[o:o + c])))
        o += c
    return out


def assert_dets_equal(got, want, box_rtol=0.0, what=""):
    """Scores / class_conf / class (cols 4..6) bit-exact, order included; boxes within box_rtol (0 = bit-exact)."""
    assert len(got) == len(want), what
    for i, (g, w) in enumerate(zip(got, want)):
        if w is None:
            assert g is None, f"{what} image {i}: expected None, got {None if g is None else tuple(g.shape)}"
            continue
        assert g is not None, f"{what} image {i}: expected {tuple(w.shape)}, got None"
        g = g.detach().cpu()
        assert g.shape == w.shape, f"{what} image {i}: {tuple(g.shape)} vs {tuple(w.shape)}"
        assert g.dtype == torch.float32
        assert torch.equal(g[:, 4:], w[:, 4:]), f"{what} image {i}: score/class columns differ"
        if box_rtol == 0.0:
            assert torch.equal(g[:, :4], w[:, :4]), f"{what} image {i}: boxes differ " \
                f"(max abs {float((g[:, :4] - w[:, :4]).abs().max()):.3e})"
        else:
            torch.testing.assert_close(g[:, :4], w[:, :4], rtol=box_rtol, atol=1e-30, msg=lambda m: f"{what} image {i}: {m}")


def prediction_with_class_sizes(sizes_per_image, nc, seed):
    """(B, N, 5+nc) decoded-looking tensor in which class c of image b holds exactly sizes_per_image[b][c] candidates
    (boxes clustered so that suppression and MERGE clusters occur), rows shuffled."""
    g = torch.Generator().manual_seed(seed)
    n = max(sum(s) for s in sizes_per_image)
    pred = torch.zeros(len(sizes_per_image), n, 5 + nc)
    for b, sizes in enumerate(sizes_per_image):
        cls = torch.cat([torch.full((k,), c, dtype=torch.long) for c, k in enumerate(sizes)])
        m = len(cls)
        centre = 300 * torch.rand(nc, 2, generator=g) + 100
        pred[b, :m, 0:2] = centre[cls] + 12 * torch.randn(m, 2, generator=g)
        pred[b, :m, 2:4] = 40 + 25 * torch.rand(m, 2, generator=g)
        pred[b, :m, 4] = 0.3 + 0.7 * torch.rand(m, generator=g)
        pred[b, torch.arange(m), 5 + cls] = 0.5 + 0.5 * torch.rand(m, generator=g)
        perm = torch.randperm(n, generator=g)
        pred[b] = pred[b, perm]                       # rows beyond m are all-zero: score 0, dropped by the filter
    return pred


def expected_candidates(dense, conf, min_wh=ops.MIN_WH):
    """Per image: (rows, meta (score, cls_conf bits; class; row), box bits) of what the reference emits on the decoded
    tensor: first arg-max of the sigmoid columns, score = fl(sigma(obj) * cls_conf)."""
    d = dense.cpu().numpy()
    with np.errstate(invalid="ignore", over="ignore"):
        cls_s = d[..., 5:]
        cls = np.argmax(cls_s, -1)
        cls_conf = np.take_along_axis(cls_s, cls[..., None], -1)[..., 0]
        score = d[..., 4] * cls_conf
        x, y, w, h = d[..., 0], d[..., 1], d[..., 2], d[..., 3]
        emit = (~np.isnan(d).any(-1)) & (score > np.float32(conf)) & (w > np.float32(min_wh)) & (h > np.float32(min_wh))
        emit &= np.isfinite(d[..., :4]).all(-1)
        hw, hh = w * np.float32(0.5), h * np.float32(0.5)
        box = np.stack([x - hw, y - hh, x + hw, y + hh], -1)
    per_img = []
    for b in range(d.shape[0]):
        r = np.nonzero(emit[b])[0]
        meta = np.stack([score[b, r].view(np.int32), cls_conf[b, r].view(np.int32), cls[b, r].astype(np.int32),
                         r.astype(np.int32)], -1)
        per_img.append((meta, box[b, r].view(np.int32)))
    return per_img, emit, cls


def read_candidates(buf):
    counts, _, ovf = ops.read_counts(buf)
    assert ovf == 0
    counts = counts.clone()
    out = []
    for b in range(buf.batch):
        n = int(counts[b])
        meta = buf.cand_meta[b * buf.cap:b * buf.cap + n].cpu().numpy()
        box = buf.cand_box[b * buf.cap:b * buf.cap + n].cpu().numpy().view(np.int32)
        o = np.argsort(meta[:, 3], kind="stable")
        out.append((meta[o], box[o]))
    return out


def assert_same_candidates(got, want, what):
    for b, ((gm, gb), (wm, wb)) in enumerate(zip(got, want)):
        assert gm.shape == wm.shape, f"{what} image {b}: {len(gm)} candidates, expected {len(wm)}"
        bad = np.nonzero((gm != wm).any(-1) | (gb != wb).any(-1))[0]
        assert bad.size == 0, (f"{what} image {b}: {bad.size} candidates differ, first row {wm[bad[0], 3]}: "
                               f"got class {gm[bad[0], 2]} conf {gm[bad[0], 1:2].view(np.float32)}, expected class "
                               f"{wm[bad[0], 2]} conf {wm[bad[0], 1:2].view(np.float32)}")
