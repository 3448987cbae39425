"""The evaluation loop (SURVEY.md section 8f row 2) against records the LIVE reference produced.

``tests/golden/eval_loop.npz`` (with ``eval_loop_a1.npz``) holds the ``{path: [records]}`` dicts of the inner loop of the reference's ``test_model``
(utils/utils.py:374-379; made by tests/golden/make_golden_eval.py).  CPU: the oracle's restatement of that loop reproduces
them exactly.  GPU: (1) fed the reference's decoded tensor, the drop-in ``non_max_suppression`` + ``dict_from_results``
give the same records -- scores and classes bit-exact, pixel coordinates equal except where a MERGE box (rtol 1e-5, see
DESIGN.md section 2) sits within that distance of a rounding boundary; (2) ``EvalPipeline`` -- H2D, heads, fused decode + NMS,
un-letterbox kernel, D2H, all overlapped -- gives the same records up to the decode's 1e-5.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import yolo_oracle
from pytorch_yolo_b200 import synth
from tests.helpers import GOLDEN_DIR, load_golden

DEV = "cuda:0"
SPP_SMALL = synth.WORKLOADS["mini-96"]


def _golden():
    g = {**load_golden("eval_loop"), **load_golden("eval_loop_a1")}
    tiny = load_golden("tiny416_randinit")
    model_a = dict(anchors=SPP_SMALL["anchors"], nc=SPP_SMALL["nc"], cur_shape=(96, 96), batches=[])
    for bi in range(2):
        heads = [torch.from_numpy(g[f"a{bi}_head{k}"]) for k in range(3)]
        shapes = [tuple(int(v) for v in s) for s in g[f"a{bi}_shapes"]]
        model_a["batches"].append((heads, [f"a{bi}_{i}.jpg" for i in range(len(shapes))], shapes))
    model_b = dict(anchors=synth.TINY_ANCHORS, nc=80, cur_shape=(416, 416),
                   batches=[([torch.from_numpy(tiny["head0"]), torch.from_numpy(tiny["head1"])], ["b0_0.jpg"],
                             [tuple(int(v) for v in g["b_shapes"][0])])])
    return (float(g["conf"]), float(g["nms"]),
            ((model_a, json.loads(str(g["records_a"]))), (model_b, json.loads(str(g["records_b"])))))


def _compare(got: dict, want: dict, exact_scores: bool, max_pixel_mismatch: float):
    assert sorted(got) == sorted(want)
    n = bad = 0
    for path, wrecs in want.items():
        grecs = got[path]
        assert len(grecs) == len(wrecs), f"{path}: {len(grecs)} records, reference has {len(wrecs)}"
        for gr, wr in zip(grecs, wrecs):
            assert gr["type"] == wr["type"], path
            if exact_scores:
                assert gr["score"] == wr["score"], path
            else:
                assert abs(gr["score"] - wr["score"]) <= 1e-5 * abs(wr["score"]), path
            for k in ("left", "top", "right", "bottom"):
                assert abs(gr[k] - wr[k]) <= 1, (path, k, gr[k], wr[k])
                n += 1
                bad += gr[k] != wr[k]
    assert bad <= max_pixel_mismatch * n, f"{bad} of {n} pixel coordinates differ from the reference's"


def test_oracle_eval_loop_matches_reference_records():
    conf, nms, cases = _golden()
    for model, want in cases:
        data = {}
        for heads, paths, shapes in model["batches"]:
            pred = yolo_oracle.decode_heads(heads, model["anchors"], model["nc"], max(model["cur_shape"]))
            det = yolo_oracle.non_max_suppression(pred, conf, nms)
            data = yolo_oracle.records_from_results(data, det, paths, shapes, model["cur_shape"])
        assert data == want


@pytest.mark.gpu
def test_drop_in_nms_and_records_on_reference_decode():
    from pytorch_yolo_b200.utils.utils import dict_from_results, non_max_suppression
    conf, nms, cases = _golden()
    for model, want in cases:
        data = {}
        for heads, paths, shapes in model["batches"]:
            pred = yolo_oracle.decode_heads(heads, model["anchors"], model["nc"], max(model["cur_shape"]))   # == the reference's p
            det = non_max_suppression(pred.to(DEV), conf, nms)
            data = dict_from_results(data, det, paths, shapes, model["cur_shape"])
        _compare(data, want, exact_scores=True, max_pixel_mismatch=0.002)


class _StubModel:
    """What EvalPipeline needs of a reference model: ``yolo_layers`` and ``_forward_encoder`` (the backbone is out of
    scope: it is replaced by a lookup of the committed head tensors, keyed by the batch id stored in the image tensor)."""

    def __init__(self, anchors, nc, batches):
        from pytorch_yolo_b200 import YOLOLayer
        self.yolo_layers = [YOLOLayer(a, nc, anchors).eval() for a in anchors]
        self.heads = [[h.to(DEV) for h in heads] for heads, _, _ in batches]

    def _forward_encoder(self, x):
        return tuple(self.heads[int(x[0, 0, 0, 0].item())])


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [1, 2])
def test_eval_pipeline_matches_reference_records(depth):
    from pytorch_yolo_b200.pipeline import EvalPipeline
    conf, nms, cases = _golden()
    for model, want in cases:
        stub = _StubModel(model["anchors"], model["nc"], model["batches"])
        h, w = model["cur_shape"]

        def batches():
            for bi, (heads, paths, shapes) in enumerate(model["batches"]):
                yield torch.full((heads[0].shape[0], 3, h, w), float(bi)), paths, shapes

        got = EvalPipeline(stub, DEV, conf, nms, depth=depth).run(batches())
        if model is cases[1][0]:
            # random-init tiny model: thousands of anchors score 0.2605 +- 1e-6, so the decode's 1e-6 relative error decides
            # which box leads each cluster; record-level equality is only defined on identical decoded input (the test
            # above).  What must hold here: same images, same class, about as many records, same score level.
            assert sorted(got) == sorted(want)
            for path, wrecs in want.items():
                assert abs(len(got[path]) - len(wrecs)) <= max(2, 0.1 * len(wrecs))
                assert {r["type"] for r in got[path]} == {r["type"] for r in wrecs}
                assert abs(got[path][0]["score"] - wrecs[0]["score"]) <= 1e-5 * wrecs[0]["score"]
            continue
        _compare(got, want, exact_scores=False, max_pixel_mismatch=0.01)
