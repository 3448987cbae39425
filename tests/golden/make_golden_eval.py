"""Golden records of the reference's evaluation loop (SURVEY.md section 8f row 2).

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden_eval.py

Runs the inner loop of the reference's ``test_model`` (utils/utils.py:374-379) -- model output ``p`` =
``torch.cat`` of the ``YOLOLayer.forward`` results, ``non_max_suppression(p, 0.1, 0.1)`` (test_model's default
thresholds, utils.py:359; stable-argsort tie rule as in make_golden.py), ``_dict_from_results`` -- with the LIVE,
unmodified reference functions, on two "models":

* A: three-scale SPP-anchor heads of the mini-96 workload, two batches of three images (seeded synthetic heads stand in
  for the backbone, which is out of scope), letterboxed 96x96 inputs of three different original shapes;
* B: the random-init YOLOv3-tiny 416x416 forward of BASELINE config 1 (its head tensors are already committed in
  tiny416_randinit.npz), one batch of one image.

Stores the head tensors of A, the shapes / paths and the resulting ``{path: [records]}`` dicts as JSON.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_loader                      # noqa: E402
from pytorch_yolo_b200 import synth                # noqa: E402
from tests.golden.make_golden import ref_decode    # noqa: E402

CONF, NMS = 0.1, 0.1                               # test_model defaults (utils.py:359)
BATCHES_A = (("B", 3, 31, ((480, 640), (96, 96), (333, 500))),
             ("A", 3, 32, ((1080, 1920), (97, 1333), (64, 48))))


def ref_loop(ref, data, pred, paths, shapes, cur_shape):
    """utils.py:378-379 on one batch."""
    with ref_loader.stable_argsort():
        det = ref.non_max_suppression(pred, CONF, NMS)
    return ref.dict_from_results(data, det, paths, shapes, cur_shape)


def main():
    torch.set_num_threads(1)
    ref = ref_loader.load()
    w = synth.WORKLOADS["mini-96"]
    arrays, data_a = {}, {}
    for bi, (kind, batch, seed, shapes) in enumerate(BATCHES_A):
        heads = synth.synth_heads("mini-96", batch, kind, seed)
        pred = ref_decode(ref, heads, w["anchors"], w["nc"], w["img_size"])
        paths = [f"a{bi}_{i}.jpg" for i in range(batch)]
        data_a = ref_loop(ref, data_a, pred, paths, shapes, (96, 96))
        for k, h in enumerate(heads):
            arrays[f"a{bi}_head{k}"] = h.numpy()
        arrays[f"a{bi}_shapes"] = np.array(shapes)
    g = np.load(os.path.join(HERE, "tiny416_randinit.npz"))
    heads_b = [torch.from_numpy(g["head0"]), torch.from_numpy(g["head1"])]
    pred_b = ref_decode(ref, heads_b, synth.TINY_ANCHORS, 80, 416)
    data_b = ref_loop(ref, {}, pred_b, ["b0_0.jpg"], ((375, 500),), (416, 416))
    path = os.path.join(HERE, "eval_loop.npz")
    # the second batch's heads go to a file of their own: each file stays under 1 MB
    side = {k: arrays.pop(k) for k in list(arrays) if k.startswith("a1_")}
    np.savez_compressed(os.path.join(HERE, "eval_loop_a1.npz"), **side)
    np.savez_compressed(path, conf=np.float64(CONF), nms=np.float64(NMS), records_a=np.array(json.dumps(data_a)),
                        records_b=np.array(json.dumps(data_b)), b_shapes=np.array(((375, 500),)), **arrays)
    print(f"eval_loop: {os.path.getsize(path) / 1024:.0f} KiB; records A {sum(len(v) for v in data_a.values())} in "
          f"{len(data_a)} images, B {sum(len(v) for v in data_b.values())}")


if __name__ == "__main__":
    main()
