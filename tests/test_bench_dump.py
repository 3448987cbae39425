"""bench.py --dump-outputs: the result of the last timed step, written as float32 / float64 .npy files, equals what the
path returns for that step's (seeded) input; --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import yolo_oracle
from pytorch_yolo_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("detections", "kept_per_image", "image_index")


def _bench(*args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def _load(path, names):
    out = {n: np.load(os.path.join(path, n + ".npy")) for n in names}
    for n, a in out.items():
        assert a.dtype in (np.float32, np.float64), n
    return out


def _assert_dump_equals(dump, dets, rows=None):
    index = dump["image_index"].astype(np.int64)
    kept = [0 if dets[i] is None else len(dets[i]) for i in index]
    assert dump["kept_per_image"].tolist() == kept
    want = torch.cat([dets[i].cpu() for i in index if dets[i] is not None] + [torch.empty(0, 7)])
    assert np.array_equal(dump["detections"].view(np.int32), want.numpy().view(np.int32))       # bit for bit
    if rows is not None:
        want_rows = torch.cat([rows[i].cpu().double() for i in index if rows[i] is not None]
                              + [torch.empty(0, dtype=torch.float64)])
        assert np.array_equal(dump["anchor_rows"], want_rows.numpy())


def test_dump_sample_is_fixed_and_bounded(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1024 + 10 * (50 * 36 + 16))       # room for 10 images of capacity 50
    g = torch.Generator().manual_seed(3)
    dets = [None if i % 7 == 0 else torch.rand(int(torch.randint(1, 50, (1,), generator=g)), 7, generator=g)
            for i in range(40)]
    rows = [None if d is None else torch.randint(0, 1000, (len(d),), dtype=torch.int32, generator=g) for d in dets]
    bench.dump_outputs(str(tmp_path / "a"), dets, rows, 50)
    bench.dump_outputs(str(tmp_path / "b"), [None if d is None else d + 1 for d in dets], rows, 50)
    a = _load(tmp_path / "a", NAMES + ("anchor_rows",))
    b = _load(tmp_path / "b", NAMES + ("anchor_rows",))
    assert np.array_equal(a["image_index"], b["image_index"])                 # the sample does not depend on the values
    index = a["image_index"]
    assert len(index) == 10 and np.all(np.diff(index) > 0) and index[-1] < 40
    _assert_dump_equals(a, dets, rows)
    assert sum(os.path.getsize(tmp_path / "a" / (n + ".npy")) for n in NAMES + ("anchor_rows",)) <= bench.DUMP_LIMIT_BYTES


def test_reference_arm_dumps_its_last_step(tmp_path):
    line = _bench("--impl", "reference", "--workload", "tiny-416", "--batch", "3", "--steps", "2", "--warmup", "1",
                  "--dump-outputs", str(tmp_path))
    assert line["steps"] == 2
    dump = _load(tmp_path, NAMES)
    w = synth.WORKLOADS["tiny-416"]
    heads = synth.synth_heads("tiny-416", 3, "B", seed=1234)
    want = yolo_oracle.non_max_suppression(yolo_oracle.decode_heads(heads, w["anchors"], w["nc"], w["img_size"]), 0.3, 0.5)
    assert dump["image_index"].tolist() == [0, 1, 2] and dump["kept_per_image"].sum() > 0
    _assert_dump_equals(dump, want)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(tmp_path):
    from pytorch_yolo_b200 import ops
    from pytorch_yolo_b200.detect import detect
    wl, batch, steps = "tiny-416", 8, 3
    line = _bench("--gpus", "1", "--only", "--workload", wl, "--batch", str(batch), "--steps", str(steps), "--warmup", "1",
                  "--dump-outputs", str(tmp_path))
    assert line["steps"] == steps
    dump = _load(tmp_path, NAMES + ("anchor_rows",))
    # the timed loop cycles through n_sets resident input sets (bench.Case): step k reads set k % n_sets
    n_sets = min(64, max(1, int(-(-160e6 // (synth.head_bytes_per_image(wl) * batch)))))
    assert (steps - 1) % n_sets != 0                      # the last step does not read the first set
    w = synth.WORKLOADS[wl]
    heads = synth.synth_heads(wl, batch, "B", seed=1234 + (steps - 1) % n_sets, device="cuda:0")
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    dets, rows = detect(heads, specs, w["nc"], 0.3, 0.5, return_rows=True)
    assert dump["image_index"].tolist() == list(range(batch)) and dump["kept_per_image"].sum() > 0
    _assert_dump_equals(dump, dets, rows)
