#!/usr/bin/env python
"""bench.py -- YOLO decode+NMS images/s on B200, with the HBM roofline of the decode/compaction kernel.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] ...
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of synthetic head tensors: fused decode + confidence
filter + compaction, the three NMS kernels and the read-back of the per-image counts.  Rank 0 prints ONE
JSON line.  Weak scaling: every GPU processes ``--batch`` images per step (global batch = batch * N); kept
rows of all ranks land in rank 0's memory through NVLink peer stores and rank 0 waits, every step, for the
completion stamps of all ranks (device-side flags; no collective on the hot path).

Extra keys next to the contract's: ``roofline`` (decode_compact_kernel timed alone), ``e2e`` (pinned host heads ->
H2D -> path -> D2H rows), ``cpu_baseline`` (the UNMODIFIED reference functions from oracle/_ref on the host cores),
``configs`` (the other BASELINE.json configs, bounded), ``drop_in`` (the reference-shaped API: YOLOLayer.forward per
scale + torch.cat + non_max_suppression), ``head_fusion`` (SURVEY 8f-3), ``gather_check`` (N > 1: the gathered rows
on rank 0 against every rank's locally computed result).

``oracle/`` is imported only by the ``cpu_baseline`` leg and by ``--impl reference``.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "YOLO decode+NMS images/sec"
UNIT = "images/s"
DEFAULTS = dict(workload="spp-608", batch=64, kind="B", conf=0.3, nms=0.5)
# images per CPU measurement: the whole batch where the reference gets through it in seconds (same config as the GPU
# arm), a bounded sample of it otherwise (SURVEY 8d: about 10-30 s of CPU work per leg)
WARM_SECONDS = 0.04          # minimum duration of the untimed warm-up (see Case.timed)
DEFAULT_STEPS = 2000
DUMP_LIMIT_BYTES = 64 << 20  # --dump-outputs: all files together
CPU_SAMPLE_BATCH = {"spp-608": 64, "spp-1024": 8, "tiny-416": 256}
# the other BASELINE.json configs, measured in the same run (bounded): (label, workload, batch/GPU, kind, conf, nms)
EXTRA_CONFIGS = [
    ("cfg3 tiny-416 b1024", "tiny-416", 1024, "B", 0.3, 0.5),
    ("cfg4 spp-608 b64 mAP-eval conf 0.001", "spp-608", 64, "B", 0.001, 0.5),
    ("cfg5 spp-1024 b256", "spp-1024", 256, "B", 0.3, 0.5),
]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help=f"timed steps (default {DEFAULT_STEPS}; --impl reference: as many as --ref-budget-s allows)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULTS["workload"])
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step")
    ap.add_argument("--kind", default=DEFAULTS["kind"], help="synthetic input: A (iid logits) or B (+ planted objects)")
    ap.add_argument("--conf", type=float, default=DEFAULTS["conf"])
    ap.add_argument("--nms", type=float, default=DEFAULTS["nms"])
    ap.add_argument("--variant", default="auto", choices=["auto", "ldg", "tma", "tma2d"], help="decode_compact kernel variant")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-priority", action="store_true", help="NMS kernels on the lane's own stream (no high-priority side stream)")
    ap.add_argument("--depth", type=int, default=None,
                    help="batches in flight (streams): NMS of batch i overlaps decode of i+1; default 3")
    ap.add_argument("--seg-warps", type=int, default=0, help="residency of the NMS segment kernel, warps per SM (0 = default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-head-fusion", action="store_true", help="skip the extra 'head_fusion' measurement (SURVEY 8f-3)")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra 'configs' key (BASELINE configs 1, 3, 4, 5)")
    ap.add_argument("--no-drop-in", action="store_true", help="skip the extra 'drop_in' key (reference-shaped API path)")
    ap.add_argument("--only", action="store_true", help="headline only: no extras at all")
    ap.add_argument("--config-steps", type=int, default=30)
    ap.add_argument("--cpu-runs", type=int, default=5)
    ap.add_argument("--cpu-kind", default="reference", choices=["reference", "port"])
    ap.add_argument("--ref-budget-s", type=float, default=150.0,
                    help="--impl reference without --steps: wall-clock budget of the timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def default_batch(workload):
    return {"spp-608": 64, "tiny-416": 1024, "spp-1024": 256}.get(workload, 8)


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def sample(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80}
        for k, bit in names.items():
            if r & bit:
                self.reasons.add(k)

    def run(self):
        if not self.ok:
            return
        while not self._halt.is_set():
            try:
                self.sample()
            except Exception:  # noqa: BLE001
                break
            self._halt.wait(self.period)

    def finish(self):
        self._halt.set()
        if self.ok:
            self.join(timeout=2)
            try:
                self.sample()
            except Exception:  # noqa: BLE001
                pass
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_index: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_index])
        except Exception:  # noqa: BLE001
            pass
    return local_index


# ------------------------------------------------------------------------------------------- CPU legs
def cpu_run(kind, workload, batch, synth_kind, conf, nms, runs, warm=1, budget_s=None):
    """Times the reference path on the host cores: ``kind == "reference"`` runs the UNMODIFIED reference functions
    (YOLOLayer.forward per scale + torch.cat + non_max_suppression, loaded by path from oracle/_ref or the reference
    checkout); ``"port"`` runs the oracle restatement.  Returns (images/s of the median run, per-run seconds, kind used,
    the detections of the last run)."""
    from pytorch_yolo_b200 import synth
    w = synth.WORKLOADS[workload]
    heads = synth.synth_heads(workload, batch, synth_kind, seed=1234)
    fn = None
    if kind == "reference":
        from oracle import ref_loader
        if ref_loader.available():
            import warnings
            warnings.filterwarnings("ignore", message="torch.meshgrid")
            ref = ref_loader.load()
            layers = [ref.YOLOLayer(a, w["nc"], w["anchors"]).eval() for a in w["anchors"]]

            def fn():
                io = [l(h, w["img_size"])[0] for l, h in zip(layers, heads)]       # yolov3_spp.py:151-153
                pred = torch.cat(io, 1)                                             # yolov3_spp.py:163-164
                return ref.non_max_suppression(pred, conf, nms)                    # utils.py:200-293
        else:
            kind = "port"
    if fn is None:
        from oracle import yolo_oracle

        def fn():
            pred = yolo_oracle.decode_heads(heads, w["anchors"], w["nc"], w["img_size"])
            return yolo_oracle.non_max_suppression(pred, conf, nms)
    times = []
    t_start = time.perf_counter()
    with torch.no_grad():
        for i in range(warm + runs):
            t0 = time.perf_counter()
            dets = fn()
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
            if budget_s is not None and times and time.perf_counter() - t_start + dt > budget_s:
                break
    return batch / statistics.median(times), times, kind, dets


def cpu_tiny_model_run(runs=10):
    """BASELINE config 1 on the host cores: the reference's YOLOv3-tiny (random init, seed 0), 416x416 batch 1, full
    forward + decode + non_max_suppression(conf 0.1) -- SURVEY.md 8d.  Returns a dict or None without the reference."""
    from oracle import ref_loader
    if not ref_loader.available():
        return None
    import warnings
    warnings.filterwarnings("ignore", message="torch.meshgrid")
    ref = ref_loader.load()
    torch.manual_seed(0)
    model = ref.YOLOv3Tiny().eval()
    x = torch.rand(1, 3, 416, 416)
    tf, tn = [], []
    with torch.no_grad():
        for i in range(runs + 2):
            t0 = time.perf_counter()
            pred, _ = model(x)
            t1 = time.perf_counter()
            out = ref.non_max_suppression(pred, 0.1, 0.5)
            t2 = time.perf_counter()
            if i >= 2:
                tf.append(t1 - t0)
                tn.append(t2 - t1)
    kept = 0 if out[0] is None else len(out[0])
    f, n = statistics.median(tf), statistics.median(tn)
    return {"forward_ms": 1e3 * f, "nms_ms": 1e3 * n, "images_per_s": 1.0 / (f + n), "kept": kept,
            "what": "reference YOLOv3Tiny random-init forward (encoder + YOLOLayer decode) + non_max_suppression, CPU"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (unmodified functions from oracle/_ref) on
    the host cores, same metric / unit / config as the GPU arm; each step is one batch (a bounded sample of it for the
    workloads the CPU needs minutes per batch for)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    full_b = args.batch
    sample_b = min(full_b, CPU_SAMPLE_BATCH.get(args.workload, 8))
    warm = max(1, min(args.warmup, 2))
    ips, times, kind, dets = cpu_run(args.cpu_kind, args.workload, sample_b, args.kind, args.conf, args.nms,
                                     runs=args.steps or DEFAULT_STEPS, warm=warm,
                                     budget_s=args.ref_budget_s if args.steps is None else None)
    if args.dump_outputs:
        from pytorch_yolo_b200 import synth
        dump_outputs(args.dump_outputs, dets, None, synth.anchors_per_image(args.workload))
    sample = (f"{args.workload} SYNTH-{args.kind} {sample_b} of {full_b} images per step, conf {args.conf} nms {args.nms}, "
              f"{len(times)} timed steps (median), torch threads {torch.get_num_threads()}")
    line = {
        "metric": METRIC, "value": ips, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
        "steps": len(times), "warmup": warm, "ms_per_step": 1e3 * statistics.median(times) * full_b / sample_b,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, full_b),
        "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, batch):
    from pytorch_yolo_b200 import synth
    return {"workload": f"{args.workload} ({synth.anchors_per_image(args.workload)} anchors/img, 80 classes) "
                        f"SYNTH-{args.kind} heads, batch {batch}/GPU, conf {args.conf} nms {args.nms}",
            "batch_per_gpu": batch, "conf_thres": args.conf, "nms_thres": args.nms,
            "l2": "inputs exceed L2 (no flush needed)" if synth.head_bytes_per_image(args.workload) * batch > 126e6
                  else "inputs rotate through >L2 worth of buffers",
            "sharding": "images across GPUs, kept rows to rank 0 by NVLink peer stores"}


def dump_outputs(path, dets, rows, cap):
    """--dump-outputs: what the caller of the timed path received from its last step, as .npy files in `path`, so that
    two builds can be compared output for output (the inputs depend only on the arguments).
      detections.npy      float32 (n, 7)  kept rows (x1, y1, x2, y2, obj, cls_conf, cls) of the dumped images, in order
      kept_per_image.npy  float64         number of those rows per dumped image
      image_index.npy     float64         which images of the batch were dumped
      anchor_rows.npy     float64 (n,)    anchor row each kept row came from (GPU arm only)
    `dets` / `rows`: per image an (n, 7) / (n,) tensor or None; `cap`: most rows one image can keep.  All images are
    dumped when their largest possible result fits DUMP_LIMIT_BYTES, else a fixed seeded sample of them, which depends
    only on the batch size and `cap`."""
    import numpy as np
    per_image = cap * (7 * 4 + (8 if rows is not None else 0)) + 16
    take = min(len(dets), (DUMP_LIMIT_BYTES - 1024) // per_image)       # 1024: the .npy headers
    if take == len(dets):
        index = torch.arange(len(dets))
    else:
        index = torch.randperm(len(dets), generator=torch.Generator().manual_seed(0))[:take].sort().values
    index = index.tolist()
    kept = [0 if dets[i] is None else len(dets[i]) for i in index]
    arrays = {
        "detections": torch.cat([dets[i].cpu() for i in index if dets[i] is not None] + [torch.empty(0, 7)]).numpy(),
        "kept_per_image": np.array(kept, dtype=np.float64),
        "image_index": np.array(index, dtype=np.float64),
    }
    if rows is not None:
        arrays["anchor_rows"] = torch.cat([rows[i].cpu().double() for i in index if rows[i] is not None]
                                          + [torch.empty(0, dtype=torch.float64)]).numpy()
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------- one workload on the GPU(s)
class Case:
    """One workload set up on this rank: resident head tensors, the (sharded) pipeline with every lane's graph captured
    at construction, and the step loop."""

    def __init__(self, workload, batch, kind, conf, nms, dev, rank, world, depth=None, variant="auto", use_graph=True,
                 priority=True, seg_warps=0):
        import torch.distributed as dist
        from pytorch_yolo_b200 import ops, synth
        from pytorch_yolo_b200.detect import PipelinedDetector
        from pytorch_yolo_b200.sharded import ShardedDetector
        self.workload, self.B, self.kind, self.conf, self.nms = workload, batch, kind, conf, nms
        self.dev, self.rank, self.world, self.variant = dev, rank, world, variant
        self.dist = dist if world > 1 else None
        self.w = w = synth.WORKLOADS[workload]
        self.bytes_per_img = synth.head_bytes_per_image(workload)
        # deeper pipelines hide the fixed per-batch latencies of small batches; big batches gain nothing and lose cache
        self.depth = depth if depth is not None else 3      # measured best on every BASELINE config (profiles/r02_a_pipeline_depth.txt)
        self.specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        # inputs: resident in HBM; when one batch is smaller than L2, rotate through enough distinct batches
        self.n_sets = min(64, max(1, int(-(-160e6 // (self.bytes_per_img * batch)))))
        self.head_sets = [synth.synth_heads(workload, batch, kind, seed=1234 + 7919 * rank + s, device=dev)
                          for s in range(self.n_sets)]
        torch.cuda.synchronize(dev)
        kw = dict(depth=self.depth, variant=variant)
        if seg_warps and world == 1:
            kw["seg_warps_per_sm"] = seg_warps
        if world > 1:
            # one sharded pipeline; with several input sets the pointers change per step -> eager launches
            self.det = ShardedDetector(self.specs, w["nc"], batch * world, dev, conf, nms,
                                       use_graph=use_graph and self.n_sets == 1, **kw)
            self.pipes = [self.det.pipe] * self.n_sets
            if use_graph and self.n_sets == 1:
                self.det.bind(self.head_sets[0])
        else:
            self.det = None
            # one pipeline (one captured graph per lane) per input set so that graph replay sees static pointers
            self.pipes = [PipelinedDetector(self.specs, w["nc"], batch, dev, conf, nms, use_graph=use_graph,
                                            nms_priority=priority and self.depth > 1, **kw) for _ in range(self.n_sets)]
            if use_graph:
                for p, hs in zip(self.pipes, self.head_sets):
                    p.bind(hs)                   # all lanes captured here: nothing but graph replays in the timed loop
        self.lane0 = self.pipes[0].lanes[0]
        torch.cuda.synchronize(dev)

    def run_steps(self, k, after_last_submit=None):
        """k steps with `depth` batches in flight: submit step i, then wait for step i - depth + 1.  N > 1: the wait is
        the gather -- on rank 0 it covers the rows of every rank (device-side stamps).  `after_last_submit` runs once all k
        steps are enqueued, before the host waits for the last `depth` of them (the timed loop enqueues its end event
        there: the event then marks the completion of the GPU work, not the moment the host got round to recording it)."""
        pending, last = [], None
        for i in range(k):
            hs = self.head_sets[i % self.n_sets]
            if self.det is not None:
                pending.append(self.det.submit(hs))
                if len(pending) >= self.depth:
                    self.det.gather(pending.pop(0), as_list=False)
            else:
                p = self.pipes[i % self.n_sets]
                pending.append((p, p.submit(hs)))
                if len(pending) >= self.depth:
                    q, t = pending.pop(0)
                    last = q.counts(t)[0]
        if after_last_submit is not None:
            after_last_submit()
        for item in pending:
            if self.det is not None:
                self.det.gather(item, as_list=False)
            else:
                last = item[0].counts(item[1])[0]
        if self.det is not None:
            last = self.det.pipe.lanes[(self.det.pipe._next - 1) % self.depth].buf.meta_host[:self.B]
        return last

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize(self.dev)

    def timed(self, steps, warmup, sampler=None):
        """(elapsed ms max over ranks, per-rank ms per step, candidates per launch on this rank).
        Warm-up: at least `warmup` steps AND at least WARM_SECONDS of work -- a 20-step timed region lasts under 2 ms,
        and the first tens of milliseconds after a start run 8-15 % slower than the steady state on this pool's B200s
        (profiles/r02_f_warmup_length.txt).  The number of warm-up steps actually run is kept in `self.warm_steps`
        (the same on every rank: the rank-0 count is broadcast)."""
        n0 = max(warmup, 3, self.depth)
        t0 = time.perf_counter()
        cand = int(self.run_steps(n0).sum())
        per_step = max((time.perf_counter() - t0) / n0, 1e-6)
        extra = min(5000, max(0, int((WARM_SECONDS - (time.perf_counter() - t0)) / per_step)))
        if self.dist is not None:
            t = torch.tensor([extra], device=self.dev)
            self.dist.broadcast(t, 0)
            extra = int(t.item())
        if extra:
            self.run_steps(extra)
        self.warm_steps = n0 + extra
        stream = torch.cuda.current_stream(self.dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        if self.dist is not None:
            # the barrier releases the processes tens to hundreds of microseconds apart (host wake-up), which is a large
            # part of a 1.7 ms timed region and lands in whichever rank started first (it waits for the others' stamps /
            # acks).  One more collective, this time only ENQUEUED: every rank's stream -- and so its start event --
            # resumes when the all-reduce completes, i.e. within microseconds of the other ranks'.
            self.dist.all_reduce(torch.zeros(1, device=self.dev))
        if sampler is not None:
            sampler.start()
        ev0.record(stream)

        def end_of_work():
            for p in set(self.pipes):
                p.drain()                        # the timing stream waits for the pipeline streams (all K steps enqueued)
            ev1.record(stream)

        self.run_steps(steps, end_of_work)       # every step's counts are read back (host sync per step)
        self.barrier()
        elapsed_ms = ev0.elapsed_time(ev1)
        by_rank = [elapsed_ms / steps]
        if self.dist is not None:
            t = torch.tensor([elapsed_ms], device=self.dev)
            every = [torch.zeros_like(t) for _ in range(self.world)]
            self.dist.all_gather(every, t)
            by_rank = [float(x.item()) / steps for x in every]
            elapsed_ms = max(float(x.item()) for x in every)          # the job is as slow as its slowest rank
        return elapsed_ms, by_rank, cand

    def last_result(self, steps):
        """What the caller got from the last of `steps` timed steps: (per-image (n, 7) detections, anchor rows), None
        for an image without any.  N > 1: the gathered global batch on rank 0, None on the other ranks."""
        if self.det is not None:
            return self.det.gather(self.det.pipe._next - 1, return_rows=True)
        p = self.pipes[(steps - 1) % self.n_sets]          # run_steps' choice for step steps - 1
        return p.collect(p._next - 1, return_rows=True)

    def kernel_roofline(self, cand_total, peak, peak_src, reps):
        """The dominant kernel (decode_compact) timed alone with CUDA events on its stream."""
        from pytorch_yolo_b200 import ops
        buf, nc, dev = self.lane0.buf, self.w["nc"], self.dev
        stream = torch.cuda.current_stream(dev)
        for s in range(min(3, self.n_sets)):
            ops.decode_compact(self.head_sets[s], self.specs, nc, self.conf, buf, variant=self.variant)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        k0.record(stream)
        for i in range(reps):
            ops.decode_compact(self.head_sets[i % self.n_sets], self.specs, nc, self.conf, buf, variant=self.variant)
        k1.record(stream)
        torch.cuda.synchronize(dev)
        kern_ms = k0.elapsed_time(k1) / reps
        algo_bytes = self.B * self.bytes_per_img + 32 * cand_total
        achieved = algo_bytes / (kern_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.isfile(tpath):
            try:
                traffic = json.load(open(tpath)).get(f"{self.workload}:{self.B}:{self.conf}")
            except Exception:  # noqa: BLE001
                traffic = None
        return {"bound": "hbm", "kernel": "decode_compact_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "variant": self.variant, "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": kern_ms, "candidates_per_launch": cand_total}

    def gather_check(self):
        """N > 1, outside any timed region: one more step through the sharded pipeline; every rank also computes its
        slice locally (plain Detector, local buffers) and sends per-image (kept count, checksum of the row bits and
        anchor rows) to rank 0, which compares them with what the peer stores left in its gather buffer."""
        from pytorch_yolo_b200.detect import Detector
        dist, dev = self.dist, self.dev
        local = Detector(self.specs, self.w["nc"], self.B, dev, self.conf, self.nms, use_graph=False)
        local.launch(self.head_sets[0])
        _, kept = local.counts()
        kept_d = kept.to(dev).long()

        def checksum(out, rows, counts):
            n_img, cap = out.shape[0], out.shape[1]
            mask = (torch.arange(cap, device=dev).view(1, cap) < counts.view(n_img, 1))
            bits = out.contiguous().view(torch.int32).long().sum(2) * 31 + rows.long()
            return (bits * mask).sum(1)

        mine = torch.stack((kept_d, checksum(local.out, local.out_row, kept_d)), 1)           # (B, 2) int64
        every = [torch.zeros_like(mine) for _ in range(self.world)]
        dist.all_gather(every, mine)
        res = self.det.gather(self.det.submit(self.head_sets[0]), as_list=False)
        verdict = None
        if self.rank == 0:
            out, row, cnt = res
            cnt_d = cnt.to(dev).long()
            got = torch.stack((cnt_d, checksum(out, row, cnt_d)), 1)
            want = torch.cat(every, 0)
            bad = (got != want).any(1).nonzero().view(-1).tolist()
            verdict = "ok" if not bad else f"MISMATCH on {len(bad)} of {len(want)} images (first: {bad[:5]})"
        del local
        return verdict

    def close(self):
        if self.det is not None:
            self.det.close()
        self.pipes, self.head_sets, self.det, self.lane0 = [], [], None, None
        gc.collect()
        torch.cuda.empty_cache()


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------- head fusion (SURVEY 8f-3)
def head_fusion_probe(args, w, specs, B, dev, peak_gbs):
    """Extra measurement, not part of `value`: the head 1x1 convolutions fused with decode + compaction on the tensor
    cores (csrc/head.cu) against the unfused sequence -- torch's cuDNN convolution (TF32) writing the head tensors, then
    decode_compact reading them -- on synthetic feature maps of the workload's shapes.  CUDA events, 20 repetitions."""
    from pytorch_yolo_b200 import ops, synth
    feats, convs = synth.synth_head_convs(args.workload, B, device=dev)
    nc = w["nc"]
    rows = sum(s.rows for s in specs)
    offs, o = [], 0
    for s in specs:
        offs.append(o)
        o += s.rows
    hws = [ops.fold_head(c, dev) for c in convs]
    buf = ops.Buffers(dev, B, rows, nc)
    # planes that are not a multiple of 4 floats (19x19, 13x13): read in place by the one-pass kernel's loader warps;
    # the three-pass mode (and the "padded" comparison below) goes through the padded copy
    padded = [None if ops.head_supported(h.c_in, s, nc) else torch.zeros(B, h.c_in, ops.padded_pitch(s), device=dev)
              for h, s in zip(hws, specs)]
    padded3 = [None if ops.head_supported(h.c_in, s, nc, fp32x3=True) else torch.zeros(B, h.c_in, ops.padded_pitch(s), device=dev)
               for h, s in zip(hws, specs)]

    def fused():
        xs = [x if p is None else ops.pad_feature(x, out=p) for x, p in zip(feats, padded)]
        ops.head_decode_compact(xs, hws, specs, offs, rows, nc, args.conf, buf)

    def timeit(fn, reps=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps * 1e3

    t_fused = timeit(fused)
    cand = int(buf.meta[:B].sum())
    ovf = int(buf.meta[B])
    # fp32-accurate mode (three TF32 passes over split operands) against cuDNN's convolution with TF32 switched off
    hws3 = [ops.fold_head(c, dev, fp32x3=True) for c in convs]

    def fused3():
        xs = [x if p is None else ops.pad_feature(x, out=p) for x, p in zip(feats, padded3)]
        ops.head_decode_compact(xs, hws3, specs, offs, rows, nc, args.conf, buf)

    def fused_padded():                       # the round-1 way: every unaligned scale through the padded copy
        xs = [x if p is None else ops.pad_feature(x, out=p) for x, p in zip(feats, padded3)]
        ops.head_decode_compact(xs, hws, specs, offs, rows, nc, args.conf, buf)

    t_padded = timeit(fused_padded) if any(p is not None for p in padded3) else None
    t_fused3 = timeit(fused3)
    cand3 = int(buf.meta[:B].sum())
    old_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            t_conv32 = timeit(lambda: [c(x) for c, x in zip(convs, feats)], reps=10)
    finally:
        torch.backends.cudnn.allow_tf32 = old_tf32
    with torch.no_grad():
        t_conv = timeit(lambda: [c(x) for c, x in zip(convs, feats)])
        heads = [c(x) for c, x in zip(convs, feats)]
        t_dec = timeit(lambda: ops.decode_compact(heads, specs, nc, args.conf, buf))
    x_bytes = sum(x.numel() * 4 for x in feats)
    flops = sum(2.0 * B * s.ny * s.nx * h.n_out * h.c_in for s, h in zip(specs, hws))
    return {"what": "1x1 head conv (TF32 tcgen05) + decode + compaction in one kernel, all scales in one launch; "
                    "planes that are not a multiple of 4 floats (19x19, 13x13) are read in place by two loader warps (cp.async)",
            "fused_us": t_fused, "fused_with_padded_copy_us": t_padded, "unfused_us": t_conv + t_dec, "unfused_conv_cudnn_us": t_conv, "unfused_decode_compact_us": t_dec,
            "speedup": (t_conv + t_dec) / t_fused, "feature_bytes": x_bytes, "feature_gbs": x_bytes / t_fused / 1e3,
            "frac_of_hbm_peak": x_bytes / t_fused / 1e3 / peak_gbs, "tf32_tflops": flops / t_fused / 1e6,
            "candidates": cand, "overflow": ovf, "padded_scales": [p is not None for p in padded],
            "loader_warp_scales": [p is None and (s.ny * s.nx) % 4 != 0 for p, s in zip(padded, specs)],
            "fp32x3": {"what": "same kernel, fp32-accurate products (3 TF32 passes, operand split) vs cuDNN convolution with "
                               "allow_tf32 = False + decode_compact", "fused_us": t_fused3, "unfused_conv_cudnn_fp32_us": t_conv32,
                       "speedup": (t_conv32 + t_dec) / t_fused3, "tf32_tflops_issued": 3 * flops / t_fused3 / 1e6,
                       "candidates": cand3},
            "allow_tf32_reference": bool(torch.backends.cudnn.allow_tf32)}


def head_fusion_step_probe(args, w, specs, B, dev, rank, world, steps=20, depth=2):
    """The fused-head path as a pipelined, sharded step (SURVEY 8f-3 + 8e): every rank turns ITS feature maps into kept
    detections -- padded copy of the unaligned scale, tensor-core head kernel, NMS -- with `depth` batches in flight; at
    N > 1 the kept rows go to rank 0 by NVLink peer stores exactly like the headline path (ShardedDetector over
    HeadDetector lanes) and rank 0 checks its own slice of one gathered step against a local single-GPU run.
    Feature maps resident in HBM; CUDA events; max over ranks."""
    import torch.distributed as dist
    from pytorch_yolo_b200 import synth
    from pytorch_yolo_b200.detect import PipelinedDetector
    from pytorch_yolo_b200.head import HeadDetector
    from pytorch_yolo_b200.sharded import ShardedDetector
    feats, convs = synth.synth_head_convs(args.workload, B, device=dev, seed=4242)      # the same weights on every rank ...
    gen = torch.Generator(device=dev)
    gen.manual_seed(99 + rank)
    for f in feats:
        f.normal_(generator=gen)                                                          # ... different images
    nc = w["nc"]
    if world > 1:
        det = ShardedDetector(specs, nc, B * world, dev, args.conf, args.nms, depth=depth, heads=convs, use_graph=True)
        det.bind(feats)
        submit, wait, lanes = det.submit, (lambda t: det.gather(t, as_list=False)), det.pipe.lanes
    else:
        det = PipelinedDetector(specs, nc, B, dev, args.conf, args.nms, depth=depth, use_graph=True,
                                factory=lambda lane: HeadDetector(convs, specs, nc, B, dev, args.conf, args.nms,
                                                                  use_graph=True, nms_priority=True))
        det.bind(feats)
        submit, wait, lanes = det.submit, det.counts, det.lanes

    def run(k):
        pending = []
        for _ in range(k):
            pending.append(submit(feats))
            if len(pending) >= depth:
                wait(pending.pop(0))
        for t in pending:
            wait(t)

    run(max(3, depth))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(steps)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    out = {"what": "feature maps -> kept detections: pad copy + fused head kernel + NMS, pipelined; kept rows to rank 0 by "
                   "peer stores at N > 1", "n_gpus": world, "steps": steps, "batches_in_flight": depth,
           "ms_per_step": ms / steps, "images_per_s": B * world * steps / (ms * 1e-3),
           "kernels_per_step": lanes[0].kernels_per_step}
    if world > 1:
        ok = "ok"
        if rank == 0:
            got, got_rows = det.gather(det.submit(feats), return_rows=True)
        else:
            det.gather(det.submit(feats))
        if rank == 0:
            single = HeadDetector(convs, specs, nc, B, dev, args.conf, args.nms)
            want, want_rows = single.run(feats, return_rows=True, clone=True)
            for i in range(B):
                g, o = got[i], want[i]
                if (g is None) != (o is None) or (g is not None and not (torch.equal(g, o) and torch.equal(got_rows[i], want_rows[i]))):
                    ok = f"mismatch at image {i}"
                    break
        out["gather_check"] = ok
        det.close()
    return out


# ------------------------------------------------------------------------------------------- the reference-shaped API path
def drop_in_probe(case, peak, reps=10):
    """The unmodified-API path a pure drop-in user gets: ``YOLOLayer.forward`` per scale (one dense-decode launch each),
    the model's own ``torch.cat(io, 1)`` (yolov3_spp.py:163-164) and ``non_max_suppression`` (compact_from_dense + the
    NMS kernels + the host sync the list return needs) -- next to the one-launch ``decode_layers`` and the dense kernel
    timed alone (2 x T algorithmic bytes)."""
    from pytorch_yolo_b200 import YOLOLayer, decode_layers, non_max_suppression, ops
    w, dev, B = case.w, case.dev, case.B
    heads = case.head_sets[0]
    layers = [YOLOLayer(a, w["nc"], w["anchors"]).eval().to(dev) for a in w["anchors"]]

    def per_layer():
        io = [l(h, w["img_size"])[0] for l, h in zip(layers, heads)]
        pred = torch.cat(io, 1)
        return non_max_suppression(pred, case.conf, case.nms)

    def one_launch():
        pred, _ = decode_layers(layers, heads, w["img_size"])
        return non_max_suppression(pred, case.conf, case.nms)

    def timeit(fn, n):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n

    with torch.no_grad():
        t_layer = timeit(per_layer, reps)
        t_one = timeit(one_launch, reps)
        out = torch.empty(B, sum(s.rows for s in case.specs), w["nc"] + 5, device=dev)
        t_dense = timeit(lambda: ops.decode_dense(heads, case.specs, w["nc"], out=out), 20)
    dense_bytes = 2 * B * case.bytes_per_img
    return {"what": "reference-shaped API on the same heads: YOLOLayer.forward x scales + torch.cat + non_max_suppression "
                    "(list return, host sync); 'decode_layers' = all scales in one dense launch, no cat",
            "per_layer_cat_nms_ms": t_layer, "per_layer_cat_nms_images_per_s": B / (t_layer * 1e-3),
            "decode_layers_nms_ms": t_one, "decode_layers_nms_images_per_s": B / (t_one * 1e-3),
            "decode_dense_kernel_ms": t_dense, "decode_dense_gbs": dense_bytes / (t_dense * 1e-3) / 1e9,
            "decode_dense_frac_of_hbm_peak": dense_bytes / (t_dense * 1e-3) / 1e9 / peak}


def tiny_b1_probe(dev, reps=200):
    """BASELINE config 1 on the GPU: decode + NMS of the reference's own random-init YOLOv3-tiny heads (416x416, batch 1,
    conf 0.1 -- the committed golden fixture, produced by the reference's encoder) through the fused path.  0.86 MB of
    input: L2-resident and launch-bound, no roofline fraction is quoted (SURVEY.md 8d)."""
    import numpy as np
    from pytorch_yolo_b200 import ops, synth
    from pytorch_yolo_b200.detect import Detector
    path = os.path.join(ROOT, "tests", "golden", "tiny416_randinit.npz")
    if not os.path.isfile(path):
        return None
    z = np.load(path)
    heads = [torch.from_numpy(z["head0"]).to(dev), torch.from_numpy(z["head1"]).to(dev)]
    w = synth.WORKLOADS["tiny-416"]
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    det = Detector(specs, w["nc"], 1, dev, float(z["conf"]), float(z["nms"]), use_graph=True)
    det.bind(heads)
    for _ in range(5):
        det.run(heads)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(reps):
        det.launch(heads)
        _, kept = det.counts()
    dt = (time.perf_counter() - t0) / reps
    return {"images_per_s": 1.0 / dt, "latency_us": dt * 1e6, "kept": int(kept[0]), "kept_reference": int(z["counts"][0]),
            "what": "fused decode+NMS of the reference's random-init tiny-416 heads, batch 1, one graph launch + count read-back "
                    "per image (wall clock: launch-bound)"}


# ------------------------------------------------------------------------------------------- GPU arm
def main():
    args = parse_args()
    if args.batch is None:
        args.batch = default_batch(args.workload)
    if args.only:
        args.no_cpu_baseline = args.no_e2e = args.no_head_fusion = args.no_configs = args.no_drop_in = True
    if args.impl == "reference":
        return run_reference(args)
    args.steps = args.steps or DEFAULT_STEPS

    import torch.distributed as dist
    from pytorch_yolo_b200 import hostmem, ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        dist.init_process_group("nccl", device_id=dev)
    peak, peak_src = hbm_peak()
    B = args.batch
    use_graph = not args.no_graph

    case = Case(args.workload, B, args.kind, args.conf, args.nms, dev, rank, world, depth=args.depth, variant=args.variant,
                use_graph=use_graph, priority=not args.no_priority, seg_warps=args.seg_warps)
    sampler = ClockSampler(physical_gpu_index(local_rank))
    elapsed_ms, by_rank, cand_total = case.timed(args.steps, args.warmup, sampler)
    clocks = sampler.finish()
    if args.dump_outputs:
        # before anything else runs on the lanes' buffers
        res = case.last_result(args.steps)
        if rank == 0:
            dump_outputs(args.dump_outputs, *res, case.lane0.buf.out_cap)
    value = B * world * args.steps / (elapsed_ms * 1e-3)
    roofline = case.kernel_roofline(cand_total, peak, peak_src, reps=max(20, min(args.steps, 200)))
    lane0 = case.lane0
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": case.warm_steps,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, B), "clocks": clocks,
        "gpu_launches": lane0.kernels_per_step * args.steps, "roofline": roofline,
        "cuda_graph": bool(lane0.use_graph), "batches_in_flight": case.depth, "ms_per_step_by_rank": by_rank,
        "nms_stream_priority": bool(lane0._side is not None),
        "step_floor_frac": (B * case.bytes_per_img / (peak * 1e9)) / (elapsed_ms * 1e-3 / args.steps),
    }
    if distributed:
        try:
            line["gather_check"] = case.gather_check()
        except Exception as e:  # noqa: BLE001
            line["gather_check"] = "error: " + repr(e)[:200]

    # ---- the next row of the scope table (8f-3), measured beside the headline: head convolution fused in
    if rank == 0 and world == 1 and not args.no_head_fusion and "head_cin" in case.w:
        try:
            line["head_fusion"] = head_fusion_probe(args, case.w, case.specs, B, dev, peak)
        except Exception as e:  # noqa: BLE001  (the headline must not depend on this extra)
            line["head_fusion"] = {"error": repr(e)[:300]}

    if not args.no_head_fusion and "head_cin" in case.w:       # every rank, every N: the sharded fused-head step
        try:
            step = head_fusion_step_probe(args, case.w, case.specs, B, dev, rank, world)
        except Exception as e:  # noqa: BLE001
            step = {"error": repr(e)[:300]}
        line.setdefault("head_fusion", {})["pipeline"] = step

    if rank == 0 and world == 1 and not args.no_drop_in:
        try:
            line["drop_in"] = drop_in_probe(case, peak)
        except Exception as e:  # noqa: BLE001
            line["drop_in"] = {"error": repr(e)[:300]}

    # ---- end to end through the public API with HOST buffers (pinned, on the GPU's NUMA node), H2D + D2H inside the
    # timed region; two batches in flight, so the H2D copy of batch i+1 overlaps the kernels and the D2H of batch i
    if not args.no_e2e:
        try:
            line["e2e"] = e2e_probe(case, args, hostmem, ops, local_rank)
        except Exception as e:  # noqa: BLE001
            line["e2e"] = {"error": repr(e)[:300]}

    case.close()
    del case, lane0

    # ---- the other BASELINE.json configs, bounded, in the same record (and under torchrun at N > 1)
    if not args.no_configs:
        line["configs"] = extra_configs(args, dev, rank, world, peak, peak_src)

    # ---- CPU baseline beside it (rank 0, N=1 only): the unmodified reference functions on a bounded sample
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sb = min(B, CPU_SAMPLE_BATCH.get(args.workload, 8))
        ips, times, kind, _ = cpu_run(args.cpu_kind, args.workload, sb, args.kind, args.conf, args.nms, runs=args.cpu_runs)
        line["cpu_baseline"] = {"value": ips, "unit": UNIT, "cores": cores, "kind": kind,
                                "sample": f"{args.workload} SYNTH-{args.kind} batch {sb}, {len(times)} runs (median), "
                                          f"{sum(times):.1f} s of CPU work, torch threads {torch.get_num_threads()}: "
                                          "YOLOLayer.forward x scales + torch.cat + non_max_suppression"}

    if rank == 0:
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def e2e_probe(case, args, hostmem, ops, local_rank):
    import torch.distributed as dist
    from pytorch_yolo_b200.detect import PipelinedDetector
    dev, B, world, rank = case.dev, case.B, case.world, case.rank
    distributed = world > 1
    phys = physical_gpu_index(local_rank)
    host_heads = [hostmem.pinned_like(h.cpu(), local_rank) for h in case.head_sets[0]]
    h2d = sum(h.numel() * 4 for h in host_heads)
    e2e_steps = max(3, min(args.steps, 30))
    stream = torch.cuda.current_stream(dev)
    numa = hostmem.gpu_numa_node(local_rank)
    if not distributed:
        pipe = PipelinedDetector(case.specs, case.w["nc"], B, dev, case.conf, case.nms, depth=2, use_graph=True, variant=case.variant)
        host_out = [hostmem.pinned_empty((B, case.lane0.buf.out_cap, ops.DET_COLS), torch.float32, local_rank) for _ in range(2)]

        def run(k):
            pend, kept, d2h = [], None, 0
            for i in range(k):
                pend.append(pipe.submit_host(host_heads))
                if len(pend) >= 2:
                    t = pend.pop(0)
                    kept, d2h = pipe.collect_host(t, host_out[t % 2])
            for t in pend:
                kept, d2h = pipe.collect_host(t, host_out[t % 2])
            return kept, d2h
        run(3)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        kept, d2h = run(e2e_steps)
        pipe.drain()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        e2e_ms = e0.elapsed_time(e1)
        kept_rows = int(kept.sum())
    else:
        det, depth = case.det, case.depth
        # per-lane device staging = the resident head set (static pointers: the captured graphs stay valid)
        stage = case.head_sets[0]
        host_all = hostmem.pinned_empty((B * world, case.lane0.buf.out_cap, ops.DET_COLS), torch.float32, local_rank) if rank == 0 else None
        state = {"d2h": 0, "kept": 0}

        def step():
            for d, h in zip(stage, host_heads):
                d.copy_(h, non_blocking=True)
            res = det.gather(det.submit(stage), as_list=False)
            if rank == 0:
                out, _, cnt = res
                n_max = max(1, int(cnt.max()))
                host_all[:, :n_max].copy_(out[:, :n_max], non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
                state["d2h"] = host_all[:, :n_max].numel() * 4 + cnt.numel() * 4
                state["kept"] = int(cnt.sum())
        for _ in range(3):
            step()
        case.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(e2e_steps):
            step()
        det.pipe.drain()
        e1.record(stream)
        case.barrier()
        e2e_ms = e0.elapsed_time(e1)
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        d2h, kept_rows = state["d2h"], state["kept"]
        h2d = h2d * world
    return {"value": B * world * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
            "kept_rows_per_step": kept_rows, "pinned_numa_node": numa, "physical_gpu": phys,
            "path": "pinned host heads (GPU-local NUMA node) -> H2D -> Detector (C ABI) -> D2H counts + kept rows"
                    + ("; 2 batches in flight" if not distributed else "; kept rows of all ranks read back by rank 0")}


def extra_configs(args, dev, rank, world, peak, peak_src):
    """BASELINE.json configs other than the headline, each timed for --config-steps steps through the same pipeline."""
    out = []
    main_key = (args.workload, args.batch, args.kind, args.conf, args.nms)
    for label, wl, b, kind, conf, nms in EXTRA_CONFIGS:
        if (wl, b, kind, conf, nms) == main_key:
            continue
        rec = {"config": label, "workload": wl, "batch_per_gpu": b, "kind": kind, "conf_thres": conf, "nms_thres": nms}
        try:
            c = Case(wl, b, kind, conf, nms, dev, rank, world, variant=args.variant, use_graph=not args.no_graph,
                     priority=not args.no_priority)
            steps = max(5, args.config_steps)
            ms, by_rank, cand = c.timed(steps, 5)
            roof = c.kernel_roofline(cand, peak, peak_src, reps=20)
            rec.update({"value": b * world * steps / (ms * 1e-3), "unit": UNIT, "steps": steps, "ms_per_step": ms / steps,
                        "roofline_frac": roof["frac"], "kernel_ms": roof["kernel_ms"], "candidates_per_launch": cand,
                        "step_floor_frac": (b * c.bytes_per_img / (peak * 1e9)) / (ms * 1e-3 / steps),
                        "batches_in_flight": c.depth, "n_gpus": world})
            if world > 1:
                rec["gather_check"] = c.gather_check()
            c.close()
            del c
        except Exception as e:  # noqa: BLE001
            rec["error"] = repr(e)[:300]
        out.append(rec)
    if rank == 0 and world == 1:
        rec = {"config": "cfg1 tiny-416 b1 random-init (reference's CPU-runnable case)", "workload": "tiny-416", "batch_per_gpu": 1}
        try:
            rec["gpu"] = tiny_b1_probe(dev)
            if not args.no_cpu_baseline:
                torch.set_num_threads(os.cpu_count() or 1)
                rec["cpu_reference"] = cpu_tiny_model_run()
        except Exception as e:  # noqa: BLE001
            rec["error"] = repr(e)[:300]
        out.append(rec)
    return out


if __name__ == "__main__":
    main()
