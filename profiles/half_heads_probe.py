"""decode_compact on fp16 and bf16 heads against fp32 heads, on BASELINE configs 2 to 5.

For each config:
- the bytes the gated kernel ("auto") touches from the objectness gate at 32-byte granules, for 4-byte and 2-byte
  elements (profiles/gated_decode_probe.py's touched_bytes);
- the decode_compact kernel time on fp32, fp16 and bf16 heads, timed alternately with CUDA events;
- the Detector graph step (decode_compact + NMS kernels + count read-back, with the host waiting for every step as a
  serving loop does) on fp32 heads, on fp16 heads, and on fp16 heads upcast into static fp32 tensors first (``copy_``, the
  same pass as ``.float()``): what a caller of an fp16 model had to do before 16-bit heads were accepted.
Two input sets with different seeds alternate launch by launch (each with its own Detector and graph), so a launch never
finds the previous launch's bytes in L2.

    python profiles/half_heads_probe.py [--pairs 5] [--reps 30] [--only cfg2,cfg4]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from profiles.gated_decode_probe import CONFIGS, touched_bytes  # noqa: E402
from pytorch_yolo_b200 import ops, synth  # noqa: E402
from pytorch_yolo_b200.detect import Detector  # noqa: E402

NMS = 0.5


def stats(ts):
    ts = sorted(ts)
    return ts[len(ts) // 2], ts[0], ts[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--only", default="", help="comma-separated config labels' first words, e.g. cfg2,cfg4")
    args = ap.parse_args()
    dev = "cuda:0"
    print(torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                           text=True, timeout=30)
        print(q.stdout.strip())
    except Exception as e:  # noqa: BLE001
        print("nvidia-smi:", e)
    for label, wl, batch, conf in CONFIGS:
        if args.only and label.split()[0] not in args.only.split(","):
            continue
        w = synth.WORKLOADS[wl]
        nc = w["nc"]
        specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        sets = {torch.float32: [synth.synth_heads(wl, batch, "B", seed=1234 + s, device=dev) for s in range(2)]}
        for dt in (torch.float16, torch.bfloat16):
            sets[dt] = [[h.to(dt) for h in hs] for hs in sets[torch.float32]]
        dense32 = batch * synth.head_bytes_per_image(wl)
        t4 = touched_bytes(sets[torch.float32][0], specs, nc, conf, 32, esize=4)
        t2 = touched_bytes(sets[torch.float16][0], specs, nc, conf, 32, esize=2)
        buf = ops.Buffers(dev, batch, synth.anchors_per_image(wl), nc)

        def kernel_us(dt):
            hs = sets[dt]
            for i in range(3):
                ops.decode_compact(hs[i % 2], specs, nc, conf, buf)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.reps):
                ops.decode_compact(hs[i % 2], specs, nc, conf, buf)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.reps * 1e3

        # Detector graph steps: one detector per input set, bound to that set's static tensors
        static_up = [[torch.empty(h.shape, dtype=torch.float32, device=dev) for h in hs] for hs in sets[torch.float16]]
        steps = {
            "fp32": ([Detector(specs, nc, batch, dev, conf, NMS) for _ in range(2)], sets[torch.float32], None),
            "fp16": ([Detector(specs, nc, batch, dev, conf, NMS) for _ in range(2)], sets[torch.float16], None),
            "fp16 upcast first": ([Detector(specs, nc, batch, dev, conf, NMS) for _ in range(2)], static_up,
                                  sets[torch.float16]),
        }

        def step_us(key):
            dets, inputs, src = steps[key]

            def one(i):
                k = i % 2
                if src is not None:
                    for d, s in zip(inputs[k], src[k]):
                        d.copy_(s)
                dets[k].launch(inputs[k])
                dets[k].counts()

            for i in range(4):
                one(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.reps):
                one(i)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.reps * 1e3

        kres = {dt: [] for dt in sets}
        sres = {k: [] for k in steps}
        for _ in range(args.pairs):
            for dt in sets:
                kres[dt].append(kernel_us(dt))
            for k in steps:
                sres[k].append(step_us(k))
        def result(d):
            _, kept = d.counts()
            return kept.tolist(), [d.out[i, :n].cpu() for i, n in enumerate(kept.tolist())]

        same = True          # the same detections whichever way the step was fed (the contract, at the benchmark's scale)
        for k in range(2):
            (ca, ra), (cb, rb) = result(steps["fp16"][0][k]), result(steps["fp16 upcast first"][0][k])
            same &= ca == cb and all(torch.equal(a, b) for a, b in zip(ra, rb))
        print(f"\n{label}: dense bytes fp32 {dense32 / 1e6:.1f} MB, 16-bit {dense32 / 2e6:.1f} MB; gated touches "
              f"{t4 / 1e6:.1f} MB (fp32) / {t2 / 1e6:.1f} MB (fp16) at 32 B granules")
        print(f"  decode_compact kernel, {args.pairs} x {args.reps} launches (median / min / max us):")
        for dt, ts in kres.items():
            med, lo, hi = stats(ts)
            tb = (t4 if dt == torch.float32 else t2) / med / 1e6
            print(f"    {str(dt).replace('torch.', ''):9s} {med:7.1f}  {lo:7.1f}  {hi:7.1f}   (touched bytes / median: {tb:.2f} TB/s)")
        k32 = stats(kres[torch.float32])[0]
        print(f"    fp16 / fp32: {stats(kres[torch.float16])[0] / k32:.3f}   bf16 / fp32: {stats(kres[torch.bfloat16])[0] / k32:.3f}")
        print(f"  Detector graph step, {args.pairs} x {args.reps} steps (median / min / max us):")
        for k, ts in sres.items():
            med, lo, hi = stats(ts)
            print(f"    {k:18s} {med:7.1f}  {lo:7.1f}  {hi:7.1f}")
        f16, up = stats(sres["fp16"])[0], stats(sres["fp16 upcast first"])[0]
        print(f"    fp16 step / upcast-first step: {f16 / up:.3f}   fp16 and upcast-first results bit-equal: {same}",
              flush=True)
        del sets, buf, steps, static_up
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
