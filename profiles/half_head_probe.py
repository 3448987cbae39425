"""The fused head on fp16 and bf16 feature maps against the fp32 fused head and the unfused 16-bit route, at the two head
shapes the benchmark times (spp-608 batch 64, tiny-416 batch 1024; synth.synth_head_convs inputs, conf 0.3).

Per shape and element type:
- the fused head kernel alone (yolo_b200_head_decode_compact, candidates only; 16-bit odd planes pre-padded);
- the same with the 16-bit plane-padding copies in front (what HeadDetector enqueues);
- the unfused 16-bit route: the module's own convolution under torch.autocast of that type (cuDNN) + decode_compact;
- the graph-replayed HeadDetector step (candidates + NMS + count read-back, the host waiting for every step as a serving
  loop does) for fp32 fused, 16-bit fused and 16-bit unfused.
Two input sets with different seeds alternate launch by launch, so no launch finds X in L2 (one set of X is 331 MB and up).
Kernel times come with the X bytes they read per second and the tensor-core rate they issue (2 * positions * c_in * NPAD,
NPAD = 256 accumulator columns for 80 classes), each set against the data-sheet bound it would be limited by.

    python profiles/half_head_probe.py [--pairs 5] [--reps 20]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pytorch_yolo_b200 import ops, synth  # noqa: E402
from pytorch_yolo_b200.head import HeadDetector  # noqa: E402

SHAPES = [("spp-608", 64), ("tiny-416", 1024)]
CONF, NMS = 0.3, 0.5
HBM = 7.7e12                                   # B/s, HGX B200 data sheet, one GPU
PEAK = {torch.float32: 1.125e15, torch.float16: 2.25e15, torch.bfloat16: 2.25e15}   # dense TF32 / FP16 / BF16 FLOP/s
NAME = {torch.float32: "fp32", torch.float16: "fp16", torch.bfloat16: "bf16"}


def stats(ts):
    ts = sorted(ts)
    return ts[len(ts) // 2], ts[0], ts[-1]


def timed(fn, reps):
    for i in range(4):
        fn(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dev = "cuda:0"
    print(torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                           text=True, timeout=30)
        print(q.stdout.strip())
    except Exception as e:  # noqa: BLE001
        print("nvidia-smi:", e)
    for wl, batch in SHAPES:
        w = synth.WORKLOADS[wl]
        nc = w["nc"]
        specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        offs, o = [], 0
        for s in specs:
            offs.append(o)
            o += s.rows
        rows = o
        feats0, convs = synth.synth_head_convs(wl, batch, seed=4321, device=dev)
        feats1, _ = synth.synth_head_convs(wl, batch, seed=4322, device=dev)
        sets32 = [feats0, feats1]
        buf = ops.Buffers(dev, batch, rows, nc)
        positions = sum(batch * s.ny * s.nx for s in specs)
        macs = sum(batch * s.ny * s.nx * c for s, c in zip(specs, w["head_cin"]))
        print(f"\n{wl} batch {batch}, conf {CONF}: {positions} positions, c_in {tuple(w['head_cin'])}")
        kres, sres, info = {}, {}, {}
        runs = {}
        for dt in (torch.float32, torch.float16, torch.bfloat16):
            sets = sets32 if dt == torch.float32 else [[x.to(dt) for x in fs] for fs in sets32]
            hws = [ops.fold_head(c, dev, dtype=dt) for c in convs]
            # what HeadDetector feeds the kernel: fp32 reads every plane in place, 16-bit pads odd planes first
            pad = [dt != torch.float32 and (s.ny * s.nx) % 2 == 1 for s in specs]
            padded = [[ops.pad_feature(x) if p else x for x, p in zip(fs, pad)] for fs in sets]
            pbufs = [torch.empty_like(x) if p else None for x, p in zip(padded[0], pad)]
            xbytes = sum(x.numel() * x.element_size() for x in sets[0])
            info[dt] = xbytes

            def fused(i, sets=sets, padded=padded, hws=hws):
                ops.head_decode_compact(padded[i % 2], hws, specs, offs, rows, nc, CONF, buf)

            def fused_pad(i, sets=sets, hws=hws, pbufs=pbufs):
                xs = [x if p is None else ops.pad_feature(x, out=p) for x, p in zip(sets[i % 2], pbufs)]
                ops.head_decode_compact(xs, hws, specs, offs, rows, nc, CONF, buf)

            runs[f"{NAME[dt]} fused kernel"] = (fused, dt)
            if any(pad):
                runs[f"{NAME[dt]} fused + pad copies"] = (fused_pad, dt)
            if dt != torch.float32:
                def unfused(i, sets=sets, dt=dt):
                    with torch.no_grad(), torch.autocast("cuda", dtype=dt):
                        heads = [c(x) for c, x in zip(convs, sets[i % 2])]
                    ops.decode_compact(heads, specs, nc, CONF, buf)
                runs[f"{NAME[dt]} unfused (cuDNN + decode)"] = (unfused, dt)

            # graph-replayed steps, one detector per input set
            def detector(unfused_route):
                d = HeadDetector(convs, specs, nc, batch, dev, CONF, NMS, use_graph=True, feature_dtype=dt)
                if unfused_route:
                    d.fused, d.padded = [False] * len(specs), [None] * len(specs)
                return d

            for label, unf in ((f"{NAME[dt]} fused", False),) + (((f"{NAME[dt]} unfused", True),) if dt != torch.float32 else ()):
                dets = [detector(unf) for _ in range(2)]
                statics = [[x.clone() for x in fs] for fs in sets]

                def step(i, dets=dets, statics=statics):
                    dets[i % 2].launch(statics[i % 2])
                    dets[i % 2].counts()
                sres[label] = (step, dets)
        for k in runs:
            kres[k] = []
        for k in sres:
            sres[k] = (sres[k][0], sres[k][1], [])
        for _ in range(args.pairs):
            for k, (fn, _) in runs.items():
                kres[k].append(timed(fn, args.reps))
            for k, (fn, _, ts) in sres.items():
                ts.append(timed(fn, args.reps))
        print(f"  kernels, {args.pairs} x {args.reps} launches alternating two input sets (median / min / max us):")
        for k, (fn, dt) in runs.items():
            med, lo, hi = stats(kres[k])
            line = f"    {k:28s} {med:7.1f}  {lo:7.1f}  {hi:7.1f}"
            if "fused kernel" in k:
                flops = 2.0 * 256 * macs
                t_mem, t_mma = info[dt] / HBM, flops / PEAK[dt]
                line += (f"   X {info[dt] / 1e6:.0f} MB -> {info[dt] / med / 1e6:.2f} TB/s;  {flops / med / 1e6:.0f} TF/s issued;"
                         f"  data-sheet floor {max(t_mem, t_mma) * 1e6:.0f} us ({'HBM' if t_mem > t_mma else 'tensor'}-bound)")
            print(line)
        print(f"  HeadDetector graph step, {args.pairs} x {args.reps} steps (median / min / max us):")
        for k, (fn, dets, ts) in sres.items():
            med, lo, hi = stats(ts)
            print(f"    {k:28s} {med:7.1f}  {lo:7.1f}  {hi:7.1f}   kernels per step {dets[0].kernels_per_step}")
        f32 = stats(sres["fp32 fused"][2])[0]
        for dt in (torch.float16, torch.bfloat16):
            n = NAME[dt]
            print(f"    {n} fused / fp32 fused: {stats(sres[f'{n} fused'][2])[0] / f32:.3f}   "
                  f"{n} fused / {n} unfused: {stats(sres[f'{n} fused'][2])[0] / stats(sres[f'{n} unfused'][2])[0]:.3f}",
                  flush=True)
        del runs, sres, sets32, feats0, feats1, buf
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
