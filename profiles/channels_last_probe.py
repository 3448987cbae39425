"""channels_last heads and feature maps: the NHWC kernels against today's handling of such tensors (a copy to NCHW, then the
NCHW kernel) and against the NCHW kernels on NCHW tensors, and the NCHW kernels of this build against a parent build.

Decode (synth SYNTH-B heads, the BASELINE configs 2-5), per element type fp32 / fp16:
- the gated NCHW kernel on NCHW heads;
- channels_last heads the way the parent handles them: .contiguous() + the gated kernel (variant "ldg" takes that route);
- the NHWC kernel on the channels_last heads;
- the Detector graph step (candidates + NMS + count read-back, the host waiting for every step) for each of the three.
Fused head (synth.synth_head_convs, conf 0.3, spp-608 b64 and tiny-416 b1024), per fp32 / fp16 / bf16:
- the NCHW kernel with the plane-padding copies HeadDetector enqueues (16-bit odd planes);
- channels_last maps copied to NCHW first, then the same;
- the NHWC kernel;
- the HeadDetector graph step for each.
NCHW before / after (--parent-lib, a build of the parent commit): the gated decode kernel and the fused head kernel on NCHW
inputs, the two libraries alternating window by window in this process.
Two input sets with different seeds alternate launch by launch, so no launch finds its bytes in L2 (the smallest set,
tiny-416 b1024 fp16 heads, is 180 MB).  Every figure is the median of --pairs windows of --reps launches (min / max beside).

    python profiles/channels_last_probe.py [--pairs 5] [--reps 20] [--parent-lib build/variants/parent.so]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pytorch_yolo_b200 import _lib, ops, synth  # noqa: E402
from pytorch_yolo_b200.detect import Detector  # noqa: E402
from pytorch_yolo_b200.head import HeadDetector  # noqa: E402

DEV = "cuda:0"
CL = torch.channels_last
DECODE = [("cfg2 spp-608 b64", "spp-608", 64, 0.3), ("cfg3 tiny-416 b1024", "tiny-416", 1024, 0.3),
          ("cfg4 spp-608 b64 conf 0.001", "spp-608", 64, 0.001), ("cfg5 spp-1024 b256", "spp-1024", 256, 0.3)]
HEAD = [("spp-608", 64), ("tiny-416", 1024)]
NAME = {torch.float32: "fp32", torch.float16: "fp16", torch.bfloat16: "bf16"}
HBM = 7.7e12


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


def measure(runs, pairs, reps, title):
    res = {k: [] for k in runs}
    for _ in range(pairs):
        for k, fn in runs.items():
            res[k].append(timed(fn, reps))
    print(f"  {title}, {pairs} x {reps} launches alternating two input sets (median / min / max us):")
    for k in runs:
        med, lo, hi = stats(res[k])
        print(f"    {k:44s} {med:8.1f} {lo:8.1f} {hi:8.1f}", flush=True)
    return {k: stats(v)[0] for k, v in res.items()}


def heads_for(wl, batch, seed):
    """SYNTH-B heads on the device; batches above 64 repeat a 64-image block (the CPU generator is slow at GBs)."""
    block = min(batch, 64)
    hs = [h.to(DEV) for h in synth.synth_heads(wl, block, "B", seed=seed)]
    return [h.repeat(batch // block, 1, 1, 1) for h in hs]


def decode_section(args):
    print("\n== decode_compact: channels_last heads ==")
    for label, wl, batch, conf in DECODE:
        w = synth.WORKLOADS[wl]
        nc = w["nc"]
        specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        rows = sum(s.rows for s in specs)
        sets32 = [heads_for(wl, batch, seed) for seed in (17, 18)]
        for dt in (torch.float32, torch.float16):
            nchw = [[h.to(dt) for h in s] for s in sets32]
            cl = [[h.contiguous(memory_format=CL) for h in s] for s in nchw]
            nbytes = sum(h.numel() * h.element_size() for h in nchw[0])
            buf = ops.Buffers(DEV, batch, rows, nc)
            runs = {
                f"{NAME[dt]} NCHW gated kernel": lambda i: ops.decode_compact(nchw[i % 2], specs, nc, conf, buf),
                f"{NAME[dt]} channels_last: copy + gated kernel": lambda i: ops.decode_compact(cl[i % 2], specs, nc, conf, buf,
                                                                                             variant="ldg"),
                f"{NAME[dt]} channels_last: NHWC kernel": lambda i: ops.decode_compact(cl[i % 2], specs, nc, conf, buf),
            }
            dets = {}
            for key, inputs, variant in (("NCHW", nchw, "auto"), ("copy", cl, "ldg"), ("NHWC", cl, "auto")):
                ds = [Detector(specs, nc, batch, DEV, conf, 0.5, use_graph=True, variant=variant) for _ in range(2)]
                for d, s in zip(ds, inputs):
                    d.bind(s)
                dets[key] = (ds, inputs)
            for key, label2 in (("NCHW", "NCHW heads"), ("copy", "channels_last, copy + gated"), ("NHWC", "channels_last, NHWC")):
                ds, inputs = dets[key]

                def step(i, ds=ds, inputs=inputs):
                    ds[i % 2].launch(inputs[i % 2])
                    ds[i % 2].counts()
                runs[f"{NAME[dt]} Detector graph step, {label2}"] = step
            print(f"\n {label} {NAME[dt]}: heads {nbytes / 1e6:.0f} MB")
            med = measure(runs, args.pairs, args.reps, "calls")
            k = f"{NAME[dt]} channels_last: NHWC kernel"
            print(f"    NHWC kernel: {nbytes / med[k] / 1e6:.2f} TB/s of head bytes ({nbytes / med[k] / 1e6 / (HBM / 1e12):.2f} of"
                  f" the 7.7 TB/s data sheet); NHWC / copy route {med[k] / med[f'{NAME[dt]} channels_last: copy + gated kernel']:.3f}")
            del runs, dets, nchw, cl, buf
            torch.cuda.empty_cache()
        del sets32
        torch.cuda.empty_cache()


def head_section(args):
    print("\n== fused head: channels_last feature maps ==")
    for wl, batch in HEAD:
        w = synth.WORKLOADS[wl]
        nc = w["nc"]
        specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        offs, o = [], 0
        for s in specs:
            offs.append(o)
            o += s.rows
        rows = o
        f0, convs = synth.synth_head_convs(wl, batch, seed=4321, device=DEV)
        f1, _ = synth.synth_head_convs(wl, batch, seed=4322, device=DEV)
        for dt in (torch.float32, torch.float16, torch.bfloat16):
            nchw = [[x.to(dt) for x in f] for f in (f0, f1)]
            cl = [[x.contiguous(memory_format=CL) for x in s] for s in nchw]
            hws = [ops.fold_head(c, DEV, dtype=dt) for c in convs]
            pad = [not ops.head_supported(hw.c_in, s, nc, dtype=dt) for hw, s in zip(hws, specs)]
            pbufs = [ops.pad_feature(x) if p else None for x, p in zip(nchw[0], pad)]
            buf = ops.Buffers(DEV, batch, rows, nc)
            nbytes = sum(x.numel() * x.element_size() for x in nchw[0])

            def nchw_call(xs, pbufs=pbufs, hws=hws, buf=buf):
                xs = [x if p is None else ops.pad_feature(x, out=p) for x, p in zip(xs, pbufs)]
                ops.head_decode_compact(xs, hws, specs, offs, rows, nc, 0.3, buf)

            runs = {
                f"{NAME[dt]} NCHW kernel + pad copies": lambda i, f=nchw_call: f(nchw[i % 2]),
                f"{NAME[dt]} channels_last: copy + NCHW": lambda i, f=nchw_call: f([x.contiguous() for x in cl[i % 2]]),
                f"{NAME[dt]} channels_last: NHWC kernel": lambda i, hws=hws, buf=buf: ops.head_decode_compact(
                    cl[i % 2], hws, specs, offs, rows, nc, 0.3, buf),
            }
            ds = [HeadDetector(convs, specs, nc, batch, DEV, 0.3, 0.5, use_graph=True, feature_dtype=dt) for _ in range(2)]
            statics = [[x.clone() for x in s] for s in nchw]
            for d, s in zip(ds, statics):
                d.bind(s)
            dcl = [HeadDetector(convs, specs, nc, batch, DEV, 0.3, 0.5, use_graph=True, feature_dtype=dt) for _ in range(2)]
            for d, s in zip(dcl, cl):
                d.bind(s)

            def step_nchw(i, ds=ds, statics=statics):
                ds[i % 2].launch(statics[i % 2])
                ds[i % 2].counts()

            def step_copy(i, ds=ds, statics=statics, cl=cl):
                for s, x in zip(statics[i % 2], cl[i % 2]):
                    s.copy_(x)
                ds[i % 2].launch(statics[i % 2])
                ds[i % 2].counts()

            def step_nhwc(i, dcl=dcl, cl=cl):
                dcl[i % 2].launch(cl[i % 2])
                dcl[i % 2].counts()
            runs[f"{NAME[dt]} HeadDetector graph step, NCHW maps"] = step_nchw
            runs[f"{NAME[dt]} HeadDetector graph step, channels_last, copy"] = step_copy
            runs[f"{NAME[dt]} HeadDetector graph step, channels_last, NHWC"] = step_nhwc
            print(f"\n {wl} b{batch} {NAME[dt]}: feature maps {nbytes / 1e6:.0f} MB, padded scales {pad}")
            med = measure(runs, args.pairs, args.reps, "calls")
            k = f"{NAME[dt]} channels_last: NHWC kernel"
            print(f"    NHWC kernel: {nbytes / med[k] / 1e6:.2f} TB/s of X; NHWC / NCHW kernel "
                  f"{med[k] / med[f'{NAME[dt]} NCHW kernel + pad copies']:.3f}; NHWC / copy route "
                  f"{med[k] / med[f'{NAME[dt]} channels_last: copy + NCHW']:.3f}")
            del runs, ds, dcl, statics, nchw, cl, buf, pbufs
            torch.cuda.empty_cache()
        del f0, f1
        torch.cuda.empty_cache()


def parent_section(args):
    """The NCHW kernels of this build and of the parent build, alternating window by window."""
    print(f"\n== NCHW kernels: this build vs the parent build ({args.parent_lib}) ==")
    mine = _lib.load()
    parent = C.CDLL(os.path.abspath(args.parent_lib))
    for name, (res, argt) in _lib._SIGNATURES.items():
        fn = getattr(parent, name)
        fn.restype, fn.argtypes = res, argt

    def with_lib(lib, fn):
        def run(i):
            _lib._lib = lib
            try:
                fn(i)
            finally:
                _lib._lib = mine
        return run

    for label, wl, batch, conf in DECODE:
        w = synth.WORKLOADS[wl]
        nc = w["nc"]
        specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        sets = [heads_for(wl, batch, seed) for seed in (17, 18)]
        buf = ops.Buffers(DEV, batch, sum(s.rows for s in specs), nc)
        call = lambda i, sets=sets, buf=buf: ops.decode_compact(sets[i % 2], specs, nc, conf, buf)
        res = {k: [] for k in ("parent", "this")}
        for _ in range(args.pairs):
            res["parent"].append(timed(with_lib(parent, call), args.reps))
            res["this"].append(timed(with_lib(mine, call), args.reps))
        print(f"  decode_compact gated fp32, {label}: parent {'%.1f %.1f %.1f' % stats(res['parent'])}   "
              f"this {'%.1f %.1f %.1f' % stats(res['this'])}   (median min max us)", flush=True)
        del sets, buf
        torch.cuda.empty_cache()
    for wl, batch in HEAD:
        w = synth.WORKLOADS[wl]
        nc = w["nc"]
        specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
        offs, o = [], 0
        for s in specs:
            offs.append(o)
            o += s.rows
        f0, convs = synth.synth_head_convs(wl, batch, seed=4321, device=DEV)
        f1, _ = synth.synth_head_convs(wl, batch, seed=4322, device=DEV)
        for dt in (torch.float32, torch.float16):
            sets = [[ops.pad_feature(x) if not ops.head_supported(x.shape[1], s, nc, dtype=dt) else x
                     for x, s in zip([y.to(dt) for y in f], specs)] for f in (f0, f1)]
            hws = [ops.fold_head(c, DEV, dtype=dt) for c in convs]
            buf = ops.Buffers(DEV, batch, o, nc)
            call = lambda i, sets=sets, hws=hws, buf=buf: ops.head_decode_compact(sets[i % 2], hws, specs, offs, o, nc, 0.3, buf)
            res = {k: [] for k in ("parent", "this")}
            for _ in range(args.pairs):
                res["parent"].append(timed(with_lib(parent, call), args.reps))
                res["this"].append(timed(with_lib(mine, call), args.reps))
            print(f"  fused head {NAME[dt]}, {wl} b{batch}: parent {'%.1f %.1f %.1f' % stats(res['parent'])}   "
                  f"this {'%.1f %.1f %.1f' % stats(res['this'])}   (median min max us)", flush=True)
            del sets, buf
            torch.cuda.empty_cache()
        del f0, f1
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--parent-lib", default=None, help="libyolo_b200.so built from the parent commit")
    ap.add_argument("--only", choices=["decode", "head", "parent"], default=None)
    args = ap.parse_args()
    print(torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                           capture_output=True, text=True, timeout=30)
        print(q.stdout.strip())
    except Exception as e:  # noqa: BLE001
        print("nvidia-smi:", e)
    if args.only in (None, "decode"):
        decode_section(args)
    if args.only in (None, "head"):
        head_section(args)
    if args.parent_lib and args.only in (None, "parent"):
        parent_section(args)


if __name__ == "__main__":
    main()
