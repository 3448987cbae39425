"""Gated decode_compact ("auto") against the dense LDG kernel ("ldg_dense") on BASELINE configs 2 to 5.

For each config: the bytes the gated kernel touches, counted on the device from the objectness gate at 32-byte and 64-byte
granules, and both kernels timed alternately with CUDA events.  Two input sets with different seeds alternate launch by
launch, so a launch never finds the previous launch's bytes in L2 (the touched bytes of one set are about L2's size);
the gated kernel is also timed on one set, as bench.py's roofline does.

    python profiles/gated_decode_probe.py [--pairs 7] [--reps 30] [--only cfg2,cfg4]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pytorch_yolo_b200 import ops, synth  # noqa: E402

CONFIGS = [("cfg2 spp-608 b64 conf 0.3", "spp-608", 64, 0.3), ("cfg3 tiny-416 b1024 conf 0.3", "tiny-416", 1024, 0.3),
           ("cfg4 spp-608 b64 conf 0.001", "spp-608", 64, 0.001), ("cfg5 spp-1024 b256 conf 0.3", "spp-1024", 256, 0.3)]
POSITIONS_PER_UNIT = 4      # positions per unit when the plane is a multiple of 4 elements, else 1


def touched_bytes(heads, specs, nc, conf, gran, esize=4):
    """Bytes in `gran`-byte granules the gated kernel requests: the whole objectness plane, and in each other plane the
    granules holding a unit (4 or 1 positions) with a position that passes the gate.  Planes are counted one by one.
    ``esize``: bytes per head element (4 for fp32 heads, 2 for fp16 / bf16 heads)."""
    no = nc + 5
    total = 0
    for h, s in zip(heads, specs):
        plane = s.ny * s.nx
        vec = POSITIONS_PER_UNIT if plane % 4 == 0 else 1
        v = h.view(-1, no, plane)                                          # slabs x channels x positions
        so = torch.sigmoid(v[:, 4].float())
        gate = (so * 1.0001) > conf
        unit = gate.view(v.shape[0], plane // vec, vec).any(-1)
        loaded = unit.repeat_interleave(vec, dim=1)                         # slabs x positions
        slabs = v.shape[0]
        pos_b = torch.arange(plane, device=h.device) * esize
        total += slabs * ((plane * esize + gran - 1) // gran) * gran      # objectness plane (upper bound by one granule)
        # plane c of slab s starts at byte ((s*no + c)*plane*esize); its phase within a granule is one of gran/esize values
        n_gran = (gran + plane * esize + gran - 1) // gran
        per_phase = {}
        for phase in range(0, gran, esize):
            if (plane * esize) % gran == 0 and phase:
                break
            g = (phase + pos_b) // gran
            hit = torch.zeros(slabs, n_gran, dtype=torch.int32, device=h.device)
            hit.scatter_reduce_(1, g.expand(slabs, -1), loaded.int(), reduce="amax")
            per_phase[phase] = hit.sum(1)                                    # granules per slab
        sidx = torch.arange(slabs, device=h.device, dtype=torch.int64)
        for c in range(no):
            if c == 4:
                continue
            ph = ((sidx * no + c) * plane * esize) % gran
            cnt = torch.zeros(slabs, dtype=torch.int64, device=h.device)
            for phase, n in per_phase.items():
                cnt += torch.where(ph == phase, n.long(), 0)
            total += int(cnt.sum()) * gran
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=7)
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
        sets = [synth.synth_heads(wl, batch, "B", seed=1234 + s, device=dev) for s in range(2)]
        dense_bytes = batch * synth.head_bytes_per_image(wl)
        t32 = touched_bytes(sets[0], specs, nc, conf, 32)
        t64 = touched_bytes(sets[0], specs, nc, conf, 64)
        buf = ops.Buffers(dev, batch, synth.anchors_per_image(wl), nc)

        def timeit(variant, n_sets):
            for i in range(3):
                ops.decode_compact(sets[i % n_sets], specs, nc, conf, buf, variant=variant)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.reps):
                ops.decode_compact(sets[i % n_sets], specs, nc, conf, buf, variant=variant)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / args.reps * 1e3              # us per launch

        res = {"ldg_dense": [], "auto": [], "auto_one_set": []}
        for _ in range(args.pairs):
            res["ldg_dense"].append(timeit("ldg_dense", 2))
            res["auto"].append(timeit("auto", 2))
            res["auto_one_set"].append(timeit("auto", 1))
        print(f"\n{label}: dense bytes {dense_bytes / 1e6:.1f} MB, gated touches {t32 / 1e6:.1f} MB at 32 B "
              f"({t32 / dense_bytes:.3f}), {t64 / 1e6:.1f} MB at 64 B ({t64 / dense_bytes:.3f})")
        for k, ts in res.items():
            ts = sorted(ts)
            med = ts[len(ts) // 2]
            nbytes = dense_bytes if k == "ldg_dense" else t32
            line = (f"  {k:13s} median {med:7.1f} us  min {ts[0]:7.1f}  max {ts[-1]:7.1f}  "
                    f"({'dense' if k == 'ldg_dense' else 'touched@32B'} bytes / median: {nbytes / med / 1e6:.2f} TB/s")
            if k != "ldg_dense":
                line += f", touched@64B: {t64 / med / 1e6:.2f} TB/s"
            print(line + ")", flush=True)
        print(f"  speed-up of auto (median) over ldg_dense: {sorted(res['ldg_dense'])[args.pairs // 2] / sorted(res['auto'])[args.pairs // 2]:.2f}x")
        del sets, buf
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
