"""Worst relative error of the device sigmoid and of the w/h decode, per binade of |x|, against float64.

sigmoidf_rn (csrc/common.cuh) is evaluated on every fp32 with 2^-8 <= |x| < 128 by decode_dense (LDG kernel, aligned plane);
decode_wh = (expf(t) * anchor_vec) * stride on every fp32 with 2^-8 <= |t| < 64 and 64 <= t <= 88.72 (anchor 1 px,
stride 8).  For each binade: the largest relative error for negative and for positive arguments, and the largest ratio of
the sigmoid's error to the bound SIG_A + SIG_B |x| that tests/test_gpu_decode_numerics.py enforces.

    python profiles/sigmoid_error_probe.py
"""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pytorch_yolo_b200 import ops  # noqa: E402
from tests.test_gpu_decode_numerics import (CHUNK, SIG_A, SIG_B, TINY, U, bits_to_f32, dense_sigmoid, f32_bits,  # noqa: E402
                                            sigma64)

DEV = "cuda:0"


def binade_chunks(k, limit=None):
    lo, hi = f32_bits(2.0 ** k), f32_bits(2.0 ** (k + 1))
    if limit is not None:
        hi = min(hi, f32_bits(limit) + 1)
    for c0 in range(lo, hi, CHUNK):
        yield bits_to_f32(c0, min(c0 + CHUNK, hi))


def sigmoid_worst(x):
    s = dense_sigmoid(x, 64, 64, "ldg").double()
    ref = sigma64(x)
    bound = SIG_A + SIG_B * x.double().abs()
    keep = ref >= TINY * (1 + bound)
    rel = torch.where(keep, (s - ref).abs() / ref, 0.0)
    return float(rel.max()), float((rel / bound).max())


def wh_worst(t):
    spec = ops.scale_spec([(1.0, 1.0)], 64, 64, 512)
    plane = 64 * 64
    n = t.numel()
    b = -(-n // plane)
    h = torch.zeros(b, 6, plane, device=DEV)
    tt = torch.zeros(b * plane, device=DEV)
    tt[:n] = t
    h[:, 2] = tt.view(b, plane)
    out = ops.decode_dense([h.view(b, 6, 64, 64)], [spec], 1, variant="ldg")
    got = out[:, :, 2].reshape(-1)[:n].double()
    ref = torch.exp(t.double()) * float(spec.anchor_vec[0, 0]) * spec.stride
    return float(((got - ref).abs() / ref).max())


def main():
    print(torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                           text=True, timeout=30)
        print(q.stdout.strip())
    except Exception as e:  # noqa: BLE001
        print("nvidia-smi:", e)
    print(f"\nsigmoidf_rn, bound {SIG_A} + {SIG_B} |x| (results below 2^-126 excluded: flushed to zero)")
    print(f"{'|x| in':>16} {'max rel, x < 0':>15} {'max rel, x > 0':>15} {'bound at top':>13} {'max err/bound':>14}")
    for k in range(-8, 7):
        worst = {-1: 0.0, 1: 0.0}
        ratio = 0.0
        for x in binade_chunks(k):
            for sign in (-1, 1):
                r, q = sigmoid_worst(sign * x)
                worst[sign] = max(worst[sign], r)
                ratio = max(ratio, q)
        print(f"[2^{k:>2}, 2^{k + 1:>2}) {worst[-1]:15.3e} {worst[1]:15.3e} {SIG_A + SIG_B * 2.0 ** (k + 1):13.3e} {ratio:14.3f}",
              flush=True)
    print(f"\ndecode_wh, bound 2^-22 + 2^-23 = {2.0 ** -22 + 2 * U:.3e} (expf 2 ulp, two fp32 products)")
    print(f"{'|t| in':>16} {'max rel, t < 0':>15} {'max rel, t > 0':>15}")
    for k in range(-8, 7):
        neg = f"{max(wh_worst(-t) for t in binade_chunks(k)):15.3e}" if k < 6 else f"{'-':>15}"   # exp(-64) ~ 1.6e-28
        pos = max(wh_worst(t) for t in binade_chunks(k, 88.72 if k == 6 else None))
        top = "88.72" if k == 6 else f"2^{k + 1:>2}"
        print(f"[2^{k:>2}, {top:>5}) {neg} {pos:15.3e}", flush=True)


if __name__ == "__main__":
    main()
