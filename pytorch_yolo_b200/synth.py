"""Synthetic head tensors of the shapes BASELINE.json names (SURVEY.md App. C).

The backbone is out of scope, so benchmarks and parity tests feed the detection
path with raw head tensors ``(B, na*(5+nc), ny, nx)`` fp32 NCHW, one per scale in
*model order* (SPP family: stride 32, 16, 8 -- reference ``models/yolov3_spp.py:151-156``;
tiny family: stride 16, 32 -- ``models/yolov3_tiny.py:89-100``).

* ``SYNTH-A``: i.i.d. logits calibrated so that a realistic fraction of anchors passes
  the confidence threshold (about 2 % at conf 0.3, about 48 % at conf 0.001).
* ``SYNTH-B``: SYNTH-A plus 50 planted objects per image, each seen by all anchors of the
  centre cell at every scale, so NMS has real clusters to merge.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence

import torch

# reference models/yolov3_spp.py:196-198 (the anchor list its __main__ uses)
SPP_ANCHORS = (((10.0, 13.0), (16.0, 30.0), (33.0, 23.0)),
               ((30.0, 61.0), (62.0, 45.0), (59.0, 119.0)),
               ((116.0, 90.0), (156.0, 198.0), (373.0, 326.0)))
# reference models/yolo_base.py:88-89 (YOLOBase default, used by the tiny family)
TINY_ANCHORS = (((10.0, 14.0), (23.0, 27.0), (37.0, 58.0)),
                ((81.0, 82.0), (135.0, 169.0), (344.0, 319.0)))

WORKLOADS: Dict[str, dict] = {
    # name: img_size, grid sizes in model order, anchors per scale, classes
    # head_cin: input channels of the 1x1 head convolutions (reference models/yolov3_tiny.py:38,42; yolov3_spp.py:86,99,111)
    "tiny-416": dict(img_size=416, grids=(26, 13), anchors=TINY_ANCHORS, nc=80, head_cin=(256, 512)),
    "spp-608": dict(img_size=608, grids=(19, 38, 76), anchors=SPP_ANCHORS, nc=80, head_cin=(1024, 512, 256)),
    "spp-1024": dict(img_size=1024, grids=(32, 64, 128), anchors=SPP_ANCHORS, nc=80, head_cin=(1024, 512, 256)),
    # every plane a multiple of four floats (tensor-map describable): the shape the TMA decode variants are compared on
    "spp-640": dict(img_size=640, grids=(20, 40, 80), anchors=SPP_ANCHORS, nc=80, head_cin=(1024, 512, 256)),
    # small shapes for tests (odd plane sizes exercise the unaligned path)
    "mini-96": dict(img_size=96, grids=(3, 6, 12), anchors=SPP_ANCHORS, nc=80),
    "mini-160": dict(img_size=160, grids=(5, 10, 20), anchors=SPP_ANCHORS, nc=80),
}


def anchors_per_image(workload: str) -> int:
    w = WORKLOADS[workload]
    return sum(len(a) * g * g for a, g in zip(w["anchors"], w["grids"]))


def head_bytes_per_image(workload: str) -> int:
    w = WORKLOADS[workload]
    return anchors_per_image(workload) * (5 + w["nc"]) * 4


def synth_heads(workload: str, batch: int, kind: str = "A", seed: int = 1234,
                device: str | torch.device = "cpu") -> List[torch.Tensor]:
    """SYNTH-A / SYNTH-B heads.  Deterministic for a given (workload, batch, kind, seed, device type)."""
    w = WORKLOADS[workload]
    nc, img = w["nc"], w["img_size"]
    dev = torch.device(device)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    heads = []
    for anchors, g in zip(w["anchors"], w["grids"]):
        na = len(anchors)
        h = torch.empty(batch, na, 5 + nc, g, g, dtype=torch.float32, device=dev)
        h[:, :, 0:2].normal_(0.0, 1.0, generator=gen)
        h[:, :, 2:4].normal_(0.0, 0.5, generator=gen)
        h[:, :, 4].normal_(-7.0, 3.0, generator=gen)
        h[:, :, 5:].normal_(-2.0, 2.0, generator=gen)
        heads.append(h)
    if kind.upper() == "B":
        _plant_objects(heads, w, gen, n_obj=50)
    elif kind.upper() != "A":
        raise ValueError(f"unknown synthetic kind {kind!r}")
    return [h.view(batch, -1, h.shape[-2], h.shape[-1]) for h in heads]


def _plant_objects(heads: Sequence[torch.Tensor], w: dict, gen: torch.Generator, n_obj: int) -> None:
    nc, img = w["nc"], float(w["img_size"])
    batch = heads[0].shape[0]
    dev = heads[0].device

    def rnd(*shape):
        return torch.rand(*shape, generator=gen, device=dev)

    def nrm(*shape):
        return torch.randn(*shape, generator=gen, device=dev)

    cx = (0.1 + 0.8 * rnd(batch, n_obj)) * img
    cy = (0.1 + 0.8 * rnd(batch, n_obj)) * img
    lo, hi = math.log(16.0), math.log(192.0)
    bw = torch.exp(lo + (hi - lo) * rnd(batch, n_obj))
    bh = torch.exp(lo + (hi - lo) * rnd(batch, n_obj))
    cls = torch.randint(0, nc, (batch, n_obj), generator=gen, device=dev)
    bi = torch.arange(batch, device=dev).view(batch, 1).expand(batch, n_obj)
    for h, anchors, g in zip(heads, w["anchors"], w["grids"]):
        s = img / g
        gx = torch.clamp((cx / s).floor().long(), 0, g - 1)
        gy = torch.clamp((cy / s).floor().long(), 0, g - 1)
        fx = torch.clamp(cx / s - gx, 0.05, 0.95)
        fy = torch.clamp(cy / s - gy, 0.05, 0.95)
        # objects of one image in one cell: the last one is planted, as by one write after the other (an indexed
        # assignment with repeated indices leaves the winner to the thread schedule: inputs would differ run to run)
        cell = gy * g + gx
        keep = ~(cell.unsqueeze(2) == cell.unsqueeze(1)).triu(1).any(2)
        kb, ky, kx = bi[keep], gy[keep], gx[keep]
        for a, (aw, ah) in enumerate(anchors):
            h[kb, a, 0, ky, kx] = (torch.logit(fx) + 0.3 * nrm(batch, n_obj))[keep]
            h[kb, a, 1, ky, kx] = (torch.logit(fy) + 0.3 * nrm(batch, n_obj))[keep]
            h[kb, a, 2, ky, kx] = (torch.log(bw / aw) + 0.1 * nrm(batch, n_obj))[keep]
            h[kb, a, 3, ky, kx] = (torch.log(bh / ah) + 0.1 * nrm(batch, n_obj))[keep]
            h[kb, a, 4, ky, kx] = (2.0 + 1.5 * nrm(batch, n_obj))[keep]
            logits = -5.0 + nrm(batch, n_obj, nc)
            logits.scatter_(2, cls.unsqueeze(2), 4.0 + nrm(batch, n_obj, 1))
            h[kb.unsqueeze(1), a, 5 + torch.arange(nc, device=dev).view(1, nc), ky.unsqueeze(1), kx.unsqueeze(1)] = logits[keep]


def synth_prediction(batch: int, n_rows: int, nc: int = 80, seed: int = 0, img: float = 608.0,
                     tie_levels: int = 0, device="cpu") -> torch.Tensor:
    """A decoded-looking ``(B, N, 5+nc)`` tensor for NMS-only tests (boxes cluster so IoUs are non-trivial).

    ``tie_levels > 0`` quantises objectness / class columns to that many levels to force exact score ties.
    """
    gen = torch.Generator(device="cpu")
    gen.manual_seed(seed)
    n_centres = max(4, n_rows // 12)
    centres = torch.rand(batch, n_centres, 2, generator=gen) * img
    which = torch.randint(0, n_centres, (batch, n_rows), generator=gen)
    xy = torch.gather(centres, 1, which.unsqueeze(2).expand(-1, -1, 2)) + 6.0 * torch.randn(batch, n_rows, 2, generator=gen)
    wh = torch.exp(3.2 + 0.6 * torch.randn(batch, n_centres, 2, generator=gen))
    wh = torch.gather(wh, 1, which.unsqueeze(2).expand(-1, -1, 2)) * torch.exp(0.15 * torch.randn(batch, n_rows, 2, generator=gen))
    obj = torch.sigmoid(-1.0 + 2.5 * torch.randn(batch, n_rows, 1, generator=gen))
    cls = torch.sigmoid(-3.0 + 2.0 * torch.randn(batch, n_rows, nc, generator=gen))
    fav = (which % nc).unsqueeze(2)
    cls.scatter_(2, fav, torch.sigmoid(1.0 + torch.randn(batch, n_rows, 1, generator=gen)))
    if tie_levels > 0:
        obj = torch.round(obj * tie_levels) / tie_levels
        cls = torch.round(cls * tie_levels) / tie_levels
    return torch.cat((xy, wh, obj, cls), 2).float().contiguous().to(device)


def synth_head_convs(workload: str, batch: int, seed: int = 4321, device: str | torch.device = "cuda"):
    """Synthetic inputs of the fused head path (SURVEY.md section 8f-3): per scale a unit-variance feature map
    (B, head_cin, g, g) and a plain 1x1 convolution whose weight rows are scaled so that the head tensor follows SYNTH-A
    (xy ~ N(0,1), wh ~ N(0,0.5^2), obj ~ N(-7,3^2), cls ~ N(-2,2^2)).  Returns (feature maps, conv modules)."""
    w = WORKLOADS[workload]
    nc = w["nc"]
    dev = torch.device(device)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    feats, convs = [], []
    for anchors, g, cin in zip(w["anchors"], w["grids"], w["head_cin"]):
        na = len(anchors)
        std = torch.tensor(([1.0, 1.0, 0.5, 0.5, 3.0] + [2.0] * nc) * na, device=dev)
        mean = torch.tensor(([0.0, 0.0, 0.0, 0.0, -7.0] + [-2.0] * nc) * na, device=dev)
        conv = torch.nn.Conv2d(cin, na * (5 + nc), 1, bias=True).to(dev).eval()
        with torch.no_grad():
            conv.weight.copy_((torch.randn(na * (5 + nc), cin, generator=gen, device=dev) * (std[:, None] / cin ** 0.5)).view_as(conv.weight))
            conv.bias.copy_(mean)
        feats.append(torch.randn(batch, cin, g, g, generator=gen, device=dev))
        convs.append(conv)
    return feats, convs
