"""Feature maps -> detections with the head convolution fused in (SURVEY.md section 8f-3).

Every detection branch of the reference models ends in a 1x1 convolution that produces the ``na*(5+nc)``-channel
head tensor -- ``ConvBlock(c, 255, size=1)`` = conv + BatchNorm + LeakyReLU(0.1) in ``YOLOv3SPP`` (reference
models/yolov3_spp.py:86,99,111), a plain ``nn.Conv2d(c, 255, 1)`` in ``YOLOv3Tiny`` / ``YOLOv3`` (models/yolov3_tiny.py:38,42,
models/yolov3.py:38,54) -- immediately followed by ``YOLOLayer`` and, in evaluation, ``non_max_suppression``.
:class:`HeadDetector` takes the *inputs* of those convolutions and runs, per scale,

* the tcgen05 kernel (``yolo_b200_head_decode_compact``: TF32 tensor-core GEMM with the decode + confidence filter +
  compaction as its epilogue) where the geometry allows it, so the head tensor never touches HBM;
* grids whose plane is not a multiple of 4 floats (19x19, 13x13: TMA needs a 16-byte row pitch) are read in place by two
  loader warps of the same kernel (4-byte asynchronous copies into the swizzled layout); the three-pass mode first copies
  them into a plane-padded buffer (``ops.pad_feature``);
* whatever is still not covered (c_in not a multiple of 32, anchor counts other than 3, more than 256 output channels) runs
  the module's own convolution followed by the LDG decode kernel, appended to the same candidate buffers;

then the segmented NMS.  ``split_head`` cuts a reference branch (an ``nn.Sequential`` ending in the head convolution) into
trunk and head.  The head values carry TF32 rounding (10-bit mantissa products, fp32 accumulation) -- the precision cuDNN
uses for the reference's own convolution on this GPU under torch's default ``allow_tf32`` -- so detections agree with the
unfused path up to scores within ~1e-3 of a threshold; fed the same head tensor the two paths are bit-identical
(tests/test_gpu_head.py).

fp16 / bf16 feature maps (``feature_dtype``, what a ``.half()`` model or autocast hands over) run the same kernel with a
``kind::f16`` main loop: exact products of the 16-bit operands (the weights are folded in fp64 and rounded to that type),
fp32 accumulation, and the same fp32 epilogue.  Such scales need c_in % 64 == 0; odd planes (19x19, 13x13) go through
the 16-bit padded copy; uncovered scales run the module's own convolution under ``torch.autocast`` of that type.

channels_last feature maps (a ``torch.channels_last`` model) are read in place by the same kernel with a K-major A operand,
at every plane size: no padded copy.  The unfused scales' module outputs are then channels_last too, and
``decode_compact`` reads them in place.
"""
from __future__ import annotations

import contextlib
from typing import List, Optional, Sequence, Tuple

import torch
from torch import nn

from . import ops
from .detect import Detector


def split_head(branch: nn.Sequential) -> Tuple[nn.Sequential, nn.Module]:
    """(trunk, head) of a detection branch whose last child is the head's 1x1 ConvBlock / Conv2d."""
    children = list(branch.children())
    if not children:
        raise ValueError("empty branch")
    return nn.Sequential(*children[:-1]), children[-1]


class HeadDetector(Detector):
    """Persistent fused pipeline ``feature maps -> kept detections`` for batches of one shape: a :class:`Detector` whose
    candidate stage is the tensor-core head kernel instead of ``decode_compact`` (same buffers, NMS, graph capture,
    pipelining and multi-GPU gather -- ``PipelinedDetector(..., factory=...)`` / ``ShardedDetector(..., heads=...)``).

    ``heads``: the head modules in model scale order (folded once, in eval mode, with :func:`ops.fold_head`);
    ``specs``: their :class:`ops.ScaleSpec`.  ``run(feats)`` returns the reference's ``non_max_suppression`` result.
    ``feature_dtype``: the dtype of the feature maps ``run`` takes -- float32, or float16 / bfloat16 for a ``.half()`` model
    or one run under autocast (weights folded to that type; one-pass precision only).
    """

    def __init__(self, heads: Sequence[nn.Module], specs: Sequence[ops.ScaleSpec], nc: int, batch: int, device,
                 conf_thres: float = 0.5, nms_thres: float = 0.5, cap: Optional[int] = None, pad_unaligned: bool = True,
                 use_graph: bool = False, precision: str = "tf32", unaligned: str = "auto",
                 feature_dtype: torch.dtype = torch.float32, **kw):
        if len(heads) != len(specs):
            raise ValueError("one head module per scale is required")
        if unaligned not in ("auto", "pad", "unfused"):
            raise ValueError("unaligned is 'auto' (19x19 / 13x13 planes read in place where the kernel can, else through the "
                             "padded copy), 'pad' (always the padded copy) or 'unfused' (the module's own convolution + "
                             "decode_compact for such scales)")
        if unaligned == "unfused":
            pad_unaligned = False
        if precision not in ("tf32", "fp32x3"):
            raise ValueError("precision is 'tf32' (one tensor-core pass, what cuDNN does under allow_tf32) or 'fp32x3' "
                             "(three passes over split operands: fp32-accurate head values)")
        if feature_dtype not in ops.FEATURE_DTYPE_FLAGS:
            raise TypeError(f"feature_dtype must be float32, float16 or bfloat16, got {feature_dtype}")
        if precision == "fp32x3" and feature_dtype != torch.float32:
            raise ValueError(f"precision='fp32x3' splits fp32 operands: it takes float32 feature maps, not {feature_dtype}")
        super().__init__(specs, nc, batch, device, conf_thres, nms_thres, cap=cap, use_graph=use_graph, **kw)
        self.modules_ = list(heads)
        self.precision = precision
        self.feature_dtype = feature_dtype
        self.weights = [ops.fold_head(m, self.device, fp32x3=precision == "fp32x3", dtype=feature_dtype) for m in self.modules_]
        self.row_offs: List[int] = []
        off = 0
        for s in self.specs:
            self.row_offs.append(off)
            off += s.rows
        # a plane that is not a multiple of 4 floats (19x19, 13x13; 16-bit: an odd plane) is copied into a padded
        # (B, C, pitch) buffer first: one read + write of the feature map instead of materialising and re-reading the head
        # tensor
        self.padded: List[Optional[torch.Tensor]] = []
        self.fused = []
        x3 = precision == "fp32x3"
        dt = feature_dtype
        for w, s in zip(self.weights, self.specs):
            direct = ops.head_supported(w.c_in, s, nc, fp32x3=x3, dtype=dt)
            if direct and unaligned != "auto" and (s.ny * s.nx) % (4 if dt == torch.float32 else 8):
                direct = False                         # "pad" / "unfused": do not read unaligned planes in place
            via_pad = not direct and pad_unaligned and ops.head_supported(w.c_in, s, nc, ops.padded_pitch(s, dt), dtype=dt)
            self.fused.append(direct or via_pad)
            self.padded.append(torch.zeros(batch, w.c_in, ops.padded_pitch(s, dt), dtype=dt, device=self.device)
                               if via_pad else None)
        # kernels per step: [pad copies] + fused head (+ cuDNN / decode_compact for uncovered scales) + 3 NMS kernels
        self.kernels_per_step = 3 + (1 if any(self.fused) else 0) + sum(p is not None for p in self.padded) + \
            (1 if not all(self.fused) else 0)

    def _pick(self, seq, flag: bool):
        return [v for v, f in zip(seq, self.fused) if f == flag]

    def _produce(self, feats) -> None:
        feats = list(feats)
        if len(feats) != len(self.specs):
            raise ValueError("one feature map per scale is required")
        for k, x in enumerate(feats):
            if isinstance(x, torch.Tensor) and x.dtype != self.feature_dtype:
                raise TypeError(f"feature map {k} is {x.dtype}, but this HeadDetector was built for "
                                f"feature_dtype={self.feature_dtype}")
        first = True
        if any(self.fused):
            # channels_last maps are read in place at every plane size (one NHWC call, no padded copy)
            if not all(ops.is_channels_last(x) for x in self._pick(feats, True)):
                feats = [x if p is None else ops.pad_feature(x, out=p) for x, p in zip(feats, self.padded)]
            ops.head_decode_compact(self._pick(feats, True), self._pick(self.weights, True), self._pick(self.specs, True),
                                    self._pick(self.row_offs, True), self.rows, self.nc, self.conf_thres, self.buf)
            first = False
        if not all(self.fused):
            # 16-bit feature maps: the module's own convolution in that precision, for a .half() module and for an fp32
            # module alike (decode_compact reads the 16-bit head tensors)
            amp = (torch.autocast("cuda", dtype=self.feature_dtype) if self.feature_dtype != torch.float32
                   else contextlib.nullcontext())
            with torch.no_grad(), amp:
                rest = [m(x) for m, x in zip(self._pick(self.modules_, False), self._pick(feats, False))]
            if self.feature_dtype != torch.float32:
                rest = [r.to(self.feature_dtype) for r in rest]      # one dtype per decode_compact call
            ops.decode_compact(rest, self._pick(self.specs, False), self.nc, self.conf_thres, self.buf,
                               row_offs=self._pick(self.row_offs, False), rows_per_img=self.rows, accumulate=not first)

def head_forward(feat: torch.Tensor, module_or_weights, spec: ops.ScaleSpec, nc: int, fp32x3: bool = False) -> torch.Tensor:
    """The head tensor alone, from the tensor-core kernel: ``module(feat)`` for a 1x1 ConvBlock / Conv2d in eval mode
    (what ``YOLOLayer.forward`` receives), always fp32.  A module is folded to the feature map's dtype.  Used by the parity
    tests and as a convolution-only entry point."""
    hw = module_or_weights if isinstance(module_or_weights, ops.HeadWeights) else \
        ops.fold_head(module_or_weights, feat.device, fp32x3, dtype=feat.dtype)
    out = torch.empty(feat.shape[0], hw.n_out, spec.ny, spec.nx, dtype=torch.float32, device=feat.device)
    ops.head_decode_compact([feat], [hw], [spec], [0], spec.rows, nc, 0.0, None, head_outs=[out], candidates=False)
    return out


# ----------------------------------------------------------------------------------------------------------------
# Model-level drop-in: any reference model (a YOLOBase subclass: ``_forward_encoder`` returns the head tensors in scale
# order, ``yolo_layers`` the matching YOLOLayers -- reference models/yolo_base.py:87-150, yolov3_spp.py:119-168,
# yolov3_tiny.py:67-100) evaluated as  trunk -> fused head + decode + NMS  without touching its code.
def find_heads(model: nn.Module, example: torch.Tensor, with_dtype: bool = False):
    """The module that produces each head tensor: per branch returned by ``model._forward_encoder(example)`` the largest
    sub-module whose output *is* that tensor and which :func:`ops.fold_head` accepts (a 1x1 Conv2d, or a ConvBlock of
    1x1 Conv2d + BatchNorm2d + LeakyReLU).  Returns ``[(qualified name, module, input shape, output shape), ...]``;
    ``with_dtype``: each entry ends with the dtype of the module's input as well (that of the example forward, so an
    autocast context around the call counts)."""
    seen = {}
    hooks = []

    def make_hook(name):
        def hook(mod, inputs, output):
            if isinstance(output, torch.Tensor) and inputs and isinstance(inputs[0], torch.Tensor):
                # the output is kept alive until the walk is over: ids of freed tensors get reused
                seen.setdefault(id(output), []).append((name, mod, tuple(inputs[0].shape), tuple(output.shape), output,
                                                        inputs[0].dtype))
        return hook

    for name, mod in model.named_modules():
        if name:
            hooks.append(mod.register_forward_hook(make_hook(name)))
    try:
        with torch.no_grad():
            branches = model._forward_encoder(example)
    finally:
        for h in hooks:
            h.remove()
    found = []
    for b in branches:
        best = None
        for name, mod, in_shape, out_shape, out, in_dtype in seen.get(id(b), []):
            if out is not b:
                continue
            try:
                ops.fold_head(mod, "cpu")
            except (ValueError, AttributeError):
                continue
            n_leaves = sum(1 for _ in mod.modules())
            if best is None or n_leaves > best[0]:
                best = (n_leaves, name, mod, in_shape, out_shape, in_dtype)
        if best is None:
            raise ValueError("no 1x1 head convolution found for one of the detection branches")
        found.append(best[1:] if with_dtype else best[1:5])
    return found


class FusedHeadModel:
    """``FusedHeadModel(model, example)(x)`` == ``non_max_suppression(model(x)[0], conf_thres, nms_thres)`` with the head
    convolutions, the decode, the confidence filter and the NMS on the B200-native kernels.  The model's own modules run
    up to the inputs of the head convolutions (the heads are swapped for ``nn.Identity`` during the call and restored
    afterwards: no copy of the weights).  ``example``: a tensor of the batch shape the detector is built for.
    The detector takes the dtype the head modules receive in the example forward: fp16 for a ``.half()`` model, the
    autocast type for a model built and called under ``torch.autocast`` -- build and call it in the same context."""

    def __init__(self, model: nn.Module, example: torch.Tensor, conf_thres: float = 0.5, nms_thres: float = 0.5,
                 cap: Optional[int] = None):
        self.model = model.eval()
        heads = find_heads(model, example, with_dtype=True)
        dtypes = {d for *_, d in heads}
        if len(dtypes) != 1:
            raise ValueError(f"the head modules receive different dtypes ({sorted(map(str, dtypes))}): one is required")
        layers = list(model.yolo_layers)
        if len(layers) != len(heads):
            raise ValueError("one YOLO layer per detection branch is expected")
        img_size = max(example.shape[-2:])                                    # models/yolov3_spp.py:142
        nc = int(layers[0].n_classes)
        self.specs = [ops.scale_spec([tuple(map(float, a)) for a in torch.as_tensor(l.anchors).tolist()], o[2], o[3], img_size)
                      for l, (_, _, _, o, _) in zip(layers, heads)]
        self._slots = []
        for name, mod, _, _, _ in heads:
            parent_name, _, attr = name.rpartition(".")
            self._slots.append((model.get_submodule(parent_name) if parent_name else model, attr, mod))
        self.detector = HeadDetector([m for _, m, *_ in heads], self.specs, nc, example.shape[0], example.device,
                                     conf_thres, nms_thres, cap=cap, feature_dtype=dtypes.pop())

    def features(self, x: torch.Tensor):
        """The inputs of the head convolutions, computed by the model's own modules."""
        ident = nn.Identity()
        try:
            for parent, attr, _ in self._slots:
                setattr(parent, attr, ident)
            with torch.no_grad():
                return list(self.model._forward_encoder(x))
        finally:
            for parent, attr, mod in self._slots:
                setattr(parent, attr, mod)

    def __call__(self, x: torch.Tensor, return_rows: bool = False):
        return self.detector.run(self.features(x), return_rows=return_rows, clone=True)
