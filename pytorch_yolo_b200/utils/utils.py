"""Drop-in for ``pytorch_yolo.utils.utils.non_max_suppression`` (reference utils/utils.py:200-293).

Same signature, same return value (python list, one entry per image: ``None`` or an fp32 ``(n, 7)``
tensor ``(x1, y1, x2, y2, obj*cls_conf, cls_conf, cls)`` on the prediction's device, ordered by
column 4 descending), same side effect (``prediction[..., 4]`` is multiplied in place by the max class
confidence, utils.py:213).  The work is done by ``compact_from_dense`` + the segmented NMS kernels.

Documented behaviour where the reference is undefined:
* score ties keep ascending anchor-row order (the reference's argsort is unstable);
* ``nms_thres >= 1`` raises ``ValueError`` (the reference loops forever);
* tensors must be float32 on a CUDA device -- there is no CPU path.

The fused path (``detect``, ``detect_layers``, ``Detector``, ``PipelinedDetector``, ``ShardedDetector``, ``EvalPipeline``)
also takes fp16 and bf16 head tensors, as a ``.half()`` or autocast model produces them, and decodes them in fp32: the
results are bit-identical to those from ``[h.float() for h in heads]``.  That deviates from the reference on 16-bit
input, which computes ``io`` in 16 bits and rounds after every op (box corners at 608 px carry ulps of 0.25-0.5 px).
``non_max_suppression``, ``decode_layers`` and ``YOLOLayer.forward`` keep taking float32 only.
"""
from __future__ import annotations

import ctypes as C

import torch

from .. import _lib, ops


def _nms_tensor(pred: torch.Tensor, conf_thres: float, nms_thres: float, return_rows: bool, cap=None):
    ops._require_cuda(pred, "prediction")
    if pred.dim() != 3:
        raise ValueError(f"prediction must be (B, N, 5+nc), got {tuple(pred.shape)}")
    work = pred if pred.is_contiguous() else pred.contiguous()
    batch, rows, no = work.shape
    if batch == 0:
        return ([], []) if return_rows else []
    buf = ops.get_buffers(work.device, batch, rows if cap is None else cap, no - 5)
    ops.compact_from_dense(work, conf_thres, buf, write_back=True)
    if work is not pred:
        pred[..., 4].copy_(work[..., 4])            # keep the in-place side effect on the caller's memory
    out, out_row = buf.new_outputs()
    ops.nms(buf, nms_thres, out, out_row, seg_warps_per_sm=32)     # one-shot call: the kernel has the GPU to itself
    _, kept, overflow = ops.read_counts(buf)
    if overflow:
        raise ops.YoloB200Error(f"candidate capacity {buf.cap} per image exceeded; raise `cap`")
    return ops.ragged(out, out_row, kept, with_rows=return_rows)


def non_max_suppression(prediction, conf_thres=0.5, nms_thres=0.5, return_rows=False):
    """See module docstring.  ``prediction``: (B, N, 5+nc) tensor or a list of (N, 5+nc) tensors."""
    if not nms_thres < 1:
        raise ValueError("nms_thres must be < 1: the reference never terminates otherwise (utils.py:266-275)")
    if isinstance(prediction, torch.Tensor):
        return _nms_tensor(prediction, conf_thres, nms_thres, return_rows)
    prediction = list(prediction)                     # list of per-image tensors, as the reference accepts
    if any(p.dim() != 2 for p in prediction):
        raise ValueError("list entries must be (N, 5+nc) tensors")
    if len(prediction) > 1 and all(p.shape == prediction[0].shape and p.device == prediction[0].device for p in prediction):
        # same-shaped images: one batched launch chain and one host sync instead of one per image; the in-place side
        # effect (utils.py:213) is copied back into every caller tensor
        work = torch.stack(prediction)
        res = _nms_tensor(work, conf_thres, nms_thres, return_rows)
        torch._foreach_copy_([p[:, 4] for p in prediction], list(work[:, :, 4].unbind(0)))
        return res
    dets, rows = [], []
    for pred in prediction:
        r = _nms_tensor(pred.unsqueeze(0), conf_thres, nms_thres, True)
        dets.append(r[0][0])
        rows.append(r[1][0])
    return (dets, rows) if return_rows else dets


# ---------------------------------------------------------------------------------------------------------------
# Post-NMS epilogue: reference utils/utils.py:296-327 (SURVEY.md section 8f, first "next" row)
def letterbox_params(img1_shape, img0_shape):
    """(pad_x, pad_y, gain) exactly as the reference's python arithmetic computes them (utils.py:298-300)."""
    gain = max(img1_shape) / max(img0_shape)
    pad_x = (img1_shape[1] - img0_shape[1] * gain) / 2
    pad_y = (img1_shape[0] - img0_shape[0] * gain) / 2
    return pad_x, pad_y, gain


def _scale_rows(coords: torch.Tensor, img1_shape, img0_shape, do_round: bool) -> torch.Tensor:
    ops._require_cuda(coords, "coords")
    if coords.dim() != 2 or coords.shape[1] < 4 or coords.stride(1) != 1:
        raise ValueError("coords must be an (n, >=4) tensor with unit column stride (a view of detection rows is fine)")
    pad_x, pad_y, gain = letterbox_params(img1_shape, img0_shape)
    n = coords.shape[0]
    if n:
        lib = _lib.load()
        with torch.cuda.device(coords.device):
            _lib.check(lib.yolo_b200_scale_coords(coords.data_ptr(), n, coords.stride(0) if n > 1 else max(4, coords.shape[1]),
                                                  pad_x, pad_y, gain, 1 if do_round else 0,
                                                  ops._stream_ptr(coords.device)), "yolo_b200_scale_coords")
    return coords


def scale_coords(img1_shape, coords, img0_shape):
    """Drop-in for the reference's ``scale_coords`` (utils.py:296-303): rescales xyxy ``coords`` (n, 4) from the
    network input shape ``img1_shape`` (h, w) to the original ``img0_shape`` in place and returns it."""
    return _scale_rows(coords, img1_shape, img0_shape, do_round=False)


def dict_from_results(data, targets, imgs_path, orig_shapes, cur_shape):
    """Drop-in for the reference's ``_dict_from_results`` (utils.py:306-327): scales + rounds every image's boxes on
    the device (one small kernel per image, in place like the reference), reads all rows back in one copy and
    appends ``{'type','score','left','top','right','bottom'}`` records per image path."""
    live = [(i, p) for i, p in enumerate(targets) if p is not None]
    if not live:
        return data
    for i, pred in live:
        _scale_rows(pred, cur_shape, orig_shapes[i], do_round=True)               # utils.py:313
    flat = torch.cat([p for _, p in live]).cpu().tolist()
    k = 0
    for i, pred in live:
        rows = flat[k:k + len(pred)]
        k += len(pred)
        recs = [{'type': int(cls), 'score': float(conf), 'left': int(x1), 'top': int(y1), 'right': int(x2),
                 'bottom': int(y2)} for x1, y1, x2, y2, conf, _cc, cls in rows]
        data.setdefault(imgs_path[i], []).extend(recs)
    return data


_dict_from_results = dict_from_results
