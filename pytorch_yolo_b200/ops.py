"""Torch-facing wrappers over the C ABI (``include/yolo_b200.h``).

PyTorch is plumbing here: it owns device memory and streams; every computation is a kernel in
``libyolo_b200.so``.  There is no CPU path -- tensors that are not on a CUDA device raise.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import DET_COLS, MAX_ANCHORS, MAX_SCALES, Scale, YoloB200Error, check

MIN_WH = 2.0           # reference utils/utils.py:207
MAX_PER_CLASS = 100    # reference utils/utils.py:247-250


_FP32 = (torch.float32,)
# head dtypes decode_compact reads, and the variant bit that tells the library (include/yolo_b200.h)
HEAD_DTYPE_BITS = {torch.float32: 0, torch.float16: _lib.VARIANT_F16, torch.bfloat16: _lib.VARIANT_BF16}


def _require_cuda(t: torch.Tensor, what: str) -> None:
    _require_device(t, what)
    _require_dtype(t, what, _FP32)


def _require_device(t: torch.Tensor, what: str) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{what}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise YoloB200Error(f"{what} is on {t.device}: pytorch_yolo_b200 has no CPU path "
                            "(the kernels are sm_100a CUDA); move the tensor to a CUDA device")


def _require_dtype(t: torch.Tensor, what: str, dtypes) -> None:
    if t.dtype not in dtypes:
        raise TypeError(f"{what}: expected {' or '.join(str(d).replace('torch.', '') for d in dtypes)}, got {t.dtype}")


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


@dataclass
class ScaleSpec:
    """Host-side description of one YOLO layer (reference models/yolo_layer.py:101-111)."""
    anchors: Tuple[Tuple[float, float], ...]
    ny: int
    nx: int
    stride: float
    anchor_vec: torch.Tensor      # (na, 2) fp32 on CPU = anchors / stride, computed like the reference does

    @property
    def na(self) -> int:
        return len(self.anchors)

    @property
    def rows(self) -> int:
        return self.na * self.ny * self.nx


def scale_spec(anchors, ny: int, nx: int, img_size) -> ScaleSpec:
    stride = img_size / max(nx, ny)                                            # yolo_layer.py:102
    vec = torch.tensor(anchors, dtype=torch.float32).view(-1, 2) / stride       # yolo_layer.py:109
    if vec.shape[0] > MAX_ANCHORS:
        raise ValueError(f"at most {MAX_ANCHORS} anchors per scale are supported, got {vec.shape[0]}")
    return ScaleSpec(tuple((float(a), float(b)) for a, b in anchors), int(ny), int(nx), float(stride), vec)


def _fill_scales(heads: Sequence[torch.Tensor], specs: Sequence[ScaleSpec], nc: int, dtypes=_FP32):
    if not 1 <= len(heads) <= MAX_SCALES or len(heads) != len(specs):
        raise ValueError(f"need 1..{MAX_SCALES} heads with one spec each, got {len(heads)} / {len(specs)}")
    arr = (Scale * len(heads))()
    batch = heads[0].shape[0]
    dev = heads[0].device
    row_off = 0
    keep = []
    for k, (h, sp) in enumerate(zip(heads, specs)):
        _require_device(h, f"head {k}")
        _require_dtype(h, f"head {k}", dtypes)
        if h.device != dev or h.shape[0] != batch:
            raise ValueError("all heads must share device and batch size")
        if h.dtype != heads[0].dtype:
            raise ValueError(f"all heads of one call must share a dtype: head 0 is {heads[0].dtype}, head {k} {h.dtype}")
        if h.dim() != 4 or h.shape[1] != sp.na * (nc + 5) or h.shape[2] != sp.ny or h.shape[3] != sp.nx:
            raise ValueError(f"head {k}: expected (B, {sp.na * (nc + 5)}, {sp.ny}, {sp.nx}), got {tuple(h.shape)}")
        if not h.is_contiguous():
            h = h.contiguous()          # the reference's .view at yolo_layer.py:67 needs contiguity as well
        keep.append(h)
        s = arr[k]
        s.head = h.data_ptr()
        s.ny, s.nx, s.na, s.row_off, s.stride = sp.ny, sp.nx, sp.na, row_off, sp.stride
        av = sp.anchor_vec.tolist()
        for a in range(sp.na):
            s.anchor_vec[a][0], s.anchor_vec[a][1] = av[a][0], av[a][1]
        row_off += sp.rows
    return arr, keep, batch, row_off, dev


# ----------------------------------------------------------------------------------------------
DENSE_VARIANTS = {"auto": 0, "ldg": 1, "tma": 2}


def decode_dense(heads: Sequence[torch.Tensor], specs: Sequence[ScaleSpec], nc: int,
                 out: Optional[torch.Tensor] = None, variant: str = "auto") -> torch.Tensor:
    """All scales -> one (B, N, 5+nc) tensor (YOLOLayer.forward eval + torch.cat), one launch.
    ``variant``: "auto" | "ldg" | "tma" (identical results; see include/yolo_b200.h)."""
    lib = _lib.load()
    arr, keep, batch, rows, dev = _fill_scales(heads, specs, nc)
    if out is None:
        out = torch.empty(batch, rows, nc + 5, dtype=torch.float32, device=dev)
    elif out.shape != (batch, rows, nc + 5) or not out.is_contiguous() or out.device != dev:
        raise ValueError("out must be a contiguous (B, N, 5+nc) tensor on the heads' device")
    with torch.cuda.device(dev):
        check(lib.yolo_b200_decode_dense_ex(arr, len(keep), batch, nc, rows, out.data_ptr(), DENSE_VARIANTS[variant],
                                            _stream_ptr(dev)), "yolo_b200_decode_dense")
    return out


class Buffers:
    """Device buffers of one (batch, capacity, classes) problem: candidates, counters, NMS workspace.

    Everything the C ABI needs is caller-owned; this object is that caller.  ``meta`` holds, in one
    int32 tensor, ``count[B] | overflow[1] | out_count[B] | sync_err[1]`` so a single D2H copy reads all of it (and one
    memset zeroes count + overflow).  ``sync_err`` is only written by the multi-GPU step flags (a timed-out wait).
    """

    def __init__(self, device, batch: int, cap: int, nc: int, max_per_class: int = MAX_PER_CLASS):
        lib = _lib.load()
        self.device = torch.device(device)
        self.batch, self.cap, self.nc, self.mpc = batch, cap, nc, max_per_class
        self.out_cap = min(cap, nc * max_per_class)
        self.cand_box = torch.empty(max(1, batch * cap), 4, dtype=torch.float32, device=self.device)
        self.cand_meta = torch.empty(max(1, batch * cap), 4, dtype=torch.int32, device=self.device)
        self.meta = torch.zeros(2 * batch + 2, dtype=torch.int32, device=self.device)
        ws = lib.yolo_b200_nms_workspace_bytes(batch, cap, nc, max_per_class)
        self.workspace = torch.empty(max(256, ws), dtype=torch.uint8, device=self.device)
        self.meta_host = torch.zeros(2 * batch + 2, dtype=torch.int32).pin_memory()
        self.meta_np = self.meta_host.numpy()       # same memory: reading one flag must not cost a tensor op per step

    @property
    def count_ptr(self) -> int:
        return self.meta.data_ptr()

    @property
    def overflow_ptr(self) -> int:
        return self.meta.data_ptr() + 4 * self.batch

    @property
    def out_count_ptr(self) -> int:
        return self.meta.data_ptr() + 4 * (self.batch + 1)

    @property
    def sync_err_ptr(self) -> int:
        return self.meta.data_ptr() + 4 * (2 * self.batch + 1)

    def new_outputs(self):
        out = torch.empty(self.batch, self.out_cap, DET_COLS, dtype=torch.float32, device=self.device)
        out_row = torch.empty(self.batch, self.out_cap, dtype=torch.int32, device=self.device)
        return out, out_row


_buffer_cache = {}
_buffer_lock = threading.Lock()


def get_buffers(device, batch: int, cap: int, nc: int, max_per_class: int = MAX_PER_CLASS) -> Buffers:
    """Scratch buffers of the one-shot entry points (``non_max_suppression``, ``detect``), cached per problem shape AND per
    (calling thread, current stream): two threads or two streams never share candidate / workspace memory, so the one-shot
    calls are re-entrant like the C ABI underneath them.  Calls on one stream are ordered by the stream itself."""
    dev = torch.device(device)
    key = (dev, batch, cap, nc, max_per_class, threading.get_ident(), torch.cuda.current_stream(dev).cuda_stream)
    with _buffer_lock:
        buf = _buffer_cache.get(key)
        if buf is None:
            if len(_buffer_cache) > 8:
                _buffer_cache.clear()      # dropped buffers stay alive until the work queued on them has run (caching allocator)
            buf = _buffer_cache[key] = Buffers(device, batch, cap, nc, max_per_class)
    return buf


DECODE_VARIANTS = {"auto": 0, "ldg": 1, "tma": 2, "tma2d": 3, "ldg_dense": 4}


def decode_compact(heads, specs, nc: int, conf_thres: float, buf: Buffers, min_wh: float = MIN_WH,
                   variant: str = "auto", row_offs: Optional[Sequence[int]] = None,
                   rows_per_img: Optional[int] = None, accumulate: bool = False) -> None:
    """Fused decode + filter + compaction into ``buf`` (no (B, N, 5+nc) tensor is materialised).
    ``heads``: float32, float16 or bfloat16, one dtype for all.  16-bit heads are converted to fp32 as the kernel loads
    them, so the candidates are bit-identical to those of ``[h.float() for h in heads]``; the TMA variants read float32
    only.
    ``variant``: "auto" | "ldg" | "tma" | "tma2d" | "ldg_dense" (identical results; see include/yolo_b200.h).
    ``row_offs`` / ``rows_per_img`` / ``accumulate``: decode only some scales of a model and append to the candidates
    already in ``buf`` (the other scales went through :func:`head_decode_compact`)."""
    lib = _lib.load()
    arr, keep, batch, rows, dev = _fill_scales(heads, specs, nc, tuple(HEAD_DTYPE_BITS))
    if row_offs is not None:
        for k, off in enumerate(row_offs):
            arr[k].row_off = int(off)
        rows = int(rows_per_img)
    if batch != buf.batch or nc != buf.nc or dev != buf.device:
        raise ValueError("buffer does not match the problem")
    with torch.cuda.device(dev):
        check(lib.yolo_b200_decode_compact_ex(arr, len(keep), batch, nc, rows, conf_thres, min_wh,
                                              buf.cand_box.data_ptr(), buf.cand_meta.data_ptr(), buf.cap,
                                              buf.count_ptr, buf.overflow_ptr,
                                              DECODE_VARIANTS[variant] | (_lib.VARIANT_ACCUMULATE if accumulate else 0)
                                              | HEAD_DTYPE_BITS[keep[0].dtype],
                                              _stream_ptr(dev)),
              "yolo_b200_decode_compact")


# ----------------------------------------------------------------------------------------------
# Head 1x1 convolution fused with decode + compaction (tcgen05 kernel, csrc/head.cu)
@dataclass
class HeadWeights:
    """A head convolution folded for the fused kernel (what ConvBlock.fuse computes, reference
    models/yolo_base.py:46-57): ``weight`` (256, c_in) on the device with pad rows zero, ``bias`` on the host."""

    weight: torch.Tensor
    bias: torch.Tensor             # (n_out,) fp32 CPU
    negative_slope: float
    n_out: int
    fp32x3: bool = False           # weight holds 512 rows: the weights, then their low parts (three-pass fp32-accurate mode)

    @property
    def c_in(self) -> int:
        return self.weight.shape[1]

    def bias_array(self):
        """The bias as the ``const float*`` host array the C ABI takes (built once)."""
        arr = self.__dict__.get("_bias_c")
        if arr is None:
            arr = self.__dict__["_bias_c"] = (C.c_float * self.n_out)(*self.bias.tolist())
        return arr


def tf32_trunc(t: torch.Tensor) -> torch.Tensor:
    """What the tensor core keeps of an fp32 operand: sign, exponent and the top 10 mantissa bits."""
    return (t.contiguous().view(torch.int32) & -8192).view(torch.float32)


def fold_head(module: torch.nn.Module, device=None, fp32x3: bool = False) -> HeadWeights:
    """Fold a reference head -- ``ConvBlock(c_in, na*(5+nc), size=1)`` = Conv2d(bias=False) + BatchNorm2d + LeakyReLU(0.1)
    (models/yolov3_spp.py:86,99,111) or a plain ``nn.Conv2d(c_in, na*(5+nc), 1)`` (models/yolov3_tiny.py:38,42) -- into one
    (256, c_in) weight matrix (rows beyond the head's channels zero), one bias vector and an activation slope.
    BatchNorm uses its running statistics (eval mode)."""
    leaves = [m for m in module.modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.BatchNorm2d, torch.nn.LeakyReLU))]
    convs = [m for m in leaves if isinstance(m, torch.nn.Conv2d)]
    bns = [m for m in leaves if isinstance(m, torch.nn.BatchNorm2d)]
    acts = [m for m in leaves if isinstance(m, torch.nn.LeakyReLU)]
    if len(convs) != 1 or len(bns) > 1 or len(acts) > 1:
        raise ValueError("a head is one 1x1 Conv2d, optionally followed by one BatchNorm2d and one LeakyReLU")
    conv = convs[0]
    if conv.kernel_size != (1, 1) or conv.stride != (1, 1) or conv.padding != (0, 0) or conv.groups != 1:
        raise ValueError("the fused head kernel covers 1x1, stride-1, ungrouped convolutions")
    with torch.no_grad():
        w = conv.weight.detach().double().reshape(conv.out_channels, conv.in_channels).cpu()
        b = conv.bias.detach().double().cpu() if conv.bias is not None else torch.zeros(conv.out_channels, dtype=torch.float64)
        if bns:
            bn = bns[0]
            g = (bn.weight.detach().double().cpu() if bn.affine else torch.ones_like(b)) / torch.sqrt(bn.running_var.detach().double().cpu() + bn.eps)
            w = w * g[:, None]
            b = (b - bn.running_mean.detach().double().cpu()) * g + (bn.bias.detach().double().cpu() if bn.affine else 0.0)
    n_out = conv.out_channels
    if n_out > 256:
        raise ValueError("the fused head kernel holds at most 256 output channels per scale")
    wp = torch.zeros(512 if fp32x3 else 256, conv.in_channels, dtype=torch.float32)      # the C ABI takes 256 rows, pad rows zero
    wp[:n_out] = w.float()
    if fp32x3:                                                           # rows 256..: w - trunc_tf32(w), exact in fp32
        wp[256:256 + n_out] = wp[:n_out] - tf32_trunc(wp[:n_out])
    dev = device if device is not None else conv.weight.device
    return HeadWeights(wp.to(dev).contiguous(), b.float().contiguous(), float(acts[0].negative_slope) if acts else 1.0, n_out,
                       fp32x3)


def head_supported(c_in: int, spec: ScaleSpec, nc: int, row_pitch: int = 0, fp32x3: bool = False) -> bool:
    """Does the tensor-core kernel take this scale?  Contiguous planes that are not a multiple of 4 floats (19x19, 13x13) are
    read in place by the one-pass kernel; the three-pass mode needs them padded (``row_pitch = padded_pitch(spec)``)."""
    return bool(_lib.load().yolo_b200_head_supported_ex(c_in, spec.ny, spec.nx, row_pitch, spec.na, nc,
                                                        _lib.HEAD_FP32X3 if fp32x3 else 0))


def padded_pitch(spec: ScaleSpec) -> int:
    """Floats per channel plane after padding to the 16-byte TMA row pitch (361 -> 364, 169 -> 172)."""
    return (spec.ny * spec.nx + 3) // 4 * 4


def pad_feature(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, C, ny, nx) -> (B, C, pitch) with every channel plane padded to a multiple of 4 floats: the form in which the
    fused head kernel accepts feature maps whose plane is not (19x19, 13x13).  One read and one write of the map."""
    _require_cuda(x, "feature map")
    b, c, ny, nx = x.shape
    pitch = (ny * nx + 3) // 4 * 4
    if out is None:
        out = torch.empty(b, c, pitch, dtype=x.dtype, device=x.device)
    elif out.shape != (b, c, pitch) or not out.is_contiguous() or out.device != x.device or out.dtype != torch.float32:
        raise ValueError(f"out must be a contiguous fp32 (B, C, {pitch}) tensor on the feature map's device")
    x = x if x.is_contiguous() else x.contiguous()
    with torch.cuda.device(x.device):
        check(_lib.load().yolo_b200_pad_planes(x.data_ptr(), out.data_ptr(), b * c, ny * nx, pitch, _stream_ptr(x.device)),
              "yolo_b200_pad_planes")
    return out


def head_decode_compact(feats: Sequence[torch.Tensor], weights: Sequence[HeadWeights], specs: Sequence[ScaleSpec],
                        row_offs: Sequence[int], rows_per_img: int, nc: int, conf_thres: float, buf: Optional[Buffers],
                        min_wh: float = MIN_WH, accumulate: bool = False,
                        head_outs: Optional[Sequence[Optional[torch.Tensor]]] = None, candidates: bool = True,
                        _profile_flags: int = 0, cta_pair: bool = False) -> None:
    """1x1 head convolution (+ folded BatchNorm + LeakyReLU) on the tensor cores, decoded and compacted straight from the
    accumulator into ``buf``.  ``feats[k]``: (B, c_in, ny, nx) input of head k; ``row_offs[k]``: first row of scale k in the
    concatenated prediction.  ``head_outs[k]`` (optional) receives the activated head tensor (B, na*(5+nc), ny, nx).
    ``cta_pair`` selects the tcgen05 ``cta_group::2`` variant of the kernel (identical results)."""
    lib = _lib.load()
    n = len(feats)
    if not 1 <= n <= MAX_SCALES or not (len(weights) == len(specs) == len(row_offs) == n):
        raise ValueError("one weight set, spec and row offset per head is required")
    arr = (_lib.Head * n)()
    keep = []
    dev = feats[0].device
    batch = feats[0].shape[0]
    for k, (x, hw, sp) in enumerate(zip(feats, weights, specs)):
        _require_cuda(x, f"feature map {k}")
        pitch = 0
        if x.dim() == 3 and x.shape[0] == batch and x.shape[1] == hw.c_in and x.shape[2] >= sp.ny * sp.nx:
            pitch = x.shape[2]                       # (B, c_in, pitch): planes padded by pad_feature
        elif x.dim() != 4 or x.shape[1] != hw.c_in or x.shape[2] != sp.ny or x.shape[3] != sp.nx or x.shape[0] != batch:
            raise ValueError(f"feature map {k}: expected (B, {hw.c_in}, {sp.ny}, {sp.nx}) or a padded (B, {hw.c_in}, pitch), "
                             f"got {tuple(x.shape)}")
        if hw.n_out != sp.na * (nc + 5):
            raise ValueError(f"head {k}: {hw.n_out} output channels, expected {sp.na * (nc + 5)}")
        if hw.weight.device != dev:
            raise ValueError("weights must live on the feature maps' device")
        x = x if x.is_contiguous() else x.contiguous()
        bias_c = hw.bias_array()
        keep += [x, bias_c]
        h = arr[k]
        h.x, h.weight, h.bias_host = x.data_ptr(), hw.weight.data_ptr(), bias_c
        ho = head_outs[k] if head_outs is not None else None
        if ho is not None:
            if ho.shape != (batch, hw.n_out, sp.ny, sp.nx) or not ho.is_contiguous() or ho.device != dev or ho.dtype != torch.float32:
                raise ValueError(f"head_outs[{k}] must be a contiguous fp32 (B, {hw.n_out}, {sp.ny}, {sp.nx}) tensor")
            h.head_out = ho.data_ptr()
        h.c_in, h.negative_slope, h.x_row_pitch = hw.c_in, hw.negative_slope, pitch
        s = h.scale
        s.ny, s.nx, s.na, s.row_off, s.stride = sp.ny, sp.nx, sp.na, int(row_offs[k]), sp.stride
        av = sp.anchor_vec.tolist()
        for a in range(sp.na):
            s.anchor_vec[a][0], s.anchor_vec[a][1] = av[a][0], av[a][1]
    flags = (_lib.HEAD_ACCUMULATE if accumulate else 0) | (0 if candidates else _lib.HEAD_NO_CANDIDATES)
    if any(hw.fp32x3 for hw in weights):
        if not all(hw.fp32x3 for hw in weights):
            raise ValueError("fold every head of one call with the same fp32x3 setting")
        flags |= _lib.HEAD_FP32X3
    flags |= _profile_flags & 0xF00          # YOLO_B200_HEAD_PROFILE_* (kernel studies only)
    if cta_pair:
        flags |= 4                           # YOLO_B200_HEAD_CTA_PAIR
    if buf is None:
        if candidates:
            raise ValueError("candidate buffers are required unless candidates=False")
        scratch = torch.zeros(batch + 1, dtype=torch.int32, device=dev)
        keep.append(scratch)
        ptrs = (None, None, 1, scratch.data_ptr(), scratch.data_ptr() + 4 * batch)
    else:
        if batch != buf.batch or nc != buf.nc or dev != buf.device:
            raise ValueError("buffer does not match the problem")
        ptrs = (buf.cand_box.data_ptr(), buf.cand_meta.data_ptr(), buf.cap, buf.count_ptr, buf.overflow_ptr)
    with torch.cuda.device(dev):
        check(lib.yolo_b200_head_decode_compact(arr, n, batch, nc, rows_per_img, conf_thres, min_wh,
                                                ptrs[0], ptrs[1], ptrs[2], ptrs[3], ptrs[4], flags, _stream_ptr(dev)),
              "yolo_b200_head_decode_compact")


def compact_from_dense(pred: torch.Tensor, conf_thres: float, buf: Buffers, write_back: bool = True,
                       min_wh: float = MIN_WH) -> None:
    """Filter + compaction of a decoded (B, N, 5+nc) tensor; writes obj*cls back into column 4 like the reference."""
    lib = _lib.load()
    _require_cuda(pred, "prediction")
    if pred.dim() != 3 or not pred.is_contiguous():
        raise ValueError("prediction must be a contiguous (B, N, 5+nc) tensor")
    batch, rows, no = pred.shape
    if batch != buf.batch or no - 5 != buf.nc or pred.device != buf.device:
        raise ValueError("buffer does not match the problem")
    with torch.cuda.device(pred.device):
        check(lib.yolo_b200_compact_from_dense(pred.data_ptr(), batch, rows, no - 5, conf_thres, min_wh,
                                               1 if write_back else 0,
                                               buf.cand_box.data_ptr(), buf.cand_meta.data_ptr(), buf.cap,
                                               buf.count_ptr, buf.overflow_ptr, _stream_ptr(pred.device)),
              "yolo_b200_compact_from_dense")


def nms(buf: Buffers, nms_thres: float, out: torch.Tensor, out_row: torch.Tensor,
        out_ptrs: Optional[Tuple[int, int, int]] = None, step: Optional[Tuple[int, int]] = None,
        seg_warps_per_sm: int = 0) -> None:
    """Segmented MERGE-NMS of the candidates in ``buf``.  ``out_ptrs`` overrides the destination
    (out, out_row, out_count) with raw device pointers, e.g. a peer GPU's buffers.  ``step`` = (step_seq, step_stamp)
    device pointers: the completion stamp of the multi-GPU gather (include/yolo_b200.h, yolo_b200_nms_opts).
    ``seg_warps_per_sm``: residency of the segment kernel (0 = library default, tuned for several batches in flight;
    32 is fastest for a call that has the GPU to itself)."""
    lib = _lib.load()
    if not nms_thres < 1.0:
        raise ValueError("nms_thres must be < 1: the reference never terminates otherwise (utils.py:266-275)")
    if out_ptrs is None:
        if out.shape[0] != buf.batch or out.shape[1] < buf.out_cap or not out.is_contiguous():
            raise ValueError("out must be (B, >= out_cap, 7) contiguous")
        out_ptrs = (out.data_ptr(), out_row.data_ptr(), buf.out_count_ptr)
        out_cap = out.shape[1]
    else:
        out_cap = buf.out_cap
    opts = None
    if step is not None or seg_warps_per_sm:
        opts = _lib.NmsOpts(0, int(seg_warps_per_sm), step[0] if step else None, step[1] if step else None)
    with torch.cuda.device(buf.device):
        check(lib.yolo_b200_nms_ex(buf.cand_box.data_ptr(), buf.cand_meta.data_ptr(), buf.count_ptr,
                                   buf.batch, buf.cap, buf.nc, nms_thres, buf.mpc,
                                   out_ptrs[0], out_ptrs[1], out_cap, out_ptrs[2],
                                   buf.workspace.data_ptr(), buf.workspace.numel(),
                                   C.byref(opts) if opts is not None else None, _stream_ptr(buf.device)),
              "yolo_b200_nms")


def flag_wait(flags_ptr: int, n_flags: int, seq_ptr: int, bias: int, err_ptr: int, device, timeout_s: float = 20.0) -> None:
    """Enqueue a wait for ``n_flags`` step flags (yolo_b200_flag_wait) on the current stream of ``device``."""
    with torch.cuda.device(device):
        check(_lib.load().yolo_b200_flag_wait(flags_ptr, n_flags, seq_ptr, bias, err_ptr, timeout_s, _stream_ptr(device)),
              "yolo_b200_flag_wait")


def flag_post(flag_ptr: int, seq_ptr: int, bias: int, device) -> None:
    """Enqueue the publication of a step flag (yolo_b200_flag_post) on the current stream of ``device``."""
    with torch.cuda.device(device):
        check(_lib.load().yolo_b200_flag_post(flag_ptr, seq_ptr, bias, _stream_ptr(device)), "yolo_b200_flag_post")


def read_counts(buf: Buffers):
    """The one D2H of the path: candidate counts, kept counts and the overflow flag."""
    buf.meta_host.copy_(buf.meta, non_blocking=True)
    torch.cuda.current_stream(buf.device).synchronize()
    m = buf.meta_host
    b = buf.batch
    return m[:b], m[b + 1:2 * b + 1], int(m[b])


def ragged(out: torch.Tensor, out_row: Optional[torch.Tensor], kept_counts, with_rows: bool = False):
    """(B, out_cap, 7) + counts -> the reference's return value: list of (n, 7) tensors or None.
    The views are cut by ONE ``split_with_sizes`` per tensor (kept rows and the unused tail of every image alternate): a
    Python slice per image costs 2-3 us, which for a batch of 64 was half of the drop-in call's host time."""
    counts = kept_counts.tolist()
    cap = out.shape[1]
    if out.is_contiguous() and (not with_rows or out_row.is_contiguous()):
        sizes = [x for n in counts for x in (n, cap - n)]
        parts = out.view(-1, out.shape[2]).split_with_sizes(sizes)
        dets: List[Optional[torch.Tensor]] = [p if n else None for p, n in zip(parts[0::2], counts)]
        if not with_rows:
            return dets
        parts = out_row.view(-1).split_with_sizes(sizes)
        return dets, [p if n else None for p, n in zip(parts[0::2], counts)]
    dets = []
    rows: List[Optional[torch.Tensor]] = []
    for i, n in enumerate(counts):
        dets.append(out[i, :n] if n else None)
        if with_rows:
            rows.append(out_row[i, :n] if n else None)
    return (dets, rows) if with_rows else dets
