"""The fused hot path: heads -> detections, without the dense (B, N, 5+nc) tensor.

``detect`` is the one-shot call; ``Detector`` keeps the device buffers (and optionally a captured
CUDA graph) for repeated batches of one shape, which is how a serving / evaluation loop such as the
reference's ``test_model`` (utils/utils.py:357-393) would drive it.
"""
from __future__ import annotations

import contextlib
from typing import Callable, List, Optional, Sequence

import torch

from . import ops


def detect(heads: Sequence[torch.Tensor], specs: Sequence[ops.ScaleSpec], nc: int,
           conf_thres: float = 0.5, nms_thres: float = 0.5, cap: Optional[int] = None,
           return_rows: bool = False):
    """decode + filter + compaction + NMS; returns the reference's list of (n,7) tensors / None."""
    if not nms_thres < 1:
        raise ValueError("nms_thres must be < 1: the reference never terminates otherwise (utils.py:266-275)")
    batch = heads[0].shape[0]
    if batch == 0:
        return ([], []) if return_rows else []
    rows = sum(s.rows for s in specs)
    buf = ops.get_buffers(heads[0].device, batch, rows if cap is None else min(cap, rows), nc)
    ops.decode_compact(heads, specs, nc, conf_thres, buf)
    out, out_row = buf.new_outputs()
    ops.nms(buf, nms_thres, out, out_row, seg_warps_per_sm=32)     # one-shot call: the kernel has the GPU to itself
    _, kept, overflow = ops.read_counts(buf)
    if overflow:
        raise ops.YoloB200Error(f"candidate capacity {buf.cap} per image exceeded; raise `cap`")
    return ops.ragged(out, out_row, kept, with_rows=return_rows)


def _high_priority_stream(device) -> torch.cuda.Stream:
    """A stream of the highest priority the device offers (its kernels' CTAs are dispatched ahead of pending CTAs of
    normal-priority streams -- also when the launches are replayed from a captured graph)."""
    return torch.cuda.Stream(device, priority=-100)      # torch clamps to the device's range (greatest = -5 on B200)


class Detector:
    """Persistent fused pipeline for batches of one shape: owns candidate buffers, NMS workspace and
    result buffers, and (optionally) replays the whole launch sequence -- decode_compact, the three NMS
    kernels and the count read-back -- as one CUDA graph.

    ``out_ptrs`` redirects the result (out, out_row, out_count device pointers, possibly in a peer GPU's
    memory) -- used by :mod:`pytorch_yolo_b200.sharded` for the NVLink ragged gather, together with ``step``
    (completion stamp), ``pre_hook`` / ``post_hook`` (extra work enqueued before the decode kernel / after the NMS
    kernels, inside the captured graph).
    ``nms_priority``: the NMS kernels and the count read-back run on a high-priority side stream that forks from /
    joins the caller's stream, so that, with several batches in flight, the small latency-bound NMS kernels of batch i
    are dispatched ahead of the thousands of pending CTAs of batch i+1's decode kernel.
    Results returned by :meth:`run` are views into the detector's result buffers and stay valid until the
    next call (pass ``clone=True`` to own them).
    """

    kernels_per_step = 4       # decode_compact, bucket_by_class, nms_segment, nms_finalize

    def __init__(self, specs: Sequence[ops.ScaleSpec], nc: int, batch: int, device,
                 conf_thres: float = 0.5, nms_thres: float = 0.5, cap: Optional[int] = None,
                 use_graph: bool = True, out_ptrs=None, variant: str = "auto", nms_priority: bool = False,
                 step=None, pre_hook: Optional[Callable[[], None]] = None, post_hook: Optional[Callable[[], None]] = None,
                 seg_warps_per_sm: int = 0):
        if not nms_thres < 1:
            raise ValueError("nms_thres must be < 1: the reference never terminates otherwise (utils.py:266-275)")
        self.specs, self.nc, self.batch = list(specs), nc, batch
        self.device = torch.device(device)
        self.conf_thres, self.nms_thres = float(conf_thres), float(nms_thres)
        self.rows = sum(s.rows for s in self.specs)
        self.buf = ops.Buffers(self.device, batch, self.rows if cap is None else min(cap, self.rows), nc)
        self.out, self.out_row = self.buf.new_outputs()
        self.out_ptrs = out_ptrs
        self.use_graph = use_graph
        self.variant = variant
        self.step, self.pre_hook, self.post_hook = step, pre_hook, post_hook
        self.seg_warps_per_sm = seg_warps_per_sm           # residency of the NMS segment kernel (0 = library default)
        self._side = _high_priority_stream(self.device) if nms_priority else None
        self._graph: Optional[torch.cuda.CUDAGraph] = None
        self._bound = None
        self._stream = None

    # -- enqueue only (no host sync) ------------------------------------------------------------
    def _produce(self, inputs) -> None:
        """Candidates of one batch into ``self.buf`` (overridden by the fused-head detector)."""
        ops.decode_compact(inputs, self.specs, self.nc, self.conf_thres, self.buf, variant=self.variant)

    def _enqueue(self, inputs) -> None:
        cur = torch.cuda.current_stream(self.device)
        side = self._side
        on_side = (lambda: torch.cuda.stream(side)) if side is not None else contextlib.nullcontext
        if self.pre_hook is not None:
            # with a side stream the hook forks off at the start of the step and is joined only by the NMS kernels: the
            # candidate stage (decode) does not wait for it
            if side is not None:
                side.wait_stream(cur)
            with on_side():
                self.pre_hook()
        self._produce(inputs)
        if side is not None:
            side.wait_stream(cur)
        with on_side():
            ops.nms(self.buf, self.nms_thres, self.out, self.out_row, out_ptrs=self.out_ptrs, step=self.step,
                    seg_warps_per_sm=self.seg_warps_per_sm)
            if self.post_hook is not None:
                self.post_hook()
            self.buf.meta_host.copy_(self.buf.meta, non_blocking=True)     # counts, overflow and sync_err in one copy
        if side is not None:
            cur.wait_stream(side)

    def bind(self, inputs: Sequence[torch.Tensor]) -> None:
        """Capture the launch sequence for these (static) input tensors on the current stream.  Call it at set-up: it
        runs the sequence once eagerly, synchronises the stream and captures."""
        inputs = list(inputs)
        self._enqueue(inputs)                                  # warm-up: module load, attribute calls
        torch.cuda.current_stream(self.device).synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):          # the side stream forks from / joins torch's capture stream: one graph, two priorities
            self._enqueue(inputs)
        self._graph = g
        self._bound = (tuple((h.data_ptr(), h.dtype) for h in inputs), inputs)

    def launch(self, inputs: Sequence[torch.Tensor]) -> None:
        """Enqueue one step on the current stream (no host sync)."""
        self._stream = torch.cuda.current_stream(self.device)
        if self.use_graph:
            # the dtype picks the kernel: a 16-bit tensor at a freed fp32 tensor's address needs a new graph
            ptrs = tuple((h.data_ptr(), h.dtype) for h in inputs)
            if self._bound is None or self._bound[0] != ptrs:
                self.bind(inputs)
            self._graph.replay()
        else:
            self._enqueue(list(inputs))

    def counts(self):
        """Wait for the step and return (candidate counts, kept counts) as CPU int32 tensors."""
        (self._stream or torch.cuda.current_stream(self.device)).synchronize()
        m, b = self.buf.meta_host, self.batch
        self._check_meta(m, b)
        return m[:b], m[b + 1:2 * b + 1]

    def _check_meta(self, m, b) -> None:
        flags = self.buf.meta_np
        if flags[2 * b + 1]:
            raise ops.YoloB200Error(f"multi-GPU gather: a step flag did not arrive in time (code {int(flags[2 * b + 1])})")
        if flags[b]:
            raise ops.YoloB200Error(f"candidate capacity {self.buf.cap} per image exceeded; raise `cap`")

    def run(self, inputs: Sequence[torch.Tensor], return_rows: bool = False, clone: bool = False):
        self.launch(inputs)
        _, kept = self.counts()
        out, out_row = (self.out.clone(), self.out_row.clone()) if clone else (self.out, self.out_row)
        return ops.ragged(out, out_row, kept, with_rows=return_rows)

    def scale_to_original(self, cur_shape, orig_shapes, do_round: bool = True) -> None:
        """Post-NMS epilogue for the whole batch in one launch: the reference's scale_coords + .round()
        (utils/utils.py:296-303, :313) applied in place to this detector's result rows."""
        from .utils.utils import letterbox_params
        from . import _lib
        if len(orig_shapes) != self.batch:
            raise ValueError("one original shape per image is required")
        params = torch.tensor([letterbox_params(cur_shape, s) for s in orig_shapes], dtype=torch.float32).pin_memory()
        dev_params = params.to(self.device, non_blocking=True)
        lib = _lib.load()
        with torch.cuda.device(self.device):
            _lib.check(lib.yolo_b200_scale_detections(self.out.data_ptr(), self.buf.out_count_ptr, self.batch,
                                                      self.out.shape[1], dev_params.data_ptr(), 1 if do_round else 0,
                                                      ops._stream_ptr(self.device)), "yolo_b200_scale_detections")

    # -- end to end from host memory --------------------------------------------------------------
    def run_from_host(self, host_heads: Sequence[torch.Tensor], dev_heads: Sequence[torch.Tensor],
                      host_out: torch.Tensor):
        """Pinned host heads -> H2D -> hot path -> D2H of the kept rows.  Returns (kept counts, host_out view,
        h2d bytes, d2h bytes).  ``dev_heads`` are the static device staging tensors, ``host_out`` a pinned
        (B, out_cap, 7) tensor."""
        h2d = 0
        for d, h in zip(dev_heads, host_heads):
            d.copy_(h, non_blocking=True)
            h2d += h.numel() * h.element_size()
        self.launch(dev_heads)
        _, kept = self.counts()
        n_max = int(kept.max()) if self.batch else 0
        d2h = self.buf.meta_host.numel() * 4
        if n_max:
            host_out[:, :n_max].copy_(self.out[:, :n_max], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            d2h += self.batch * n_max * ops.DET_COLS * 4
        return kept, host_out, h2d, d2h


class PipelinedDetector:
    """``depth`` detectors on ``depth`` streams, used round-robin: the NMS kernels and the count read-back of
    batch i overlap the decode kernel of batch i+1 (the NMS stage is latency-bound and occupies few SMs, the
    decode stage is HBM-bound).  ``submit`` enqueues a batch and returns a ticket; ``collect(ticket)`` waits for
    that batch only and returns its ragged result.  ``factory(lane) -> Detector`` builds the lanes (default: plain
    :class:`Detector` with the NMS kernels on a high-priority side stream)."""

    def __init__(self, specs, nc, batch, device, conf_thres=0.5, nms_thres=0.5, depth: int = 2,
                 factory: Optional[Callable[[int], Detector]] = None, **kw):
        self.device = torch.device(device)
        self.depth = depth
        kw.setdefault("nms_priority", depth > 1)
        make = factory or (lambda lane: Detector(specs, nc, batch, device, conf_thres, nms_thres, **kw))
        self.lanes: List[Detector] = [make(lane) for lane in range(depth)]
        self.streams = [torch.cuda.Stream(self.device) for _ in range(depth)]
        self._staging: List[Optional[List[torch.Tensor]]] = [None] * depth
        self._next = 0
        self.kernels_per_step = self.lanes[0].kernels_per_step

    def bind(self, inputs, per_lane: bool = False) -> None:
        """Capture every lane's graph for these static input tensors now (set-up time), so that no capture, warm-up
        launch or stream synchronisation happens inside a serving / timed loop.  ``per_lane``: ``inputs[l]`` are lane
        l's own static tensors (a caller that refills the inputs while other batches are in flight)."""
        cur = torch.cuda.current_stream(self.device)
        for k, (lane, st) in enumerate(zip(self.lanes, self.streams)):
            if not lane.use_graph:
                continue
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                lane.bind(inputs[k] if per_lane else inputs)
        self.drain()

    def submit(self, inputs) -> int:
        ticket = self._next
        lane = ticket % self.depth
        st = self.streams[lane]
        st.wait_stream(torch.cuda.current_stream(self.device))     # inputs were produced on the caller's stream
        with torch.cuda.stream(st):
            self.lanes[lane].launch(inputs)
        self._next += 1
        return ticket

    def submit_host(self, host_inputs: Sequence[torch.Tensor]) -> int:
        """``submit`` for inputs in PINNED HOST memory: every lane owns device staging tensors and the host -> device
        copies run on the lane's stream, so the copy of batch i+1 overlaps the kernels and the read-back of batch i."""
        ticket = self._next
        lane = ticket % self.depth
        if self._staging[lane] is None:
            self._staging[lane] = [torch.empty(h.shape, dtype=h.dtype, device=self.device) for h in host_inputs]
        stage = self._staging[lane]
        with torch.cuda.stream(self.streams[lane]):
            for d, h in zip(stage, host_inputs):
                d.copy_(h, non_blocking=True)
            self.lanes[lane].launch(stage)
        self._next += 1
        return ticket

    def collect_host(self, ticket: int, host_out: torch.Tensor):
        """Wait for ``ticket`` and copy its kept rows into the pinned ``host_out`` (B, >= max kept, 7).
        Returns (kept counts on the host, bytes copied device -> host for this step)."""
        lane = ticket % self.depth
        d = self.lanes[lane]
        _, kept = d.counts()
        n_max = int(kept.max()) if d.batch else 0
        nbytes = d.buf.meta_host.numel() * 4
        if n_max:
            with torch.cuda.stream(self.streams[lane]):
                host_out[:, :n_max].copy_(d.out[:, :n_max], non_blocking=True)
            self.streams[lane].synchronize()
            nbytes += d.batch * n_max * ops.DET_COLS * 4
        return kept, nbytes

    def counts(self, ticket: int):
        return self.lanes[ticket % self.depth].counts()

    def collect(self, ticket: int, return_rows: bool = False, clone: bool = False):
        d = self.lanes[ticket % self.depth]
        _, kept = d.counts()
        out, out_row = (d.out.clone(), d.out_row.clone()) if clone else (d.out, d.out_row)
        return ops.ragged(out, out_row, kept, with_rows=return_rows)

    def drain(self):
        for st in self.streams:
            torch.cuda.current_stream(self.device).wait_stream(st)
