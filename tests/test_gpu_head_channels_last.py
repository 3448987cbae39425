"""GPU: the fused head kernel on channels_last feature maps (YOLO_B200_HEAD_NHWC, csrc/head.cu).

An NHWC feature map is a row-major (B*ny*nx, c_in) matrix: one 3-D tensor-map box per k-block stages 128 positions x 128
bytes of channels in the K-major SWIZZLE_128B layout, and the MMA reads A K-major.  Everything else is the NCHW kernel's.
The bars:
  * head values against fp64 (TF32, fp16, bf16, fp32x3), and bit-identical to the NCHW kernel on ``x.contiguous()``: the
    same truncated operands, k-block order and instruction shape, only the shared-memory layout of A differs;
  * candidates bit-exact against decode_compact on the head tensor the NHWC call writes;
  * HeadDetector / FusedHeadModel / graphs / pipelines on channels_last maps give the detections of NCHW maps, and launch
    no plane-padding copy.
"""
import pytest
import torch

from pytorch_yolo_b200 import ops, synth
from pytorch_yolo_b200.detect import PipelinedDetector
from pytorch_yolo_b200.head import FusedHeadModel, HeadDetector, head_forward
from tests.test_gpu_head import MiniYolo, conv_block, tf32_trunc
from tests.test_gpu_head_half import check_head_values, fused_candidates, spp_scales, unfused_candidates
from tests.test_gpu_head_steady import assert_same_candidates, assert_same_detections, row_offsets, sorted_candidates

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ANCHORS = [(10, 13), (16, 30), (33, 23)]
CL = torch.channels_last
MODES = {"tf32": (torch.float32, False), "fp16": (torch.float16, False), "bf16": (torch.bfloat16, False),
         "fp32x3": (torch.float32, True)}


def nchw_input(x, spec, nc, fp32x3):
    """The NCHW kernel's input for the same map: contiguous, or the padded copy where the plane needs one."""
    x = x.contiguous()
    if ops.head_supported(x.shape[1], spec, nc, fp32x3=fp32x3, dtype=x.dtype):
        return x
    return ops.pad_feature(x)


def bits(t):
    return t.view(torch.int32)


# ------------------------------------------------------------------------------------------------------------------
# Head values
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("batch,c_in,ny,nx", [(2, 0, 13, 13), (2, 0, 76, 76), (2, 256, 38, 38), (2, 256, 26, 26),
                                              (2, 512, 19, 19), (1, 1024, 13, 13), (3, 256, 10, 23), (1, 1024, 76, 76)])
def test_head_values_against_fp64_and_nchw(mode, batch, c_in, ny, nx):
    dtype, x3 = MODES[mode]
    c_in = c_in or (32 if dtype == torch.float32 else 64)
    spec = ops.scale_spec(ANCHORS, ny, nx, 16 * max(ny, nx))
    assert ops.head_supported(c_in, spec, 80, fp32x3=x3, dtype=dtype, memory_format=CL)
    blk = conv_block(c_in, 255, seed=c_in + ny).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(ny * nx + c_in)
    x = torch.randn(batch, c_in, ny, nx, generator=g, device=DEV).to(dtype).contiguous(memory_format=CL)
    assert ops.is_channels_last(x)
    hw = ops.fold_head(blk, DEV, fp32x3=x3, dtype=dtype)
    got = head_forward(x, hw, spec, 80)
    # contract: bit-identical to the NCHW kernel
    want = head_forward(nchw_input(x, spec, 80, x3), hw, spec, 80)
    assert torch.equal(bits(got), bits(want)), float((got - want).abs().max())
    # and within the fp64 bounds of the NCHW kernel's own tests
    if dtype != torch.float32:
        check_head_values(got, x.contiguous(), hw)
        return
    w = hw.weight[:255].double()
    xd = x.contiguous().flatten(2).double()
    ref = torch.matmul(w if x3 else tf32_trunc(hw.weight[:255]).double(), xd if x3 else tf32_trunc(x.contiguous()).double().flatten(2))
    ref = ref + hw.bias.to(DEV).double()[None, :, None]
    ref = torch.maximum(ref, ref * hw.negative_slope).view_as(got)
    s = torch.matmul(w.abs(), xd.abs()).view_as(got)
    err = (got.double() - ref).abs()
    # TF32: the fp32 accumulation of c_in / 8 rounded partial sums, <= (c_in / 8) 2^-24 S; fp32x3 adds the lost low-part
    # products (2^-21 S); a wrong layout or descriptor is off by O(S)
    bar = ((3 if x3 else 1) * c_in / 8 * 2.0 ** -24 + (2.0 ** -20 if x3 else 0.0)) * s + 1e-5
    assert bool((err <= bar).all()), float((err / s).max())


# ------------------------------------------------------------------------------------------------------------------
# Candidates
@pytest.mark.parametrize("mode", ["tf32", "fp16", "bf16", "fp32x3"])
@pytest.mark.parametrize("conf", [0.3, 0.001])
def test_candidates_bit_exact_against_decode_compact_on_own_head_tensor(mode, conf):
    dtype, x3 = MODES[mode]
    nc = 80
    specs, heads, feats = spp_scales(nc, 2, dtype, seed=60)
    feats = [x.contiguous(memory_format=CL) for x in feats]
    hws = [ops.fold_head(m, DEV, fp32x3=x3, dtype=dtype) for m in heads]
    hts = [torch.full((2, hw.n_out, s.ny, s.nx), float("nan"), device=DEV) for hw, s in zip(hws, specs)]
    with_head = sorted_candidates(fused_candidates(feats, hws, specs, nc, conf, head_outs=hts))
    want = sorted_candidates(unfused_candidates(hts, specs, nc, conf))
    assert int(want[0].sum()) > 0
    assert_same_candidates(with_head, want, "head_out instantiation vs decode_compact")
    assert_same_candidates(sorted_candidates(fused_candidates(feats, hws, specs, nc, conf)), want,
                           "production instantiation vs decode_compact")
    # an overflowing cap: the same counts and the flag
    cap = int(want[0].min()) - 1
    assert cap >= 1
    got_cnt, _, got_ovf = ops.read_counts(fused_candidates(feats, hws, specs, nc, conf, cap=cap))
    got_cnt = got_cnt.clone()
    want_cnt, _, want_ovf = ops.read_counts(unfused_candidates(hts, specs, nc, conf, cap=cap))
    assert got_ovf == want_ovf == 1 and torch.equal(got_cnt, want_cnt)


# ------------------------------------------------------------------------------------------------------------------
# Steady state at the benchmark's head shapes: every CTA runs many tiles
@pytest.mark.parametrize("wl,batch", [("spp-608", 64), ("tiny-416", 1024)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16], ids=["fp32", "fp16", "bf16"])
def test_steady_state_equals_nchw(wl, batch, dtype):
    w = synth.WORKLOADS[wl]
    nc = w["nc"]
    specs = [ops.scale_spec(a, g, g, w["img_size"]) for a, g in zip(w["anchors"], w["grids"])]
    feats, convs = synth.synth_head_convs(wl, batch, seed=4321, device=DEV)
    feats = [x.to(dtype) for x in feats]
    hws = [ops.fold_head(c, DEV, dtype=dtype) for c in convs]
    offs, rows = row_offsets(specs)
    tiles = sum(batch * -(-s.ny * s.nx // 128) for s in specs)
    assert tiles >= 10 * torch.cuda.get_device_properties(0).multi_processor_count

    def run(xs):
        buf = ops.Buffers(DEV, batch, rows, nc)
        ops.head_decode_compact(xs, hws, specs, offs, rows, nc, 0.3, buf)
        return sorted_candidates(buf)

    want = run([nchw_input(x, s, nc, False) for x, s in zip(feats, specs)])
    cl = [x.contiguous(memory_format=CL) for x in feats]
    del feats
    assert int(want[0].sum()) > 0
    assert_same_candidates(run(cl), want, f"{wl} b{batch} channels_last vs NCHW")


# ------------------------------------------------------------------------------------------------------------------
# Detectors and models
def detector_inputs(dtype, batch=2, seed=80):
    nc = 80
    specs, heads, feats = spp_scales(nc, batch, dtype, seed=seed)
    return specs, heads, feats


def test_channels_last_step_launches_no_pad_copy():
    """fp16 spp-608 maps: the NCHW step pads the odd 19x19 plane into the detector's padded buffer first; the channels_last
    step leaves that buffer alone and gives the same detections."""
    specs, heads, feats = detector_inputs(torch.float16)
    det = HeadDetector(heads, specs, 80, 2, DEV, 0.3, 0.5, feature_dtype=torch.float16)
    assert det.fused == [True, True, True] and det.padded[0] is not None and det.padded[1:] == [None, None]
    assert det.kernels_per_step == 5                                            # the NCHW plan, unchanged
    cl = [x.contiguous(memory_format=CL) for x in feats]
    pad = det.padded[0]
    pad.view(torch.int16).fill_(0x7E01)                                         # an fp16 NaN pattern nothing writes
    got = det.run(cl, return_rows=True, clone=True)
    torch.cuda.synchronize()
    assert bool((pad.view(torch.int16) == 0x7E01).all())
    want = det.run(feats, return_rows=True, clone=True)
    assert not bool((pad.view(torch.int16) == 0x7E01).all())                    # the NCHW step wrote it
    assert assert_same_detections(got, want) > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16], ids=["fp32", "fp16", "bf16"])
def test_head_detector_graph_replay_and_pipeline(dtype):
    specs, heads, _ = detector_inputs(dtype)
    batch = 2
    det = HeadDetector(heads, specs, 80, batch, DEV, 0.3, 0.5, use_graph=True, feature_dtype=dtype)
    ref = HeadDetector(heads, specs, 80, batch, DEV, 0.3, 0.5, use_graph=False, feature_dtype=dtype)
    static = None
    for step in range(3):
        _, _, feats = detector_inputs(dtype, seed=90 + step)
        if static is None:
            static = [x.contiguous(memory_format=CL) for x in feats]
        else:
            for s, x in zip(static, feats):
                s.copy_(x)
        want = ref.run(feats, return_rows=True, clone=True)
        assert assert_same_detections(det.run(static, return_rows=True, clone=True), want) > 0
    pipe = PipelinedDetector(specs, 80, batch, DEV, depth=3,                   # one lane per batch: none is overwritten
                             factory=lambda lane: HeadDetector(heads, specs, 80, batch, DEV, 0.3, 0.5, use_graph=True,
                                                               feature_dtype=dtype, nms_priority=True))
    sets = [detector_inputs(dtype, seed=100 + k)[2] for k in range(3)]
    cl_sets = [[x.contiguous(memory_format=CL) for x in s] for s in sets]      # alive until the lanes have read them
    tickets = [pipe.submit(s) for s in cl_sets]
    for t, s in zip(tickets, sets):
        want = ref.run(s, return_rows=True, clone=True)
        assert assert_same_detections(pipe.collect(t, return_rows=True, clone=True), want) > 0


@pytest.mark.parametrize("kind", ["fp32", "half", "bf16_autocast"])
def test_fused_head_model_on_a_channels_last_model(kind):
    torch.manual_seed(3)
    model = MiniYolo().to(DEV).eval()
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.2)
                m.running_var.uniform_(0.5, 1.5)
        model.branch2[1].bias[4::85] -= 3.0
    model = model.to(memory_format=CL)
    x = torch.rand(2, 3, 52, 52, device=DEV).contiguous(memory_format=CL)
    if kind == "half":
        model, x = model.half(), x.half()
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if kind == "bf16_autocast" else torch.no_grad()
    with ctx:
        fused = FusedHeadModel(model, x, conf_thres=0.05, nms_thres=0.5)
        feats = fused.features(x)
        assert all(ops.is_channels_last(f) for f in feats)
        got = fused.detector.run(feats, return_rows=True, clone=True)
        want = fused.detector.run([f.contiguous() for f in feats], return_rows=True, clone=True)
        assert_same_detections(fused(x, return_rows=True), want)
    assert assert_same_detections(got, want) > 0
