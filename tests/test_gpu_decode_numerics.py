"""The decode arithmetic against float64, and the class pick on near-ties in every kernel that has one.

A. sigmoidf_rn (csrc/common.cuh) over every fp32 with 2^-8 <= |x| <= 128, through decode_dense (every column from 4 on is
   the sigmoid of the head value), on the paths that evaluate it: the LDG and TMA dense kernels on an aligned plane and
   the scalar LDG kernel on a 13x13 plane.  The relative error is held to the bound
   stated in common.cuh, SIG_A + SIG_B * |x|, and the kernels must agree bit for bit.
B. decode_wh = (expf(t) * anchor_vec) * stride and decode_xy = (sigma(t) + g) * stride against float64.
C. The class pick.  Kernels scan raw logits for (max, second max, first arg-max) and rescan in sigmoid space when
   fl(sigma(m2) * kSlack) >= sigma(m).  The inputs here are near-ties (ulp-apart logits, exact duplicates, +inf beside
   large finite logits, NaN in a non-max class, logits where the sigmoid collapses to 1.0), so the rescan decides most
   candidates.  Every implementation (decode_compact's LDG, dense LDG and TMA kernels, compact_from_dense, the fused head
   kernel's TMEM loop) must equal the first arg-max of the sigmoid columns decode_dense writes, bit for bit.
"""
import numpy as np
import pytest
import torch
from torch import nn

from pytorch_yolo_b200 import ops
from tests.helpers import assert_same_candidates, expected_candidates, read_candidates

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Relative error bound of sigmoidf_rn (common.cuh): 2^-22 (ex2.approx) + 2^-24 (fl(1 + e)) + 2^-23 (rcp.approx) = 4.17e-7,
# and |x| * (2^-24 + 1.34e-8) from the rounded product x * fl(-log2 e) and the rounding of log2 e to fp32.
SIG_A, SIG_B = 4.2e-7, 7.3e-8
KSLACK = float(np.float32(1.00003))       # kSlack of finish_anchor (decode.cu) and finish_anchor_tmem (head.cu)
U = 2.0 ** -24                             # unit roundoff of fp32
TINY = 2.0 ** -126                         # smallest normal fp32: sigmoidf_rn flushes results below it to 0
FLT_MAX = float(np.finfo(np.float32).max)
SIG_NC = 80                                # decode_dense on 5 + 80 channels: 81 sigmoid columns per row
# the LDG and TMA kernels on an aligned plane, the scalar LDG kernel on a 13x13 plane ("tma" takes aligned planes only)
SIG_PATHS = [("ldg", 64, 64), ("tma", 64, 64), ("ldg", 13, 13), ("auto", 13, 13)]
CHUNK = 1 << 24


def sig_bound(x):
    return SIG_A + SIG_B * x.abs()


def sigma64(x):
    return 1.0 / (1.0 + torch.exp(-x.double()))


def bits_to_f32(lo, hi, step=1):
    """fp32 values with bit patterns lo, lo + step, ... < hi (increasing for non-negative patterns)."""
    return torch.arange(lo, hi, step, dtype=torch.int64, device=DEV).to(torch.int32).view(torch.float32)


def f32_bits(v):
    return int(np.float32(v).view(np.int32))


def dense_sigmoid(x, ny, nx, variant):
    """sigmoidf_rn of the 1-D fp32 device tensor x, evaluated by decode_dense: x fills the objectness and class planes of
    (B, 85, ny, nx) heads, and columns 4.. of the output are their sigmoids."""
    n = x.numel()
    plane = ny * nx
    per_img = (SIG_NC + 1) * plane
    b = -(-n // per_img)
    sig = torch.zeros(b * per_img, device=DEV)
    sig[:n] = x
    h = torch.cat([torch.zeros(b, 4, plane, device=DEV), sig.view(b, SIG_NC + 1, plane)], 1).view(b, SIG_NC + 5, ny, nx)
    spec = ops.scale_spec([(10.0, 13.0)], ny, nx, 32 * max(ny, nx))
    out = ops.decode_dense([h], [spec], SIG_NC, variant=variant)
    return out[:, :, 4:].transpose(1, 2).reshape(-1)[:n]


def all_paths(x):
    """sigmoidf_rn(x) from every path, asserted bit-identical; returns one of them."""
    got = [dense_sigmoid(x, ny, nx, v) for v, ny, nx in SIG_PATHS]
    for (v, ny, nx), s in zip(SIG_PATHS[1:], got[1:]):
        assert torch.equal(s.view(torch.int32), got[0].view(torch.int32)), f"{v} {ny}x{nx} differs from ldg 64x64"
    return got[0]


@pytest.fixture(scope="module")
def sigmoid_sweep():
    """Every fp32 with 2^-8 <= |x| <= 128 and a strided sample of smaller |x|, each chunk in increasing order of x.
    Reductions run on the device; the host only sees per-chunk scalars and the windows around non-monotone steps."""
    def chunks():
        lo, hi = f32_bits(2.0 ** -8), f32_bits(128.0) + 1
        for c0 in range(lo, hi, CHUNK):
            pos = bits_to_f32(c0, min(c0 + CHUNK, hi))
            yield pos
            yield -pos.flip(0)
        small = bits_to_f32(0, lo, 997)
        yield small
        yield -small.flip(0)

    st = {"n": 0, "bad": [], "eps": [], "eps_x": [], "ratio": [], "ratio_x": [], "smax": [], "dips": 0, "windows": []}
    for x in chunks():
        s = all_paths(x)
        ref = sigma64(x)
        rel = (s.double() - ref).abs() / ref
        bound = sig_bound(x.double())
        ftz = ref < TINY * (1.0 + bound)                  # results at the flush-to-zero edge may be 0
        ok = (rel <= bound) | (ftz & (s == 0))
        st["n"] += x.numel()
        st["bad"].append((~ok).sum())
        r = torch.where(ftz, 0.0, rel / bound)
        k = r.argmax()
        st["ratio"].append(r[k]); st["ratio_x"].append(x[k])
        e = torch.where(ftz | (x.abs() > 88.0), 0.0, rel)
        k = e.argmax()
        st["eps"].append(e[k]); st["eps_x"].append(x[k])
        st["smax"].append(s.max())
        dip = torch.nonzero(s[1:] < s[:-1]).flatten()     # x increases along the chunk: sigma must not decrease
        st["dips"] += dip.numel()
        dip = dip[dip + 12 < x.numel()][:256]
        if dip.numel():
            w = dip[:, None] + torch.arange(12, device=DEV)
            st["windows"] += list(zip(x[w].cpu().numpy(), s[w].cpu().numpy()))
    out = {"n": st["n"], "dips": st["dips"], "windows": st["windows"]}
    out["bad"] = int(torch.stack(st["bad"]).sum())
    for key in ("eps", "ratio"):
        v = torch.stack(st[key])
        k = int(v.argmax())
        out[key], out[key + "_x"] = float(v[k]), float(st[key + "_x"][k])
    out["smax"] = float(torch.stack(st["smax"]).max())
    return out


# ---------------------------------------------------------------------------------------------------------------------
# A. sigmoid

def test_sigmoid_within_bound_over_the_fp32_range(sigmoid_sweep):
    sw = sigmoid_sweep
    print(f"\nsigmoidf_rn: {sw['n']} values, max rel err (|x| <= 88) {sw['eps']:.3e} at x = {sw['eps_x']!r}, "
          f"max err / bound {sw['ratio']:.3f} at x = {sw['ratio_x']!r}, max sigma {sw['smax']!r} "
          f"({'<= 1' if sw['smax'] <= 1.0 else '> 1'}), non-monotone steps {sw['dips']}")
    assert sw["n"] > 2.5e8
    assert sw["bad"] == 0, f"{sw['bad']} values outside {SIG_A} + {SIG_B} |x| (worst ratio {sw['ratio']} at {sw['ratio_x']})"
    assert sw["ratio"] <= 1.0


def test_sigmoid_premises_of_the_objectness_gate_and_the_class_pick(sigmoid_sweep):
    sw = sigmoid_sweep
    # obj_gate (decode.cu) assumes sigma <= 1 + 2^-23
    assert sw["smax"] <= 1.0 + 2.0 ** -23
    # the class pick: a class k can beat the raw-logit arg-max in sigmoid space only if sigma(m2) >= sigma(m) (1 - eps) /
    # (1 + eps); the rescan test fl(sigma(m2) * kSlack) >= sigma(m) must hold then, rounding of the product included
    eps = sw["eps"]
    assert 2 * eps < KSLACK - 1
    assert KSLACK * (1 - U) >= (1 + eps) / (1 - eps)


def test_sigmoid_special_values():
    f = np.finfo(np.float32)
    vals = [0.0, -0.0, float(f.tiny), -float(f.tiny), 1e-45, -1e-45, 2.0 ** -140, -(2.0 ** -140), float(f.max),
            -float(f.max), float("inf"), -float("inf"), float("nan"), 88.0, -88.0, 88.72, -88.72, 89.0, -89.0, 200.0, -200.0]
    x = torch.tensor(vals, dtype=torch.float32, device=DEV)
    # and a strided sample of |x| > 128 up to FLT_MAX
    big = bits_to_f32(f32_bits(128.0), f32_bits(float(f.max)) + 1, 4099)
    x = torch.cat([x, big, -big])
    s = all_paths(x).cpu()
    xs = x.cpu()
    assert torch.isnan(s[12])
    assert s[10] == 1.0 and s[11] == 0.0
    fin = torch.isfinite(xs)
    ref = sigma64(xs[fin])
    sf = s[fin].double()
    bound = sig_bound(xs[fin].double().clamp(-128, 128))
    ok = ((sf - ref).abs() <= bound * ref) | ((ref < TINY * (1 + bound)) & (sf == 0))
    assert bool(ok.all()), list(zip(xs[fin][~ok].tolist(), sf[~ok].tolist()))
    assert bool((s[fin][xs[fin] > 17.0] == 1.0).all()) and bool((s[fin][xs[fin] < -88.73] == 0.0).all())


def test_sigmoid_against_torch_cpu_at_the_parity_tolerance(sigmoid_sweep):
    """The criterion the oracle tests use for decode_dense: |sigma_dev - sigma_cpu| <= 1e-5 sigma_cpu + 1e-30."""
    g = torch.Generator().manual_seed(3)
    x = torch.cat([torch.rand(1 << 20, generator=g) * 256.0 - 128.0,
                   torch.tensor([sigmoid_sweep["eps_x"], sigmoid_sweep["ratio_x"], -87.3, -88.0, 88.0, 0.0])]).float()
    s = all_paths(x.to(DEV)).cpu()
    want = torch.sigmoid(x)
    assert bool(((s - want).abs() <= 1e-5 * want + 1e-30).all())


# ---------------------------------------------------------------------------------------------------------------------
# B. box arithmetic

ANCHOR_PX = [(1.0, 1.5), (10.0, 13.0), (116.0, 90.0), (373.0, 326.0)]     # w overflows at t = 88.72 - ln(anchor)
BOX_CASES = [(64, 64, 512, v) for v in ("ldg", "tma")] + [(40, 48, 768, v) for v in ("ldg", "tma")] + \
    [(13, 13, 416, v) for v in ("ldg", "auto")]                          # strides 8, 16 (non-square), 32


def box_sweep():
    """t over [-30, 88] (every 61st fp32) and every fp32 in [88, 89]."""
    pos = bits_to_f32(0, f32_bits(88.0), 61)
    neg = -bits_to_f32(0, f32_bits(30.0) + 1, 61)
    edge = bits_to_f32(f32_bits(88.0), f32_bits(89.0) + 1)
    return torch.cat([neg, pos, edge])


@pytest.mark.parametrize("ny,nx,img,variant", BOX_CASES)
def test_box_decode_against_fp64(ny, nx, img, variant):
    spec = ops.scale_spec(ANCHOR_PX, ny, nx, img)
    na, plane = spec.na, ny * nx
    t = box_sweep()
    n = t.numel()
    b = -(-n // (na * plane))
    h = torch.zeros(b, na, 6, plane, device=DEV)
    tt = torch.zeros(b * na * plane, device=DEV)
    tt[:n] = t
    tt = tt.view(b, na, plane)
    h[:, :, 0] = tt
    h[:, :, 1] = tt.flip(0)                                   # another value for y at each position
    h[:, :, 2] = tt
    h[:, :, 3] = tt
    out = ops.decode_dense([h.view(b, na * 6, ny, nx)], [spec], 1, variant=variant).view(b, na, plane, 6)
    stride = spec.stride
    av = spec.anchor_vec.double().to(DEV)                        # fp32 values, exact in fp64

    # w, h: expf within 2 ulp, then two fp32 products
    bnd = 2.0 ** -22 + 2 * U + 1e-12
    for c in (2, 3):
        got = out[..., c].double()
        ref = torch.exp(tt.double()) * av[:, c - 2].view(1, na, 1) * stride
        over = ref > FLT_MAX * (1 + bnd)
        under = ref < FLT_MAX * (1 - bnd)
        close = (got - ref).abs() <= bnd * ref
        assert bool((got[over] == float("inf")).all())
        assert bool((close[under] & torch.isfinite(got[under])).all())
        assert bool((close | torch.isinf(got))[~over & ~under].all())
        if c == 2:
            assert int(over.sum()) > 0 and int(under[:, 0][tt[:, 0] > 88.0].sum()) > 0   # both sides of the edge swept

    # x, y: (sigma(t) + g) * stride, sigma within the bound of A, then the add and the product
    g_idx = torch.arange(plane, device=DEV)
    for c, g in ((0, (g_idx % nx).double()), (1, (g_idx // nx).double())):
        tv = h[:, :, c]
        got = out[..., c].double()
        sg = sigma64(tv)
        exact = (sg + g) * stride
        err = (stride * (sig_bound(tv.double()) * sg + U * (sg + g)) + U * exact) * (1 + 1e-5)
        assert bool(((got - exact).abs() <= err).all()), c
    assert int(g.max()) == ny - 1 and int((g_idx % nx).max()) == nx - 1


# ---------------------------------------------------------------------------------------------------------------------
# C. class pick

def ulp32(v):
    return np.abs(np.spacing(np.float32(v))).astype(np.float64)


def dip_triples(windows):
    """From windows around non-monotone steps of the device sigmoid (x0 < x1 < ..., s0 > s1): (l, m2, m) = (x0, x1, xj)
    with s1 < sj <= s0.  The first sigmoid arg-max is l while the raw-logit arg-max is m and sigma(m2) < sigma(m): only
    kSlack > 1 sends such an anchor to the rescan."""
    out = []
    for xs, ss in windows:
        for j in range(2, len(xs)):
            if ss[1] < ss[j] <= ss[0]:
                out.append((xs[0], xs[1], xs[j]))
                break
    return out


def near_tie_logits(rng, n, nc, triples=()):
    """(n, nc) fp32 class logits, one near-tie pattern per row."""
    out = np.full((n, nc), -60.0, np.float32)
    if nc == 1:
        out[:, 0] = rng.uniform(-12, 40, n)
        out[rng.random(n) < 0.1, 0] = np.nan                   # ignored: one class means column 5 := 1
        return out
    kinds = rng.integers(0, 6, n)
    for r in range(n):
        L = np.float32(rng.uniform(-12.0, 40.0))
        kind = kinds[r]
        if kind == 5 and (not triples or nc < 3):
            kind = 0
        if kind in (0, 3):                                      # ulp-apart logits at random classes
            k = min(nc, int(rng.integers(2, 7)))
            idx = rng.choice(nc, k, replace=False)
            js = rng.integers(0, 7, k)
            js[0] = 0
            out[r, idx] = (np.float64(L) - js * ulp32(L)).astype(np.float32)
            if kind == 3:                                       # NaN in a class that is not the max: the row must drop
                rest = [c for c in range(nc) if c != idx[0]]
                out[r, rng.choice(rest)] = np.nan
        elif kind == 1:                                         # exact duplicates at the first, a middle and the last class
            out[r, [0, nc // 2, nc - 1]] = L
            out[r, rng.integers(0, nc)] = np.float32(np.float64(L) - ulp32(L))
            out[r, [0, nc // 2, nc - 1][rng.integers(0, 3)]] = L
        elif kind == 2:                                         # +inf beside large finite logits: sigma is 1.0 for all
            idx = rng.choice(nc, min(nc, 4), replace=False)
            out[r, idx] = np.array([np.inf, 17.0, 25.0, 40.0], np.float32)[:len(idx)]
        elif kind == 4:                                         # a clear winner: no rescan
            L = np.float32(rng.uniform(-12.0, 6.0))
            idx = rng.choice(nc, 2, replace=False)
            out[r, idx] = [L, L - np.float32(1.0)]
        else:                                                   # a non-monotone step of the device sigmoid
            l, m2, m = triples[int(rng.integers(0, len(triples)))]
            idx = np.sort(rng.choice(nc, 3, replace=False))
            out[r, idx[0]], out[r, idx[2]] = l, m               # l before m: l is the first sigmoid arg-max
            out[r, idx[1]] = m2
    return out


def tie_heads(specs, nc, batch, seed, triples=()):
    rng = np.random.default_rng(seed)
    heads = []
    for s in specs:
        plane = s.ny * s.nx
        n = batch * s.na * plane
        rows = np.empty((n, 5 + nc), np.float32)
        rows[:, 0:2] = rng.normal(0.0, 0.5, (n, 2))
        rows[:, 2:4] = rng.normal(0.0, 0.3, (n, 2))
        rows[:, 4] = rng.uniform(3.0, 8.0, n)
        rows[:, 5:] = near_tie_logits(rng, n, nc, triples)
        h = torch.from_numpy(rows).view(batch, s.na, plane, 5 + nc).permute(0, 1, 3, 2).reshape(batch, -1, s.ny, s.nx)
        heads.append(h.contiguous())
    return heads


def class_logits(heads, specs, nc):
    """(B, N, nc) raw class logits in the row order of decode_dense."""
    parts = []
    for h, s in zip(heads, specs):
        b = h.shape[0]
        parts.append(h.detach().cpu().view(b, s.na, 5 + nc, s.ny * s.nx)[:, :, 5:].permute(0, 1, 3, 2).reshape(b, -1, nc))
    return torch.cat(parts, 1).numpy()


def assert_reach_and_fp64(dense, logits, emit, cls, nc, what):
    """The cases exist for the rescan: enough emitted anchors must take it, and enough of those must resolve to a class
    other than the raw-logit arg-max.  Every picked class is within 2 eps of the best in float64."""
    if nc == 1:
        assert int(emit.sum()) >= 50
        return
    s = dense.cpu().numpy()[..., 5:]
    with np.errstate(invalid="ignore"):
        raw = np.argmax(np.where(np.isnan(logits), -np.inf, logits), -1)
        rest = np.where(np.arange(nc) == raw[..., None], -np.inf, logits)
        k2 = np.argmax(rest, -1)
    sm = np.take_along_axis(s, raw[..., None], -1)[..., 0]
    sm2 = np.take_along_axis(s, k2[..., None], -1)[..., 0]
    rescan = emit & (sm2 * np.float32(KSLACK) >= sm)
    differs = rescan & (cls != raw)
    n_emit, n_rescan, n_diff = int(emit.sum()), int(rescan.sum()), int(differs.sum())
    print(f"\n{what}: {n_emit} candidates, {n_rescan} take the rescan, {n_diff} of them pick another class than the "
          f"raw-logit arg-max")
    assert n_rescan >= max(50, 0.25 * n_emit), what
    assert n_diff >= max(50, 0.25 * n_rescan), what
    lg = logits[emit].astype(np.float64)
    picked = np.take_along_axis(lg, cls[emit][:, None], -1)[:, 0]
    with np.errstate(over="ignore"):
        s64 = 1.0 / (1.0 + np.exp(-lg))
        sp = 1.0 / (1.0 + np.exp(-picked))
    eps = SIG_A + SIG_B * np.minimum(np.abs(np.concatenate([picked[:, None], lg], 1)).max(1), 88.0)
    assert bool((sp >= s64.max(1) * (1 - 2 * eps)).all()), what


DECODE_VARIANTS = ["auto", "ldg", "ldg_dense", "tma", "tma2d"]
ANCHORS3 = [(10.0, 13.0), (16.0, 30.0), (33.0, 23.0)]


@pytest.mark.parametrize("conf", [0.3, 1e-12])
@pytest.mark.parametrize("ny,nx", [(16, 16), (13, 13)])
@pytest.mark.parametrize("nc", [1, 2, 3, 20, 37, 80])
def test_class_pick_on_near_ties_in_every_decode_kernel(nc, ny, nx, conf, sigmoid_sweep):
    batch = 5                                                  # 3 * 5 slabs: the last LDG CTA and TMA tile are partial
    specs = [ops.scale_spec(ANCHORS3, ny, nx, 32 * max(ny, nx))]
    triples = dip_triples(sigmoid_sweep["windows"])
    heads = tie_heads(specs, nc, batch, seed=100 * nc + ny, triples=triples)
    dev_heads = [h.to(DEV) for h in heads]
    dense = ops.decode_dense(dev_heads, specs, nc)
    want, emit, cls = expected_candidates(dense, conf)
    assert_reach_and_fp64(dense, class_logits(heads, specs, nc), emit, cls, nc, f"nc {nc} {ny}x{nx} conf {conf}")
    if nc == 1:
        assert all(bool((m[:, 2] == 0).all()) and bool((m[:, 1].view(np.float32) == 1.0).all()) for m, _ in want)
    buf = ops.Buffers(DEV, batch, specs[0].rows, nc)
    for v in DECODE_VARIANTS:
        ops.decode_compact(dev_heads, specs, nc, conf, buf, variant=v)
        assert_same_candidates(read_candidates(buf), want, v)
    ops.compact_from_dense(dense.clone(), conf, buf, write_back=False)
    assert_same_candidates(read_candidates(buf), want, "compact_from_dense")


# ---- the fused head kernel: the same near-ties carried by the head tensor ----

def tf32_exact(v):
    return (torch.as_tensor(v, dtype=torch.float32).view(torch.int32) & -8192).view(torch.float32)


def tie_head_module(c_in, nc, leaky, seed):
    """A 1x1 head whose class rows are one-hot on input channel 0 (weight 1: the accumulator is exactly x[0] in the one-pass
    and the three-pass mode) with biases that differ by ulps; activate() adds them in fp32 after the MMA.  The other class
    rows are far below (weight 0, bias -60), box rows 0, objectness 6."""
    rng = np.random.default_rng(seed)
    no = nc + 5
    w = np.zeros((3 * no, c_in), np.float32)
    b = np.zeros(3 * no, np.float32)
    for a, delta in enumerate((2.0 ** -22, 2.0 ** -18, 2.0 ** -14)):
        b[a * no + 4] = 6.0
        b[a * no + 5:(a + 1) * no] = -60.0
        if a == 0:
            cls = sorted({0, nc // 2, nc - 1})
            js = np.arange(len(cls))                            # the largest logit at the highest index
        else:
            cls = rng.choice(nc, min(nc, 6), replace=False)
            js = rng.integers(0, 5, len(cls))
        for c, j in zip(cls, js):
            w[a * no + 5 + c, 0] = 1.0
            b[a * no + 5 + c] = np.float32(0.5 + j * delta)
    conv = nn.Conv2d(c_in, 3 * no, 1, bias=True)
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(w).view(3 * no, c_in, 1, 1))
        conv.bias.copy_(torch.from_numpy(b))
    mod = nn.Sequential(conv, nn.LeakyReLU(0.1)) if leaky else conv
    return mod.eval(), w, b


HEAD_CASES = [  # (name, nc, ny, nx, leaky, cta_pair, fp32x3)
    ("single-80-plain", 80, 20, 20, False, False, False),
    ("single-80-leaky-13x13", 80, 13, 13, True, False, False),
    ("single-20-leaky", 20, 20, 20, True, False, False),
    ("single-37-plain", 37, 20, 20, False, False, False),
    ("pair-80-plain", 80, 32, 32, False, True, False),
    ("pair-80-leaky", 80, 20, 20, True, True, False),
    ("x3-80-leaky", 80, 20, 20, True, False, True),
    ("x3-37-plain", 37, 20, 20, False, False, True),
]


@pytest.mark.parametrize("name,nc,ny,nx,leaky,cta_pair,fp32x3", HEAD_CASES, ids=[c[0] for c in HEAD_CASES])
def test_class_pick_on_near_ties_in_the_fused_head(name, nc, ny, nx, leaky, cta_pair, fp32x3):
    batch, c_in, conf = 4, 64, 0.3
    spec = ops.scale_spec(ANCHORS3, ny, nx, 32 * max(ny, nx))
    mod, w, b = tie_head_module(c_in, nc, leaky, seed=nc + ny)
    hw = ops.fold_head(mod, DEV, fp32x3=fp32x3)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(batch, c_in, ny, nx, generator=g)
    # channel 0 carries the class logits' level: tf32-exact values from -12 to 40, through the sigmoid's collapse to 1.0
    x[:, 0] = tf32_exact(torch.rand(batch, ny, nx, generator=g) * 52.0 - 12.0)
    x = x.to(DEV)
    ho = torch.empty(batch, 3 * (nc + 5), ny, nx, device=DEV)
    buf = ops.Buffers(DEV, batch, spec.rows, nc)
    ops.head_decode_compact([x], [hw], [spec], [0], spec.rows, nc, conf, buf, head_outs=[ho], cta_pair=cta_pair)
    fused = read_candidates(buf)

    # the head tensor is what the construction promises: fl(x0 * w + b), then the activation
    acc = np.where(w[:, 0][None, :, None, None] != 0, x[:, 0:1].cpu().numpy(), np.float32(0.0)).astype(np.float32)
    want_h = acc + b[None, :, None, None]
    if leaky:
        want_h = np.maximum(want_h, want_h * np.float32(0.1))
    assert np.array_equal(ho.cpu().numpy().view(np.int32), want_h.view(np.int32))

    dense = ops.decode_dense([ho], [spec], nc)
    want, emit, cls = expected_candidates(dense, conf)
    assert_reach_and_fp64(dense, class_logits([ho], [spec], nc), emit, cls, nc, name)
    assert_same_candidates(fused, want, f"{name} fused")
    ops.decode_compact([ho], [spec], nc, conf, buf)
    assert_same_candidates(read_candidates(buf), want, f"{name} decode_compact on head_outs")
