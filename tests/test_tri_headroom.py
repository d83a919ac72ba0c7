"""Headroom of precision mode 1 ("f16f8") on the CPU: the contract "the range monitor accepts =>
the layer is within 1e-4 of fp64".

The tri-plane exponents are measured on an engine's first input and then frozen.  A later input
s times larger runs with those stale exponents; MNCEngine.range_ok() decides whether the result is
still good enough.  fp16 saturates only 16x above the calibrated maximum, but the e4m3 correction
planes give out at about 4x, so a threshold at fp16's limit accepts layers several times worse
than calibrated.  Here each layer is restated exactly -- the planes of dense.tri_from_f32 (the
device conversion, bit for bit: tests/test_gpu_round2.py), the three products of the kernels
(Xh.Wh + Xl.Wc + Xc.Wl) summed in fp64, the output re-encoded with its stale exponent -- and the
engine's own range_ok() is asked about the input and output maxima."""
import pytest
import torch
import torch.nn.functional as F

SCALES = (2.0 ** -10, 2.0 ** -4, 1, 2, 4, 6, 8, 12, 15)


def _planes(t):
    f8 = lambda p: p.view(torch.float8_e4m3fn).double()
    return t.h.double(), f8(t.l), f8(t.c)


def _tri_layer(x, wt, kind):
    """The kernels' arithmetic in fp64: x Tri (activations), wt Tri (weights) -> pre-ReLU fp64."""
    xh, xl, xc = _planes(x)
    wh, wl, wc = _planes(wt)
    if kind == "fc":
        acc = xh @ wh.T + xl @ wc.T + xc @ wl.T
    else:
        acc = sum(F.conv2d(a, b, padding=1) for a, b in ((xh, wh), (xl, wc), (xc, wl)))
    return acc * 2.0 ** -(x.exp + wt.exp)


def _post(y, pool):
    y = y.clamp_min(0)
    return F.max_pool2d(y, 2, 2, ceil_mode=True) if pool else y


def _monitor_accepts(amax_in, e_in, amax_out, e_out):
    """MNCEngine.range_ok() on an engine whose kernels published these two maxima."""
    from mnc_b200.engine import MNCEngine
    eng = MNCEngine.__new__(MNCEngine)
    eng.tri = True
    eng.exp = {"in": e_in, "out": e_out}
    eng._amax_slot = {"in": 0, "out": 1}
    eng._amax_all = torch.tensor([amax_in, amax_out], dtype=torch.float32).view(torch.int32)
    eng._calibrated = True
    eng.range_violations = 0
    return eng.range_ok()


def headroom_table(kind, dist, pool=False, seed=0):
    """[(s, input scaled max, output scaled max, accepted, relative error)] for one layer."""
    from mnc_b200 import dense
    g = torch.Generator().manual_seed(seed)
    if kind == "fc":
        M, K, N = 512, 4608, 256
        shape, w = (M, K), torch.randn(N, K, generator=g) * (2.0 / K) ** 0.5
        wt = dense.tri_from_f32(w, weight=True)
        ref_fn = lambda xs: xs.double() @ w.double().T
    else:
        C, H, W = 64, 75, 125
        shape, w = (1, C, H, W), torch.randn(C, C, 3, 3, generator=g) * (2.0 / (9 * C)) ** 0.5
        # conv_weight_to_tri's planes, back in Caffe's (Cout, Cin, kh, kw) order for conv2d
        t = dense.conv_weight_to_tri(w)
        back = lambda p: p.view(C, 3, 3, C).permute(0, 3, 1, 2).contiguous()
        wt = dense.Tri(back(t.h), back(t.l), back(t.c), t.exp)
        ref_fn = lambda xs: F.conv2d(xs.double(), w.double(), padding=1)
    x = torch.rand(shape, generator=g) if dist == "uniform" else torch.randn(shape, generator=g).clamp_min(0)
    # calibration on the s = 1 input, the way MNCEngine._scaled measures it
    e_in = dense.exp_for(float(x.abs().max()))
    y1 = _post(_tri_layer(dense.tri_from_f32(x, exp=e_in), wt, kind), pool)
    e_out = dense.exp_for(float(y1.abs().max()))
    rows = []
    for s in SCALES:
        xs = x * s
        ref = _post(ref_fn(xs), pool)
        y = _post(_tri_layer(dense.tri_from_f32(xs, exp=e_in), wt, kind), pool)
        got = dense.tri_from_f32(y.float(), exp=e_out).float().double()
        err = float((got - ref).abs().max() / ref.abs().max())
        a_in, a_out = float(xs.abs().max()), float(y.abs().max())
        rows.append((s, a_in * 2.0 ** e_in, a_out * 2.0 ** e_out,
                     _monitor_accepts(a_in, e_in, a_out, e_out), err))
    return rows


def format_table(rows):
    return "\n".join("s=%-9g in %8.0f  out %8.0f  %-8s err %.2e" % (s, a, b, "accepted" if ok else "rejected", e)
                     for s, a, b, ok, e in rows)


@pytest.mark.parametrize("kind,pool", [("fc", False), ("conv", False), ("conv", True)])
@pytest.mark.parametrize("dist", ["uniform", "relu_randn"])
def test_monitor_accepts_only_accurate_layers(kind, pool, dist):
    rows = headroom_table(kind, dist, pool)
    msg = "%s%s, %s activations:\n%s" % (kind, " pooled" if pool else "", dist, format_table(rows))
    for s, _, _, ok, err in rows:
        if ok:
            assert err <= 1e-4, msg
    # the calibrated input itself and 2x over it are always accepted and accurate
    assert all(ok and err <= 3e-5 for s, _, _, ok, err in rows if s in (1, 2)), msg
    # and the range past fp16's own limit is never accepted
    assert not any(ok for s, a, b, ok, _ in rows if max(a, b) > 65504), msg
