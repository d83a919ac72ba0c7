"""Host-side wrappers of the dense (conv / inner-product) C-ABI entry points.

Activations and weights are "split" tensors: a torch bf16 tensor of shape [2, ...] holding the
(hi, lo) planes with x ~= hi + lo.
"""
import ctypes

import torch

from ._lib import lib, ptr, cur_stream, check, c_int, c_ll


def split(x):
    """fp32 tensor -> bf16 [2, *x.shape] (hi, lo) with hi = rn(x), lo = rn(x - hi)."""
    x = x.float()
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.stack([hi, lo]).contiguous()


def merge(s):
    """fp32 value of a split-bf16 tensor ([2, ...]) or of a Tri."""
    if isinstance(s, Tri):
        return s.float()
    return s[0].float() + s[1].float()


def conv_weight_to_split(w):
    """Caffe conv weight (Cout, Cin, 3, 3) -> split [2, Cout, 9*Cin], K index = tap*Cin + c."""
    cout, cin, kh, kw = w.shape
    return split(w.permute(0, 2, 3, 1).reshape(cout, kh * kw * cin))


def fc_weight_to_split(w, chw=None):
    """Caffe InnerProduct weight (N, K) with K flattened as (c, h, w)
    (inner_product_layer.cpp:14-34) -> split [2, N, K'] with K' flattened as (h, w, c), the
    order our NHWC RoI features use.  chw=None keeps K as is."""
    if chw is not None:
        c, h, wd = chw
        w = w.reshape(w.shape[0], c, h, wd).permute(0, 2, 3, 1).reshape(w.shape[0], -1)
    return split(w)


# ------------------------------------------------------------------ precision mode 1 ("tri-plane")
class Tri:
    """A tensor in the tri-plane format of csrc/igemm_tc.cu: x * 2^exp = h + l / l_scale, with a
    low-precision copy c = x * 2^exp * c_scale (activations: l_scale 2^6, c_scale 2^-5; weights:
    l_scale 2^5, c_scale 2^-6).  h: fp16, l / c: e4m3 bytes (uint8 tensors), all of one shape."""
    __slots__ = ("h", "l", "c", "exp")

    def __init__(self, h, l, c, exp):
        self.h, self.l, self.c, self.exp = h, l, c, int(exp)

    @property
    def shape(self):
        return self.h.shape

    def view(self, *shape):
        return Tri(self.h.view(*shape), self.l.view(*shape), self.c.view(*shape), self.exp)

    def flat(self, n):
        return Tri(self.h.view(-1)[:n], self.l.view(-1)[:n], self.c.view(-1)[:n], self.exp)

    def float(self):
        """fp32 value carried by the two precise planes: (h + l / 2^6) * 2^-exp (activations)."""
        l = self.l.view(torch.float8_e4m3fn).float()
        return (self.h.float() + l * (1.0 / 64.0)) * (2.0 ** -self.exp)

    def clone(self):
        return Tri(self.h.clone(), self.l.clone(), self.c.clone(), self.exp)

    def __getitem__(self, idx):
        return Tri(self.h[idx], self.l[idx], self.c[idx], self.exp)


def tri_alloc(shape, device, exp=0):
    n = 1
    for s_ in shape:
        n *= int(s_)
    buf = torch.empty(4 * n, dtype=torch.uint8, device=device)
    return Tri(buf[:2 * n].view(torch.float16).view(*shape), buf[2 * n:3 * n].view(*shape),
               buf[3 * n:].view(*shape), exp)


def _e4m3(x):
    return x.clamp(-448.0, 448.0).to(torch.float8_e4m3fn).view(torch.uint8)


def exp_for(amax, target_log2=12):
    """Power-of-two exponent e with amax * 2^e in (2^(target-1), 2^target]."""
    import math
    if not (amax > 0) or math.isinf(amax):
        return 0
    return target_log2 - int(math.ceil(math.log2(amax)))


def tri_from_f32(x, exp=None, weight=False):
    """torch restatement of the device conversion (tests, weights at load time)."""
    x = x.float()
    if exp is None:
        exp = exp_for(float(x.abs().max()), 13 if weight else 12)
    xs = (x * (2.0 ** exp)).clamp(-65504.0, 65504.0)
    h = xs.half()
    r = xs - h.float()
    if weight:
        return Tri(h.contiguous(), _e4m3(r * 32.0).contiguous(), _e4m3(xs * (1.0 / 64.0)).contiguous(), exp)
    return Tri(h.contiguous(), _e4m3(r * 64.0).contiguous(), _e4m3(xs * (1.0 / 32.0)).contiguous(), exp)


def conv_weight_to_tri(w):
    cout, cin, kh, kw = w.shape
    return tri_from_f32(w.permute(0, 2, 3, 1).reshape(cout, kh * kw * cin), weight=True)


def fc_weight_to_tri(w, chw=None):
    if chw is not None:
        c, h, wd = chw
        w = w.reshape(w.shape[0], c, h, wd).permute(0, 2, 3, 1).reshape(w.shape[0], -1)
    return tri_from_f32(w, weight=True)


def igemm2(a, batch, H, W, cin, w, cout, taps, bias=None, relu=False, out=None, out_f32=None,
           out_pix_stride=None, out_ch_offset=0, split_k=1, split_stride=0, bn=0, max_ctas=0,
           pool=False, out_exp=0, amax=None, img_hw=None, level=0):
    """General tensor-core launch (mnc_igemm_tc2).  a / w: split bf16 tensors ([2, ...]) or Tri;
    out: split bf16 tensor, or Tri (written with exponent out_exp), or out_f32.
    img_hw: device int32 (batch, 2) image sizes of a mixed-size batch, `level` pools below the
    input (mnc_igemm_tc3): pixels outside their image come out as zeros."""
    tri_in = isinstance(a, Tri)
    assert tri_in == isinstance(w, Tri)
    if tri_in:
        ap = (a.h, a.l, a.c)
        wp = (w.h, w.c, w.l)          # kernel order: value, copy, residual
        acc_scale = 2.0 ** -(a.exp + w.exp)
    else:
        ap, wp, acc_scale = (a[0], a[1], None), (w[0], w[1], None), 1.0
    if out_f32 is not None:
        mode, op = 1, (out_f32, None, None)
    elif isinstance(out, Tri):
        mode, op = (5 if pool else 4), (out.h, out.l, out.c)
        out.exp = int(out_exp)
    else:
        mode, op = (2 if pool else 0), (out[0], out[1], None)
    stride = out_pix_stride if out_pix_stride is not None else cout
    if timer is not None:
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    args = (c_int(int(tri_in)), ptr(ap[0]), ptr(ap[1]), ptr(ap[2]), c_int(batch),
            c_int(H), c_int(W), c_int(cin), ptr(wp[0]), ptr(wp[1]), ptr(wp[2]),
            c_int(cout), c_int(taps), ptr(bias), c_int(int(relu)), c_int(mode),
            ptr(op[0]), ptr(op[1]), ptr(op[2]), c_ll(stride), c_int(out_ch_offset),
            c_int(split_k), c_ll(split_stride), c_int(bn), c_int(max_ctas),
            ctypes.c_float(acc_scale), ctypes.c_float(2.0 ** out_exp), ptr(amax))
    if img_hw is None:
        check(lib.mnc_igemm_tc2(*args, cur_stream()), "mnc_igemm_tc2")
    else:
        check(lib.mnc_igemm_tc3(*args, ptr(img_hw_arg(img_hw, batch)), c_int(level), cur_stream()),
              "mnc_igemm_tc3")
    if timer is not None:
        ev1.record()
        timer.records.append((ev0, ev1, 2.0 * batch * H * W * cout * taps * cin,
                              "%dx%dx%d" % (batch * H * W, cout, taps * cin)))
        m_out = batch * ((H + 1) // 2) * ((W + 1) // 2) if pool else batch * H * W
        timer.manifest.append(dict(
            M=batch * H * W, N=cout, K=taps * cin, taps=taps, bn=bn, split_k=split_k,
            pooled=bool(pool), fp32_out=out_f32 is not None, tri_in=tri_in,
            flops=2.0 * batch * H * W * cout * taps * cin,
            bytes=4.0 * (batch * H * W * cin + cout * taps * cin + m_out * cout * max(split_k, 1))))



def img_hw_arg(img_hw, batch):
    """Per-image sizes of a mixed-size batch as the kernels read them: a contiguous device int32
    (batch, 2) tensor (shape and type are checked here; the values are the caller's to validate,
    engine.check_extents)."""
    if not (img_hw.is_cuda and img_hw.dtype == torch.int32 and img_hw.is_contiguous()
            and tuple(img_hw.shape) == (batch, 2)):
        raise ValueError("img_hw must be a contiguous device int32 tensor of shape (%d, 2)" % batch)
    return img_hw


class KernelTimer:
    """Optional per-launch CUDA-event timing of the implicit-GEMM kernel (bench.py's roofline):
    events are recorded on the launching stream around every igemm launch, together with the
    launch's algorithmic FLOPs (2*M*N*K on the real, unpadded dims)."""

    def __init__(self):
        self.records = []   # (start_event, end_event, flops, tag)
        self.manifest = []  # one dict per launch: shape, algorithmic FLOPs and bytes

    def totals(self):
        ms = sum(s.elapsed_time(e) for s, e, _, _ in self.records)
        return ms, sum(f for _, _, f, _ in self.records), len(self.records)


timer = None  # set to a KernelTimer to enable


def igemm(a, batch, H, W, cin, w, cout, taps, bias=None, relu=False, out=None, out_f32=None,
          out_pix_stride=None, out_ch_offset=0, split_k=1, split_stride=0, bn=0, max_ctas=0,
          impl="tc", pool=False):
    """a: split [2, batch, H, W, cin]; w: split [2, cout, taps*cin].
    Writes split `out` ([2, ..., stride]) or fp32 `out_f32`."""
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16
    if out_f32 is not None:
        mode, o0, o1 = 1, out_f32, None
        stride = out_pix_stride if out_pix_stride is not None else cout
    else:
        mode, o0, o1 = (2 if pool else 0), out[0], out[1]
        stride = out_pix_stride if out_pix_stride is not None else cout
    if timer is not None and impl == "tc":
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    if impl == "tc":
        rc = lib.mnc_igemm_tc(ptr(a[0]), ptr(a[1]), c_int(batch), c_int(H), c_int(W), c_int(cin),
                              ptr(w[0]), ptr(w[1]), c_int(cout), c_int(taps), ptr(bias),
                              c_int(int(relu)), c_int(mode), ptr(o0), ptr(o1), c_ll(stride),
                              c_int(out_ch_offset), c_int(split_k), c_ll(split_stride), c_int(bn),
                              c_int(max_ctas), cur_stream())
        check(rc, "mnc_igemm_tc")
        if timer is not None:
            ev1.record()
            timer.records.append((ev0, ev1, 2.0 * batch * H * W * cout * taps * cin,
                                  "%dx%dx%d" % (batch * H * W, cout, taps * cin)))
            # algorithmic bytes: activations in once (split bf16 = 4 B/elt), weights in once,
            # result out once (split bf16 or fp32 = 4 B/elt; pooled outputs are a quarter;
            # split-K partials are counted as written, their reduce is a separate kernel)
            m_out = batch * ((H + 1) // 2) * ((W + 1) // 2) if pool else batch * H * W
            timer.manifest.append(dict(
                M=batch * H * W, N=cout, K=taps * cin, taps=taps, bn=bn, split_k=split_k,
                pooled=bool(pool), fp32_out=out_f32 is not None,
                flops=2.0 * batch * H * W * cout * taps * cin,
                bytes=4.0 * (batch * H * W * cin + cout * taps * cin + m_out * cout * max(split_k, 1))))
    else:
        assert split_k == 1
        rc = lib.mnc_igemm_simt(ptr(a[0]), ptr(a[1]), c_int(batch), c_int(H), c_int(W),
                                c_int(cin), ptr(w[0]), ptr(w[1]), c_int(cout), c_int(taps),
                                ptr(bias), c_int(int(relu)), c_int(mode), ptr(o0), ptr(o1),
                                c_ll(stride), c_int(out_ch_offset), cur_stream())
        check(rc, "mnc_igemm_simt")


cluster_size = 2      # CTAs per work item of igemm_tc_kernel (tracked for the engine's split-K model)


def set_cluster(cl):
    """Thread-block-cluster size of the tensor-core launches (1 or 2, default 2)."""
    global cluster_size
    check(lib.mnc_igemm_set_cluster(c_int(cl)), "mnc_igemm_set_cluster")
    cluster_size = cl


def set_tma_store(on):
    """A/B and test switch: out_mode 0 epilogues through shared memory + TMA store (default on)
    or direct per-thread stores."""
    check(lib.mnc_igemm_set_tma_store(c_int(int(on))), "mnc_igemm_set_tma_store")


def set_halo_pair(on):
    """A/B: CTA pairs in the halo kernel's precision mode 1 (default on)."""
    check(lib.mnc_igemm_set_halo_pair(c_int(int(on))), "mnc_igemm_set_halo_pair")


def set_block_k(bk):
    """K elements per pipeline stage of the tensor-core launches: 64, 32 or 0 (= per-shape default)."""
    check(lib.mnc_igemm_set_block_k(c_int(bk)), "mnc_igemm_set_block_k")


def splitk_reduce(partial, splits, split_stride, rows, cols, bias=None, relu=False, out=None,
                  out_f32=None, out_row_stride=None, out_ch_offset=0, img_hw=None, level=0,
                  map_hw=None):
    """img_hw / level / map_hw = (H, W): the rows are the pixels of a conv launch over a
    (batch, H, W) map of a mixed-size batch; rows outside their image come out as zeros."""
    if out_f32 is not None:
        mode, o0, o1 = 1, out_f32, None
    else:
        mode, o0, o1 = 0, out[0], out[1]
    stride = out_row_stride if out_row_stride is not None else cols
    args = (ptr(partial), c_int(splits), c_ll(split_stride), c_ll(rows), c_int(cols), ptr(bias),
            c_int(int(relu)), c_int(mode), ptr(o0), ptr(o1), c_ll(stride), c_int(out_ch_offset))
    if img_hw is None:
        check(lib.mnc_splitk_reduce(*args, cur_stream()), "mnc_splitk_reduce")
    else:
        H, W = map_hw
        check(lib.mnc_splitk_reduce2(*args, ptr(img_hw_arg(img_hw, rows // (H * W))), c_int(level), c_int(H),
                                     c_int(W), cur_stream()), "mnc_splitk_reduce2")


def conv1_1(data, weight, bias, out):
    b, c, H, W = data.shape
    assert c == 3 and data.dtype == torch.float32
    rc = lib.mnc_conv1_1(ptr(data), c_int(b), c_int(H), c_int(W), ptr(weight), ptr(bias),
                         c_int(weight.shape[0]), ptr(out[0]), ptr(out[1]), cur_stream())
    check(rc, "mnc_conv1_1")


def conv1_1_weight_to_tc(weight):
    """fp32 [64,3,3,3] -> bf16 [128,32]: hi plane rows 0..63, lo plane rows 64..127, K padded 27->32."""
    assert tuple(weight.shape) == (64, 3, 3, 3)
    w = torch.zeros((64, 32), dtype=torch.float32, device=weight.device)
    w[:, :27] = weight.reshape(64, 27)
    sp = split(w)                      # [2, 64, 32]
    return sp.reshape(128, 32).contiguous()


def conv1_1_tc(data, w_stacked, bias, out, out_exp=0, amax=None, img_hw=None):
    """out: split bf16 [2, B, H, W, 64] or Tri (written with exponent out_exp).  img_hw: image
    sizes of a mixed-size batch (device int32 (B, 2)); outputs outside an image are zeros."""
    b, c, H, W = data.shape
    assert c == 3 and data.dtype == torch.float32 and data.is_contiguous()
    assert w_stacked.dtype == torch.bfloat16 and tuple(w_stacked.shape) == (128, 32)
    if isinstance(out, Tri):
        out.exp = int(out_exp)
        mode, op = 4, (out.h, out.l, out.c)
    else:
        mode, op = 0, (out[0], out[1], None)
    args = (ptr(data), c_int(b), c_int(H), c_int(W), ptr(w_stacked), ptr(bias), c_int(mode),
            ptr(op[0]), ptr(op[1]), ptr(op[2]), ctypes.c_float(2.0 ** out_exp), ptr(amax))
    if img_hw is None:
        check(lib.mnc_conv1_1_tc2(*args, cur_stream()), "mnc_conv1_1_tc2")
    else:
        check(lib.mnc_conv1_1_tc3(*args, ptr(img_hw_arg(img_hw, b)), cur_stream()), "mnc_conv1_1_tc3")


def maxpool2x2(a, batch, H, W, C, out):
    rc = lib.mnc_maxpool2x2_split(ptr(a[0]), ptr(a[1]), c_int(batch), c_int(H), c_int(W), c_int(C),
                                  ptr(out[0]), ptr(out[1]), cur_stream())
    check(rc, "mnc_maxpool2x2_split")


def split_to_nchw(a, batch, H, W, C, out):
    if isinstance(a, Tri):     # blob read-back path (not hot): torch does the layout change
        out.copy_(a.float().view(batch, H, W, C).permute(0, 3, 1, 2))
        return
    rc = lib.mnc_split_to_nchw(ptr(a[0]), ptr(a[1]), c_int(batch), c_int(H), c_int(W), c_int(C),
                               ptr(out), cur_stream())
    check(rc, "mnc_split_to_nchw")


def nchw_to_split(x, out):
    b, C, H, W = x.shape
    rc = lib.mnc_nchw_to_split(ptr(x), c_int(b), c_int(C), c_int(H), c_int(W), ptr(out[0]),
                               ptr(out[1]), cur_stream())
    check(rc, "mnc_nchw_to_split")


def split_to_f32(a, out):
    """out (fp32, same element order) = hi + lo (split bf16) or (h + l / 2^6) * 2^-exp (Tri)."""
    n = out.numel()
    if isinstance(a, Tri):
        rc = lib.mnc_tri_to_f32(ptr(a.h), ptr(a.l), c_ll(n), ctypes.c_float(2.0 ** -a.exp), ptr(out),
                                cur_stream())
        check(rc, "mnc_tri_to_f32")
        return
    rc = lib.mnc_split_to_f32(ptr(a[0]), ptr(a[1]), c_ll(n), ptr(out), cur_stream())
    check(rc, "mnc_split_to_f32")


def f32_to_tri(x, out, exp, amax=None):
    """Device conversion fp32 -> Tri `out` (same element order) with exponent exp."""
    out.exp = int(exp)
    rc = lib.mnc_f32_to_tri(ptr(x), c_ll(x.numel()), ctypes.c_float(2.0 ** exp), ptr(out.h), ptr(out.l),
                            ptr(out.c), ptr(amax), cur_stream())
    check(rc, "mnc_f32_to_tri")


def splitk_reduce_tri(partial, splits, split_stride, rows, cols, out, out_exp, bias=None, relu=False,
                      out_row_stride=None, out_ch_offset=0, amax=None, img_hw=None, level=0,
                      map_hw=None):
    out.exp = int(out_exp)
    stride = out_row_stride if out_row_stride is not None else cols
    args = (ptr(partial), c_int(splits), c_ll(split_stride), c_ll(rows), c_int(cols), ptr(bias),
            c_int(int(relu)), ctypes.c_float(2.0 ** out_exp), ptr(out.h), ptr(out.l), ptr(out.c),
            c_ll(stride), c_int(out_ch_offset), ptr(amax))
    if img_hw is None:
        check(lib.mnc_splitk_reduce_tri(*args, cur_stream()), "mnc_splitk_reduce_tri")
    else:
        H, W = map_hw
        check(lib.mnc_splitk_reduce_tri2(*args, ptr(img_hw_arg(img_hw, rows // (H * W))), c_int(level),
                                         c_int(H), c_int(W), cur_stream()), "mnc_splitk_reduce_tri2")
