"""Batched MNC 5-stage inference engine (the hot path of BASELINE.json's north_star).

One `MNCEngine` per GPU: weights resident in HBM as split-bf16, activations NHWC split-bf16,
every layer of models/VGG16/mnc_5stage/test.prototxt executed by a kernel of libmnc_b200.so on
torch's current stream, no host round trips inside `forward` (the reference crosses D<->H four
times per image for its Python layers: SURVEY.md section 3.2).  The reference is batch-1
(lib/pylayer/proposal_layer.py:65); here images are batched by looping the proposal stage per
image on device and stacking RoIs with their batch index (ROIWarping honours roi[0],
roi_warping_layer.cu:79,96), so the FC weights stream from HBM once per batch.

PyTorch's role: device memory and streams (a step is ~60 asynchronous launches queued in 1.2 ms
of host time against 15 ms of device time, so no CUDA graph is needed to keep the GPU busy).  Apart
from a few `torch.cat` / copies in the `detect` tail, no torch op computes on the path.
"""
import math

import torch

from . import dense, ops
from .weights import TRUNK_NAMES, POOL_AFTER, arch_of

ROIS_PER_IMAGE = 300   # cfg.TEST.RPN_POST_NMS_TOP_N (lib/mnc_config.py:130)
PRE_NMS_TOP_N = 6000   # cfg.TEST.RPN_PRE_NMS_TOP_N (:128)
RPN_NMS_THRESH = 0.7   # cfg.TEST.RPN_NMS_THRESH (:126)
RPN_MIN_SIZE = 16.0    # cfg.TEST.RPN_MIN_SIZE (:132)
MASK_SIZE = 21         # cfg.MASK_SIZE (:28)
NUM_CLASSES = 21


def _ceil_half(x):
    return (x + 1) // 2


HALO_MAX_COUT = 128    # 3x3 convs with Cout <= 128 run the halo kernel
C5_LEVEL = 4           # conv5_x, the RPN and the RoI features sit four 2x2 pools below the input

# Largest max |value| * 2^exp a tri-plane tensor may reach before its exponent counts as stale.
# Calibration puts the maximum in (2^11, 2^12].  fp16 itself saturates only at 65504, but the e4m3
# planes give out much earlier: the residual plane (x 2^6) clamps at 448 once the fp16 rounding
# step exceeds 16 (values above 2^15), the copy plane (x 2^-5) above 14336, and the layer then
# degrades toward plain fp16 (2e-4 per layer).  Up to 2^14 every layer kind stays within 1e-4 of
# fp64 (tests/test_tri_headroom.py, tests/test_gpu_tri_path.py::test_headroom_contract).
RANGE_MAX = 2.0 ** 14


def in_range(amax, exp):
    """Is a tensor whose max |value| is `amax` still carried accurately with exponent `exp`?"""
    return amax * 2.0 ** exp <= RANGE_MAX


def level_extent(n, level):
    """Rows (or columns) that an image of n input rows covers `level` 2x2 ceil-mode pools deeper:
    ceil(n / 2^level), Caffe's chain of ceil-mode halvings (pooling_layer.cpp:90-93)."""
    return (n + (1 << level) - 1) >> level


def check_extents(extents, H, W, max_batch=None):
    """Host validation of the per-image sizes of a mixed-size batch: an int (B, 2) array of
    (rows, cols) at input resolution, each >= 1 and within the (H, W) blob.  Returns it as a
    contiguous int32 CPU tensor.  Raises ValueError (nothing has been launched)."""
    import numpy as np
    e = np.asarray(extents.cpu() if isinstance(extents, torch.Tensor) else extents)
    if e.ndim != 2 or e.shape[1] != 2 or e.shape[0] < 1:
        raise ValueError("extents must have shape (B, 2), got %s" % (e.shape,))
    if max_batch is not None and e.shape[0] > max_batch:
        raise ValueError("%d images in one batch, at most %d" % (e.shape[0], max_batch))
    if not np.issubdtype(e.dtype, np.integer):
        raise ValueError("extents must be integers")
    if (e < 1).any():
        raise ValueError("every image extent must be at least 1 pixel: %s" % e.tolist())
    if (e[:, 0] > H).any() or (e[:, 1] > W).any():
        raise ValueError("image extents %s exceed the %dx%d blob" % (e.tolist(), H, W))
    return torch.from_numpy(np.ascontiguousarray(e, dtype=np.int32))


def pick_split_k(tiles_m, tiles_n, k_steps, sms, cluster=2, max_split=32, out_elems=0):
    """Split-K only when the launch cannot fill the GPU (e.g. fc6_maskest: 19 row tiles,
    K = 100352; every FC at batch 1).  A wave-quantisation-driven split (608 tiles -> 4.1 waves)
    was measured and rejected: the extra fp32 partial reduce costs what the shorter tail saves
    (profiles/README.md).  When splitting, the factor minimises waves x k-steps-per-item, counted
    the way the kernel schedules: a work item is a CTA PAIR (two adjacent 128-row tiles x one
    Cout tile x one split) and there are sms/2 of them in flight (igemm_tc.cu launch_igemm).
    (Counting single tiles against 148 SMs picked 15 splits for fc6_maskest = 150 items = three
    waves of 74, the last with 2 items; and 2 splits for fc6 at batch 1 = 88 items = two waves,
    i.e. no gain at all.)  Cost unit: one k-step of a pair item (~0.45 us); each split adds a
    launch-side constant and one fp32 copy of the output to write and re-read (M*N*8 B at ~5 TB/s)."""
    slots = max(1, sms // cluster)
    items = math.ceil(tiles_m / cluster) * tiles_n
    if items >= slots * 0.7 or k_steps < 16:
        return 1
    per_split = 0.5 + out_elems * 1.7e-6
    best, best_cost = 1, None
    for s in range(1, min(max_split, max(1, k_steps // 8)) + 1):
        waves = math.ceil(items * s / slots)
        cost = waves * math.ceil(k_steps / s) + per_split * s
        if best_cost is None or cost < best_cost:
            best, best_cost = s, cost
    return best


class MNCEngine:
    # "f16f8": precision mode 1 on every launch of the per-tap / inner-product kernel -- tri-plane
    # operands, fp16 main product + two FP8 correction products (2 tensor-work units per MAC);
    # "bf16x3": split-bf16 operands everywhere (3 units per MAC).  The halo kernel (Cout <= 128)
    # has both modes as well (HALO_TRI False keeps it on split-bf16 operands under "f16f8");
    # conv1_1 (K = 27) computes in split bf16 in both and writes the format its consumer reads.
    DEFAULT_PRECISION = "f16f8"
    HALO_TRI = True

    def __init__(self, weights, device="cuda", impl="tc", sm_count=None, precision=None):
        """weights: {caffe name: (weight, bias)} fp32 tensors in Caffe layouts (see weights.py)."""
        self.device = torch.device(device)
        self.impl = impl
        self.precision = (precision or self.DEFAULT_PRECISION) if impl == "tc" else "bf16x3"
        self.tri = self.precision == "f16f8"
        self.halo_tri = self.HALO_TRI
        self.fuse_pool = True
        # per-tensor exponents of the tri-plane activations, measured on the first forward
        self.exp = {}
        self._calibrating = False
        self._calibrated = not self.tri
        self.arch = arch_of(weights)
        self.sms = sm_count or torch.cuda.get_device_properties(self.device).multi_processor_count
        dev = self.device
        self.c5 = self.arch["trunk"][-1]
        self.fc = self.arch["fc"]
        self.me = self.arch["maskest"]
        w = {k: (v[0].to(dev).float().contiguous(), v[1].to(dev).float().contiguous())
             for k, v in weights.items()}
        # conv1_1 stays fp32 (SIMT kernel); the other convs are split [2, Cout, 9*Cin]
        self.conv1_1 = w["conv1_1"]
        # 64-channel conv1_1 runs on the tensor cores (stacked hi/lo weight tile, K padded to 32)
        self.conv1_1_tc = (dense.conv1_1_weight_to_tc(w["conv1_1"][0])
                           if impl == "tc" and w["conv1_1"][0].shape[0] == 64 else None)
        if self.conv1_1_tc is None:
            self.halo_tri = False      # only the tensor-core conv1_1 writes tri-plane output
        self.convs = []
        for name in TRUNK_NAMES[1:] + ["rpn_conv_3x3"]:
            if name in w:   # the CFM test net has no RPN (proposals are an input)
                tri = self._conv_in_tri(w[name][0].shape[0])
                cw = dense.conv_weight_to_tri(w[name][0]) if tri else dense.conv_weight_to_split(w[name][0])
                self.convs.append((name, cw, w[name][1]))
        self.trunk_convs = [c for c in self.convs if c[0] != "rpn_conv_3x3"]
        if "rpn_conv_3x3" in w:
            r = self.arch["rpn"]
            rpn_w = torch.cat([w["rpn_cls_score"][0].reshape(18, r), w["rpn_bbox_pred"][0].reshape(36, r)])
            self.rpn_head = (self._fc_w(rpn_w), torch.cat([w["rpn_cls_score"][1], w["rpn_bbox_pred"][1]]).contiguous())
        c5 = self.c5
        self.fc6 = (self._fc_w(w["fc6"][0], (c5, 7, 7)), w["fc6"][1])
        self.fc7 = (self._fc_w(w["fc7"][0]), w["fc7"][1])
        if "fc6_maskest" in w:
            self.fc6_maskest = (self._fc_w(w["fc6_maskest"][0], (c5, 14, 14)), w["fc6_maskest"][1])
            self.mask_pred = (self._fc_w(w["mask_pred"][0]), w["mask_pred"][1])
            self.fc6_mask = (self._fc_w(w["fc6_mask"][0], (c5, 7, 7)), w["fc6_mask"][1])
            self.fc7_mask = (self._fc_w(w["fc7_mask"][0]), w["fc7_mask"][1])
        # cls_score | seg_cls_score | bbox_pred share their input: one inner product for all of them
        names = [n for n in ("cls_score", "seg_cls_score", "bbox_pred") if n in w]
        self.cls_head_names = names
        cls_w = torch.cat([w[n][0] for n in names])
        cls_b = torch.cat([w[n][1] for n in names])
        self.cls_heads = (self._fc_w(cls_w), cls_b.contiguous())
        self._buf = {}
        self._amax = torch.zeros(2, dtype=torch.int32, device=dev)
        # running max |value| of every tri-plane activation tensor (float bits, one slot per exponent
        # key): written by the producing kernels on every call, read by range_ok()
        self._amax_all = torch.zeros(128, dtype=torch.int32, device=dev)
        self._amax_slot = {}
        self.range_violations = 0      # how often range_ok() found a stale exponent
        # the box branch (fc6 on the 7x7 features: tensor-bound) is issued on a side stream so that
        # the mask branch's small / HBM-bound kernels (mask_pred, sigmoid + resize, MaskPooling) run
        # under it instead of in front of it; in a captured graph the fork becomes parallel branches
        self.overlap_heads = True
        self._side = None

    def clone_state(self):
        """A second engine over the SAME weights and exponents with its own activation buffers,
        scratch, range-monitor slots, side stream and CUDA graphs: lets two steps be in flight on
        two streams (the second step's kernels fill the first one's wave tails and its
        low-occupancy proposal phase).  Clone after the first forward (the clone inherits the
        calibration; both share the exponent dictionary)."""
        import copy
        e = copy.copy(self)
        e._buf = {}
        e._amax = torch.zeros_like(self._amax)
        e._amax_all = torch.zeros_like(self._amax_all)
        e._side = None
        e._graphs = {}
        return e

    def _fc_w(self, w, chw=None):
        return dense.fc_weight_to_tri(w, chw) if self.tri else dense.fc_weight_to_split(w, chw)

    # ------------------------------------------------------------------ helpers
    def _drop_graphs(self, old):
        """Buffer `old` is being replaced by a larger one (a bigger blob or batch than any so far):
        graphs captured over it would replay into freed memory, so they go (after the work queued
        on them has finished)."""
        graphs = getattr(self, "_graphs", None)
        if old is None or not graphs:
            return
        if not torch.cuda.is_current_stream_capturing():
            torch.cuda.synchronize(self.device)
        graphs.clear()

    def _split_buf(self, key, *shape):
        t = self._buf.get(key)
        need = 1
        for s in shape:
            need *= s
        if t is None or t.numel() < 2 * need:
            self._drop_graphs(t)
            t = torch.empty(2 * need, dtype=torch.bfloat16, device=self.device)
            self._buf[key] = t
        return t[:2 * need].view(2, *shape)

    def _act_buf(self, key, *shape, tri=None, exp_key=None):
        """Activation buffer in the format its consumer wants: split bf16 [2, *shape] or Tri."""
        if not (self.tri if tri is None else tri):
            return self._split_buf(key, *shape)
        need = 1
        for s_ in shape:
            need *= s_
        t = self._buf.get("tri_" + key)
        if t is None or t.numel() < 4 * need:
            self._drop_graphs(t)
            t = torch.empty(4 * need, dtype=torch.uint8, device=self.device)
            self._buf["tri_" + key] = t
        return dense.Tri(t[:2 * need].view(torch.float16).view(*shape), t[2 * need:3 * need].view(*shape),
                         t[3 * need:4 * need].view(*shape), self.exp.get(exp_key or key, 0))

    def _scaled(self, exp_key, fn):
        """Run fn(out_exp, amax) -- the launch(es) that write the tri-plane tensor `exp_key`.  Normal
        operation: the frozen exponent.  Calibration (first forward): launch, read the measured
        max |value|, choose the exponent that puts it at 2^12 (4x headroom to RANGE_MAX, where the
        e4m3 correction planes start to saturate), relaunch if it changed."""
        if not self._calibrating:
            slot = self._amax_slot.setdefault(exp_key, len(self._amax_slot))
            fn(self.exp[exp_key], self._amax_all[slot:slot + 1] if slot < 128 else None)
            return
        slot = self._amax[:1]
        slot.zero_()
        e0 = self.exp.get(exp_key, 0)
        fn(e0, slot)
        amax = float(slot.view(torch.float32).item())
        e = dense.exp_for(amax, 12) if amax > 0 else e0
        self.exp[exp_key] = e
        if e != e0:
            fn(e, None)

    def range_ok(self, reset=True, amax=None, exp=None):
        """Were the exponents still adequate for everything computed since the last check?  A
        tensor whose maximum left the accurate range of its exponent (`in_range`) makes this return
        False and un-calibrates the engine: the next forward measures the exponents again (and
        graphs are re-captured).  amax: a host copy of `_amax_all` taken after the step (default:
        one small D2H read now); exp: the exponents the step ran with (default: the current ones)."""
        if not self.tri or not self._amax_slot:
            return True
        amax = (self._amax_all.cpu() if amax is None else amax).view(torch.float32)
        exp = self.exp if exp is None else exp
        bad = [k for k, i in self._amax_slot.items()
               if i < 128 and not in_range(float(amax[i]), exp.get(k, 0))]
        if reset:
            self._amax_all.zero_()
        if bad:
            self.range_violations += 1
            self._calibrated = False
            if hasattr(self, "_graphs"):
                self._graphs.clear()
            self.last_range_violation = bad
            return False
        return True

    def run_checked(self, step, *args, **kwargs):
        """step(*args, **kwargs) -- this engine's forward, detect or detect_graphed -- followed by
        the range check (one host sync); a batch whose activations outgrew the frozen exponents is
        computed again with exponents measured on it.  Returns what the last step returned."""
        out = step(*args, **kwargs)
        if not self.range_ok():
            out = step(*args, **kwargs)
        return out

    def forward_checked(self, data, im_info, keep_intermediate=False, extents=None):
        """`forward` with the per-call range check of `run_checked`."""
        return self.run_checked(self.forward, data, im_info, keep_intermediate, extents=extents)

    def detect_checked(self, data, im_info, im_hw, im_scale, extents=None):
        """`detect` with the per-call range check of `run_checked`."""
        return self.run_checked(self.detect, data, im_info, im_hw, im_scale, extents=extents)

    def _extents(self, data, extents):
        """The device int32 (B, 2) image sizes of a mixed-size batch (None: every image fills the
        blob).  A host array is validated (check_extents) and uploaded; a device tensor is taken
        as is -- checking its values would cost a host sync, so a caller passing device extents
        must have validated them (the kernels clamp them to the map, but invalid sizes give wrong
        results)."""
        if extents is None:
            return None
        if self.impl != "tc" or not self.fuse_pool or self.conv1_1_tc is None:
            raise NotImplementedError("mixed-size batches run on the tensor-core path with fused "
                                      "pools and the tensor-core conv1_1 only")
        B, _, H, W = data.shape
        if not (isinstance(extents, torch.Tensor) and extents.is_cuda):
            extents = check_extents(extents, H, W).to(self.device, non_blocking=True)
        if extents.dtype != torch.int32 or tuple(extents.shape) != (B, 2):
            raise ValueError("extents must be int32 of shape (%d, 2)" % B)
        return extents.contiguous()

    def _f32_buf(self, key, *shape):
        t = self._buf.get(key)
        need = 1
        for s in shape:
            need *= s
        if t is None or t.numel() < need:
            self._drop_graphs(t)
            t = torch.empty(need, dtype=torch.float32, device=self.device)
            self._buf[key] = t
        return t[:need].view(*shape)

    def _linear(self, a, M, K, wgt, N, bias, relu, out=None, out_f32=None, out_stride=None,
                out_ch_offset=0, key="lin", block_k=0, bn=0, exp_key=None):
        """y = act(a @ W^T + b) through the implicit-GEMM kernel; split-K when the tile count
        cannot fill the GPU (e.g. fc6_maskest: K = 100352, N = 256).  a / wgt / out: split-bf16
        tensors or dense.Tri (out written with the exponent of `exp_key`)."""
        tri_in = isinstance(a, dense.Tri)
        # Cout tile: 192 for the wide layers -- at M = 2400, N = 4096 it gives 19 x 22 = 418 tiles
        # (220 CTA-pair items = 2.97 waves of 74 pairs), against 2.16 (-> 3) waves at 256
        bn = bn or (64 if N <= 64 else (128 if N <= 128 else (192 if N >= 1024 else 256)))
        k_steps = K // 64
        split = (self._pick_split(math.ceil(M / 128), math.ceil(N / bn), k_steps, out_elems=M * N)
                 if self.impl == "tc" else 1)
        a4 = a.view(1, 1, M, K) if tri_in else a.view(2, 1, 1, M, K)
        tri_out = isinstance(out, dense.Tri)
        ek = exp_key or key
        if split == 1:
            if self.impl != "tc":
                dense.igemm(a4, 1, 1, M, K, wgt, N, 1, bias=bias, relu=relu, out=out, out_f32=out_f32,
                            out_pix_stride=out_stride, out_ch_offset=out_ch_offset, bn=bn, impl=self.impl)
                return

            def run(e, amax):
                dense.igemm2(a4, 1, 1, M, K, wgt, N, 1, bias=bias, relu=relu, out=out, out_f32=out_f32,
                             out_pix_stride=out_stride, out_ch_offset=out_ch_offset, bn=bn,
                             out_exp=e, amax=amax)
            if tri_out:
                self._scaled(ek, run)
            else:
                run(0, None)
            return
        part = self._f32_buf("splitk_" + key, split, M, N)
        if block_k and not tri_in:
            dense.set_block_k(block_k)
        try:
            dense.igemm2(a4, 1, 1, M, K, wgt, N, 1, out_f32=part, split_k=split, split_stride=M * N, bn=bn)
        finally:
            if block_k and not tri_in:
                dense.set_block_k(0)
        if tri_out:
            self._scaled(ek, lambda e, amax: dense.splitk_reduce_tri(
                part, split, M * N, M, N, out, e, bias=bias, relu=relu, out_row_stride=out_stride,
                out_ch_offset=out_ch_offset, amax=amax))
        else:
            dense.splitk_reduce(part, split, M * N, M, N, bias=bias, relu=relu, out=out,
                                out_f32=out_f32, out_row_stride=out_stride, out_ch_offset=out_ch_offset)

    def _pick_split(self, tiles_m, tiles_n, k_steps, max_split=32, out_elems=0):
        """Split-K factor of one tensor-core launch: see pick_split_k."""
        return pick_split_k(tiles_m, tiles_n, k_steps, self.sms, dense.cluster_size, max_split, out_elems)

    def _conv(self, x, B, H, W, cin, wgt, cout, bias, out, key, pool=False, ext=None, level=0):
        """3x3 conv + bias + ReLU (+ fused 2x2 ceil-mode max pool) -> `out` (split-bf16 or Tri),
        split-K when whole waves would idle.  ext / level: image sizes of a mixed-size batch and
        the input's depth in pools (pixels outside an image come out as zeros)."""
        if self.impl != "tc":
            dense.igemm(x, B, H, W, cin, wgt, cout, 9, bias=bias, relu=True, out=out, impl=self.impl)
            return
        bn = 64 if cout <= 64 else (128 if cout <= 128 else 256)
        split = 1 if pool else self._pick_split(B * math.ceil(H / 8) * math.ceil(W / 16),
                                                math.ceil(cout / bn), 9 * cin // 64, max_split=4,
                                                out_elems=B * H * W * cout)
        tri_out = isinstance(out, dense.Tri)
        if split == 1:
            def run(e, amax):
                dense.igemm2(x, B, H, W, cin, wgt, cout, 9, bias=bias, relu=True, out=out, pool=pool,
                             out_exp=e, amax=amax, img_hw=ext, level=level)
            if tri_out:
                self._scaled(key, run)
            else:
                run(0, None)
            return
        M = B * H * W
        part = self._f32_buf("splitk_conv", split, M, cout)
        dense.igemm2(x, B, H, W, cin, wgt, cout, 9, out_f32=part, split_k=split, split_stride=M * cout)
        if tri_out:
            self._scaled(key, lambda e, amax: dense.splitk_reduce_tri(
                part, split, M * cout, M, cout, out, e, bias=bias, relu=True, amax=amax,
                img_hw=ext, level=level, map_hw=(H, W)))
        else:
            dense.splitk_reduce(part, split, M * cout, M, cout, bias=bias, relu=True, out=out,
                                img_hw=ext, level=level, map_hw=(H, W))

    # ------------------------------------------------------------------ trunk
    def _conv_in_tri(self, cout):
        """Does the conv with `cout` output channels read tri-plane operands?"""
        return self.tri and (cout > HALO_MAX_COUT or self.halo_tri)

    def trunk(self, data, extents=None):
        """conv1_1 .. conv5_3 (test.prototxt:19-387).  data fp32 (B,3,H,W) -> NHWC conv5_3 in the
        format its consumers read (split bf16, or Tri when rpn_conv_3x3 takes tri-plane operands).
        extents: device int32 (B, 2) image sizes of a mixed-size batch (zero-padded blob); every
        layer's output is then zero outside each image, as if it had run on that image alone."""
        B, _, H, W = data.shape
        ext = self._extents(data, extents)
        level = 0
        ch = self.arch["trunk"]
        big = B * H * W * max(ch[0], ch[1])
        cur = 0
        names = [c[0] for c in self.trunk_convs]
        couts = [c[1].shape[-2] for c in self.trunk_convs]

        # the two ping-pong buffers are raw bytes: 4 per element in either format
        self._act_buf("act0", big, tri=False)
        self._act_buf("act1", big, tri=False)
        first_next = couts[0] if couts else 0
        x = self._pp_buf(cur, self._conv_in_tri(first_next), "conv1_1", B, H, W, ch[0])
        if isinstance(x, dense.Tri):
            d = data.contiguous()
            self._scaled("conv1_1", lambda e, amax: dense.conv1_1_tc(
                d, self.conv1_1_tc, self.conv1_1[1], x, out_exp=e, amax=amax, img_hw=ext))
        elif self.conv1_1_tc is not None:
            dense.conv1_1_tc(data.contiguous(), self.conv1_1_tc, self.conv1_1[1], x, img_hw=ext)
        else:
            dense.conv1_1(data, self.conv1_1[0], self.conv1_1[1], x)
        cin = ch[0]
        if "conv1_1" in POOL_AFTER:
            raise NotImplementedError
        for li, (name, wgt, bias) in enumerate(self.trunk_convs):
            cout = couts[li]
            nxt = 1 - cur
            pool_here = name in POOL_AFTER
            fuse = pool_here and self.impl == "tc" and self.fuse_pool
            Ho, Wo = (_ceil_half(H), _ceil_half(W)) if pool_here else (H, W)
            # the consumer of this layer's output decides its format
            if name == "conv5_3":
                nxt_tri = self._conv_in_tri(self.arch["rpn"]) if self.arch["rpn"] else False
            else:
                nxt_tri = self._conv_in_tri(couts[li + 1])
            if fuse or not pool_here:
                if name == "conv5_3":
                    y = self._act_buf("conv5_3", B, Ho, Wo, cout, tri=nxt_tri, exp_key="conv5_3")
                else:
                    y = self._pp_buf(nxt, nxt_tri, name, B, Ho, Wo, cout)
                self._conv(x, B, H, W, cin, wgt, cout, bias, y, name, pool=fuse, ext=ext, level=level)
                x, cur, cin, H, W = y, nxt, cout, Ho, Wo
                level += int(fuse)
                continue
            # un-fused pooling (SIMT cross-check path): split-bf16 only
            y = self._pp_buf(nxt, False, name, B, H, W, cout)
            self._conv(x, B, H, W, cin, wgt, cout, bias, y, name)
            x, cur, cin = y, nxt, cout
            nxt = 1 - cur
            y = self._pp_buf(nxt, False, name + "_pool", B, Ho, Wo, cout)
            dense.maxpool2x2(x, B, H, W, cout, y)
            x, cur, H, W = y, nxt, Ho, Wo
        return x, H, W

    def _pp_buf(self, slot, tri, exp_key, *shape):
        """View of ping-pong activation buffer `slot` (raw bytes, 4 per element) as split bf16 or Tri."""
        need = 1
        for s_ in shape:
            need *= s_
        raw = self._buf["act%d" % slot]          # bf16 tensor of 2 * big elements
        if not tri:
            return raw[:2 * need].view(2, *shape)
        b = raw.view(torch.uint8)
        return dense.Tri(b[:2 * need].view(torch.float16).view(*shape), b[2 * need:3 * need].view(*shape),
                         b[3 * need:4 * need].view(*shape), self.exp.get(exp_key, 0))

    # ------------------------------------------------------------------ one cascade stage head
    def head(self, feat14, box7, R, tag):
        """test.prototxt:509-785 on R RoIs.  feat14 [R,14,14,C5], box7 [R,7,7,C5] NHWC RoI features
        (split bf16 or Tri)."""
        c5, fc, me = self.c5, self.fc, self.me
        join = self._act_buf("join", R, 2 * fc, exp_key="join_" + tag)
        h6 = self._act_buf("h6", R, fc, exp_key="h6_box_" + tag)
        # (not worth a fork / join for a handful of RoIs: single-image latency is launch-count bound)
        fork = self.overlap_heads and not self._calibrating and R >= 4 * ROIS_PER_IMAGE
        h_me = self._act_buf("h_me", R, me, exp_key="h_me_" + tag)
        # fc6_maskest streams its 963 MB activation matrix from HBM exactly once (a single Cout
        # tile: no L2 reuse), so it wants loads in flight rather than big stages (split-bf16 mode:
        # BLOCK_K 32 gives a 4-deep ring at BN 256).  What remains (2.7 TB/s) is the DRAM efficiency
        # of 128-byte row segments 200 KB apart, the price of K-major rows with K = 100352.
        self._linear(feat14, R, 196 * c5, self.fc6_maskest[0], me, self.fc6_maskest[1], True,
                     out=h_me, key="me", block_k=32, exp_key="h_me_" + tag)
        logits = self._f32_buf("mask_logits_" + tag, R, 448)
        self._linear(h_me, R, me, self.mask_pred[0], 441, self.mask_pred[1], False,
                     out_f32=logits, out_stride=448, key="mp")
        box_done = None
        if fork:
            # fork behind mask_pred (a second persistent GEMM would only queue behind fc6's CTAs):
            # sigmoid + resize and MaskPooling then run UNDER the tensor-bound fc6
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.device)
            main = torch.cuda.current_stream(self.device)
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(self._side):
                self._side.wait_event(ev)
                # (own split-K scratch: this launch overlaps the mask branch's fc6_mask)
                self._linear(box7, R, 49 * c5, self.fc6[0], fc, self.fc6[1], True, out=h6, key="fc6_box",
                             exp_key="h6_box_" + tag)
                box_done = torch.cuda.Event()
                box_done.record(self._side)
        mask_proposal, mask14 = ops.sigmoid_mask_resize(logits, R, MASK_SIZE, 14)
        if not fork:
            self._linear(box7, R, 49 * c5, self.fc6[0], fc, self.fc6[1], True, out=h6, key="fc6_box",
                         exp_key="h6_box_" + tag)
        m7 = self._act_buf("m7", R, 7, 7, c5, exp_key="roi_feat")
        if isinstance(feat14, dense.Tri):
            ops.mask_pool_tri(feat14, mask14, R, c5, m7)
        else:
            ops.mask_pool_split(feat14, mask14, R, c5, m7)
        h6m = self._act_buf("h6m", R, fc, exp_key="h6_mask_" + tag)
        self._linear(m7, R, 49 * c5, self.fc6_mask[0], fc, self.fc6_mask[1], True, out=h6m, key="fc6",
                     exp_key="h6_mask_" + tag)
        if box_done is not None:
            torch.cuda.current_stream(self.device).wait_event(box_done)
        # Concat [fc7_mask | fc7] (test.prototxt:700-705): both halves of `join` share one exponent
        if isinstance(join, dense.Tri):
            def both(e, amax):
                for src, wb, off in ((h6, self.fc7, fc), (h6m, self.fc7_mask, 0)):
                    dense.igemm2(src.view(1, 1, R, fc), 1, 1, R, fc, wb[0], fc, 1, bias=wb[1], relu=True,
                                 out=join, out_pix_stride=2 * fc, out_ch_offset=off,
                                 bn=self._fc_bn(fc), out_exp=e, amax=amax)
            self._scaled("join_" + tag, both)
        else:
            self._linear(h6, R, fc, self.fc7[0], fc, self.fc7[1], True, out=join, out_stride=2 * fc,
                         out_ch_offset=fc, key="fc7")
            self._linear(h6m, R, fc, self.fc7_mask[0], fc, self.fc7_mask[1], True, out=join,
                         out_stride=2 * fc, out_ch_offset=0, key="fc7")
        heads = self._f32_buf("heads_" + tag, R, 128)
        self._linear(join, R, 2 * fc, self.cls_heads[0], 126, self.cls_heads[1], False,
                     out_f32=heads, out_stride=128, key="cls")
        cls_prob = ops.softmax_rows(heads[:, 0:21], 21)
        seg_cls_prob = ops.softmax_rows(heads[:, 21:42], 21)
        bbox_pred = heads[:, 42:126]
        return dict(mask_proposal=mask_proposal, mask_logits=logits, mask_resize=mask14,
                    cls_prob=cls_prob, seg_cls_prob=seg_cls_prob, bbox_pred=bbox_pred,
                    seg_cls_score=heads[:, 21:42], join=join)

    @staticmethod
    def _fc_bn(N):
        return 64 if N <= 64 else (128 if N <= 128 else (192 if N >= 1024 else 256))

    # ------------------------------------------------------------------ trunk + RPN + proposals
    def conv5_f32(self, conv5_3, B, H5, W5):
        """fp32 copy of conv5_3 (exact value of the stored planes) for the RoI gathers: 39 MB per
        batch of 8."""
        c5f = self._f32_buf("conv5_f32", B, H5, W5, self.c5)
        dense.split_to_f32(conv5_3, c5f)
        if self._calibrating:
            # RoI features are interpolations of conv5_3 (and their products with masks <= 1):
            # they take conv5_3's range
            amax = float(c5f.abs().max().item())
            self.exp["roi_feat"] = dense.exp_for(amax, 12) if amax > 0 else 0
        return c5f

    def rpn_rois(self, data, im_info, keep_intermediate=False, extents=None):
        """test.prototxt:19-476: trunk, rpn_conv_3x3, rpn_cls_score | rpn_bbox_pred, softmax,
        ProposalLayer.  -> conv5_3 (NHWC), H5, W5, fp32 conv5_3, rois (B*300,5), counts.
        extents: image sizes of a mixed-size batch (`trunk`); anchors outside an image take no
        part in its proposals."""
        B = data.shape[0]
        ext = self._extents(data, extents)
        conv5_3, H5, W5 = self.trunk(data, ext)
        c5, r = self.c5, self.arch["rpn"]
        name, wgt, bias = self.convs[-1]
        rpn = self._act_buf("rpn", B, H5, W5, r, exp_key="rpn")     # consumer: the 54-wide head
        self._conv(conv5_3, B, H5, W5, c5, wgt, r, bias, rpn, "rpn", ext=ext, level=C5_LEVEL)
        rpn_out = self._f32_buf("rpn_out", B, H5, W5, 64)
        self._linear(rpn, B * H5 * W5, r, self.rpn_head[0], 54, self.rpn_head[1], False,
                     out_f32=rpn_out, out_stride=64, key="rpn_head")
        res = ops.proposals_from_rpn(rpn_out, None, im_info, B, H5, W5, "nhwc", True,
                                     pre_nms_top_n=PRE_NMS_TOP_N, post_nms_top_n=ROIS_PER_IMAGE,
                                     nms_thresh=RPN_NMS_THRESH, min_size=RPN_MIN_SIZE,
                                     batch_index_mode=True, return_intermediate=keep_intermediate,
                                     img_hw=ext, level=C5_LEVEL)
        rois = res[0].view(B * ROIS_PER_IMAGE, 5)
        return conv5_3, H5, W5, self.conv5_f32(conv5_3, B, H5, W5), rois, res[1], res, rpn_out

    def roi_features(self, c5f, H5, W5, rois, sub, feat14, box7, extents=None):
        """ROIWarping (+ 28->14 pool when sub == 2) + 14->7 pool into the FC operand buffers.
        extents: image sizes of a mixed-size batch; a RoI samples its own image only."""
        if isinstance(feat14, dense.Tri):
            ops.roi_warp_tri(c5f, self.c5, H5, W5, rois, sub, feat14, box7, self.exp["roi_feat"],
                             img_hw=extents, level=C5_LEVEL)
        else:
            ops.roi_warp_split(c5f, self.c5, H5, W5, rois, sub, feat14, box7, img_hw=extents,
                               level=C5_LEVEL)

    # ------------------------------------------------------------------ whole forward
    def forward(self, data, im_info, keep_intermediate=False, extents=None):
        """data fp32 (B,3,H,W) device, im_info fp32 (B,3) device [h, w, scale].
        extents: None, or the int32 (B, 2) sizes of the images of a mixed-size batch, each in the
        top-left corner of the zero-padded blob (normally im_info[:, :2]): every image then gets
        the results it would get alone (device tensor: no host sync; host array: validated).
        Returns device tensors named after the blobs callers read (tools/demo.py:84-90):
        rois (B*300,5), mask_proposal (B*300,1,21,21), seg_cls_prob (B*300,21) and the `_ext`
        versions, plus roi_counts (B,) = number of real (non-padding) RoIs per image.

        Precision mode 1 needs one exponent per tri-plane activation tensor: the first call
        measures them layer by layer on its own input (a few dozen host syncs, once) and freezes
        them; every later call is the sync-free launch sequence."""
        extents = self._extents(data, extents)
        if not self._calibrated:
            self._calibrating = True
            try:
                self._forward(data, im_info, False, extents)
            finally:
                self._calibrating = False
            self._calibrated = True
        return self._forward(data, im_info, keep_intermediate, extents)

    def _forward(self, data, im_info, keep_intermediate=False, extents=None):
        B = data.shape[0]
        out = {}
        conv5_3, H5, W5, c5f, rois, roi_counts, res, rpn_out = self.rpn_rois(data, im_info, keep_intermediate,
                                                                             extents)
        c5 = self.c5
        R = B * ROIS_PER_IMAGE
        out["rois"] = rois
        out["roi_counts"] = roi_counts
        feat14 = self._act_buf("feat14", R, 14, 14, c5, exp_key="roi_feat")
        box7 = self._act_buf("box7", R, 7, 7, c5, exp_key="roi_feat")
        self.roi_features(c5f, H5, W5, rois, 2, feat14, box7, extents)
        s1 = self.head(feat14, box7, R, "s1")
        rois_ext = ops.stage_bridge(rois, s1["bbox_pred"], s1["seg_cls_prob"], im_info,
                                    ROIS_PER_IMAGE)
        out["rois_ext"] = rois_ext
        for k in ("mask_proposal", "seg_cls_prob", "cls_prob", "bbox_pred"):
            out[k] = s1[k]
        if keep_intermediate:
            out["_rpn_out"] = rpn_out.clone()
            out["_proposal"] = res[2]
            out["_conv5_3"] = conv5_3.clone()
            out["_feat14"] = feat14.clone()
            out["_box7"] = box7.clone()
            out["_mask_logits"] = s1["mask_logits"].clone()
            out["_mask_resize"] = s1["mask_resize"]
            out["_join"] = s1["join"].clone()
        self.roi_features(c5f, H5, W5, rois_ext, 1, feat14, box7, extents)
        s2 = self.head(feat14, box7, R, "s2")
        for k in ("mask_proposal", "seg_cls_prob", "cls_prob", "bbox_pred"):
            out[k + "_ext"] = s2[k]
        if keep_intermediate:
            out["_feat14_ext"] = feat14.clone()
            out["_mask_logits_ext"] = s2["mask_logits"].clone()
        return out

    def detect(self, data, im_info, im_hw, im_scale, extents=None):
        """forward + im_detect tail (tools/demo.py:92-100): boxes (B,600,4), masks (B,600,1,21,21),
        scores (B,600,21), valid (B,600) uint8.  extents: see `forward`."""
        o = self.forward(data, im_info, extents=extents)
        return self.detect_tail(o, data.shape[0], im_hw, im_scale) + (o,)

    def detect_graphed(self, data, im_info, im_hw, im_scale, rec=None, extents=None):
        """`detect` replayed from a CUDA graph: the ~60 launches of a step (shapes, buffers and
        tensor maps are static once the exponents are calibrated) are captured on first use per
        (input buffers, shape) and re-issued with one cudaGraphLaunch -- what makes the single-image
        latency (BASELINE.json configs[0]) launch-bound no more.  Inputs are read from the tensors
        given at capture time: pass the same (persistent) tensors again, or others of the same
        shape, which are then copied in.  Returns the same views as `detect` (static buffers:
        valid until the next call).  extents (see `forward`) are an input like im_info: one graph
        serves every mix of image sizes that pads to the same blob shape."""
        if not hasattr(self, "_graphs"):
            self._graphs = {}
        extents = self._extents(data, extents)
        ins = (data, im_info, im_hw, im_scale) + (() if extents is None else (extents,))
        key = (tuple(data.shape), None if rec is None else rec.data_ptr(), extents is not None)
        ent = self._graphs.get(key)
        if ent is None:
            st = [t if i == 0 else t.clone() for i, t in enumerate(ins)]
            ex = st[4] if extents is not None else None
            for _ in range(2):                       # calibrates, sizes every buffer, loads kernels
                self.detect(st[0], st[1], st[2], st[3], extents=ex)
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            # thread_local: a NCCL watchdog thread may poll events while this thread captures
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                o = self.forward(st[0], st[1], extents=ex)
                outs = self.detect_tail(o, data.shape[0], st[2], st[3], rec=rec) + (o,)
            ent = (g, st, outs, self.last_record)
            self._graphs[key] = ent
        g, st, outs, last = ent
        for dst, src in zip(st, ins):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        g.replay()
        self.last_record = last
        return outs

    def detect_tail(self, o, B, im_hw, im_scale, n=ROIS_PER_IMAGE, rec=None):
        """The `im_detect` tail on the blobs of `forward` (tools/demo.py:84-100 ==
        TesterWrapper.py:244-260) in ONE launch: rois / im_scale (fp32 division, the numpy-1.x
        evaluation of `rois[:, 1:5] / im_scales[0]`), clip_boxes to the ORIGINAL image shape im_hw,
        stage 1 rows then stage 2 rows, written into the per-step output record
        (ops.record_layout: counts | boxes | scores | masks -- the buffer the host copy and the
        all-gather take as is).  o: dict with rois, rois_ext (B*n,5), mask_proposal(_ext),
        seg_cls_prob(_ext), roi_counts (B,).  Returns views of the record + valid (B,2n) uint8."""
        msz = o["mask_proposal"].shape[-1] * o["mask_proposal"].shape[-2]
        need = ops.record_layout(B, n, msz, o["seg_cls_prob"].shape[-1])[3]
        if rec is None:
            fresh = "record" not in self._buf or self._buf["record"].numel() < need
            rec = self._f32_buf("record", need)
            if fresh:
                rec.zero_()          # the padding after counts[B] is never written by the kernel
        valid = self._buf.get("valid")
        if valid is None or valid.numel() < B * 2 * n:
            self._drop_graphs(valid)
            valid = torch.empty(B * 2 * n, dtype=torch.uint8, device=self.device)
            self._buf["valid"] = valid
        valid = valid[:B * 2 * n].view(B, 2 * n)
        _, boxes, scores, masks = ops.detect_tail(o, B, n, im_scale, im_hw, rec[:need], valid)
        self.last_record = rec[:need]
        return boxes, masks, scores, valid
