"""Public host-buffer API of the batched engine: the call a user makes.

`Detector.im_detect_batch(host_blob)` is the batched form of the reference's `im_detect`
(tools/demo.py:79-100 == lib/caffeWrapper/TesterWrapper.py:239-260): network inputs in HOST memory
(fp32 NCHW blobs exactly as `prepare_mnc_args` builds them, tools/demo.py:54-76), results back in
HOST memory -- boxes (B,600,4), masks (B,600,1,21,21), scores (B,600,21), valid (B,600).
Host<->device copies go through pinned staging buffers on the engine's stream.
`Detector.mask_voting` is the batched `gpu_mask_voting` (lib/transform/mask_transform.py:213-286).
`Detector.im_segment` goes from raw images to voted instances (and, optionally, the demo's rendered
label images) in one call, with one small result record coming back to the host.
"""
import numpy as np
import torch

from . import ops
from .engine import MNCEngine, ROIS_PER_IMAGE, MASK_SIZE, NUM_CLASSES, check_extents


class Detector:
    def __init__(self, weights, device="cuda", max_batch=8, height=600, width=1000, use_graph=True):
        self.device = torch.device(device)
        self.engine = MNCEngine(weights, device=self.device)
        # a step is ~60 launches on static buffers: replayed from a CUDA graph per input shape
        self.use_graph = use_graph
        self.max_batch = max_batch
        B, n = max_batch, 2 * ROIS_PER_IMAGE
        self._h_in = torch.empty((B, 3, height, width), dtype=torch.float32).pin_memory()
        # results come back as ONE record (ops.record_layout) + the valid flags: two D2H copies
        self._h_rec = torch.empty(ops.record_layout(B, ROIS_PER_IMAGE)[3], dtype=torch.float32).pin_memory()
        self._h_valid = torch.empty((B, n), dtype=torch.uint8).pin_memory()
        self._d_in = torch.empty((B, 3, height, width), dtype=torch.float32, device=self.device)
        # the engine's per-tensor activation maxima come back with every record (512 B): each
        # call checks them against the exponents the step ran with
        self._h_amax = torch.empty_like(self.engine._amax_all, device="cpu").pin_memory()
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def _fit_input(self, H, W):
        """Input staging follows the blob size (real images scale to 600x800 ... 901x600,
        lib/utils/blob.py:41-46); the engine's own buffers grow on demand."""
        if tuple(self._d_in.shape[2:]) != (H, W):
            B = self.max_batch
            self._h_in = torch.empty((B, 3, H, W), dtype=torch.float32).pin_memory()
            self._d_in = torch.empty((B, 3, H, W), dtype=torch.float32, device=self.device)

    def im_detect_batch(self, blob, im_info=None, im_scales=None, im_shapes=None):
        """blob: (B,3,H,W) fp32 numpy / CPU tensor (mean-subtracted BGR, as `im_list_to_blob`
        returns).  im_info: (B,3) [H, W, scale] (default: blob size, scale 1).  Synchronous."""
        blob = torch.as_tensor(blob)
        B, _, H, W = blob.shape
        assert B <= self.max_batch
        self._fit_input(H, W)
        dev = self.device
        if im_info is None:
            im_info = np.tile(np.array([[H, W, 1.0]], dtype=np.float32), (B, 1))
        info_h = torch.as_tensor(np.asarray(im_info, dtype=np.float32))
        scale_h = info_h[:, 2].contiguous() if im_scales is None else torch.as_tensor(np.asarray(im_scales, np.float32))
        if im_shapes is None:
            # boxes are clipped to the ORIGINAL image (TesterWrapper.py:254-255): blob size / scale
            hw_h = torch.round(info_h[:, :2] / scale_h[:, None]).contiguous()
        else:
            hw_h = torch.as_tensor(np.asarray(im_shapes, np.float32))
        if blob.is_pinned():
            src = blob                                   # caller already handed page-locked memory
        else:
            self._h_in[:B].copy_(blob)                   # user memory -> pinned staging
            src = self._h_in[:B]
        with torch.cuda.device(dev):
            self._d_in[:B].copy_(src, non_blocking=True)
            info = info_h.to(dev, non_blocking=True)
            out = self._detect_to_host(B, self._d_in[:B], info, hw_h.to(dev), scale_h.to(dev))
        self.h2d_bytes = blob.numel() * 4 + info_h.numel() * 4 + scale_h.numel() * 4 + hw_h.numel() * 4
        return out

    def _detect(self, data, info, hw, sc, ext=None):
        if self.use_graph:
            return self.engine.detect_graphed(data, info, hw, sc, extents=ext)
        return self.engine.detect(data, info, hw, sc, extents=ext)

    def _detect_to_host(self, B, data, info, hw, sc, ext=None):
        """One step, its results to host memory, then the range check on the activation maxima
        that came back with them: a batch whose activations outgrew the frozen exponents
        (MNCEngine.range_ok) is computed again with exponents measured on it."""
        valid = self._detect(data, info, hw, sc, ext)[3]
        out = self._results_to_host(B, valid)
        if not self.engine.range_ok(amax=self._h_amax):
            valid = self._detect(data, info, hw, sc, ext)[3]
            out = self._results_to_host(B, valid)
        return out

    def _results_to_host(self, B, valid):
        rec = self.engine.last_record
        n = rec.numel()
        self._h_rec[:n].copy_(rec, non_blocking=True)
        self._h_valid[:B].copy_(valid, non_blocking=True)
        self._h_amax.copy_(self.engine._amax_all, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self.d2h_bytes = n * 4 + valid.numel()
        _, boxes, scores, masks = ops.record_views(self._h_rec[:n], B, ROIS_PER_IMAGE)
        return boxes.numpy(), masks.numpy(), scores.numpy(), self._h_valid[:B].numpy()

    def im_detect_images(self, images_u8):
        """Batched `im_detect(im, net)` on raw images, as the reference's callers hand them over
        (tools/demo.py:143-146): uint8 BGR (B,H,W,3) host array, all of one size.  Mean
        subtraction, the 600/1000 resize rule and HWC->NCHW run on the device (mnc_prep_images),
        so only B*H*W*3 bytes cross PCIe.  Returns boxes (in original-image coordinates), masks,
        scores, valid -- host arrays -- and the scale used."""
        pinned_src = None
        if isinstance(images_u8, torch.Tensor):
            # a page-locked uint8 tensor goes to the device without the staging copy
            assert images_u8.dtype == torch.uint8 and images_u8.is_contiguous()
            if images_u8.is_pinned():
                pinned_src = images_u8
            images_u8 = images_u8.numpy()
        images_u8 = np.ascontiguousarray(images_u8)
        B, H, W, _ = images_u8.shape
        scale = ops.im_scale_for((H, W))
        out_h, out_w = int(np.rint(H * scale)), int(np.rint(W * scale))
        assert B <= self.max_batch
        self._fit_input(out_h, out_w)
        dev = self.device
        if getattr(self, "_h_u8", None) is None or self._h_u8.shape[1:] != images_u8.shape[1:]:
            self._h_u8 = torch.empty((self.max_batch, H, W, 3), dtype=torch.uint8).pin_memory()
            self._d_u8 = torch.empty((self.max_batch, H, W, 3), dtype=torch.uint8, device=dev)
        if pinned_src is None:
            self._h_u8[:B].copy_(torch.from_numpy(images_u8))
            pinned_src = self._h_u8[:B]
        info = torch.tensor([[out_h, out_w, scale]] * B, dtype=torch.float32)
        hw = torch.tensor([[H, W]] * B, dtype=torch.float32)
        sc = torch.full((B,), scale, dtype=torch.float32)
        with torch.cuda.device(dev):
            self._d_u8[:B].copy_(pinned_src, non_blocking=True)
            ops.prep_images(self._d_u8[:B], scale, out=self._d_in[:B])
            out = self._detect_to_host(B, self._d_in[:B], info.to(dev, non_blocking=True),
                                       hw.to(dev, non_blocking=True), sc.to(dev, non_blocking=True))
        self.h2d_bytes = images_u8.nbytes + (info.numel() + hw.numel() + sc.numel()) * 4
        return out + (scale,)

    def _mixed_batch(self, images):
        """Host side of a mixed-size batch: validation, per-image scales and blob sizes, the
        packed frames in pinned staging `buf` (grown on demand).  -> dict of host values."""
        images = [np.ascontiguousarray(im.numpy() if isinstance(im, torch.Tensor) else im)
                  for im in images]
        if not 1 <= len(images) <= self.max_batch:
            raise ValueError("%d images in one batch, at most %d" % (len(images), self.max_batch))
        for im in images:
            if im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3 or min(im.shape[:2]) < 1:
                raise ValueError("images must be uint8 BGR (H, W, 3) arrays, got %s %s" % (im.dtype, im.shape))
        scales = np.array([ops.im_scale_for(im.shape) for im in images], dtype=np.float64)
        src_hw = np.array([im.shape[:2] for im in images], dtype=np.int32)
        dst_hw = np.array([ops.blob_size_for(im.shape, s) for im, s in zip(images, scales)], dtype=np.int32)
        Hb, Wb = int(dst_hw[:, 0].max()), int(dst_hw[:, 1].max())
        ext = check_extents(dst_hw, Hb, Wb, self.max_batch)
        sizes = [im.nbytes for im in images]
        offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
        return dict(images=images, scales=scales, src_hw=src_hw, dst_hw=dst_hw, H=Hb, W=Wb, ext=ext,
                    offsets=offsets, nbytes=int(sum(sizes)), B=len(images))

    @staticmethod
    def _pack(mb, h_buf, dev, d_buf):
        """Grow-on-demand pinned / device byte buffers holding the packed frames of `mb`."""
        if h_buf is None or h_buf.numel() < mb["nbytes"]:
            h_buf = torch.empty(mb["nbytes"], dtype=torch.uint8).pin_memory()
            d_buf = torch.empty(mb["nbytes"], dtype=torch.uint8, device=dev)
        for im, off in zip(mb["images"], mb["offsets"]):
            h_buf[off:off + im.nbytes].copy_(torch.from_numpy(im.reshape(-1)))
        return h_buf, d_buf

    def _mixed_inputs(self, mb):
        """im_info [blob h, blob w, scale], original sizes and scales of a mixed batch (host)."""
        info = torch.tensor([[h, w, s] for (h, w), s in zip(mb["dst_hw"], mb["scales"])], dtype=torch.float32)
        hw = torch.from_numpy(mb["src_hw"].astype(np.float32))
        sc = torch.from_numpy(mb["scales"].astype(np.float32))
        return info, hw, sc

    def im_detect_mixed(self, images):
        """`im_detect` on a batch of images of DIFFERENT sizes in one step: images is a list of
        at most max_batch uint8 BGR (H_i, W_i, 3) host arrays.  Each image is scaled by its own
        600/1000 rule and placed in the top-left corner of one zero-padded blob (as the
        reference's `im_list_to_blob` pads), and every layer treats the pixels outside an image as
        outside it, so each image gets the results it would get alone.  Returns boxes (in each
        image's original coordinates), masks, scores, valid -- host arrays as `im_detect_images`
        returns them -- and the scales (B,)."""
        mb = self._mixed_batch(images)
        B, dev = mb["B"], self.device
        self._fit_input(mb["H"], mb["W"])
        self._h_pack, self._d_pack = self._pack(mb, getattr(self, "_h_pack", None), dev,
                                                getattr(self, "_d_pack", None))
        info, hw, sc = self._mixed_inputs(mb)
        with torch.cuda.device(dev):
            self._d_pack[:mb["nbytes"]].copy_(self._h_pack[:mb["nbytes"]], non_blocking=True)
            ops.prep_images_ragged(self._d_pack, mb["offsets"], mb["src_hw"], mb["scales"], mb["H"],
                                   mb["W"], out=self._d_in[:B])
            out = self._detect_to_host(B, self._d_in[:B], info.to(dev, non_blocking=True),
                                       hw.to(dev, non_blocking=True), sc.to(dev, non_blocking=True),
                                       mb["ext"].to(dev, non_blocking=True))
        self.h2d_bytes = mb["nbytes"] + (info.numel() + hw.numel() + sc.numel() + mb["ext"].numel()) * 4
        return out + (mb["scales"].copy(),)

    def im_detect_stream(self, batches):
        """Pipelined `im_detect_images`: an iterable of uint8 BGR (B,H,W,3) host batches (all of
        one size) -> a generator of (boxes, masks, scores, valid, scale) per batch, in order.  A
        batch may also be a LIST of differently sized (H_i, W_i, 3) images (`im_detect_mixed`);
        its result then carries the scales (B,) in place of the scalar.
        Two batches are in flight: while batch k computes, the frames of batch k+1 cross PCIe on a
        copy stream and the record of batch k-1 comes back on another, so the host<->device copies
        (14.4 MB in, 9 MB out per batch of 8) leave the critical path; and the two batches compute
        on two streams, each with its own engine state over the shared weights
        (MNCEngine.clone_state), so that batch k+1's kernels fill batch k's wave tails and its
        low-occupancy proposal phase.  A yielded result is valid until the next iteration (its
        pinned buffers are reused two batches later)."""
        return self._pipeline(batches)

    def im_segment(self, images, max_per_image=100, render=False, vis_thresh=0.5):
        """Raw images in, voted instances out: `im_detect` + `gpu_mask_voting`
        (lib/transform/mask_transform.py:213-286) for every image of a batch, everything resident
        on the device until one small record (plus, with render, the label images) is copied back.
        images: a uint8 BGR (B, H, W, 3) array or tensor (as `im_detect_images` takes), or a list of
        differently sized uint8 BGR (H_i, W_i, 3) images (as `im_detect_mixed` takes).  Returns a
        list of B dicts, in input order: boxes int32 (k, 4), scores fp32 (k,), classes int32 (k,),
        masks fp32 (k, 21, 21) -- every voted result, class-major as the reference's loops emit them
        -- and the image's scale.  With render=True also the demo's images at the image's own size
        (`_convert_pred_to_image` of `get_vis_dict(..., vis_thresh)`, tools/demo.py:153-164):
        inst, cls int32 (H_i, W_i) and bgr uint8 (H_i, W_i, 3); vis_thresh affects these only."""
        res, = self.im_segment_stream([images], max_per_image, render, vis_thresh)
        return res

    def im_segment_stream(self, batches, max_per_image=100, render=False, vis_thresh=0.5):
        """Pipelined `im_segment`, built as `im_detect_stream` (two batches in flight, each slot
        with its own engine state; frames in and results out on copy streams): an iterable of
        batches of either form -> a generator of `im_segment` results per batch, in order."""
        seg = dict(max_per_image=int(max_per_image), render=bool(render), vis_thresh=float(vis_thresh))
        return self._pipeline(batches, seg)

    def _pipeline(self, batches, seg=None):
        """Two batches in flight (im_detect_stream); seg: the options of im_segment_stream, or None
        for detect results."""
        pending = None
        for k, images_u8 in enumerate(batches):
            cur = self._submit(k & 1, images_u8, seg)
            if pending is not None:
                yield self._collect(pending)
            pending = cur
        if pending is not None:
            yield self._collect(pending)

    def _submit(self, slot, images_u8, seg=None):
        if isinstance(images_u8, (list, tuple)):
            return self._submit_mixed(slot, images_u8, seg)
        dev = self.device
        pinned_src = None
        if isinstance(images_u8, torch.Tensor):
            if images_u8.dtype != torch.uint8 or not images_u8.is_contiguous():
                raise ValueError("an image batch tensor must be contiguous uint8, got %s" % images_u8.dtype)
            if images_u8.is_pinned():
                pinned_src = images_u8
            images_u8 = images_u8.numpy()
        images_u8 = np.ascontiguousarray(images_u8)
        if images_u8.dtype != np.uint8 or images_u8.ndim != 4 or images_u8.shape[3] != 3 or \
                min(images_u8.shape[1:3]) < 1:
            raise ValueError("an image batch must be uint8 BGR (B, H, W, 3), got %s %s"
                             % (images_u8.dtype, images_u8.shape))
        B, H, W, _ = images_u8.shape
        if not 1 <= B <= self.max_batch:
            raise ValueError("%d images in one batch, at most %d" % (B, self.max_batch))
        scale = ops.im_scale_for((H, W))
        out_h, out_w = int(np.rint(H * scale)), int(np.rint(W * scale))
        self._fit_input(out_h, out_w)
        st, eng = self._slot(slot)
        if st.get("h_u8") is None or tuple(st["h_u8"].shape[1:]) != (H, W, 3):
            st["h_u8"] = torch.empty((self.max_batch, H, W, 3), dtype=torch.uint8).pin_memory()
            st["d_u8"] = torch.empty((self.max_batch, H, W, 3), dtype=torch.uint8, device=dev)
        if pinned_src is None:
            st["h_u8"][:B].copy_(torch.from_numpy(images_u8))      # pageable -> pinned staging (host)
            pinned_src = st["h_u8"][:B]
        info = torch.tensor([[out_h, out_w, scale]] * B, dtype=torch.float32)
        hw = torch.tensor([[H, W]] * B, dtype=torch.float32)
        sc = torch.full((B,), scale, dtype=torch.float32)
        prep = lambda: ops.prep_images(st["d_u8"][:B], scale, out=st["d_in"][:B])
        return self._issue(slot, st, eng, B, lambda: st["d_u8"][:B].copy_(pinned_src, non_blocking=True),
                           prep, info, hw, sc, None, scale, images_u8.nbytes, seg)

    def _slot(self, slot):
        """Slot `slot`'s staging buffers (input blob sized like _d_in) and engine."""
        dev = self.device
        if getattr(self, "_s_in", None) is None:
            self._s_in = torch.cuda.Stream(device=dev)
            self._s_out = torch.cuda.Stream(device=dev)
            self._slots = [None, None]
            self._s_comp = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
            self._engines = [self.engine, None]
        st = self._slots[slot]
        if st is None:
            n_rec = ops.record_layout(self.max_batch, ROIS_PER_IMAGE)[3]
            st = dict(d_rec=torch.empty(n_rec, dtype=torch.float32, device=dev),
                      h_rec=torch.empty(n_rec, dtype=torch.float32).pin_memory(),
                      d_in=torch.empty_like(self._d_in),
                      h_amax=torch.empty_like(self._h_amax).pin_memory(),
                      u8_free=None, out_done=None)
            self._slots[slot] = st
        if tuple(st["d_in"].shape) != tuple(self._d_in.shape):
            st["d_in"] = torch.empty_like(self._d_in)
        eng = self._engines[slot]
        if eng is None:          # slot 1's engine: made once slot 0's first call has calibrated
            torch.cuda.synchronize(dev)
            eng = self._engines[slot] = self.engine.clone_state()
        return st, eng

    def _submit_mixed(self, slot, images, seg=None):
        mb = self._mixed_batch(images)
        B = mb["B"]
        self._fit_input(mb["H"], mb["W"])
        st, eng = self._slot(slot)
        if st["u8_free"] is not None:
            st["u8_free"].synchronize()          # the pinned pack buffer may still be crossing
        st["h_pack"], st["d_pack"] = self._pack(mb, st.get("h_pack"), self.device, st.get("d_pack"))
        info, hw, sc = self._mixed_inputs(mb)
        nb = mb["nbytes"]
        h2d = lambda: st["d_pack"][:nb].copy_(st["h_pack"][:nb], non_blocking=True)
        prep = lambda: ops.prep_images_ragged(st["d_pack"], mb["offsets"], mb["src_hw"], mb["scales"],
                                              mb["H"], mb["W"], out=st["d_in"][:B])
        return self._issue(slot, st, eng, B, h2d, prep, info, hw, sc, mb["ext"], mb["scales"].copy(), nb, seg)

    def _issue(self, slot, st, eng, B, h2d, prep, info, hw, sc, ext, scale, in_bytes, seg=None):
        """Queue one batch on slot `slot`: frames H2D on the copy stream (h2d), preparation (prep)
        and the step on the slot's compute stream, the record D2H on the other copy stream.  With
        seg (im_segment_stream), mask voting (and rendering) follow the step on the compute stream
        and the voted record replaces the detect record on the way back."""
        dev = self.device
        with torch.cuda.device(dev), torch.cuda.stream(self._s_comp[slot]):
            main = torch.cuda.current_stream()                      # this slot's compute stream
            with torch.cuda.stream(self._s_in):                     # frames of this batch: H2D
                if st["u8_free"] is not None:
                    self._s_in.wait_event(st["u8_free"])
                h2d()
                ev_in = torch.cuda.Event()
                ev_in.record(self._s_in)
            main.wait_event(ev_in)
            prep()
            st["u8_free"] = torch.cuda.Event()
            st["u8_free"].record(main)
            if st["out_done"] is not None:
                main.wait_event(st["out_done"])                     # this slot's record was read
            n = ops.record_layout(B, ROIS_PER_IMAGE)[3]
            args = (st["d_in"][:B], info.to(dev, non_blocking=True), hw.to(dev, non_blocking=True),
                    sc.to(dev, non_blocking=True), None if ext is None else ext.to(dev, non_blocking=True))
            eng._amax_all.zero_()                                   # maxima of this step only
            outs = self._step(slot, args, B)
            job = None
            if seg is not None:
                job = self._seg_job(st, B, hw, scale, seg)
                self._vote(st, outs, job, st["d_vrec"])
            ev_done = torch.cuda.Event()
            ev_done.record(main)
            with torch.cuda.stream(self._s_out):                    # record of this batch: D2H
                self._s_out.wait_event(ev_done)
                if job is None:
                    st["h_rec"][:n].copy_(st["d_rec"][:n], non_blocking=True)
                else:
                    n = job["n_rec"]
                    st["h_vrec"][:n].copy_(st["d_vrec"][:n], non_blocking=True)
                    if seg["render"]:
                        nr = job["n_render"]
                        st["h_rbuf"][:nr].copy_(st["d_rbuf"][:nr], non_blocking=True)
                st["h_amax"].copy_(eng._amax_all, non_blocking=True)
                st["out_done"] = torch.cuda.Event()
                st["out_done"].record(self._s_out)
        self.h2d_bytes = in_bytes + (info.numel() + hw.numel() + sc.numel()) * 4
        if job is None:
            self.d2h_bytes = n * 4
        else:
            self.d2h_bytes = job["n_rec"] * 4 + st["h_amax"].numel() * 4 + job["n_render"]
        # the exponents this step ran with (a captured graph keeps those of its capture)
        return (slot, B, n, scale, args, dict(eng.exp), outs, job)

    def _seg_job(self, st, B, hw, scale, seg):
        """Device inputs and slot buffers (grown on demand) of the voting / rendering of one batch.
        hw: host fp32 (B, 2) original image sizes."""
        dev = self.device
        hw_i = hw.to(torch.int32)
        R = ops.default_vote_cap(seg["max_per_image"])
        n_rec = ops.vote_record_layout(B, R, MASK_SIZE)[-1]
        if st.get("d_vrec") is None or st["d_vrec"].numel() < n_rec:
            st["d_vrec"] = torch.empty(n_rec, dtype=torch.int32, device=dev)
            st["h_vrec"] = torch.empty(n_rec, dtype=torch.int32).pin_memory()
        pix = hw_i[:, 0].long() * hw_i[:, 1].long()
        pix_off = torch.cumsum(pix, 0) - pix
        P = int(pix.sum())
        job = dict(B=B, R=R, n_rec=n_rec, seg=seg, hw=hw_i.numpy(), pix_off=pix_off.numpy(), P=P,
                   n_render=11 * P if seg["render"] else 0, scale=scale,
                   d_hw=hw_i.to(dev, non_blocking=True))
        if seg["render"]:
            # one byte buffer, one copy back: inst int32[P] | cls int32[P] | bgr uint8[P][3]
            if st.get("d_rbuf") is None or st["d_rbuf"].numel() < 11 * P:
                st["d_rbuf"] = torch.empty(11 * P, dtype=torch.uint8, device=dev)
                st["h_rbuf"] = torch.empty(11 * P, dtype=torch.uint8).pin_memory()
            job["d_off"] = pix_off.to(dev, non_blocking=True)
            job["max_hw"] = (int(job["hw"][:, 0].max()), int(job["hw"][:, 1].max()))
        return job

    def _vote(self, st, outs, job, d_vrec, R=None):
        """Mask voting on the step outputs `outs` into the record d_vrec (R result slots per image,
        default the job's), then, if asked for, rendering into the slot's render buffer."""
        B, seg = job["B"], job["seg"]
        R = job["R"] if R is None else R
        boxes, masks, scores, valid = outs
        views = ops.vote_record_views(d_vrec, B, R, MASK_SIZE)
        ops.mask_voting(boxes, masks, scores, job["d_hw"], max_per_image=seg["max_per_image"],
                        max_results=R, box_valid=valid, out=views)
        if seg["render"]:
            P, rb = job["P"], st["d_rbuf"]
            ops.paste_voted_ragged(views, job["d_hw"], job["d_off"], job["max_hw"],
                                   rb[:4 * P].view(torch.int32), rb[4 * P:8 * P].view(torch.int32),
                                   rb[8 * P:11 * P], vis_thresh=seg["vis_thresh"])

    def _step(self, slot, args, B):
        """One step of slot `slot` into its record -> (boxes, masks, scores, valid) device views."""
        eng, st = self._engines[slot], self._slots[slot]
        if self.use_graph:
            return eng.detect_graphed(*args[:4], rec=st["d_rec"], extents=args[4])[:4]
        o = eng.forward(args[0], args[1], extents=args[4])
        return eng.detect_tail(o, B, args[2], args[3], rec=st["d_rec"])

    def _collect(self, handle):
        slot, B, n, scale, args, exp_used, outs, job = handle
        st, eng = self._slots[slot], self._engines[slot]
        st["out_done"].synchronize()
        # exponents re-measured since this batch was issued (on the other slot's batch): recompute
        # it with the current ones; activations that outgrew the exponents: re-measure and recompute
        ok = exp_used == eng.exp and eng.range_ok(reset=False, amax=st["h_amax"], exp=exp_used)
        for _ in range(2):
            if ok:
                break
            dev = self.device
            # the other slot's step may still be replaying a graph that is about to be dropped
            torch.cuda.synchronize(dev)
            if not eng._calibrated:            # the exponents (shared by both slots) will change
                for e in self._engines:
                    if e is not None and hasattr(e, "_graphs"):
                        e._graphs.clear()
            with torch.cuda.device(dev), torch.cuda.stream(self._s_comp[slot]):
                eng._amax_all.zero_()
                outs = self._step(slot, args, B)
                if job is None:
                    st["h_rec"][:n].copy_(st["d_rec"][:n])
                else:
                    self._vote(st, outs, job, st["d_vrec"])
                    self._seg_to_host(st, job)
            torch.cuda.synchronize(dev)
            ok = eng.range_ok()
        if job is not None:
            return self._seg_results(slot, outs, job)
        counts, boxes, scores, masks = ops.record_views(st["h_rec"][:n], B, ROIS_PER_IMAGE)
        # valid flags from the counts (2 x RoIs per image: stage-1 rows, then stage-2 rows)
        per_stage = (counts.numpy() / 2).astype(np.int64)
        idx = np.arange(2 * ROIS_PER_IMAGE) % ROIS_PER_IMAGE
        valid = (idx[None, :] < per_stage[:, None]).astype(np.uint8)
        return boxes.numpy(), masks.numpy(), scores.numpy(), valid, scale

    @staticmethod
    def _seg_to_host(st, job, d_vrec=None, h_vrec=None):
        n = job["n_rec"] if d_vrec is None else d_vrec.numel()
        (st["h_vrec"] if h_vrec is None else h_vrec)[:n].copy_((st["d_vrec"] if d_vrec is None else d_vrec)[:n])
        if job["n_render"]:
            st["h_rbuf"][:job["n_render"]].copy_(st["d_rbuf"][:job["n_render"]])

    def _seg_results(self, slot, outs, job):
        """The host side of a voted batch: results that did not fit the record's R slots per image
        are voted again with twice the room (ops.mask_voting_checked's rule), then the per-image
        results are cut out of the record (and the render buffer)."""
        st, B, R, seg = self._slots[slot], job["B"], job["R"], job["seg"]
        h_vrec = st["h_vrec"]
        views = ops.vote_record_views(h_vrec, B, R, MASK_SIZE)
        limit = outs[0].shape[1] * (NUM_CLASSES - 1)
        while int(views["overflow"][0]) != 0:
            if R >= limit:
                raise ops.VotingOverflow("mask voting overflow at max_results = %d" % R)
            R = min(2 * R, limit)
            n = ops.vote_record_layout(B, R, MASK_SIZE)[-1]
            d_vrec = torch.empty(n, dtype=torch.int32, device=self.device)
            h_vrec = torch.empty(n, dtype=torch.int32)
            with torch.cuda.device(self.device), torch.cuda.stream(self._s_comp[slot]):
                # the step outputs stay valid until this slot's next submit
                self._vote(st, outs, job, d_vrec, R)
                self._seg_to_host(st, job, d_vrec, h_vrec)
            self.d2h_bytes += n * 4 + job["n_render"]
            views = ops.vote_record_views(h_vrec, B, R, MASK_SIZE)
        n_res = views["n_res"].numpy()
        cls, score = views["res_class"].numpy(), views["res_score"].numpy()
        box, mask = views["result_box"].numpy(), views["result_mask"].numpy()
        if seg["render"]:
            P, rb = job["P"], st["h_rbuf"]
            inst, clsi, bgr = (rb[:4 * P].view(torch.int32).numpy(), rb[4 * P:8 * P].view(torch.int32).numpy(),
                               rb[8 * P:11 * P].numpy())
        scale = job["scale"]
        out = []
        for b in range(B):
            k = int(n_res[b])
            r = dict(boxes=box[b, :k].copy(), scores=score[b, :k].copy(), classes=cls[b, :k].copy(),
                     masks=mask[b, :k, 0].copy(),
                     scale=float(scale if np.ndim(scale) == 0 else scale[b]))
            if seg["render"]:
                (H, W), o = job["hw"][b], int(job["pix_off"][b])
                r["inst"] = inst[o:o + H * W].reshape(H, W).copy()
                r["cls"] = clsi[o:o + H * W].reshape(H, W).copy()
                r["bgr"] = bgr[3 * o:3 * (o + H * W)].reshape(H, W, 3).copy()
            out.append(r)
        return out

    def mask_voting(self, boxes, masks, scores, valid, im_hw, max_per_image=100):
        """Device-resident batched gpu_mask_voting on `engine.detect` outputs (device tensors)."""
        hw = torch.as_tensor(np.asarray(im_hw, dtype=np.int32)).to(self.device)
        return ops.mask_voting_checked(boxes, masks, scores, hw, max_per_image=max_per_image,
                                       box_valid=valid)


def unpack_voting(result, num_classes=NUM_CLASSES):
    """Voted results -> the reference's per-class format of `gpu_mask_voting`
    (mask_transform.py:270-286): (list_result_mask, list_result_box), each a list over the
    num_classes-1 foreground classes of (k,1,M,M) fp32 masks / (k,5) fp32 [box, score].
    result: one image's result of `Detector.im_segment`; or the dict of device tensors that
    `ops.mask_voting` returns for a batch, which gives a list of such pairs, one per image."""
    if "n_res" in result:
        n_res = result["n_res"].cpu().numpy()
        cls, score = result["res_class"].cpu().numpy(), result["res_score"].cpu().numpy()
        box, mask = result["result_box"].cpu().numpy(), result["result_mask"].cpu().numpy()
        return [unpack_voting(dict(boxes=box[b, :k], scores=score[b, :k], classes=cls[b, :k],
                                   masks=mask[b, :k]), num_classes)
                for b, k in enumerate(n_res.astype(np.int64))]
    masks = np.asarray(result["masks"])
    M = masks.shape[-1]
    boxes, scores, cls = np.asarray(result["boxes"]), np.asarray(result["scores"]), np.asarray(result["classes"])
    list_mask, list_box = [], []
    for c in range(1, num_classes):
        sel = np.where(cls == c)[0]
        list_mask.append(masks[sel].reshape(-1, 1, M, M).astype(np.float32))
        list_box.append(np.hstack((boxes[sel].astype(np.float32), scores[sel, None].astype(np.float32))))
    return list_mask, list_box
