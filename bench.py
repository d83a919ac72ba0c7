#!/usr/bin/env python
"""bench.py -- images/sec of the MNC 5-stage inference hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference]
  (N > 1: launched by torchrun, one rank per GPU; reads RANK/LOCAL_RANK/WORLD_SIZE/MASTER_*)

A "step" = one pass of the hot path (im_detect: trunk -> RPN proposals -> two cascade stages ->
im_detect tail, tools/demo.py:79-100) over one batch of B synthetic 600x1000 images per GPU (weak
scaling: the batch is sharded over images; the one collective is an all-gather of the per-step
output records, issued on a side stream so that it overlaps the next step's trunk).
`value`  : whole-job images/s with the inputs resident in HBM (CUDA events, max over ranks); the
           step is replayed from a CUDA graph (mnc_b200.engine.MNCEngine.detect_graphed).
`e2e`    : same metric through the public host-buffer API (mnc_b200.api.Detector.im_detect_images):
           uint8 frames in host memory -> H2D -> prep + forward -> results D2H, all inside the
           timed region; reported from page-locked and from pageable caller memory.
`roofline`: the dominant kernel (tcgen05 implicit GEMM: all conv + inner-product launches of a step):
           algorithmic FLOPs (2*M*N*K, real dims) / summed per-launch CUDA-event time (measured in
           an eager pass of the same step); `roofline_roi_warp`: the RoI-warp HBM roofline.
`micro`  : BASELINE.json configs[3] (RoI-warp / mask-pool GB/s) and configs[4] (gpu_nms 10k boxes,
           gpu_mask_voting 600 x 21; ms + bit-exactness against the reference's own kernels).
`cpu_baseline`: the oracle (port of the reference path; the reference has no runnable CPU path,
           BASELINE.md section 2) timed on this box's host cores on a bounded sample (rank 0, N=1).
--impl reference prints the same line for the CPU oracle alone.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 600, 1000
METRIC = "images/sec VGG16 MNC 5-stage @600x1000, 300 RoIs"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def physical_cores():
    """Physical cores of the box (SMT siblings counted once)."""
    try:
        seen = set()
        phys = core = None
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("physical id"):
                    phys = line.split(":")[1].strip()
                elif line.startswith("core id"):
                    core = line.split(":")[1].strip()
                elif not line.strip():
                    if phys is not None and core is not None:
                        seen.add((phys, core))
                    phys = core = None
        if seen:
            return len(seen)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                smax = max(smax, float(s[1]))
                for nm, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_time(weights, images, warmup, budget_s=45.0):
    """The CPU oracle, one image per step: `warmup` untimed images, then up to `images` timed ones.
    Bounded: once `budget_s` seconds have gone by the remaining warm-ups are skipped and the loop
    stops after the next timed image (a loaded host must not stall the GPU bench).  Returns the
    per-image seconds (>= 1 entry)."""
    from oracle import oracle as O
    times = []
    t_start = time.perf_counter()
    it = 0
    warm_left = warmup
    while len(times) < images:
        over = time.perf_counter() - t_start > budget_s
        if over and times:
            break
        im = O.synthetic_image(it, H, W)
        it += 1
        t0 = time.perf_counter()
        O.im_detect(weights, im)
        dt = time.perf_counter() - t0
        if warm_left > 0 and not over and dt < budget_s / 3:
            warm_left -= 1
            continue
        warm_left = 0
        times.append(dt)
    return times


def _summ(times):
    s = sorted(times)
    n = len(s)
    return {"median_s": s[n // 2], "p10_s": s[max(0, int(0.1 * n))], "p90_s": s[min(n - 1, int(0.9 * n))], "n": n}


_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL announces its
    version on the first communicator), so file descriptor 1 is pointed at stderr for the whole
    run and the JSON line is written to a private duplicate of the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


_T0 = time.perf_counter()


def _log(msg):
    """Progress marker on stderr (stdout carries only the JSON line)."""
    sys.stderr.write("[bench %7.1fs] %s\n" % (time.perf_counter() - _T0, msg))
    sys.stderr.flush()


def usable_cores():
    """Threads the CPU arm may use: physical cores, capped by the process's affinity mask and by
    the cgroup CPU quota (a box that hands this container 8 CPUs must not get 64 OpenMP threads)."""
    n = physical_cores()
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


def _pin_cpu_threads():
    """One software thread per physical core, before torch / OpenMP start (torchrun pins
    OMP_NUM_THREADS to 1 for its workers; oversubscribing SMT siblings made this arm swing 6x)."""
    n = usable_cores()
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ["MKL_NUM_THREADS"] = str(n)
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")
    return n


def run_reference(args, rank):
    """--impl reference: the reference's own algorithm on the host cores.  The reference has no
    runnable CPU implementation (its MNC layers are NOT_IMPLEMENTED on CPU and Caffe does not
    build here), so this is the oracle port on all physical cores; a step = one image."""
    if rank != 0:
        return
    ncpu = _pin_cpu_threads()
    import torch
    torch.set_num_threads(ncpu)
    from mnc_b200 import weights as Wt
    w = Wt.make_weights(Wt.FULL_ARCH)
    images = max(5, min(args.steps, 8))
    warm = max(2, min(args.warmup, 3))
    times = cpu_reference_time(w, images, warm, budget_s=90.0)
    st = _summ(times)
    images = len(times)
    v = 1.0 / st["median_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus,
        "steps": images, "warmup": warm, "ms_per_step": 1000.0 * st["median_s"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, 1),
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": ncpu, "kind": "port",
                         "sample": "%d images (600x1000, 300 RoIs/stage) one per step after %d "
                                   "warm-up images; value = 1 / median per-image time" % (images, warm),
                         "per_image_s": st},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference has no runnable CPU path (BASELINE.md section 2); oracle port timed on "
                "%d host threads = usable cores of this container (torch CPU fp32 conv/FC + numpy layers + C/OpenMP kernels); "
                "steps/warmup clamped to keep the run bounded" % ncpu,
    }
    _emit(line)


def workload_config(args, world):
    return {"workload": "configs[1]: VGG16 MNC 5-stage inference (im_detect), batch %d per GPU, "
                        "600x1000 synthetic, 300 RoIs/stage" % args.batch,
            "global_batch": args.batch * world, "image": [H, W], "rois_per_stage": 300,
            "parallelism": "dp%d (images sharded, 1 all-gather of records per step, overlapped)" % world,
            "steps_in_flight": 1 if args.no_graph else args.streams,
            "l2": "inputs larger than L2: every step streams 1.13 GB of weights and > 5 GB of "
                  "activations through the 126 MB L2, nothing of a step survives to the next",
            "weights": "seeded random init (mnc_b200/weights.py), fp32 -> fp16 + 2 x e4m3 planes "
                       "(every conv3x3 / inner product; conv1_1, K = 27: split bf16)"}


def median_ms(fn, iters=20, warm=3, flush=None):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ms = []
    for i in range(iters):
        if flush is not None:
            flush.fill_(i & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    return ms[len(ms) // 2]


def microbench(hbm_gbs):
    """BASELINE.json configs[3] and configs[4] (SURVEY.md section 8d inputs), one GPU."""
    import ctypes
    import numpy as np
    import torch
    from mnc_b200 import ops
    from oracle import oracle as O
    from tests import util
    res = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cpu").manual_seed(7)
    feat = torch.randn(1, 512, 38, 63, generator=g).clamp_min(0).cuda()
    rng = np.random.default_rng(8)
    x1, y1 = rng.uniform(0, 999, 2000), rng.uniform(0, 599, 2000)
    w, h = rng.uniform(16, 600, 2000), rng.uniform(16, 600, 2000)
    rois = np.stack([np.zeros(2000), x1, y1, np.clip(x1 + w, 0, 999), np.clip(y1 + h, 0, 599)], 1).astype(np.float32)
    trois = torch.from_numpy(rois).cuda()
    for P in (28, 14):
        out = torch.empty(2000, 512, P, P, device="cuda")
        ms = median_ms(lambda: ops.roi_warp_nchw(feat, trois, P, P, out=out), flush=flush)
        alg = 2000 * 512 * P * P * 4 + 512 * 38 * 63 * 4 + 2000 * 20
        res["roi_warp_P%d" % P] = {"ms": ms, "algorithmic_bytes": alg, "GBps": alg / ms / 1e6,
                                   "frac_of_hbm": alg / ms / 1e6 / hbm_gbs}
        del out
    f14 = torch.randn(2000, 512, 14, 14, device="cuda")
    m14 = torch.rand(2000, 1, 14, 14, device="cuda")
    o14 = torch.empty_like(f14)
    ms = median_ms(lambda: ops.mask_pool_nchw(f14, m14, out=o14), flush=flush)
    alg = 2 * 2000 * 512 * 196 * 4 + 2000 * 196 * 4
    res["mask_pool"] = {"ms": ms, "algorithmic_bytes": alg, "GBps": alg / ms / 1e6,
                        "frac_of_hbm": alg / ms / 1e6 / hbm_gbs}
    del f14, o14
    # ---- configs[4]: gpu_nms, 10 000 boxes, keep 300 at 0.7, vs the reference's own _nms
    boxes = util.random_boxes(10000, seed=10)
    scores = util.tie_free_scores(10000, seed=11)
    order = O.order_desc(scores)
    sorted_dets = np.ascontiguousarray(np.hstack([boxes, scores[:, None]]).astype(np.float32)[order])
    sb = torch.from_numpy(np.ascontiguousarray(sorted_dets[:, :4])).cuda()[None].contiguous()
    ms = median_ms(lambda: ops.nms_sorted(sb, None, 0.7, 300))
    keep, num = ops.nms_sorted(sb, None, 0.7, 300)
    got = keep[0, :int(num[0].item())].cpu().numpy()
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libmnc_ref.so")
    exact, against = None, None
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    if os.path.exists(ref_so):
        ref = ctypes.CDLL(ref_so)
        k_ref = np.zeros(10000, dtype=np.int32)
        n_ref = ctypes.c_int(0)
        ref._Z4_nmsPiS_PKfiifi(p(k_ref), ctypes.byref(n_ref), p(sorted_dets), 10000, 5, ctypes.c_float(0.7), 0)
        exact, against = bool(np.array_equal(got, k_ref[:300])), "reference _nms (oracle/_ref)"
    else:
        exact, against = bool(np.array_equal(got, O.nms_sorted(sorted_dets, 0.7)[:300])), "oracle"
    res["nms_10k_keep300"] = {"ms": ms, "kept": int(len(got)), "bit_exact": exact, "against": against,
                              "algorithmic_bytes": 10000 * 20 + 2 * 10000 * 157 * 8}
    # ---- configs[4]: gpu_mask_voting, 600 boxes x 21 classes at 600x1000
    from tests.test_ref_pin import _voting_inputs
    vb, vm, vs = _voting_inputs(600, 600, 1000, 11)
    tb, tm, ts = (torch.from_numpy(a).cuda()[None] for a in (vb, vm, vs))
    hw = torch.tensor([[600, 1000]], dtype=torch.int32, device="cuda")
    ms = median_ms(lambda: ops.mask_voting(tb, tm, ts, hw), iters=10)
    r = ops.mask_voting(tb, tm, ts, hw)
    inds, start, wts, cs, bar = O.mask_voting_candidates(vb, vs, 21, 100)
    k = int(r["n_res"][0])
    beg, end = r["cand_begin"][0, :k].cpu().numpy(), r["cand_end"][0, :k].cpu().numpy()
    ci, cw = r["cand_inds"][0].cpu().numpy().ravel(), r["cand_weights"][0].cpu().numpy().ravel()
    lists_ok = bool(k == len(start) and np.array_equal(np.concatenate([ci[b:e] for b, e in zip(beg, end)]), inds)
                    and np.array_equal(np.concatenate([cw[b:e] for b, e in zip(beg, end)]), wts))
    rm_o, rb_o = O.mv(vb, vm, inds, start, wts, 600, 1000)
    boxes_ok = bool(np.array_equal(r["result_box"][0, :k].cpu().numpy(), rb_o))
    res["mask_voting_600x21"] = {"ms": ms, "results": k, "candidates": int(len(inds)),
                                 "lists_bit_exact": lists_ok, "result_boxes_exact": boxes_ok,
                                 "against": "oracle (itself == reference _mv built -fmad=false, tests/test_ref_pin.py)"}
    return res


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, outs):
    """What one step of the timed path hands its caller (engine.detect_graphed: boxes, masks,
    scores, valid, and the RoI count per image) as float32 DIR/<name>.npy, so that two builds can
    be compared output for output.  If the masks would take the total over 64 MB (batch 60 and
    up), a fixed seeded sample of their rows is written instead, with the row numbers in
    masks_rows.npy."""
    import numpy as np
    boxes, masks, scores, valid, o = outs
    arrs = {name: t.float().cpu().numpy() for name, t in (
        ("boxes", boxes), ("masks", masks), ("scores", scores), ("valid", valid), ("roi_counts", o["roi_counts"]))}
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_LIMIT:
        m = arrs["masks"]
        flat = m.reshape(m.shape[0] * m.shape[1], -1)
        n = (DUMP_LIMIT - (total - m.nbytes)) // (flat.shape[1] * 4 + 8)
        rows = np.sort(np.random.default_rng(0).choice(flat.shape[0], n, replace=False))
        arrs["masks"], arrs["masks_rows"] = flat[rows], rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-micro", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-overlap-heads", action="store_true",
                    help="A/B: issue the box branch in line instead of on the side stream")
    ap.add_argument("--halo-split", action="store_true",
                    help="A/B: the halo kernel (Cout <= 128 convs) on split-bf16 operands")
    ap.add_argument("--streams", type=int, default=2, choices=[1, 2],
                    help="steps in flight: 2 = consecutive steps alternate between two streams (each "
                         "with its own activation buffers and CUDA graph over the shared weights)")
    ap.add_argument("--halo-single", action="store_true",
                    help="A/B: the halo kernel with one CTA per tile instead of CTA pairs")
    ap.add_argument("--nms-matrix", action="store_true",
                    help="A/B: proposal NMS through the n x n/64 suppression matrix (nms_mask + nms_scan) "
                         "instead of the capped form")
    ap.add_argument("--nms-single-cta", action="store_true",
                    help="A/B: the capped proposal NMS on one CTA per image instead of a cluster of 8")
    ap.add_argument("--nms-mode", type=int, default=None, choices=[0, 1, 2, 3],
                    help="A/B: capped proposal NMS form (3: cluster, 256-candidate rounds; 2: cluster, "
                         "64-candidate rounds; 1: one CTA per image; 0: suppression matrix)")
    ap.add_argument("--mv-full-sweep", action="store_true",
                    help="A/B: mask voting finds the tight boxes by one full sweep instead of two passes")
    ap.add_argument("--dump-igemm", default=None,
                    help="write the ordered list of tensor-core launches of one step "
                         "(shape, algorithmic FLOPs / bytes) as JSON, for scripts/ncu_tc_summary.py")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (rank 0's images) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    # a run that is still going after 5 minutes leaves the Python stacks of all threads on stderr
    # (the default line takes ~20 s on a warm box; one run of the round stalled without a trace)
    import faulthandler
    faulthandler.enable()
    faulthandler.dump_traceback_later(300, repeat=False, exit=False)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    ncpu = _pin_cpu_threads() if int(os.environ.get("WORLD_SIZE", "1")) == 1 else None
    import numpy as np
    import torch
    import torch.distributed as dist
    from mnc_b200 import weights as Wt, dense, _lib, ops
    from mnc_b200 import dist as mdist
    from mnc_b200.api import Detector

    rank, world, local = mdist.init_from_env()
    _log("imports done; rank %d of %d" % (rank, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B = args.batch
    w = Wt.make_weights(Wt.FULL_ARCH)
    if args.halo_split:
        from mnc_b200 import engine as _eng
        _eng.MNCEngine.HALO_TRI = False
    if args.halo_single:
        dense.set_halo_pair(0)
    if args.nms_matrix:
        ops.nms_set_lazy(0)
    if args.nms_single_cta:
        ops.nms_set_lazy(1)
    if args.nms_mode is not None:
        ops.nms_set_lazy(args.nms_mode)
    if args.mv_full_sweep:
        ops.mv_set_two_pass(False)
    _log("weights made; building the engine")
    det = Detector(w, device=dev, max_batch=B, height=H, width=W, use_graph=not args.no_graph)
    eng = det.engine
    eng.overlap_heads = not args.no_overlap_heads

    # synthetic inputs: image i of the global batch = seed 1234 + i (SURVEY.md section 8d)
    start, _ = mdist.shard_range(B * world, rank, world)
    u8 = np.stack([np.random.default_rng(1234 + start + i).integers(0, 256, size=(H, W, 3), dtype=np.uint8)
                   for i in range(B)])
    data = ops.prep_images(torch.from_numpy(u8).to(dev), 1.0)
    im_info = torch.tensor([[H, W, 1.0]] * B, dtype=torch.float32, device=dev)
    im_hw = torch.tensor([[H, W]] * B, dtype=torch.float32, device=dev)
    im_scale = torch.ones(B, dtype=torch.float32, device=dev)
    pipe = mdist.GatherPipe(dev, mdist.record_len(B))

    def step(graph=not args.no_graph, e=None):
        e = e or eng
        rec = pipe.send_buffer()
        if graph:
            outs = e.detect_graphed(data, im_info, im_hw, im_scale, rec=rec)
        else:
            o = e.forward(data, im_info)
            outs = e.detect_tail(o, B, im_hw, im_scale, rec=rec) + (o,)
        return outs, pipe.submit()

    for _ in range(args.warmup + 2):      # + 2: one graph capture per send buffer of the gather pipe
        (boxes, masks, scores, valid, o), gathered = step()
    pipe.drain()
    torch.cuda.synchronize()

    # two steps in flight: step k runs on stream k % 2 with engine k % 2 (shared weights, own
    # buffers and graph); the gather pipe's slot k % 2 is then always the same engine's record
    n_str = 1 if args.no_graph else args.streams
    engines = [eng] + [eng.clone_state() for _ in range(n_str - 1)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_str)] if n_str > 1 else [None]

    def step_k(k):
        if n_str == 1:
            return step()
        s = streams[k % n_str]
        with torch.cuda.stream(s):
            return step(e=engines[k % n_str])

    def fork():
        for s in streams:
            if s is not None:
                s.wait_stream(torch.cuda.current_stream(dev))

    def join():
        for s in streams:
            if s is not None:
                torch.cuda.current_stream(dev).wait_stream(s)

    if n_str > 1:
        fork()
        for k in range(2 * n_str + 2):    # captures the clones' graphs (one per send buffer), warms up
            step_k(k)
        join()
        pipe.drain()
        torch.cuda.synchronize()
        # the clone computes the same step: identical records
        ra = engines[0].last_record.clone()
        assert torch.equal(ra, engines[1].last_record), "two-stream engines disagree"
    counts = o["roi_counts"].cpu().numpy()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    _log("warm-up done (%d streams); timed region" % n_str)
    # ------------------------------------------------------------- timed region (device resident)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    torch.cuda.nvtx.range_push("timed")
    t_wall0 = time.perf_counter()
    ev[0].record()
    fork()
    for k in range(args.steps):
        last_outs, _ = step_k(k)
        if k + 1 < args.steps:
            ev[k + 1].record(streams[k % n_str] if n_str > 1 else None)
    join()
    pipe.drain()                           # the last step's gather is inside the timed region
    ev[args.steps].record()
    barrier()
    torch.cuda.nvtx.range_pop()
    t_wall = time.perf_counter() - t_wall0
    dev_ms = ev[0].elapsed_time(ev[args.steps])
    step_ms = sorted(ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps))
    clocks = sampler.finish() if rank == 0 else None
    tms = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    total_ms = float(tms.item())
    value = world * B * args.steps / (total_ms / 1000.0)
    if args.dump_outputs and rank == 0:
        # before the passes below reuse the engines' output buffers
        dump_outputs(args.dump_outputs, last_outs)

    # the collective alone (same buffers, main stream, nothing to overlap with)
    comm_ms = 0.0
    if world > 1:
        rec = pipe.send[0]
        out = pipe.recv[0]
        comm_ms = median_ms(lambda: mdist.all_gather_records(rec, out), iters=10)

    _log("timed region done: %.2f ms per step; eager pass" % (total_ms / args.steps))
    # ------------------------------------------------------------- eager pass: per-kernel roofline
    # (single stream: with the box branch forked to the side stream two fc6 launches share the GPU
    # and the events around each would count the overlap twice)
    dense.timer = dense.KernelTimer()
    launches0 = _lib.launch_count
    n_eager = 3
    overlap_saved, eng.overlap_heads = eng.overlap_heads, False
    for _ in range(n_eager):
        step(graph=False)
    pipe.drain()
    torch.cuda.synchronize()
    eng.overlap_heads = overlap_saved
    launches_per_step = (_lib.launch_count - launches0) // n_eager
    ktimer, dense.timer = dense.timer, None
    if args.dump_igemm and rank == 0:
        per = len(ktimer.manifest) // n_eager
        with open(args.dump_igemm, "w") as f:
            json.dump({"steps": 1, "launches": ktimer.manifest[-per:]}, f)

    _log("forward + voting")
    # ------------------------------------------------------------- forward + gpu_mask_voting
    # (the published 0.33 s/img covers im_detect only, tools/demo.py:144-147; BASELINE.md asks for
    # both numbers)
    im_hw_i = torch.tensor([[H, W]] * B, dtype=torch.int32, device=dev)

    def step_vote():
        bx, mk, sc, vl, _ = eng.detect_graphed(data, im_info, im_hw, im_scale) if not args.no_graph \
            else eng.detect(data, im_info, im_hw, im_scale)
        return ops.mask_voting(bx, mk, sc, im_hw_i, box_valid=vl)

    for _ in range(2):
        vr = step_vote()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        vr = step_vote()
    ev1.record()
    torch.cuda.synchronize()
    tv = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tv, op=dist.ReduceOp.MAX)
    vote_value = world * B * args.steps / (float(tv.item()) / 1000.0)
    n_instances = [int(x) for x in vr["n_res"].cpu().numpy()]

    _log("e2e (host buffers)")
    # ------------------------------------------------------------- e2e: host buffers in and out
    # the reference's callers hand im_detect the raw uint8 image (tools/demo.py:143-146); so does
    # this: uint8 BGR frames in host memory -> boxes / masks / scores in host memory (+ the
    # all-gather of the records when N > 1)
    def e2e_run(src, pipelined):
        def run(n):
            if pipelined:    # Detector.im_detect_stream: two batches in flight, copies off the critical path
                for res in det.im_detect_stream(src for _ in range(n)):
                    if world > 1:
                        mdist.all_gather_records(eng.last_record, pipe.recv[0])
                        torch.cuda.synchronize()
            else:            # one synchronous call per step
                for _ in range(n):
                    det.im_detect_images(src)
                    if world > 1:
                        mdist.all_gather_records(eng.last_record, pipe.recv[0])
                        torch.cuda.synchronize()
        run(3)
        barrier()
        t0 = time.perf_counter()
        run(args.steps)
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return world * B * args.steps / float(te.item())

    u8_pinned = torch.from_numpy(u8).pin_memory()
    e2e_pinned = e2e_run(u8_pinned, True)
    e2e_pageable = e2e_run(u8, True)       # a plain numpy array, as cv2.imread returns
    e2e_sync = e2e_run(u8_pinned, False)   # one blocking im_detect_images call per step

    _log("batch-1 latency")
    # ------------------------------------------------------------- batch-1 latency (configs[0])
    lat1 = None
    if world == 1:
        d1, i1, h1, s1 = data[:1].contiguous(), im_info[:1].contiguous(), im_hw[:1].contiguous(), im_scale[:1].contiguous()
        fn = (lambda: eng.detect_graphed(d1, i1, h1, s1)) if not args.no_graph else (lambda: eng.detect(d1, i1, h1, s1))
        lat1 = median_ms(fn, iters=20, warm=4)
        t0 = time.perf_counter()
        for _ in range(20):
            fn()
        host_ms1 = (time.perf_counter() - t0) * 1000.0 / 20      # host time to issue a step
        torch.cuda.synchronize()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ------------------------------------------------------------- roofline of the dominant kernel
    k_ms, k_flops, k_n = ktimer.totals()
    per_step = k_n // n_eager
    site_ms = [0.0] * per_step
    for i, (e0, e1, _, _) in enumerate(ktimer.records):
        site_ms[i % per_step] += e0.elapsed_time(e1) / n_eager
    site_tags = [ktimer.records[i][3] for i in range(per_step)]
    man = ktimer.manifest[:per_step]
    work = sum(m["flops"] * (2 if m.get("tri_in") else 3) for m in man)
    flops_step = sum(m["flops"] for m in man)
    k_ms_step = k_ms / n_eager
    peaks, peak_src = _peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    ach = flops_step / (k_ms_step / 1000.0) / 1e12 if k_ms_step > 0 else 0.0
    traffic, traffic_note = None, None
    for nm in ("r02_ncu_tc_summary.json", "r01_ncu_tc_summary.json"):
        summ = os.path.join(ROOT, "profiles", nm)
        if os.path.exists(summ):
            with open(summ) as f:
                sj = json.load(f)
            traffic = sj["mean_traffic_bytes_per_launch"]
            traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum per launch, mean over the %d "
                            "tensor-core launches of one step in the committed ncu --set full capture "
                            "(profiles/%s); algorithmic bytes of the same launches: %.3e per launch"
                            % (sj["n_launches"], nm, sj["mean_algorithmic_bytes_per_launch"]))
            break
    ms_step = total_ms / args.steps
    roofline = {
        "kernel": "igemm_tc_kernel / conv_halo_tc_kernel (tcgen05 implicit GEMM: 13 conv3x3 + 15 "
                  "inner-product launches per step)",
        "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
        "frac": ach / peak_tf, "traffic": traffic, "traffic_note": traffic_note,
        "peak_source": peak_src + ", bf16 dense sustained (kernel timed inside a long step)",
        "launches_timed": k_n, "share_of_step": k_ms_step / ms_step,
        "ms_by_launch_site": [[t, round(m, 4)] for t, m in zip(site_tags, site_ms)],
        "algorithmic_flops_per_step": flops_step,
        "tensor_work_factor": work / flops_step,
        "frac_tensor_pipe": (work / flops_step) * ach / peak_tf,
        "note": "fp32-parity arithmetic: launches with tri-plane operands issue one fp16 MMA + two "
                "FP8 MMAs (double rate) per algorithmic MAC = 2 bf16-equivalent units (conv1_1, not in "
                "this kernel's launch list, three bf16 MMAs); frac counts "
                "algorithmic FLOPs only, frac_tensor_pipe counts issued tensor work; per-launch "
                "times from CUDA events around each launch in an eager pass of the same step",
    }

    micro, roof_warp = None, None
    if world == 1 and not args.no_micro:
        _log("microbenchmarks (configs[3] / configs[4])")
        micro = microbench(hbm)
        rw = micro["roi_warp_P28"]
        roof_warp = {"kernel": "roi_warp_nchw_kernel (ROIWarping layer form, 2000 RoIs, 28x28, "
                               "512x38x63 map: BASELINE.json configs[3])",
                     "bound": "hbm", "achieved": rw["GBps"], "peak": hbm, "unit": "GB/s",
                     "frac": rw["frac_of_hbm"], "traffic": None,
                     "algorithmic_bytes": rw["algorithmic_bytes"], "peak_source": peak_src + ", copy bandwidth"}

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        torch.set_num_threads(ncpu)
        _log("cpu baseline (oracle on %d host threads, <= 5 images, 45 s budget)" % ncpu)
        times = cpu_reference_time(w, 5, 2)
        st = _summ(times)
        cpu = {"value": 1.0 / st["median_s"], "unit": "images/s", "cores": ncpu, "kind": "port",
               "sample": "%d images (600x1000, 300 RoIs/stage) after <= 2 warm-up images (45 s budget), oracle port "
                         "(torch CPU fp32 conv/FC + numpy layers + C kernels); 1 / median" % len(times),
               "per_image_s": st}

    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f16+2xf8 (fp16 main product + two e4m3 correction products on tcgen05, fp32 "
                 "accumulate, fp32-parity; conv1_1, K = 27: bf16x3)" if not args.halo_split else
                 "f16+2xf8 (Cout > 128 convs, inner products), bf16x3 (Cout <= 128 convs)",
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": e2e_pinned, "unit": "images/s", "h2d_bytes_per_step": det.h2d_bytes,
                "d2h_bytes_per_step": det.d2h_bytes,
                "value_pageable_input": e2e_pageable, "value_blocking_calls": e2e_sync,
                "api": "mnc_b200.api.Detector.im_detect_stream (value, value_pageable_input: every "
                       "step's uint8 BGR host frames -> H2D -> mean/resize/NCHW on device -> forward "
                       "(CUDA-graph replay) -> im_detect tail -> one record D2H -> host arrays; two "
                       "batches in flight so the copies overlap the previous batch's compute; value: "
                       "page-locked caller memory, value_pageable_input: a plain numpy array staged "
                       "through the Detector's pinned buffer) and Detector.im_detect_images "
                       "(value_blocking_calls: one synchronous call per step)"
                       + ("; + all-gather of the records" if world > 1 else "")},
        "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
        "clocks": clocks, "roofline": roofline, "roofline_roi_warp": roof_warp, "micro": micro,
        "cpu_baseline": cpu,
        "step_ms": {"median": step_ms[len(step_ms) // 2], "p10": step_ms[int(0.1 * len(step_ms))],
                    "p90": step_ms[min(len(step_ms) - 1, int(0.9 * len(step_ms)))]},
        "comm_ms_per_step": comm_ms,
        "comm_note": "all_gather_into_tensor of the %d-float record per rank, alone on an idle GPU; "
                     "in the timed loop it runs on a side stream under the next step's trunk"
                     % mdist.record_len(B),
        "latency_batch1_ms": lat1, "host_issue_ms_batch1": host_ms1 if world == 1 else None,
        "cuda_graph": not args.no_graph,
        "steps_in_flight": n_str,
        "steps_in_flight_note": "consecutive steps alternate between %d stream(s), each with its own "
                                "activation buffers and CUDA graph over the shared weights; the K timed "
                                "steps all complete inside the timed region" % n_str,
        "forward_plus_voting": {"value": vote_value, "unit": "images/s",
                                "instances_per_image": n_instances,
                                "note": "im_detect + batched device gpu_mask_voting (100 per image)"},
        "rois_per_image": [int(c) for c in counts],
        "published_reference": {"s_per_img": 0.33, "hardware": "Titan X", "source": "README.md:44"},
        "speedup_vs_published_titanx": value / world * 0.33,
        "wall_s_timed_region": t_wall,
    }
    _emit(line)
    _log("done")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
