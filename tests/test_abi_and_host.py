"""CPU tests: the C-ABI library loads and exports every symbol the header declares (no compute
calls without a GPU), and the host-side logic (prototxt reader, graph check, cfg, sharding,
record packing, weight container, host bbox helpers)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "mnc_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = sorted(set(re.findall(r"\b(mnc_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 30
    so = os.path.join(ROOT, "mnc_b200", "libmnc_b200.so")
    assert os.path.exists(so), "build the library first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(so)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert lib.mnc_abi_version() == 1


def test_anchor_generator_in_library_matches_known_answer():
    """host-only entry point (no kernel launch): lib/transform/anchors.py:15-35 minus one."""
    lib = ctypes.CDLL(os.path.join(ROOT, "mnc_b200", "libmnc_b200.so"))
    out = np.zeros((9, 4), dtype=np.float32)
    assert lib.mnc_generate_anchors(out.ctypes.data_as(ctypes.c_void_p)) == 0
    assert list(out[0]) == [-84, -40, 99, 55] and list(out[8]) == [-168, -344, 183, 359]
    from oracle import oracle as O
    assert np.array_equal(out.astype(np.float64), O.generate_anchors())


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    import importlib
    import mnc_b200._lib as L
    monkeypatch.setattr(L, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(ImportError):
        L._load()
    importlib.reload(L)


def test_prototxt_reader_and_graph_check(tmp_path):
    import mnc_b200.lib as lib
    lib.install()
    from caffe import mnc_graph
    g = mnc_graph.build_graph()
    types = [l["type"] for l in g]
    # layer census of models/VGG16/mnc_5stage/test.prototxt (SURVEY.md section 2.1)
    assert types.count("Convolution") == 16 and types.count("InnerProduct") == 18
    assert types.count("Pooling") == 9 and types.count("ReLU") == 24 and types.count("Softmax") == 5
    assert types.count("ROIWarping") == 2 and types.count("MaskResize") == 2
    assert types.count("MaskPooling") == 2 and types.count("Python") == 4 and types.count("Concat") == 2

    def emit(layers, inputs=("data", "im_info")):
        out = ['name: "VGG16"']
        for name in inputs:
            out += ['input: "%s"' % name, "input_shape { dim: 1 dim: 3 }"]
        for l in layers:
            s = ["layer {", '  name: "%s"' % l["name"], '  type: "%s"' % l["type"]]
            s += ['  bottom: "%s"' % b for b in l["bottom"]] + ['  top: "%s"' % t for t in l["top"]]
            for k, v in l.items():
                if isinstance(v, dict):
                    s.append("  %s {" % k)
                    for kk, vv in v.items():
                        s.append("    %s: %s  # c" % (kk, ('"%s"' % vv) if isinstance(vv, str) and kk != "pool" else vv))
                    s.append("  }")
            s.append("}")
            out.append("\n".join(s))
        return "\n".join(out)
    p = tmp_path / "test.prototxt"
    p.write_text(emit(g))
    assert len(mnc_graph.check_prototxt(str(p))) == len(g)
    bad = [dict(l) for l in g]
    bad[-1] = dict(bad[-1], inner_product_param=dict(num_output=80))
    p.write_text(emit(bad))
    with pytest.raises(ValueError):
        mnc_graph.check_prototxt(str(p))
    # the sibling test graphs (SURVEY.md section 8f row 4) are told apart by their layers
    for kind, n_layers in (("faster_rcnn", 48), ("cfm", 52)):
        gk = mnc_graph.GRAPHS[kind]()
        assert len(gk) == n_layers
        p.write_text(emit(gk, mnc_graph.GRAPH_INPUTS[kind]))
        assert mnc_graph.identify_prototxt(str(p))[0] == kind
        with pytest.raises(ValueError):
            mnc_graph.check_prototxt(str(p))          # not the 5-stage graph
    p.write_text(emit(mnc_graph.GRAPHS["cfm"](), ("data", "im_info")))
    with pytest.raises(ValueError):
        mnc_graph.identify_prototxt(str(p))           # CFM layers with the wrong inputs
    # the original project's own prototxts (models/VGG16/, copied unmodified)
    base = os.path.join(ROOT, "tests", "golden", "models", "VGG16") + os.sep
    assert len(mnc_graph.check_prototxt(base + "mnc_5stage/test.prototxt")) == 88
    assert mnc_graph.identify_prototxt(base + "faster_rcnn_end2end/test.prototxt")[0] == "faster_rcnn"
    assert mnc_graph.identify_prototxt(base + "cfm/test.prototxt")[0] == "cfm"
    with pytest.raises(ValueError):
        mnc_graph.identify_prototxt(base + "mnc_5stage/train.prototxt")


def test_cfg_constants():
    import mnc_b200.lib as lib
    lib.install()
    from mnc_config import cfg
    assert cfg.USE_GPU_NMS and cfg.MASK_SIZE == 21 and cfg.BINARIZE_THRESH == 0.4
    assert cfg.TEST.RPN_PRE_NMS_TOP_N == 6000 and cfg.TEST.RPN_POST_NMS_TOP_N == 300
    assert cfg.TEST.RPN_NMS_THRESH == 0.7 and cfg.TEST.RPN_MIN_SIZE == 16
    assert cfg.TEST.MASK_MERGE_IOU_THRESH == 0.5 and cfg.TEST.MASK_MERGE_NMS_THRESH == 0.3
    assert cfg["TEST"].SCALES == (600,) and cfg.TRAIN.MAX_SIZE == 1000


def test_host_bbox_helpers_match_oracle():
    import mnc_b200.lib as lib
    lib.install()
    from transform import bbox_transform as T
    from oracle import oracle as O
    rng = np.random.default_rng(0)
    boxes = (rng.uniform(0, 500, size=(50, 4))).astype(np.float32)
    boxes[:, 2:] += boxes[:, :2]
    d = rng.normal(0, 0.3, size=(50, 8)).astype(np.float32)
    assert np.array_equal(T.bbox_transform_inv(boxes, d), O.bbox_transform_inv(boxes, d))
    a, ka = T.clip_boxes(boxes * 2 - 100, (600, 1000, 3))
    b, kb = O.clip_boxes(boxes * 2 - 100, (600, 1000, 3))
    assert np.array_equal(a, b) and np.array_equal(ka, kb)
    assert np.array_equal(T.filter_small_boxes(boxes, 40), O.filter_small_boxes(boxes, 40))
    assert T.bbox_transform_inv(np.zeros((0, 4), np.float32), np.zeros((0, 8), np.float32)).shape == (0, 8)


def test_blob_and_layer_protocol():
    import mnc_b200.lib as lib
    lib.install()
    import caffe
    from pylayer.mask_layer import MaskLayer
    b = caffe.Blob(2, 3, 4, 5)
    assert (b.num, b.channels, b.height, b.width, b.count) == (2, 3, 4, 5, 120)
    b.reshape(7, 441)
    assert b.shape == (7, 441) and b.data.dtype == np.float32
    b.data[...] = np.arange(7 * 441).reshape(7, 441)
    top = [caffe.Blob()]
    layer = MaskLayer(phase=caffe.TEST)
    assert str(layer.phase) == "TEST"
    layer.setup([b], top)
    layer.forward([b], top)
    assert top[0].shape == (7, 1, 21, 21) and top[0].data[3, 0, 20, 20] == b.data[3, 440]


def test_shard_range_and_records():
    from mnc_b200 import dist as D
    for total, world in ((64, 8), (10, 4), (3, 8), (8, 1)):
        got = [D.shard_range(total, r, world) for r in range(world)]
        assert got[0][0] == 0 and got[-1][1] == total
        assert all(got[i][1] == got[i + 1][0] for i in range(world - 1))
        assert max(e - s for s, e in got) - min(e - s for s, e in got) <= 1
    B = 3
    boxes = torch.rand(B, 600, 4)
    masks = torch.rand(B, 600, 1, 21, 21)
    scores = torch.rand(B, 600, 21)
    valid = (torch.rand(B, 600) > 0.3).to(torch.uint8)
    rec = D.pack_records(boxes, masks, scores, valid)
    assert rec.shape == (D.record_len(B),)
    c, b2, m2, s2 = D.unpack_records(rec.view(1, -1), B)
    assert torch.equal(b2, boxes) and torch.equal(m2, masks) and torch.equal(s2, scores)
    assert torch.equal(c, valid.sum(1).to(torch.int64))


def test_weight_container():
    from mnc_b200 import weights as Wt
    w = Wt.make_weights(Wt.TINY_ARCH)
    w2 = Wt.make_weights(Wt.TINY_ARCH)
    assert all(torch.equal(w[k][0], w2[k][0]) for k in w)      # seeded
    assert Wt.arch_of(w) == Wt.TINY_ARCH
    assert w["fc6"][0].shape == (256, 64 * 49) and w["fc6_maskest"][0].shape == (64, 64 * 196)
    assert w["cls_score"][0].shape == (21, 512) and w["bbox_pred"][0].shape == (84, 512)
    assert w["rpn_cls_score"][0].shape == (18, 64, 1, 1)
    full = Wt.FULL_ARCH
    assert full["trunk"][-1] == 512 and full["fc"] == 4096   # Appendix A shapes


def test_split_representation():
    from mnc_b200 import weights  # noqa: F401  (package import must work without a GPU)
    x = torch.randn(1000) * 10
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    err = ((hi.float() + lo.float()) - x).abs() / x.abs().clamp_min(1e-6)
    assert err.max() < 2 ** -15


def test_caffemodel_roundtrip_and_protobuf_crosscheck(tmp_path):
    """`.caffemodel` reader/writer (SURVEY.md section 8f row 2): round trip of the MNC weight set,
    and a cross-check of the hand-rolled wire-format reader against the protobuf runtime on a
    message built with the same field numbers as caffe.proto."""
    from mnc_b200 import weights as Wt, caffemodel as CM
    w = Wt.make_weights(Wt.TINY_ARCH)
    p = str(tmp_path / "mnc_tiny.caffemodel")
    CM.save_caffemodel(w, p)
    layers = CM.load_caffemodel(p)
    assert set(layers.keys()) == set(w.keys())
    back = CM.weights_from_caffemodel(p)
    assert all(torch.equal(back[k][0], w[k][0]) and torch.equal(back[k][1], w[k][1]) for k in w)
    assert back["fc6"][0].shape == w["fc6"][0].shape and back["conv1_1"][0].shape == (64, 3, 3, 3)
    # legacy blobs: 4-D dims in fields 1..4, non-packed floats, V1 `layers` (field 2)
    def vint(v):
        out = bytearray()
        while True:
            b = v & 0x7F
            v >>= 7
            out.append(b | (0x80 if v else 0))
            if not v:
                return bytes(out)
    import struct
    blob = b"".join(vint((f << 3) | 0) + vint(d) for f, d in ((1, 1), (2, 1), (3, 2), (4, 3)))
    blob += b"".join(vint((5 << 3) | 5) + struct.pack("<f", float(i)) for i in range(6))
    layer = vint((4 << 3) | 2) + vint(3) + b"ip1" + vint((6 << 3) | 2) + vint(len(blob)) + blob
    net = vint((2 << 3) | 2) + vint(len(layer)) + layer
    q = tmp_path / "legacy.caffemodel"
    q.write_bytes(net)
    got = CM.load_caffemodel(str(q))
    assert list(got) == ["ip1"] and got["ip1"][0].shape == (1, 1, 2, 3)
    assert np.array_equal(got["ip1"][0].ravel(), np.arange(6, dtype=np.float32))
    with pytest.raises(KeyError):
        CM.weights_from_caffemodel(str(q))
    # sibling graphs: Faster R-CNN snapshots name the RPN conv `rpn_conv/3x3`
    # (faster_rcnn_end2end/test.prototxt:391); CFM snapshots have no RPN at all
    wf = Wt.make_sibling_weights("faster_rcnn", Wt.TINY_ARCH)
    renamed = {("rpn_conv/3x3" if k == "rpn_conv_3x3" else k): v for k, v in wf.items()}
    pf = str(tmp_path / "frcnn_tiny.caffemodel")
    CM.save_caffemodel(renamed, pf)
    bf = CM.weights_from_caffemodel(pf, "faster_rcnn")
    assert set(bf) == set(wf) and torch.equal(bf["rpn_conv_3x3"][0], wf["rpn_conv_3x3"][0])
    assert bf["cls_score"][0].shape == (21, Wt.TINY_ARCH["fc"])
    with pytest.raises(KeyError):
        CM.weights_from_caffemodel(pf, "mnc_5stage")
    wc = Wt.make_sibling_weights("cfm", Wt.TINY_ARCH)
    pc = str(tmp_path / "cfm_tiny.caffemodel")
    CM.save_caffemodel(wc, pc)
    assert set(CM.weights_from_caffemodel(pc, "cfm")) == set(wc)


def test_eval_host_helpers_match_oracle_and_voc_palette():
    """voc_ap / mask_overlap / colour map of the evaluator boundary (SURVEY.md 8f row 3) against the
    oracle restatements and the published PASCAL VOC palette (known answers)."""
    import mnc_b200.lib as L
    L.install()
    from utils.voc_eval import voc_ap
    from utils.vis_seg import _get_voc_color_map, get_vis_dict
    from transform.mask_transform import mask_overlap
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    for trial in range(5):
        hits = rng.integers(0, 2, 80)
        tp, fp = np.cumsum(hits), np.cumsum(1 - hits)
        rec, prec = tp / 57.0, tp / np.maximum(tp + fp, np.finfo(np.float64).eps)
        assert voc_ap(rec, prec, True) == O.voc_ap(rec, prec, True)
        assert voc_ap(rec, prec, False) == pytest.approx(O.voc_ap(rec, prec, False), abs=1e-15)
    assert voc_ap(np.zeros(0), np.zeros(0), True) == 0.0
    for trial in range(20):
        b1 = rng.integers(0, 40, 2); b1 = np.concatenate([b1, b1 + rng.integers(0, 30, 2)])
        b2 = rng.integers(0, 40, 2); b2 = np.concatenate([b2, b2 + rng.integers(0, 30, 2)])
        m1 = rng.uniform(size=(b1[3] - b1[1] + 1, b1[2] - b1[0] + 1)) > 0.5
        m2 = rng.uniform(size=(b2[3] - b2[1] + 1, b2[2] - b2[0] + 1)) > 0.3
        assert mask_overlap(b1, b2, m1, m2) == O.mask_overlap(b1, b2, m1, m2)
    cmap = _get_voc_color_map()
    assert np.array_equal(cmap, O.voc_color_map())
    assert cmap[1].tolist() == [128, 0, 0] and cmap[15].tolist() == [192, 128, 128]
    assert cmap[20].tolist() == [0, 64, 128] and cmap[255].tolist() == [224, 224, 192]
    dets = [np.array([[1, 2, 3, 4, 0.9], [5, 6, 7, 8, 0.2]], np.float32), np.zeros((0, 5), np.float32)]
    segs = [np.ones((2, 1, 21, 21), np.float32), np.zeros((0, 1, 21, 21), np.float32)]
    d = get_vis_dict(dets, segs, "n", ["a", "b"], vis_thresh=0.5)
    assert d["cls_name"] == [1] and d["boxes"][0][4] == np.float32(0.9) and d["masks"][0].shape == (21, 21)


def test_hdf5_reader_on_reference_test_files_and_caffemodel_h5(tmp_path):
    """mnc_b200/hdf5_min.py (SURVEY.md 8f row 2, `.caffemodel.h5`): (1) the reference's own HDF5 test
    files, whose contents its generator script defines (caffe-mnc/src/caffe/test/test_data/
    generate_sample_data.py:13-52) -- contiguous float32, and gzip-chunked float32 / uint8;
    (2) a Net::ToHDF5-shaped weight file (net.cpp:920-975: /data/<layer>/<param id>, empty groups for
    parameter-sharing layers, a /diff group) assembled byte by byte, 26 layer groups so the group
    B-tree spans several symbol-table nodes; (3) the engine weight dict from it."""
    from mnc_b200 import hdf5_min, weights as Wt, caffemodel as CM
    from tests.util import write_h5_tree
    # caffe-mnc/src/caffe/test/test_data/*.h5, copied unmodified
    base = os.path.join(ROOT, "tests", "golden", "caffe_test_data") + os.sep
    data = np.arange(10 * 8 * 6 * 5).reshape(10, 8, 6, 5).astype(np.float32)
    label = (1 + np.arange(10)[:, None]).astype(np.float32)
    d = hdf5_min.read_hdf5(base + "sample_data.h5")
    assert set(d) == {"/data", "/label", "/label2"}
    assert np.array_equal(d["/data"], data) and np.array_equal(d["/label"], label)
    assert np.array_equal(d["/label2"], label + 1)
    g = hdf5_min.read_hdf5(base + "sample_data_2_gzip.h5")
    assert np.array_equal(g["/data"], data + data.size) and g["/label"].dtype == np.uint8
    assert np.array_equal(g["/label2"], (label + 1).astype(np.uint8))
    s = hdf5_min.read_hdf5(base + "solver_data.h5")
    assert s["/data"].shape == (8, 3, 10, 10) and s["/targets"].shape == (8, 1)
    w = Wt.make_weights(Wt.TINY_ARCH)
    tree = {"data": {}, "diff": {}}
    for name, (wt, b) in w.items():
        tree["data"][name] = {"0": wt.numpy(), "1": b.numpy()}
    tree["data"]["fc6_ext"] = {}                      # parameter-sharing layer: group without datasets
    tree["data"]["relu1_1"] = {}
    p = str(tmp_path / "mnc_tiny.caffemodel.h5")
    write_h5_tree(p, tree)
    layers = hdf5_min.load_caffemodel_h5(p)
    assert set(layers) == set(w) and len(w) >= 25
    back = CM.weights_from_caffemodel(p)
    assert all(torch.equal(back[k][0], w[k][0]) and torch.equal(back[k][1], w[k][1]) for k in w)
    # layer names with '/' are nested groups in the file (faster_rcnn_end2end: "rpn_conv/3x3")
    wf = Wt.make_sibling_weights("faster_rcnn", Wt.TINY_ARCH)
    tf = {"data": {}}
    for name, (wt, b) in wf.items():
        if name == "rpn_conv_3x3":
            tf["data"]["rpn_conv"] = {"3x3": {"0": wt.numpy(), "1": b.numpy()}}
        else:
            tf["data"][name] = {"0": wt.numpy(), "1": b.numpy()}
    pf = str(tmp_path / "frcnn_tiny.caffemodel.h5")
    write_h5_tree(pf, tf)
    bf = CM.weights_from_caffemodel(pf, "faster_rcnn")
    assert set(bf) == set(wf) and torch.equal(bf["rpn_conv_3x3"][0], wf["rpn_conv_3x3"][0])
    with pytest.raises(ValueError):
        bad = tmp_path / "x.h5"
        bad.write_bytes(b"not hdf5" * 100)
        hdf5_min.read_hdf5(str(bad))


def test_voc_seg_result_files_writer(tmp_path):
    """`<cls>_det.pkl` / `<cls>_seg.pkl` as PascalVOCSeg writes them (pascal_voc_seg.py:160-193):
    masks reshaped to (n, 21, 21) and binarised at 0.4, empty entries stay empty lists."""
    import pickle
    import mnc_b200.lib as L
    L.install()
    from utils.voc_eval import write_voc_seg_results_file
    classes = ["__background__", "aeroplane", "bicycle"]
    rng = np.random.default_rng(0)
    boxes = [[[] for _ in range(2)] for _ in range(3)]
    masks = [[[] for _ in range(2)] for _ in range(3)]
    boxes[1][0] = rng.uniform(0, 50, (3, 5)).astype(np.float32)
    masks[1][0] = rng.uniform(0, 1, (3, 1, 21, 21)).astype(np.float32)
    boxes[2][1] = rng.uniform(0, 50, (1, 5)).astype(np.float32)
    masks[2][1] = rng.uniform(0, 1, (1, 441)).astype(np.float32)      # (n, sz*sz) is accepted too
    paths = write_voc_seg_results_file(boxes, masks, classes, str(tmp_path / "res"))
    assert sorted(os.path.basename(p) for p in paths) == ["aeroplane_det.pkl", "aeroplane_seg.pkl",
                                                          "bicycle_det.pkl", "bicycle_seg.pkl"]
    with open(tmp_path / "res" / "aeroplane_seg.pkl", "rb") as f:
        seg = pickle.load(f)
    with open(tmp_path / "res" / "aeroplane_det.pkl", "rb") as f:
        det = pickle.load(f)
    assert seg[0].shape == (3, 21, 21) and seg[0].dtype == bool and len(seg[1]) == 0
    assert np.array_equal(seg[0], masks[1][0].reshape(3, 21, 21) >= 0.4)
    assert np.array_equal(det[0], boxes[1][0]) and len(det[1]) == 0
    with open(tmp_path / "res" / "bicycle_seg.pkl", "rb") as f:
        assert pickle.load(f)[1].shape == (1, 21, 21)


def test_sbd_ground_truth_cache(tmp_path):
    """parse_inst / check_voc_sds_cache (voc_eval.py:306-391) on SBD-shaped .mat files: tight bounds,
    masks cropped to them, class from the class map, per-class {image: [instances]} pickles, and the
    cache is not rebuilt when complete."""
    import pickle
    import scipy.io as sio
    import mnc_b200.lib as L
    L.install()
    from utils.voc_eval import parse_inst, check_voc_sds_cache
    dev = tmp_path / "sbd"
    (dev / "inst").mkdir(parents=True)
    (dev / "cls").mkdir()
    inst = np.zeros((40, 60), np.uint8)
    cls = np.zeros((40, 60), np.uint8)
    inst[5:15, 10:30] = 1; cls[5:15, 10:30] = 2          # instance 1: class 2, a full rectangle
    inst[20:35, 40:55] = 2; cls[20:35, 40:55] = 1        # instance 2: class 1 ...
    inst[22:25, 42:45] = 0; cls[22:25, 42:45] = 0        # ... with a hole
    inst[0:3, 0:3] = 3; cls[0:3, 0:3] = 2                # instance 3: class 2 again
    for name in ("im_a", "im_b"):
        sio.savemat(str(dev / "inst" / (name + ".mat")), {"GTinst": {"Segmentation": inst, "Categories": np.array([2, 1, 2])}})
        sio.savemat(str(dev / "cls" / (name + ".mat")), {"GTcls": {"Segmentation": cls}})
    rec = parse_inst("im_a", str(dev))
    assert [int(r["mask_cls"]) for r in rec] == [2, 1, 2]
    assert rec[0]["mask_bound"].tolist() == [10, 5, 29, 14] and rec[0]["mask"].all()
    assert rec[1]["mask_bound"].tolist() == [40, 20, 54, 34] and rec[1]["mask"].shape == (15, 15)
    assert rec[1]["mask"].sum() == 15 * 15 - 9 and rec[2]["mask_bound"].tolist() == [0, 0, 2, 2]
    names = ["__background__", "aeroplane", "bicycle"]
    cache = tmp_path / "cache"
    check_voc_sds_cache(str(cache), str(dev), ["im_a", "im_b"], names)
    with open(cache / "bicycle_mask_gt.pkl", "rb") as f:
        gt = pickle.load(f)
    assert set(gt) == {"im_a", "im_b"} and len(gt["im_a"]) == 2 and gt["im_a"][0]["already_detect"] is False
    with open(cache / "aeroplane_mask_gt.pkl", "rb") as f:
        assert [len(v) for v in pickle.load(f).values()] == [1, 1]
    stamp = (cache / "bicycle_mask_gt.pkl").stat().st_mtime_ns
    check_voc_sds_cache(str(cache), str(tmp_path / "nowhere"), ["im_a"], names)   # complete: not rebuilt
    assert (cache / "bicycle_mask_gt.pkl").stat().st_mtime_ns == stamp


def test_split_k_model_counts_cta_pair_work_items():
    """engine.pick_split_k: the factor is chosen in the kernel's own scheduling unit (CTA-pair work
    items on sms/2 slots, igemm_tc.cu launch_igemm), not single tiles on all SMs."""
    import math
    from mnc_b200.engine import pick_split_k

    def pick(M, N, K, bn, **kw):
        return pick_split_k(math.ceil(M / 128), math.ceil(N / bn), K // 64, 148, 2, out_elems=M * N, **kw)

    def waves(M, N, bn, s):
        return math.ceil(M / 256) * math.ceil(N / bn) * s / 74.0

    # launches that fill the GPU are never split (fc6 / fc7 at the benchmarked batch 8)
    assert pick(2400, 4096, 25088, 192) == 1 and pick(2400, 4096, 4096, 192) == 1
    # fc6_maskest at batch 8: 10 row pairs -> 7 splits = 70 items = one wave (15 was three waves)
    s = pick(2400, 256, 100352, 256)
    assert s == 7 and waves(2400, 256, 256, s) <= 1.0
    # batch 1: fc6 (2 row pairs x 22 Cout tiles) -> 5 splits = 220 items = 2.97 waves
    s = pick(300, 4096, 25088, 192)
    assert s == 5 and 2.9 < waves(300, 4096, 192, s) <= 3.0
    # tiny K is never split; the conv path caps the factor at 4
    assert pick(300, 441, 256, 256) == 1
    assert pick_split_k(20, 2, 72, 148, 2, max_split=4, out_elems=2394 * 512) <= 4
    # single-CTA scheduling (cluster 1) keeps the old counting
    assert pick_split_k(19, 1, 1568, 148, 1, out_elems=2400 * 256) in range(2, 33)


def test_bench_cpu_arm_is_bounded_and_counts_usable_cores(monkeypatch):
    """bench.py's CPU arm: the thread count honours the affinity mask / cgroup quota and the image
    loop stops at its time budget with at least one timed image."""
    import sys
    import types
    import bench
    n = bench.usable_cores()
    assert 1 <= n <= bench.physical_cores()
    assert n <= len(__import__("os").sched_getaffinity(0))
    calls = []
    clock = [0.0]
    fake = types.SimpleNamespace(synthetic_image=lambda it, H, W: it,
                                 im_detect=lambda w, im: (calls.append(im), clock.__setitem__(0, clock[0] + 20.0)))
    import oracle
    monkeypatch.setattr(oracle, "oracle", fake, raising=False)
    monkeypatch.setitem(sys.modules, "oracle.oracle", fake)
    monkeypatch.setattr(bench.time, "perf_counter", lambda: clock[0])
    times = bench.cpu_reference_time(None, images=5, warmup=2, budget_s=45.0)
    # every image "takes" 20 s: slower than budget / 3, so no image is spent on warm-up, and the loop
    # stops once the 45 s budget is exceeded: images at t = 0, 20, 40 are timed, the 4th never starts
    assert len(times) == 3 and all(abs(t - 20.0) < 1e-9 for t in times) and len(calls) == 3
    clock[0] = 0.0
    fast = types.SimpleNamespace(synthetic_image=lambda it, H, W: it,
                                 im_detect=lambda w, im: clock.__setitem__(0, clock[0] + 1.0))
    monkeypatch.setitem(sys.modules, "oracle.oracle", fast)
    monkeypatch.setattr(oracle, "oracle", fast, raising=False)
    times = bench.cpu_reference_time(None, images=5, warmup=2, budget_s=45.0)
    assert len(times) == 5                       # 2 warm-ups + 5 timed images fit the budget
