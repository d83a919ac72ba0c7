"""caffe.Net for the MNC 5-stage test graph, on the fused B200 engine."""
from collections import OrderedDict

import numpy as np


def kind_of_weights(weights):
    """Graph kind implied by which layers a weight dict holds."""
    if "rpn_conv_3x3" not in weights:
        return "cfm"
    return "mnc_5stage" if "fc6_maskest" in weights else "faster_rcnn"


def load_weights(prototxt=None, weights=None, return_kind=False):
    """Resolve the arguments of caffe.Net into the engine's {layer: (weight, bias)} dict.  The
    prototxt must be one of the supported test graphs (mnc_graph.identify_prototxt); without one
    the graph kind follows from the layers present in `weights`."""
    import torch
    from mnc_b200.weights import make_weights, make_sibling_weights
    from . import mnc_graph
    kind = mnc_graph.identify_prototxt(prototxt)[0] if prototxt is not None else None
    if weights is None:
        kind = kind or "mnc_5stage"
        weights = make_weights() if kind == "mnc_5stage" else make_sibling_weights(kind)
    elif isinstance(weights, str) and weights.endswith((".caffemodel", ".caffemodel.h5", ".h5")):
        from mnc_b200.caffemodel import weights_from_caffemodel
        weights = weights_from_caffemodel(weights, kind or "mnc_5stage")   # by layer name
    elif isinstance(weights, str):
        weights = torch.load(weights, map_location="cpu")
    if kind is None:
        kind = kind_of_weights(weights)
    elif kind != kind_of_weights(weights):
        raise ValueError("weights hold the %s layer set, prototxt is the %s graph" % (
            kind_of_weights(weights), kind))
    return (weights, kind) if return_kind else weights


_OUTPUTS = {"mnc_5stage": ["cls_prob", "cls_prob_ext", "bbox_pred_ext"],
            "faster_rcnn": ["cls_prob", "bbox_pred"],
            "cfm": ["mask_prob", "cls_prob", "seg_cls_prob", "bbox_pred"]}


class Net(object):
    """Net(prototxt, weights, phase).

    prototxt : path to one of the reference's test graphs -- models/VGG16/mnc_5stage/test.prototxt,
               faster_rcnn_end2end/test.prototxt or cfm/test.prototxt (checked layer by layer
               against mnc_graph) -- or None (graph implied by the weights; default 5-stage).
    weights  : {caffe layer name: (weight, bias)} dict, a binary `.caffemodel`
               or HDF5 `.caffemodel.h5` (mnc_b200/caffemodel.py, hdf5_min.py), a torch-saved file of
               such a dict, or None for the seeded random initialiser (mnc_b200/weights.py).
    """

    def __init__(self, prototxt=None, weights=None, phase=1):
        import torch
        from mnc_b200.engine import MNCEngine
        from mnc_b200.siblings import FasterRCNNEngine, CFMEngine
        from . import Blob, _state, mnc_graph
        if phase != 1:
            raise NotImplementedError("inference (caffe.TEST) only")
        weights, kind = load_weights(prototxt, weights, return_kind=True)
        self.kind = kind
        self._graph = mnc_graph.GRAPHS[kind]()
        self._device = torch.device("cuda", _state["device"])
        cls = {"mnc_5stage": MNCEngine, "faster_rcnn": FasterRCNNEngine, "cfm": CFMEngine}[kind]
        with torch.cuda.device(self._device):
            self._engine = cls(weights, device=self._device)
        self.name = "VGG16"
        self.inputs = list(mnc_graph.GRAPH_INPUTS[kind])
        self.blobs = OrderedDict()
        self.blobs["data"] = Blob(1, 3, 224, 224)     # input_shape of test.prototxt:3-9
        if kind == "cfm":
            self.blobs["rois"] = Blob(1, 5)           # cfm/test.prototxt:11-15
            self.blobs["masks"] = Blob(1, 1, 14, 14)  # :17-23
        else:
            self.blobs["im_info"] = Blob(1, 3)        # :11-15
        for layer in self._graph:
            for t in layer["top"]:
                if t not in self.blobs:
                    self.blobs[t] = Blob()
        self.outputs = list(_OUTPUTS[kind])

    def _set_inputs(self, kwargs):
        if kwargs:
            if set(kwargs.keys()) != set(self.inputs):
                raise Exception("Input blob arguments do not match net inputs.")
            for in_, blob in kwargs.items():
                if blob.shape[0] != self.blobs[in_].num:
                    raise Exception("Input is not batch sized")
                self.blobs[in_].data[...] = blob

    def _forward_siblings(self):
        import torch
        from mnc_b200 import dense
        dev = self._device
        t = lambda name: torch.from_numpy(np.ascontiguousarray(self.blobs[name].data, dtype=np.float32)).to(dev)
        with torch.cuda.device(dev):
            if self.kind == "faster_rcnn":
                if self.blobs["data"].data.shape[0] != 1:
                    raise AssertionError("Only single item batches are supported")
                o = self._engine.forward_checked(t("data"), t("im_info"), keep_intermediate=True)
                n = int(o["roi_counts"][0].item())
                host = {"rois": o["rois"][:n], "cls_prob": o["cls_prob"][:n], "bbox_pred": o["bbox_pred"][:n]}
            else:
                o = self._engine.run_checked(self._engine.forward, t("data"), t("rois"), t("masks"),
                                             keep_intermediate=True)
                R = self.blobs["rois"].data.shape[0]
                host = {"mask_prob": o["mask_prob"].view(R, -1), "cls_prob": o["cls_prob"],
                        "seg_cls_prob": o["seg_cls_prob"], "bbox_pred": o["bbox_pred"]}
            conv5 = o["_conv5_3"]
            B, H5, W5, C5 = tuple(conv5.shape)[-4:]   # split bf16 [2, B, H, W, C] or dense.Tri
            c5 = torch.empty((B, C5, H5, W5), dtype=torch.float32, device=dev)
            dense.split_to_nchw(conv5, B, H5, W5, C5, c5)
            host["conv5_3"] = c5
            for k, v in host.items():
                arr = v.contiguous().cpu().numpy()
                if k == "rois":
                    arr[:, 0] = 0
                self.blobs[k].data = arr
        return {k: self.blobs[k].data for k in self.outputs}

    def forward(self, blobs=None, start=None, end=None, **kwargs):
        """pycaffe.py:62-108: inputs by keyword, returns {output blob name: array}."""
        import torch
        from mnc_b200 import dense
        if start is not None or end is not None:
            raise NotImplementedError("partial forward is not supported by the fused engine")
        self._set_inputs(kwargs)
        if self.kind != "mnc_5stage":
            return self._forward_siblings()
        data = self.blobs["data"].data
        im_info = self.blobs["im_info"].data
        if data.shape[0] != 1:
            raise AssertionError("Only single item batches are supported")  # proposal_layer.py:65
        dev = self._device
        with torch.cuda.device(dev):
            d = torch.from_numpy(np.ascontiguousarray(data, dtype=np.float32)).to(dev)
            info = torch.from_numpy(np.ascontiguousarray(im_info, dtype=np.float32)).to(dev)
            o = self._engine.forward_checked(d, info, keep_intermediate=True)
            n = int(o["roi_counts"][0].item())
            conv5 = o["_conv5_3"]
            B, H5, W5, C5 = tuple(conv5.shape)[-4:]   # split bf16 [2, B, H, W, C] or dense.Tri
            c5 = torch.empty((B, C5, H5, W5), dtype=torch.float32, device=dev)
            dense.split_to_nchw(conv5, B, H5, W5, C5, c5)
            host = {
                "conv5_3": c5,
                "rois": o["rois"][:n], "rois_ext": o["rois_ext"][:n],
                "mask_proposal": o["mask_proposal"][:n], "mask_proposal_ext": o["mask_proposal_ext"][:n],
                "seg_cls_prob": o["seg_cls_prob"][:n], "seg_cls_prob_ext": o["seg_cls_prob_ext"][:n],
                "cls_prob": o["cls_prob"][:n], "cls_prob_ext": o["cls_prob_ext"][:n],
                "bbox_pred": o["bbox_pred"][:n], "bbox_pred_ext": o["bbox_pred_ext"][:n],
            }
            for k, v in host.items():
                arr = v.contiguous().cpu().numpy()
                if k.startswith("rois"):
                    arr[:, 0] = 0  # single-image net: batch index 0 (proposal_layer.py:159)
                self.blobs[k].data = arr
        return {k: self.blobs[k].data for k in self.outputs}
