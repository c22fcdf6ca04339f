#!/usr/bin/env python
"""Generate tests/golden/*.npz from the REFERENCE ITSELF (run in the build container only).

    python tests/golden/make_golden.py

Imports the reference's own modules from /root/reference:
  * models/generate_anchors.py            -- imported unmodified (numpy + six only)
  * models/bbox_transform.py, models/proposal_layer.py
                                          -- imported unmodified under a numpy-only stand-in
                                             for the `chainer` package (Chainer is not
                                             installable here: no network).  The stand-in
                                             only supplies Variable / cuda.get_array_module /
                                             cuda.get_device_from_array / cuda.to_cpu, i.e. the
                                             CPU branch the reference takes with numpy inputs.
  * models/cpu_nms.pyx                    -- the reference's compiled extension
                                             (oracle/build_ref.py -> oracle/_ref/).
`np.float` (removed NumPy alias used at models/proposal_layer.py:66) is aliased to `float`.

The vectors are committed; the GPU box never needs /root/reference.
Inputs that are large are NOT stored: they are regenerated from the seed by
tests/golden_inputs.py (same code used here), and a checksum of the input is stored instead.
"""
import contextlib
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import build_ref          # noqa: E402
import golden_inputs as gi  # noqa: E402

REF = "/root/reference"


def install_chainer_standin():
    """Numpy-only stand-in for the handful of chainer symbols the two reference modules touch."""
    if not hasattr(np, "float"):
        np.float = float      # models/proposal_layer.py:66
    chainer = types.ModuleType("chainer")
    cuda = types.ModuleType("chainer.cuda")

    class Variable(object):
        def __init__(self, data, volatile=False):
            self.data = data
        shape = property(lambda s: s.data.shape)
        ndim = property(lambda s: s.data.ndim)
        dtype = property(lambda s: s.data.dtype)

    class _CupyNdarray(object):   # never instantiated: `isinstance(x, cuda.cupy.ndarray)` is False
        pass

    class _Dev(object):
        id = -1
        def __enter__(self):
            return self
        def __exit__(self, *a):
            return False

    cupy = types.SimpleNamespace(ndarray=_CupyNdarray)
    cuda.cupy = cupy
    cuda.get_array_module = lambda *a: np
    cuda.get_device_from_array = lambda *a: _Dev()
    cuda.to_cpu = lambda a: a
    cuda.to_gpu = lambda a, d=None: a
    chainer.Variable = Variable
    chainer.cuda = cuda
    sys.modules["chainer"] = chainer
    sys.modules["chainer.cuda"] = cuda
    return Variable


def import_reference():
    Variable = install_chainer_standin()
    ref_nms = build_ref.load()
    assert ref_nms is not None, "reference cpu_nms could not be built"
    sys.path.insert(0, REF)
    import models  # noqa: F401  (the reference's package)
    sys.modules["models.cpu_nms"] = ref_nms
    gpu_stub = types.ModuleType("models.gpu_nms")
    gpu_stub.gpu_nms = None     # imported at models/proposal_layer.py:27, never called (Q2)
    sys.modules["models.gpu_nms"] = gpu_stub
    from models import generate_anchors as ga
    from models import bbox_transform as bt
    from models import proposal_layer as pl
    return Variable, ref_nms, ga, bt, pl


def write_cpu_nms_clustered(ref_nms):
    """cpu_nms keep lists on larger clustered cases (1500 boxes, 40 clusters) at the three thresholds the project uses."""
    out = {}
    for name, (seed, thr) in gi.NMS_CLUSTERED_CASES.items():
        dets = gi._clustered_dets(1500, seed)
        out[name + "_keep"] = np.asarray(ref_nms.cpu_nms(dets, thr), dtype=np.int64)
        out[name + "_checksum"] = gi.checksum(dets)
    np.savez_compressed(os.path.join(HERE, "cpu_nms_clustered.npz"), **out)


def main():
    Variable, ref_nms, ga, bt, pl = import_reference()
    out = {}

    # ---- 1. anchors (SURVEY.md Q9)
    out["anchors_default_call"] = ga.generate_anchors()                                   # scales (4,8,16,32)
    out["anchors_proposal_layer"] = ga.generate_anchors(ratios=(0.5, 1, 2), scales=(8, 16, 32))
    out["anchors_r3_s2"] = ga.generate_anchors(base_size=15, ratios=(0.25, 1, 4), scales=(2, 64))
    np.savez(os.path.join(HERE, "anchors.npz"), **out)

    # ---- 2. bbox_transform_inv / clip / filter
    out = {}
    for name, (n, k, seed) in {"rpn": (4000, 1, 11), "head": (300, 21, 12)}.items():
        boxes, trans = gi.box_transform_case(n, k, seed)
        pred = bt.bbox_transform_inv(boxes, trans)
        out[name + "_inv"] = pred
        clipped = bt.clip_boxes(pred.copy(), np.array([600, 1000]))
        out[name + "_clip"] = clipped
        if k == 1:
            out[name + "_filter16"] = bt.filter_boxes(clipped, 16)
        out[name + "_checksum"] = gi.checksum(boxes, trans)
    out["empty_inv"] = bt.bbox_transform_inv(np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32))
    np.savez(os.path.join(HERE, "bbox_transform.npz"), **out)

    # ---- 3. cpu_nms
    out = {}
    for name in gi.NMS_CASES:
        dets, thr = gi.nms_case(name)
        keep = ref_nms.cpu_nms(dets, thr)
        out[name + "_keep"] = np.asarray(keep, dtype=np.int64)
        out[name + "_thr"] = np.float64(thr)
        out[name + "_checksum"] = gi.checksum(dets)
    np.savez(os.path.join(HERE, "cpu_nms.npz"), **out)
    write_cpu_nms_clustered(ref_nms)

    # ---- 4. ProposalLayer.__call__
    out = {}
    for name in gi.PROPOSAL_CASES:
        prob, pred, info, train = gi.proposal_case(name)
        layer = pl.ProposalLayer()
        layer.train = train
        rois, probs = layer(Variable(prob), Variable(pred), Variable(info))
        out[name + "_rois"] = rois
        out[name + "_probs"] = probs
        out[name + "_checksum"] = gi.checksum(prob, pred)
        # all-anchor grid known answer for the same map
        out[name + "_all_bbox_head"] = layer._generate_all_bbox(prob.shape[2], prob.shape[3])[:40]
        out[name + "_all_bbox_sum"] = np.float64(layer._generate_all_bbox(prob.shape[2], prob.shape[3]).sum())
        print(name, "rois", rois.shape, "probs", probs.shape)
    np.savez(os.path.join(HERE, "proposal_layer.npz"), **out)

    # ---- 5. training path: bbox_overlaps (compiled bbox.pyx), keep_inside, bbox_transform, AnchorTargetLayer.__call__
    ref_bbox = build_ref.load_bbox()
    assert ref_bbox is not None, "reference bbox.pyx could not be built"
    sys.modules["models.bbox"] = ref_bbox
    from models import anchor_target_layer as atl
    out = {}
    boxes, _ = gi.box_transform_case(500, 1, 21)
    query, _ = gi.box_transform_case(17, 1, 22)
    out["overlaps_500x17"] = ref_bbox.bbox_overlaps(np.ascontiguousarray(boxes, dtype=np.float64),
                                                    np.ascontiguousarray(query, dtype=np.float64))
    out["overlaps_checksum"] = gi.checksum(boxes, query)
    ex, _ = gi.box_transform_case(300, 1, 23)
    gt_, _ = gi.box_transform_case(300, 1, 24)
    out["bbox_transform_f64xf32"] = bt.bbox_transform(ex.astype(np.float64), gt_)       # the dtype mix AnchorTargetLayer uses
    out["bbox_transform_checksum"] = gi.checksum(ex, gt_)
    real_choice = np.random.choice
    for name in gi.ANCHOR_TARGET_CASES:
        fh, fw, gt, info, seed = gi.anchor_target_case(name)
        calls = []

        def recording_choice(a, size=None, replace=True, p=None):
            r = real_choice(a, size=size, replace=replace, p=p)
            calls.append((np.asarray(a).copy(), np.asarray(r).copy()))
            return r
        np.random.choice = recording_choice
        try:
            np.random.seed(seed)
            layer = atl.AnchorTargetLayer()
            labels, targets, inds_inside, n_all = layer(fh, fw, Variable(gt), Variable(info))
        finally:
            np.random.choice = real_choice
        out[name + "_labels"] = labels
        out[name + "_targets"] = targets
        out[name + "_inds_inside"] = inds_inside
        out[name + "_n_all"] = np.int64(n_all)
        # the subsampling draws, in call order: [pool, chosen] (fg first if it happened, then bg)
        out[name + "_n_choice_calls"] = np.int64(len(calls))
        for ci, (pool, chosen) in enumerate(calls):
            out[name + "_choice%d_pool" % ci] = pool
            out[name + "_choice%d_chosen" % ci] = chosen
        out[name + "_checksum"] = gi.checksum(gt, info)
        print(name, "labels", labels.shape, "fg", int((labels == 1).sum()), "bg", int((labels == 0).sum()),
              "choice calls", len(calls), targets.dtype)
    np.savez_compressed(os.path.join(HERE, "anchor_target_layer.npz"), **out)

    # ---- 6. ProposalTargetLayer.__call__ (RCNN training path)
    from models import proposal_target_layer as ptl
    out = {}
    for name in gi.PROPOSAL_TARGET_CASES:
        props, gt, seed = gi.proposal_target_case(name)
        calls = []

        def recording_choice2(a, size=None, replace=True, p=None):
            r = real_choice(a, size=size, replace=replace, p=p)
            calls.append((np.asarray(a).copy(), np.asarray(r).copy()))
            return r
        np.random.choice = recording_choice2
        try:
            np.random.seed(seed)
            layer = ptl.ProposalTargetLayer()
            use_gt, ext, keep = layer(props, Variable(gt))
        finally:
            np.random.choice = real_choice
        out[name + "_use_gt_boxes"] = use_gt
        out[name + "_bbox_reg_targets"] = ext
        out[name + "_keep_inds"] = keep
        out[name + "_n_choice_calls"] = np.int64(len(calls))
        for ci, (pool, chosen) in enumerate(calls):
            out[name + "_choice%d_pool" % ci] = pool
            out[name + "_choice%d_chosen" % ci] = chosen
        out[name + "_checksum"] = gi.checksum(props, gt)
        print(name, "keep", keep.shape, keep.dtype, "targets", ext.shape, ext.dtype, "choice calls", len(calls))
    np.savez_compressed(os.path.join(HERE, "proposal_target_layer.npz"), **out)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
