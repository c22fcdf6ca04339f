"""Seeded input generators shared by tests/golden/make_golden.py (which feeds them to the
REFERENCE to produce the committed golden outputs) and by the tests (which feed the same
inputs to the oracle and to the CUDA path).  Large inputs are regenerated from the seed
instead of being committed; `checksum` guards against generator drift."""
import zlib

import numpy as np

f32 = np.float32


def checksum(*arrays):
    c = 0
    for a in arrays:
        c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    return np.int64(c)


def _unique_f32(rng, draw, n):
    """n float32 values from draw(k), all distinct (tie-free scores, SURVEY.md Q6)."""
    v = draw(n).astype(f32)
    for _ in range(100):
        _, first = np.unique(v, return_index=True)
        dup = np.setdiff1d(np.arange(n), first)
        if dup.size == 0:
            return v
        v[dup] = draw(dup.size).astype(f32)
    raise RuntimeError("could not make scores unique")


# --------------------------------------------------------------------------- bbox_transform
def box_transform_case(n, k, seed):
    rng = np.random.default_rng(seed)
    xy = rng.uniform(-50, 900, size=(n, 2))
    wh = rng.uniform(4, 400, size=(n, 2))
    boxes = np.hstack([xy, xy + wh]).astype(f32)
    trans = (rng.standard_normal((n, 4 * k)) * 0.6).astype(f32)
    return boxes, trans


# --------------------------------------------------------------------------- cpu_nms
def _clustered_dets(n, seed, ncl=40, W=1000.0, H=600.0):
    rng = np.random.default_rng(seed)
    c = rng.uniform([0, 0], [W, H], size=(ncl, 2))
    s = rng.uniform(30, 300, size=(ncl, 2))
    idx = rng.integers(0, ncl, size=n)
    ctr = c[idx] + rng.standard_normal((n, 2)) * 12
    wh = s[idx] * np.exp(rng.standard_normal((n, 2)) * 0.15)
    x1y1 = np.clip(ctr - wh / 2, 0, [W - 1, H - 1])
    x2y2 = np.clip(ctr + wh / 2, 0, [W - 1, H - 1])
    sc = _unique_f32(rng, lambda m: rng.uniform(0, 1, size=m), n)
    return np.hstack([x1y1, x2y2, sc[:, None]]).astype(f32)


def _integer_dets(n, seed, grid=24):
    """Integer-coordinate boxes on a small grid: exact rational IoUs such as 7/10, 3/10, 1/2
    are frequent, which is what separates `(double)ovr >= thr` (cpu_nms.pyx:66) from
    `ovr >= (float)thr` and from nms_kernel.cu's `>` (SURVEY.md Q3/Q4)."""
    rng = np.random.default_rng(seed)
    x1 = rng.integers(0, grid, size=(n, 2))
    wh = rng.integers(1, grid, size=(n, 2))
    sc = _unique_f32(rng, lambda m: rng.uniform(0, 1, size=m), n)
    d = np.hstack([x1, x1 + wh, sc[:, None]]).astype(f32)
    # hand-made exact cases first (highest scores so they are evaluated against each other):
    #   A=(0,0,9,9) area 100;  B=(0,0,9,6) area 70 -> IoU 7/10;  C=(0,0,9,2) area 30 -> 3/10 with A
    #   D=(0,0,9,4) area 50 -> 1/2 with A
    d[0] = [100, 100, 109, 109, 0.99]
    d[1] = [100, 100, 109, 106, 0.98]
    d[2] = [100, 100, 109, 102, 0.97]
    d[3] = [100, 100, 109, 104, 0.96]
    return d


NMS_CASES = {
    "n0": (0, 0.7), "n1": (1, 0.7), "n63": (63, 0.7), "n64": (64, 0.7), "n65": (65, 0.7),
    "n300_t03": (300, 0.3), "n2000_t07": (2000, 0.7), "n6000_t07": (6000, 0.7),
    "identical_t07": (100, 0.7), "disjoint_t03": (128, 0.3),
    "int_t07": (600, 0.7), "int_t03": (600, 0.3), "int_t05": (600, 0.5),
}


# name: (seed of _clustered_dets(1500, seed), threshold)
NMS_CLUSTERED_CASES = {"s%d_t%02d" % (seed, round(10 * thr)): (seed, thr)
                       for seed in range(100, 105) for thr in (0.3, 0.5, 0.7)}


def nms_case(name):
    n, thr = NMS_CASES[name]
    seed = zlib.crc32(name.encode()) & 0xFFFF
    if name.startswith("identical"):
        rng = np.random.default_rng(seed)
        sc = _unique_f32(rng, lambda m: rng.uniform(0, 1, size=m), n)
        d = np.tile(np.array([[10, 20, 110, 220, 0]], dtype=f32), (n, 1))
        d[:, 4] = sc
        return d, thr
    if name.startswith("disjoint"):
        rng = np.random.default_rng(seed)
        i = np.arange(n)
        x1 = (i % 16) * 50.0
        y1 = (i // 16) * 50.0
        sc = _unique_f32(rng, lambda m: rng.uniform(0, 1, size=m), n)
        return np.stack([x1, y1, x1 + 30, y1 + 30, sc], axis=1).astype(f32), thr
    if name.startswith("int_"):
        return _integer_dets(n, seed), thr
    if n == 0:
        return np.zeros((0, 5), dtype=f32), thr
    return _clustered_dets(n, seed, ncl=max(1, min(40, n // 8 + 1))), thr


# --------------------------------------------------------------------------- ProposalLayer
PROPOSAL_CASES = {
    # name: (feat_h, feat_w, (img_h, img_w), train_mode, kind, seed)
    "t14_train": (14, 14, (224, 224), True, "uniform", 1),     # tests/test_proposal_layer.py:20-32
    "t14_test": (14, 14, (224, 224), False, "uniform", 2),
    "c0_test": (38, 50, (600, 600), False, "softmax", 3),      # forward.py:93 passes (H, H) (Q7)
    "c0w_test": (38, 50, (600, 800), False, "softmax", 4),
    "c1_test": (38, 63, (600, 1000), False, "softmax", 5),     # headline config
    "c1_train": (38, 63, (600, 1000), True, "softmax", 6),
    "c1_wide_test": (38, 63, (600, 1000), False, "wide", 7),   # large deltas: min-size filter bites
}


def proposal_case(name, A=9):
    fh, fw, info, train, kind, seed = PROPOSAL_CASES[name]
    rng = np.random.default_rng(1000 + seed)
    n = A * fh * fw
    if kind == "uniform":
        prob = rng.uniform(0, 1, size=(1, 2 * A, fh, fw)).astype(f32)
        fg = _unique_f32(rng, lambda m: rng.uniform(0, 1, size=m), n)
        pred = rng.uniform(0, 1, size=(1, 4 * A, fh, fw)).astype(f32)
    else:
        logits = rng.standard_normal((1, 2 * A, fh, fw)) * 1.5
        e = np.exp(logits - logits.max(axis=1, keepdims=True))
        prob = (e / e.sum(axis=1, keepdims=True)).astype(f32)
        fg0 = prob[0, A:].reshape(-1).copy()
        fg = _unique_f32(rng, lambda m: rng.uniform(1e-4, 0.6, size=m), n)
        # keep the softmax values where they are already unique, patch duplicates only
        _, first = np.unique(fg0, return_index=True)
        uniq_mask = np.zeros(n, dtype=bool)
        uniq_mask[first] = True
        fg = np.where(uniq_mask, fg0, fg).astype(f32)
        assert np.unique(fg).size == n
        std = 1.2 if kind == "wide" else 0.35
        pred = (rng.standard_normal((1, 4 * A, fh, fw)) * std).astype(f32)
    prob[0, A:] = fg.reshape(A, fh, fw)
    assert np.unique(prob[0, A:]).size == n
    return prob, pred, np.array([info], dtype=np.int32), train


# --------------------------------------------------------------------------- AnchorTargetLayer (training path)
ANCHOR_TARGET_CASES = {
    # name: (feat_h, feat_w, (img_h, img_w), n_gt, kind, seed)
    "t14_ref_test": (14, 14, (224, 224), 3, "reference_test", 0),   # tests/test_anchor_target_layer.py:18-30
    "c1_g1": (38, 63, (600, 1000), 1, "random", 1),
    "c1_g8": (38, 63, (600, 1000), 8, "random", 2),
    "c1_g40_manyfg": (38, 63, (600, 1000), 40, "anchor_like", 3),   # > 128 positives: fg subsampling runs
    "c1_g3_outside": (38, 63, (600, 1000), 3, "one_outside", 4),    # a gt no inside anchor overlaps (gt_max == 0 quirk)
    "c0_g5_square_info": (38, 50, (600, 600), 5, "random", 5),      # img_info (H, H) as forward.py passes it (Q7)
    "t10_small": (10, 12, (160, 192), 2, "random", 6),               # few inside anchors; bg <= 256: no bg subsampling
}


def anchor_target_case(name):
    """-> feat_h, feat_w, gt_boxes float32 (1, G, 5) [x1,y1,x2,y2,cls], img_info int32 (1, 2) [h, w], numpy seed."""
    fh, fw, (ih, iw), g, kind, seed = ANCHOR_TARGET_CASES[name]
    rng = np.random.default_rng(2000 + seed)
    if kind == "reference_test":
        gt = np.array([[10, 10, 60, 200, 0], [50, 100, 210, 210, 1], [160, 40, 200, 70, 2]], dtype=f32)
    else:
        if kind == "anchor_like":
            # boxes shaped like the anchors themselves (128/256/512 px, ratios 0.5/1/2) so many anchors reach IoU 0.7
            size = rng.choice([128.0, 256.0], size=g)
            ratio = rng.choice([0.5, 1.0, 2.0], size=g)
            w = size / np.sqrt(ratio)
            h = size * np.sqrt(ratio)
            cx = rng.uniform(w / 2, iw - w / 2)
            cy = rng.uniform(np.minimum(h / 2, ih / 2), np.maximum(ih - h / 2, ih / 2))
        else:
            w = rng.uniform(20, iw * 0.6, size=g)
            h = rng.uniform(20, ih * 0.6, size=g)
            cx = rng.uniform(w / 2, iw - w / 2)
            cy = rng.uniform(h / 2, ih - h / 2)
        x1 = np.clip(np.floor(cx - w / 2), 0, iw - 2)
        y1 = np.clip(np.floor(cy - h / 2), 0, ih - 2)
        x2 = np.clip(np.floor(cx + w / 2), x1 + 1, iw - 1)
        y2 = np.clip(np.floor(cy + h / 2), y1 + 1, ih - 1)
        cls = rng.integers(0, 20, size=g)
        gt = np.stack([x1, y1, x2, y2, cls], axis=1).astype(f32)
        if kind == "one_outside":
            gt[1, :4] = [iw + 50, ih + 50, iw + 90, ih + 120]       # beyond every inside anchor
    info = np.array([[ih, iw]], dtype=np.int32)
    return fh, fw, gt[None], info, 7000 + seed


# --------------------------------------------------------------------------- ProposalTargetLayer (RCNN training path)
PROPOSAL_TARGET_CASES = {
    # name: (n_proposals, n_gt, kind, seed)
    "ref_test": (300, 3, "reference_test", 0),        # tests/test_proposal_target_layer.py:20-33: gt + integer jitter
    "few_fg": (300, 4, "random", 1),                  # random proposals: few reach IoU 0.5, many backgrounds
    "n50": (50, 2, "jitter", 2),                      # fewer proposals than ROIS_PER_IMAGE
    "class0": (200, 3, "class0", 3),                  # a gt of class 0: its rows get no regression targets
}


def proposal_target_case(name):
    """-> proposals float32 (N,4), gt_boxes float32 (1,G,5), numpy seed."""
    n, g, kind, seed = PROPOSAL_TARGET_CASES[name]
    rng = np.random.default_rng(3000 + seed)
    gt = np.array([[10, 10, 60, 200, 1], [50, 100, 210, 210, 2], [160, 40, 200, 70, 3], [20, 150, 120, 215, 7]], dtype=f32)[:g]
    if kind == "class0":
        gt[1, 4] = 0
    if kind == "random":
        xy = rng.uniform(0, 160, size=(n, 2))
        wh = rng.uniform(10, 120, size=(n, 2))
        props = np.hstack([xy, np.minimum(xy + wh, 223)]).astype(f32)
        props[: n // 6] = (gt[rng.integers(0, g, n // 6), :4] + rng.integers(-8, 8, (n // 6, 4))).astype(f32)
    else:
        jitter = rng.integers(-10, 10, size=(n, 4))
        props = (gt[rng.integers(0, g, size=n), :4] + jitter).astype(f32)
    return props, gt[None], 9000 + seed
