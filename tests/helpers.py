"""Shared helpers for the parity tests (the oracle is the checker, never the product)."""
import os

import numpy as np
import torch

from oracle import mmd_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LEVELS = ("p3", "p4", "p5", "p6", "p7")

# name -> (C, conv_channels, n_cells, first, B, s3, seed)   (must mirror oracle/make_golden.py main())
STACK_CASES = {
    "cell_c16": (16, [8, 12, 20], 1, False, 2, 16, 1),
    "first_c16": (16, [8, 12, 20], 1, True, 2, 16, 2),
    "stack3_c16": (16, [8, 12, 20], 3, True, 2, 32, 3),
    "stack2_c16_odd": (16, [8, 12, 20], 2, True, 1, 48, 4),
    "stack2_c112": (112, [48, 120, 352], 2, True, 2, 16, 5),
    "cell_c112": (112, [48, 120, 352], 1, False, 2, 16, 6),
}
# name -> (kind, C, num_anchors, num_classes, num_layers, B, s3, seed)   (must mirror oracle/make_golden.py main())
HEAD_CASES = {"reg_c112": ("reg", 112, 9, 20, 3, 2, 16, 9), "cls_c112": ("cls", 112, 9, 20, 3, 2, 16, 10)}
# name -> (annotation kind, B, image size, classes, seed)   (must mirror oracle/make_golden.py FOCAL_CASES)
FOCAL_CASES = {"focal_mixed": ("mixed", 4, 128, 20, 21), "focal_dense": ("dense", 2, 128, 20, 22), "focal_none": ("none", 2, 128, 20, 23)}
# pseudo-label generation (must mirror oracle/make_golden.py PSEUDO_*): name -> (B, image size, classes, seed, teachers)
PSEUDO_VALID_IDS = [2, 4, 6, 7, 9, 11, 14, 16, 19]
PSEUDO_CASES = {"pseudo_a": (4, 128, 20, 100, 3)}
PSEUDO_CFG = dict(conf_threshold=0.3, nms_threshold=0.5, ignore_labels=(4,))
MTA_CASES = {"mta_c112": (2, 112, [12, 6, 3], 7), "mta_c16": (3, 16, [16, 8, 4, 2, 1], 8)}


def golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def pyramid_inputs(B, C, s3, seed, dtype=torch.float32):
    sizes = [s3, s3 // 2, s3 // 4, s3 // 8, max(s3 // 16, 1)]
    return [O.synth((B, C, s, s), seed + i, 1.0, 0.1 * i, dtype) for i, s in enumerate(sizes)]


def backbone_inputs(B, conv_channels, s3, seed, dtype=torch.float32):
    return [O.synth((B, c, s3 >> i, s3 >> i), seed + i, 1.0, 0.0, dtype) for i, c in enumerate(conv_channels)]


def stack_case_inputs(name, dtype=torch.float32):
    C, cc, n_cells, first, B, s3, seed = STACK_CASES[name]
    params = O.synth_stack_params(C, cc, n_cells, seed, first_cell_first_time=first, dtype=dtype)
    xs = backbone_inputs(B, cc, s3, seed + 50, dtype) if first else pyramid_inputs(B, C, s3, seed + 50, dtype)
    return params, xs


def pseudo_case_inputs(name):
    """-> anchors [1,N,4] (the reference's), [(classification, regression)] per teacher, label id of every valid prediction id."""
    B, size, K, seed, nt = PSEUDO_CASES[name]
    anchors = torch.from_numpy(golden(name)["anchors"])
    logits = [O.synth_teacher_logits(B, anchors, K, seed + 10 * t, size=size) for t in range(nt)]
    return anchors, logits, {i: n for n, i in enumerate(PSEUDO_VALID_IDS)}


def focal_case_inputs(name, dtype=torch.float32):
    """-> classification [B,N,K], regression [B,N,4], anchors [1,N,4] (the reference's, stored in the fixture), annotations."""
    kind, B, size, K, seed = FOCAL_CASES[name]
    anchors = torch.from_numpy(golden(name)["anchors"])
    c, r = O.synth_detections(B, anchors.shape[1], K, seed, dtype)
    return c, r, anchors, O.synth_annotations(kind, B, size, K)


def head_case_inputs(name, dtype=torch.float32):
    kind, C, A, K, L, B, s3, seed = HEAD_CASES[name]
    params = O.synth_head_params(C, A * (4 if kind == "reg" else K), L, seed, dtype=dtype)
    return params, pyramid_inputs(B, C, s3, seed + 50, dtype)


def head_case_gouts(name, y, a):
    seed = HEAD_CASES[name][7]
    return O.synth(tuple(y.shape), seed + 70, 1.0, 0.0), O.synth(tuple(a.shape), seed + 71, 1.0, 0.0)


def stack_case_gouts(name, outs):
    seed = STACK_CASES[name][6]
    return [O.synth(tuple(t.shape), seed + 70 + i, 1.0, 0.0).to(t.dtype) for i, t in enumerate(outs)]


def structured_features(B, C, sizes, seed, dtype=torch.float32):
    fs = []
    for i, s in enumerate(sizes):
        base = O.synth((B, C, s, s), seed + i, 1.0, 0.0)
        mod = torch.exp(1.5 * O.synth((B, 1, s, s), seed + 100 + i, 1.0, 0.0))
        fs.append((base * mod).to(dtype))
    return fs


def rel_l2(a, b):
    a = torch.as_tensor(a).double().flatten()
    b = torch.as_tensor(b).double().flatten()
    d = (a - b).norm().item()
    n = b.norm().item()
    return d / n if n > 0 else d


# Tile shapes (TW, TH) of the tiled BiFPN node kernels (bifpn_fwd_v4.cu / bifpn_bwd_v4.cu, pick_geom), tried in this order;
# a level that fits none of them runs on the run-time-geometry kernels (bifpn_fwd_tc.cu / bifpn_bwd_tc.cu).
TILE_GEOMS = ((16, 8), (12, 8), (8, 8), (12, 6), (6, 6))


def pick_geom(H, W):
    """Python mirror of pick_geom(): the (TW, TH) tile of an H x W level, or None for the run-time-geometry kernels."""
    for tw, th in TILE_GEOMS:
        if W % tw == 0 and H % th == 0:
            return tw, th
    return None


def worst_tile_rel_l2(a, b, tile):
    """Largest rel-L2 of a against b over the (TH x TW) tiles of each sample ([B, C, H, W] tensors, all channels of a tile
    together): one wrong or missing tile reads ~1 here, whatever the size of the rest of the tensor."""
    tw, th = tile
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    B, C, Hh, W = b.shape
    assert Hh % th == 0 and W % tw == 0, (tuple(b.shape), tile)
    per = lambda t: t.reshape(B, C, Hh // th, th, W // tw, tw).pow(2).sum(dim=(1, 3, 5))
    num, den = per(a - b), per(b)
    return float((num / den.clamp_min(1e-300)).sqrt().max())


def max_rel(a, b):
    """max |a-b| / max|b| : the 'relative' error used for the 1e-4 bar on dense tensors."""
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    m = b.abs().max().item()
    d = (a - b).abs().max().item()
    return d / m if m > 0 else d


def efficientdet_anchors(size):
    """The anchor table of the reference's `Anchors(anchor_scale=4.)` (src/YetAnotherEfficientDet.py:71-152) for a size x
    size image, [1, N, 4] (y1, x1, y2, x2): strides 8..128, 3 scales x 3 ratios per position.  tests/test_gpu_focal.py
    checks the same construction against the stored reference anchors."""
    ys = []
    for lvl in range(3, 8):
        stride = 2 ** lvl
        for sc in (2 ** 0, 2 ** (1.0 / 3.0), 2 ** (2.0 / 3.0)):
            for ra in ((1.0, 1.0), (1.4, 0.7), (0.7, 1.4)):
                half_x, half_y = 4.0 * stride * sc * ra[0] / 2.0, 4.0 * stride * sc * ra[1] / 2.0
                x = np.arange(stride / 2, size, stride)
                xv, yv = np.meshgrid(x, x)
                ys.append((lvl, np.stack((yv.reshape(-1) - half_y, xv.reshape(-1) - half_x, yv.reshape(-1) + half_y,
                                          xv.reshape(-1) + half_x), axis=1)))
    per_level = [np.stack([b for l, b in ys if l == lvl], axis=1).reshape(-1, 4) for lvl in range(3, 8)]
    return torch.from_numpy(np.concatenate(per_level, axis=0).astype(np.float32)).unsqueeze(0)


def pseudo_config(size, **over):
    """The reference's config section for the pseudo-label path (a dict works like the configparser section)."""
    cfg = {"conf_threshold": str(PSEUDO_CFG["conf_threshold"]), "nms_threshold": str(PSEUDO_CFG["nms_threshold"]),
           "image_size": str(size), "student": "YetAnotherEfficientDet",
           "ignore_labels": ",".join(str(i) for i in PSEUDO_CFG["ignore_labels"])}
    cfg.update(over)
    return cfg


def pseudo_valid_classes_dict():
    """valid_classes_dict as oracle/make_golden.py::run_pseudo_case builds it."""
    return {"predictions_txt2i": {"c%d" % i: i for i in PSEUDO_VALID_IDS}, "predictions_i2txt": {i: "c%d" % i for i in PSEUDO_VALID_IDS},
            "labels_txt2i": {"c%d" % i: n for n, i in enumerate(PSEUDO_VALID_IDS)}}
