#!/usr/bin/env python
"""Golden vectors for the small host-side helpers of the `mutils` surface (tests/test_mutils_surface_cpu.py): the outputs of the REFERENCE's
own utils/model_utils.py functions, imported unmodified through ref_shims.py (nothing copied), on the seeded inputs defined here (the test
builds the same inputs).  Outputs checked for bit identity are stored as digests (digest.py), the others as values.
Run where the reference tree is present:  python tests/golden/make_mutils_golden.py [out.npz]  ->  tests/golden/mutils_surface.npz"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shims as RS  # noqa: E402
from digest import digest  # noqa: E402

SUM_AXES = [(0, 2, 3, 4), (1,), (0, 2)]


def _boxes(rs, n, dim):
    lo = rs.uniform(0, 100, size=(n, dim))
    hi = lo + rs.uniform(1, 40, size=(n, dim))
    return np.concatenate([lo[:, :2], hi[:, :2]] + ([lo[:, 2:], hi[:, 2:]] if dim == 3 else []), axis=1)[:, [0, 1, 2, 3] + ([4, 5] if dim == 3 else [])]


def iou_inputs(dim):
    """boxes a [300], b [17], volumes of a and of b[0], a clip window and boxes reaching outside it"""
    rs = np.random.RandomState(dim)
    a, b = _boxes(rs, 300, dim), _boxes(rs, 17, dim)
    vol = np.prod(a[:, [2, 3] + ([5] if dim == 3 else [])] - a[:, [0, 1] + ([4] if dim == 3 else [])], axis=1)
    vb = float(np.prod(b[0, [2, 3] + ([5] if dim == 3 else [])] - b[0, [0, 1] + ([4] if dim == 3 else [])]))
    win = (64, 80) if dim == 2 else (64, 80, 48)
    return {"a": a, "b": b, "vol": vol, "vb": np.array([vb]), "win": np.array(win), "wild": a * 1.7 - 30}


def tensor_inputs():
    rs = np.random.RandomState(5)
    out = {"t1": rs.permutation(50)[:20], "t2": rs.permutation(50)[:25], "x": rs.rand(2, 3, 4, 5, 6)}
    out["pred"], out["y"] = rs.randint(0, 3, (2, 1, 8, 8, 4)), rs.randint(0, 3, (2, 1, 8, 8, 4))
    out["p2"] = torch.softmax(torch.from_numpy(rs.randn(2, 2, 8, 8)), 1).numpy()
    out["y2"] = torch.nn.functional.one_hot(torch.from_numpy(rs.randint(0, 2, (2, 8, 8))), 2).movedim(-1, 1).double().numpy()
    out["m2"] = (rs.rand(2, 8, 8) > 0.3).astype(np.float64)
    out["p3"] = torch.softmax(torch.from_numpy(rs.randn(1, 2, 4, 4, 4)), 1).numpy()
    out["y3"] = torch.nn.functional.one_hot(torch.from_numpy(rs.randint(0, 2, (1, 4, 4, 4))), 2).movedim(-1, 1).double().numpy()
    return out


def unmold_inputs():
    rs = np.random.RandomState(6)
    return {"m2": rs.rand(28, 28).astype(np.float32), "box2": np.array([3, 5, 40, 33]), "shape2": np.array([64, 64]),
            "m3": rs.rand(14, 14, 5).astype(np.float32), "box3": np.array([2, 4, 30, 25, 1, 9]), "shape3": np.array([32, 32, 16])}


def main():
    RS.install_import_shims()
    import utils.model_utils as ref                                           # the reference module, unmodified
    out = {}
    for dim in (2, 3):
        i = iou_inputs(dim)
        iou = ref.compute_iou_2D if dim == 2 else ref.compute_iou_3D
        out["iou%d__overlaps" % dim] = digest(ref.compute_overlaps(i["a"], i["b"]))
        out["iou%d__iou" % dim] = digest(iou(i["b"][0], i["a"], float(i["vb"][0]), i["vol"]))
        out["iou%d__clip" % dim] = digest(ref.clip_boxes_numpy(i["wild"], tuple(i["win"].tolist())))
    t = tensor_inputs()
    out["tensor__intersect1d"] = ref.intersect1d(torch.from_numpy(t["t1"]), torch.from_numpy(t["t2"])).numpy()
    for j, axes in enumerate(SUM_AXES):
        out["tensor__sum_%d" % j] = ref.sum_tensor(torch.from_numpy(t["x"]), axes).numpy()
        out["tensor__sum_keepdim_shape_%d" % j] = np.array(ref.sum_tensor(torch.from_numpy(t["x"]), axes, keepdim=True).shape)
    out["tensor__dice"] = np.asarray(ref.get_dice_per_batch_and_class(t["pred"], t["y"], 3))
    out["tensor__dice_mask"] = np.array([float(ref.batch_dice_mask(*(torch.from_numpy(t[k]) for k in ("p2", "y2", "m2"))))])
    u = unmold_inputs()
    out["unmold__out2"] = digest(ref.unmold_mask_2D(u["m2"], u["box2"].tolist(), tuple(u["shape2"].tolist())))
    out["unmold__out3"] = digest(ref.unmold_mask_3D(u["m3"], u["box3"].tolist(), tuple(u["shape3"].tolist())))
    out = {k: np.array(json.dumps(v)) if isinstance(v, list) else v for k, v in out.items()}     # digests as JSON strings
    np.savez_compressed(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "mutils_surface.npz"), **out)


if __name__ == "__main__":
    main()
