"""The small host-side helpers that complete the `mutils` surface (model_utils.py: compute_iou_*, compute_overlaps, clip_boxes_numpy,
intersect1d, sum_tensor, get_dice_per_batch_and_class, batch_dice_mask, unmold_mask_*) against the reference's own functions: their outputs
on the seeded inputs of make_mutils_golden.py are stored in tests/golden/mutils_surface.npz (bit-identical ones as digests)."""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_mutils_golden as MG  # noqa: E402
from digest import digest  # noqa: E402

from medicaldetectiontoolkit_b200 import model_utils as M  # noqa: E402


@pytest.fixture(scope="module")
def ref(golden_dir):
    g = np.load(os.path.join(golden_dir, "mutils_surface.npz"))
    return {k: json.loads(str(g[k])) if g[k].dtype.kind == "U" else g[k] for k in g.files}


@pytest.mark.parametrize("dim", [2, 3])
def test_numpy_iou_helpers_bit_identical(ref, dim):
    i = MG.iou_inputs(dim)
    a, b = i["a"], i["b"]
    assert digest(M.compute_overlaps(a, b)) == ref["iou%d__overlaps" % dim]
    f = M.compute_iou_2D if dim == 2 else M.compute_iou_3D
    assert digest(f(b[0], a, float(i["vb"][0]), i["vol"])) == ref["iou%d__iou" % dim]
    assert digest(M.clip_boxes_numpy(i["wild"], tuple(i["win"].tolist()))) == ref["iou%d__clip" % dim]


def test_tensor_helpers(ref):
    t = {k: torch.from_numpy(v) for k, v in MG.tensor_inputs().items()}
    assert torch.equal(M.intersect1d(t["t1"], t["t2"]), torch.from_numpy(ref["tensor__intersect1d"]))
    for j, axes in enumerate(MG.SUM_AXES):
        assert torch.allclose(M.sum_tensor(t["x"], axes), torch.from_numpy(ref["tensor__sum_%d" % j]), rtol=1e-13, atol=0)
        assert list(M.sum_tensor(t["x"], axes, keepdim=True).shape) == ref["tensor__sum_keepdim_shape_%d" % j].tolist()
    assert np.allclose(M.get_dice_per_batch_and_class(t["pred"].numpy(), t["y"].numpy(), 3), ref["tensor__dice"], rtol=1e-14)
    assert abs(float(M.batch_dice_mask(t["p2"], t["y2"], t["m2"])) - float(ref["tensor__dice_mask"][0])) < 1e-14
    assert abs(float(M.batch_dice_mask(t["p3"], t["y3"], None)) - float(M.batch_dice(t["p3"], t["y3"]))) < 1e-15


def test_unmold_masks(ref):
    u = MG.unmold_inputs()
    assert digest(M.unmold_mask_2D(u["m2"], u["box2"].tolist(), tuple(u["shape2"].tolist()))) == ref["unmold__out2"]
    assert digest(M.unmold_mask_3D(u["m3"], u["box3"].tolist(), tuple(u["shape3"].tolist()))) == ref["unmold__out3"]
