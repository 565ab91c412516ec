"""Patient-level prediction pipeline (medicaldetectiontoolkit_b200/predictor.py: Predictor) against the reference's unmodified `Predictor`
(predictor.py:27-510) driven by the SAME deterministic stand-in network on the CPU (tests/golden/predictor_standin.py; the reference's
outputs are stored in tests/golden/predictor.npz by make_predictor_golden.py, segmentations as digests): chunked forwarding, re-tiling of
boxes and segmentation into patient coordinates (float16 sums, overlap counts), patch ids / centre factors / overlap counts per box, the
three test-time mirrorings, and the consolidation calls.  The consolidation kernels need a GPU, so here `weighted_box_clustering` /
`nms_2to3D` are bound to the CPU restatement of the kernels' formulation (oracle/consolidate_oracle.py, itself pinned to reference goldens in test_consolidate_cpu.py)."""
import copy
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from medicaldetectiontoolkit_b200 import predictor as P  # noqa: E402
from digest import digest  # noqa: E402
from predictor_standin import Logger, StandInNet, make_cf, patient, plain, whole_image  # noqa: E402


@pytest.fixture(scope="module")
def ref_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "predictor.npz"))

    def case(name):
        """the reference Predictor's result of one case; 'seg_preds' is the digest [shape, dtype, sha256] of its segmentation"""
        return json.loads(str(g[name]))
    return case


@pytest.fixture()
def cpu_consolidation(monkeypatch):
    import consolidate_oracle as CO
    monkeypatch.setattr(P, "weighted_box_clustering", CO.weighted_box_clustering)
    monkeypatch.setattr(P, "nms_2to3D", CO.nms_2to3D)


def _same_boxes(ours, theirs, rtol=1e-12):
    assert len(ours) == len(theirs)
    for bo, bt in zip(ours, theirs):
        assert len(bo) == len(bt)
        for o, t in zip(bo, bt):
            assert sorted(o.keys()) == sorted(t.keys())
            for k in o:
                if isinstance(o[k], str):
                    assert o[k] == t[k], k
                else:
                    np.testing.assert_allclose(np.asarray(o[k], dtype=np.float64), np.asarray(t[k], dtype=np.float64), rtol=rtol, atol=1e-12, err_msg=k)


@pytest.mark.parametrize("dim", [3, 2])
def test_spatial_tiling_equals_the_reference(ref_golden, tmp_path, dim):
    batch = patient(dim, seed=dim)
    b = ref_golden("tiling%d" % dim)
    ours = P.Predictor(make_cf(dim, tmp_path), StandInNet(dim), Logger(), 'val')
    ours.patched_patient = True
    a = ours.spatial_tiling_forward(copy.deepcopy(batch), batch['patch_crop_coords'])
    _same_boxes(a['boxes'], b['boxes'])
    assert a['seg_preds'].dtype == np.float16 and digest(a['seg_preds']) == b['seg_preds']
    assert a['monitor_values'] == b['monitor_values']
    # whole-image prediction (no patch crops): the image is one patch with overlap 1
    _same_boxes(ours.spatial_tiling_forward(copy.deepcopy(whole_image(batch)))['boxes'], b['whole_boxes'])


@pytest.mark.parametrize("dim", [3, 2])
def test_predict_patient_val_mode_equals_the_reference(ref_golden, tmp_path, cpu_consolidation, dim):
    batch = patient(dim, seed=10 + dim)
    a = P.Predictor(make_cf(dim, tmp_path), StandInNet(dim), Logger(), 'val').predict_patient(copy.deepcopy(batch))
    b = ref_golden("val%d" % dim)
    _same_boxes(a['boxes'], b['boxes'], rtol=1e-9)            # after weighted box clustering (and the 2D -> 3D merge for dim 2)
    assert digest(a['seg_preds']) == b['seg_preds'] and a['monitor_values'] == b['monitor_values']


def test_test_mode_mirroring_and_test_set_loop(ref_golden, tmp_path, cpu_consolidation):
    import torch
    cf = make_cf(3, tmp_path, test_aug=True)
    np.save(os.path.join(str(tmp_path), 'epoch_ranking.npy'), np.array([4, 9, 2]))
    batch = patient(3, seed=7)
    ours, b = P.Predictor(cf, StandInNet(3), Logger(), 'test'), ref_golden("test3")
    assert ours.n_ens == b['n_ens'] == 8 and plain(list(ours.epoch_ranking)) == b['epoch_ranking']
    a = ours.predict_patient(copy.deepcopy(batch))
    _same_boxes(a['boxes'], b['boxes'])
    assert a['seg_preds'].shape == (1, 4, 48, 48, 24) and digest(a['seg_preds']) == b['seg_preds']
    assert ours.__class__.__name__ == 'Predictor' and \
        plain(P.get_mirrored_patch_crops(batch['patch_crop_coords'], batch['original_img_shape'])) == b['mirrored_crops']

    # the temporal-ensembling loop with stand-in checkpoints (the reference consolidates in a 6-process pool; here: in-process)
    class Net(StandInNet):
        def load_state_dict(self, sd):
            self.loaded = getattr(self, 'loaded', 0) + 1

        def eval(self):
            return self
    for ep in (4, 9):
        os.makedirs(os.path.join(str(tmp_path), '{}_best_checkpoint'.format(ep)), exist_ok=True)
        torch.save({}, os.path.join(str(tmp_path), '{}_best_checkpoint'.format(ep), 'params.pth'))
    net = Net(3)
    pred = P.Predictor(cf, net, Logger(), 'test')
    gen = {'n_test': 1, 'test': iter([copy.deepcopy(batch), copy.deepcopy(batch)])}
    out = pred.predict_test_set(gen, return_results=True)
    assert net.loaded == 2 and len(out) == 1 and out[0][1] == 'p3'
    dets = [bx for bx in out[0][0][0] if bx['box_type'] == 'det']
    assert dets and all(set(bx) == {'box_type', 'box_coords', 'box_score', 'box_pred_class_id'} for bx in dets)
    assert os.path.isfile(os.path.join(str(tmp_path), 'raw_pred_boxes_list.pickle'))
    again = pred.load_saved_predictions(apply_wbc=True)
    assert len(again) == 1 and len([bx for bx in again[0][0][0] if bx['box_type'] == 'det']) == len(dets)
