"""Deterministic stand-in network, config and patients shared by make_predictor_golden.py (fed to the REFERENCE's Predictor) and
tests/test_predictor_cpu.py (fed to ours)."""
import types

import numpy as np


class Logger:
    def info(self, *a, **k):
        pass


class StandInNet:
    """deterministic function of the input patch: a few boxes per batch element + a label map; fresh dicts on every call"""

    def __init__(self, dim):
        self.dim = dim

    def parameters(self):
        return iter(())

    def _element(self, patch):
        rs = np.random.RandomState(int(np.abs(patch).sum() * 1000) % (2 ** 31))
        sp = patch.shape[1:]
        boxes = []
        for _ in range(rs.randint(1, 5)):
            lo = [rs.randint(0, s - 6) for s in sp]
            hi = [l + rs.randint(3, min(s - l, 12)) for l, s in zip(lo, sp)]
            coords = [lo[0], lo[1], hi[0], hi[1]] + ([lo[2], hi[2]] if self.dim == 3 else [])
            boxes.append({'box_coords': np.array(coords, dtype=np.int32), 'box_score': float(rs.uniform(0.1, 0.99)), 'box_type': 'det',
                          'box_pred_class_id': int(rs.randint(1, 3))})
        return boxes

    def test_forward(self, batch, return_masks=True):
        data = batch['data']
        return {'boxes': [self._element(p) for p in data], 'seg_preds': (data[:, :1] > 0.6).astype(np.uint8)}

    def train_forward(self, batch, is_validation=False):
        out = self.test_forward(batch)
        for b in out['boxes']:
            b.append({'box_coords': np.zeros(2 * self.dim), 'box_label': 1, 'box_type': 'gt'})
        out['monitor_values'] = {'loss': float(batch['data'].mean()), 'class_loss': float(batch['data'].std())}
        return out


def make_cf(dim, tmp, test_aug=False):
    return types.SimpleNamespace(dim=dim, batch_size=3, patch_size=[32, 32, 16][:dim], test_aug=test_aug, class_dict={1: 'a', 2: 'b'}, wcs_iou=1e-5,
                                 merge_2D_to_3D_preds=dim == 2, merge_3D_iou=0.1, return_masks_in_test=False, fold_dir=str(tmp), fold=0, test_n_epochs=2,
                                 hold_out_test_set=False, folds=[0], exp_dir=str(tmp))


def patient_3d(rs):
    shape = (1, 1, 48, 48, 24)
    crops = [[y, y + 32, x, x + 32, z, z + 16] for y in (0, 16) for x in (0, 16) for z in (0, 8)]
    vol = rs.rand(*shape).astype(np.float32)
    data = np.stack([vol[0, :, c[0]:c[1], c[2]:c[3], c[4]:c[5]] for c in crops])
    return {'data': data, 'patch_crop_coords': crops, 'original_img_shape': shape, 'pid': 'p3',
            'patient_bb_target': np.array([[[5, 5, 20, 20, 2, 9]]]), 'patient_roi_labels': np.array([[1]])}


def patient_2d(rs):
    n_slices = 5
    shape = (n_slices, 1, 48, 48)
    crops = [[y, y + 32, x, x + 32, z, z + 1] for z in range(n_slices) for y in (0, 16) for x in (0, 16)]
    vol = rs.rand(*shape).astype(np.float32)
    data = np.stack([vol[c[4], :, c[0]:c[1], c[2]:c[3]] for c in crops])
    return {'data': data, 'patch_crop_coords': crops, 'original_img_shape': shape, 'pid': 'p2',
            'patient_bb_target': np.array([[[5, 5, 20, 20]]] * n_slices), 'patient_roi_labels': np.array([[1]] * n_slices)}


def patient(dim, seed):
    rs = np.random.RandomState(seed)
    return patient_3d(rs) if dim == 3 else patient_2d(rs)


def whole_image(batch):
    """whole-image prediction input (no patch crops): the image is one patch with overlap 1"""
    return {'data': batch['data'][:2], 'original_img_shape': (2,) + batch['data'].shape[1:], 'pid': 'w'}


def plain(o):
    """o with numpy arrays / scalars and tuples turned into lists and Python numbers (the JSON form of the goldens)"""
    if isinstance(o, dict):
        return {k: plain(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [plain(v) for v in o]
    if isinstance(o, np.ndarray):
        return o.tolist()
    if isinstance(o, np.generic):
        return o.item()
    return o
