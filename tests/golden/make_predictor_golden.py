#!/usr/bin/env python
"""Golden outputs of the REFERENCE's unmodified `Predictor` (predictor.py, imported through ref_shims.py; nothing copied) driven by the
deterministic stand-in network of predictor_standin.py, for tests/test_predictor_cpu.py.  Each case is stored as one JSON string (floats
round-trip exactly): box lists, monitor values, other small results and the digest of the segmentation output (digest.py).
Run where the reference tree is present:  python tests/golden/make_predictor_golden.py [out.npz]  ->  tests/golden/predictor.npz"""
import copy
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import predictor_standin as S  # noqa: E402
import ref_shims as RS  # noqa: E402
from digest import digest  # noqa: E402


def main():
    RS.install_import_shims()
    import predictor as ref                                                   # the reference module, unmodified
    out = {}

    def put(name, res, **extra):
        out[name] = np.array(json.dumps(S.plain(dict(boxes=res['boxes'], monitor_values=res.get('monitor_values'), seg_preds=digest(res['seg_preds']),
                                                     **extra))))

    with tempfile.TemporaryDirectory() as tmp:
        for dim in (3, 2):
            batch = S.patient(dim, seed=dim)
            p = ref.Predictor(S.make_cf(dim, tmp), S.StandInNet(dim), S.Logger(), 'val')
            p.patched_patient = True
            res = p.spatial_tiling_forward(copy.deepcopy(batch), batch['patch_crop_coords'])
            whole = p.spatial_tiling_forward(copy.deepcopy(S.whole_image(batch)))
            put("tiling%d" % dim, res, whole_boxes=whole['boxes'])
        for dim in (3, 2):
            batch = S.patient(dim, seed=10 + dim)
            put("val%d" % dim, ref.Predictor(S.make_cf(dim, tmp), S.StandInNet(dim), S.Logger(), 'val').predict_patient(copy.deepcopy(batch)))
        np.save(os.path.join(tmp, 'epoch_ranking.npy'), np.array([4, 9, 2]))
        batch = S.patient(3, seed=7)
        p = ref.Predictor(S.make_cf(3, tmp, test_aug=True), S.StandInNet(3), S.Logger(), 'test')
        put("test3", p.predict_patient(copy.deepcopy(batch)), n_ens=p.n_ens, epoch_ranking=list(p.epoch_ranking),
            mirrored_crops=ref.get_mirrored_patch_crops(batch['patch_crop_coords'], batch['original_img_shape']))
    np.savez_compressed(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "predictor.npz"), **out)


if __name__ == "__main__":
    main()
