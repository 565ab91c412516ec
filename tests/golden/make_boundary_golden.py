#!/usr/bin/env python
"""Golden facts of the REFERENCE's own model graphs (models/retina_unet.py, models/mrcnn.py, imported unmodified through ref_shims.py; nothing
copied) for tests/test_boundary.py:
  graph/<model>:        the graph built on this package's drop-ins (ref_shims.dropin_setup): state-dict keys and shapes in order, and how
                        many of its modules are this package's Conv3d
  weight_init/<model>/<init>: the stock reference net (nn.Conv3d, its own backbone.py) built under torch.manual_seed(5) with cf.weight_init
                        = <init>: state-dict keys in order with the digest (digest.py: shape, dtype, SHA-256) of each tensor
Run where the reference tree is present:  python tests/golden/make_boundary_golden.py [out.npz]  ->  tests/golden/boundary.npz (one JSON string)"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [HERE, os.path.dirname(os.path.dirname(HERE))]
import ref_shims as RS  # noqa: E402
from digest import digest  # noqa: E402

GRAPH_MODELS = ("retina_unet", "mrcnn")
WEIGHT_INIT_CASES = [("retina_unet", "kaiming_normal"), ("mrcnn", "xavier_uniform"), ("mrcnn", "kaiming_uniform")]
WEIGHT_INIT_PATCH = (32, 32, 16)
WEIGHT_INIT_SEED = 5


def main():
    from medicaldetectiontoolkit_b200 import conv as b200_conv
    from medicaldetectiontoolkit_b200.configs import make_cf
    out = {"graph": {}, "weight_init": {}}
    for model in GRAPH_MODELS:
        mutils, saved, cf = RS.dropin_setup(model)
        try:
            with RS.torch04_semantics(cpu=True):
                net = RS.load_ref_module(model).net(cf, RS.Logger())
            out["graph"][model] = {"state_dict": [[k, list(v.shape)] for k, v in net.state_dict().items()],
                                   "n_b200_conv3d": sum(isinstance(m, b200_conv.Conv3d) for m in net.modules())}
        finally:
            RS.dropin_teardown(mutils, saved)
    for model, init in WEIGHT_INIT_CASES:
        RS.install_import_shims()
        cf = make_cf(model, 3, WEIGHT_INIT_PATCH)
        cf.weight_init = init
        try:
            with RS.torch04_semantics(cpu=True):
                ref = RS.load_ref_module(model)
                torch.manual_seed(WEIGHT_INIT_SEED)
                rnet = ref.net(RS.ref_cf(cf), RS.Logger())
            out["weight_init"]["%s/%s" % (model, init)] = [[k] + digest(v) for k, v in rnet.state_dict().items()]
        finally:
            RS.drop_cuda_functions()
    np.savez_compressed(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "boundary.npz"), json=np.array(json.dumps(out)))


if __name__ == "__main__":
    main()
