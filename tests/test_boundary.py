"""Boundary proof through the reference's OWN graph (INTEGRATION.md §1): the unmodified models/retina_unet.py and models/mrcnn.py built with
`medicaldetectiontoolkit_b200.install_dropin()` + the two `mutils` attribute patches + `cf.backbone_path` pointing at this package's
backbone.py (tests/golden/ref_shims.py: dropin_setup).

Pinned by stored facts of the reference's graphs (tests/golden/boundary.npz, make_boundary_golden.py): the reference's import sites resolve
to libmdt_b200's drop-ins, and the graph it builds on them has OUR FPN / conv modules with the reference's state-dict keys; the weight
initialisation is bit-identical to the reference's.  Where the reference tree is present, the reference's forward running on our kernels
(needs a GPU as well) and the two models outside the hot path are also built from the reference's files."""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)
REF = os.environ.get("REF", "/root/reference")
needs_reference = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "models")), reason="reference tree not present")

import make_boundary_golden as BG  # noqa: E402
import ref_shims as RS  # noqa: E402
from digest import digest  # noqa: E402


@pytest.fixture(scope="module")
def golden():
    return json.loads(str(np.load(os.path.join(GOLD, "boundary.npz"))["json"]))


@pytest.mark.parametrize("model", ["retina_unet", "mrcnn"])
def test_reference_graph_resolves_to_the_dropins(golden, model):
    import medicaldetectiontoolkit_b200 as mdt
    import medicaldetectiontoolkit_b200.cuda_functions.nms_2D.pth_nms as d2
    import medicaldetectiontoolkit_b200.cuda_functions.nms_3D.pth_nms as d3
    from medicaldetectiontoolkit_b200 import backbone as b200_backbone
    from medicaldetectiontoolkit_b200 import conv as b200_conv
    from medicaldetectiontoolkit_b200 import mrcnn as b200_mrcnn
    from medicaldetectiontoolkit_b200 import native_ops
    from medicaldetectiontoolkit_b200 import retina_unet as b200_ru
    from medicaldetectiontoolkit_b200.configs import make_cf
    mdt.install_dropin()
    try:
        # the reference's import sites (models/retina_unet.py:26-27, models/mrcnn.py:24-27)
        from cuda_functions.nms_2D.pth_nms import nms_gpu as nms_2D
        from cuda_functions.nms_3D.pth_nms import nms_gpu as nms_3D
        from cuda_functions.roi_align_2D.roi_align.crop_and_resize import CropAndResizeFunction as ra2D
        from cuda_functions.roi_align_3D.roi_align.crop_and_resize import CropAndResizeFunction as ra3D
        assert nms_3D is d3.nms_gpu and nms_2D is d2.nms_gpu
        assert ra3D is native_ops.CropAndResizeFunction and ra2D is native_ops.CropAndResizeFunction2D
    finally:
        RS.drop_cuda_functions()
    want = golden["graph"][model]
    ours = (b200_ru if model == "retina_unet" else b200_mrcnn).net(make_cf(model, 3, (64, 64, 32)), None)
    fpn = ours.Fpn if model == "retina_unet" else ours.fpn
    assert fpn.__class__.__name__ == "FPN"
    assert os.path.samefile(fpn.__class__.__init__.__code__.co_filename, b200_backbone.__file__)
    n_b200 = sum(isinstance(m, b200_conv.Conv3d) for m in ours.modules())
    n_torch = sum(isinstance(m, torch.nn.Conv3d) for m in ours.modules())
    assert n_b200 == want["n_b200_conv3d"] > 60 and n_torch == 0                              # every conv of the reference graph is ours
    ref_sd = {k: tuple(shape) for k, shape in want["state_dict"]}
    our_sd = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    if model == "mrcnn":   # the reference's nn.ConvTranspose3d vs our _Deconv2x: same keys and shapes
        assert ref_sd["mask.deconv.weight"] == our_sd["mask.deconv.weight"]
    assert ref_sd == our_sd


@needs_reference
@pytest.mark.parametrize("model", ["retina_unet", "mrcnn"])
def test_reference_graph_built_live_on_the_dropins(golden, model):
    """the reference's unmodified models/*.py, built through ref_shims.dropin_setup: its FPN is this package's backbone.py, every conv is ours,
    and its state dict and conv count are the stored ones that test_reference_graph_resolves_to_the_dropins compares the mirror with"""
    from medicaldetectiontoolkit_b200 import backbone as b200_backbone
    from medicaldetectiontoolkit_b200 import conv as b200_conv
    from medicaldetectiontoolkit_b200 import native_ops
    mutils, saved, cf = RS.dropin_setup(model)
    try:
        with RS.torch04_semantics(cpu=True):
            ref = RS.load_ref_module(model)
            net = ref.net(cf, RS.Logger())
        import medicaldetectiontoolkit_b200.cuda_functions.nms_3D.pth_nms as d3
        assert ref.nms_3D is d3.nms_gpu
        if model == "mrcnn":
            assert ref.ra3D is native_ops.CropAndResizeFunction
        fpn = net.Fpn if model == "retina_unet" else net.fpn
        assert os.path.samefile(fpn.__class__.__init__.__code__.co_filename, b200_backbone.__file__)
        assert sum(isinstance(m, torch.nn.Conv3d) for m in net.modules()) == 0
        want = golden["graph"][model]
        assert sum(isinstance(m, b200_conv.Conv3d) for m in net.modules()) == want["n_b200_conv3d"]
        assert [[k, list(v.shape)] for k, v in net.state_dict().items()] == want["state_dict"]
    finally:
        RS.dropin_teardown(mutils, saved)


@needs_reference
@pytest.mark.gpu
def test_reference_forward_on_b200_kernels_matches_the_mirror():
    """the reference's unmodified retina_unet.net.forward running on libmdt_b200 (drop-ins) == our retina_unet.net, same weights"""
    import detweights
    import golden_inputs as GI
    from medicaldetectiontoolkit_b200 import retina_unet as b200_ru
    mutils, saved, cf = RS.dropin_setup("retina_unet")
    try:
        with RS.torch04_semantics(cpu=False):
            ref = RS.load_ref_module("retina_unet")
            orig_unique = np.unique
            np.unique = lambda a, *x, **k: orig_unique(a.cpu().numpy() if torch.is_tensor(a) else a, *x, **k)   # retina_unet.py:205 on a CUDA tensor
            try:
                net = ref.net(cf, RS.Logger()).cuda()
                GI.tame_(detweights.fill_(net), "retina_unet")
                img = torch.from_numpy(GI.synthetic_batch(cf, 2, seed=5)['data']).cuda()
                with torch.no_grad():
                    det_r, cl_r, bb_r, seg_r = net.forward(img)
            finally:
                np.unique = orig_unique
        ours = b200_ru.net(cf, None)
        GI.tame_(detweights.fill_(ours), "retina_unet")
        ours = ours.cuda()
        with torch.no_grad():
            det_o, cl_o, bb_o, seg_o = ours.forward(img)
        for a, b in ((cl_r, cl_o), (bb_r, bb_o), (seg_r, seg_o)):
            assert float((a - b).abs().max() / b.abs().max()) <= 1e-5
        assert det_r.shape == det_o.shape
    finally:
        RS.dropin_teardown(mutils, saved)


@pytest.mark.parametrize("model,init", BG.WEIGHT_INIT_CASES)
def test_weight_init_equals_the_reference(golden, model, init):
    """cf.weight_init (utils/model_utils.py:695-728): the UNMODIFIED reference net (stock nn.Conv3d, its own backbone.py) and the mirror, built
    under the same seed, end up with bit-identical parameters — same module order, same fans, same RNG consumption."""
    from medicaldetectiontoolkit_b200 import mrcnn as b200_mrcnn
    from medicaldetectiontoolkit_b200 import retina_unet as b200_ru
    from medicaldetectiontoolkit_b200.configs import make_cf
    cf = make_cf(model, 3, BG.WEIGHT_INIT_PATCH)
    cf.weight_init = init
    torch.manual_seed(BG.WEIGHT_INIT_SEED)
    osd = (b200_ru if model == "retina_unet" else b200_mrcnn).net(cf, None).state_dict()
    want = golden["weight_init"]["%s/%s" % (model, init)]
    assert list(osd) == [w[0] for w in want]
    for k, shape, dtype, sha in want:
        assert digest(osd[k]) == [shape, dtype, sha], k


@needs_reference
@pytest.mark.parametrize("model", ["ufrcnn", "detection_unet"])
def test_other_reference_models_build_on_the_dropins(model):
    """SURVEY §2 row 15: models/ufrcnn.py and models/detection_unet.py are outside the hot-path scope but share the import sites
    (ufrcnn.py:24-27, the backbone path and mutils.NDConvGenerator): the unmodified reference files build entirely on libmdt_b200 modules"""
    from medicaldetectiontoolkit_b200 import backbone as b200_backbone
    from medicaldetectiontoolkit_b200 import conv as b200_conv
    mutils, saved, cf = RS.dropin_setup("mrcnn" if model == "ufrcnn" else "retina_unet")
    try:
        cf.model = model
        if model == "ufrcnn":
            cf.num_seg_classes, cf.operate_stride1, cf.frcnn_mode = 2, True, True
        with RS.torch04_semantics(cpu=True):
            net = RS.load_ref_module(model).net(cf, RS.Logger())
        fpn = net.Fpn if hasattr(net, "Fpn") else net.fpn
        assert os.path.samefile(fpn.__class__.__init__.__code__.co_filename, b200_backbone.__file__)
        assert sum(isinstance(m, b200_conv.Conv3d) for m in net.modules()) > 60
        assert sum(isinstance(m, torch.nn.Conv3d) for m in net.modules()) == 0
    finally:
        RS.dropin_teardown(mutils, saved)
