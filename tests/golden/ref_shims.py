"""Load the reference's UNMODIFIED model files (models/retina_unet.py, models/mrcnn.py, models/retina_net.py) on the CPU of the build
container.  TEST INFRASTRUCTURE: used by make_model_golden.py to generate the committed fixtures and by the optional boundary tests;
never by the product package.  Nothing is copied from the reference: it is imported from REF (default /root/reference, read-only).

The shims are the five of SURVEY.md §8c:
  1. stub `matplotlib*` (utils/exp_utils.py:23 imports plotting.py which imports matplotlib, absent here)
  2. inject `cuda_functions.*` modules (the real ones need torch.utils.ffi / TH): `nms_gpu` and `CropAndResizeFunction` backed by the C
     oracle (oracle/mdt_oracle.c, itself pinned on the GPU to the reference's own kernels) — or by any pair of callables given
  3. `.cuda()` = identity for CPU runs (models hard-code `.cuda()`, e.g. retina_unet.py:374,395-400)
  4. torch-0.4 integer `/` (floor for the non-negative indices at retina_unet.py:212, mrcnn.py index math)
  5. absolute `cf.backbone_path` (default_configs.py:35 is relative to the reference root)
plus byte-mask indexing (`tensor[ByteTensor]`, model_utils.py:645-654 and mrcnn.py) mapped to bool-mask indexing.
"""
import contextlib
import importlib.util
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("REF", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "tests"), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)


class Logger:
    def info(self, *a, **k):
        pass


# ----------------------------------------------------------------------------------------------------------- oracle-backed CPU ops
def oracle_nms(dim):
    """pth_nms.nms_gpu(dets, thresh) (cuda_functions/nms_3D/pth_nms.py:5-17): sort by score, greedy NMS, indices into the input order"""
    import _oracle as O

    def nms_gpu(dets, thresh):
        scores = dets[:, -1]
        _, order = scores.sort(0, descending=True)
        d = dets[order].contiguous().detach().numpy()
        keep = O.nms(d, float(thresh), dim)
        return order[torch.from_numpy(keep).long()].contiguous()

    return nms_gpu


def oracle_roi_align(dim):
    """callable class CropAndResizeFunction(ch, cw[, cz], extrapolation_value)(image, boxes, box_ind), autograd to image
    (cuda_functions/roi_align_3D/roi_align/crop_and_resize.py:10-51)"""
    import _oracle as O

    class _Fn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, image, boxes, box_ind, crop):
            ctx.save_for_backward(boxes, box_ind)
            ctx.in_shape = tuple(image.shape)
            # the C side reads sizes [0 .. 1 + dim] only (crop_and_resize_gpu.c:17-24): trailing singleton axes (the channel-last GT masks of
            # mrcnn.py:556-559 arrive as [n, 1, y, x, z, 1]) are part of the same contiguous memory
            image = image.detach().contiguous().reshape(image.shape[:2 + dim])
            ctx.im_size = tuple(image.shape)
            out = O.crop_and_resize_forward(image.numpy(), boxes.detach().numpy(), box_ind.detach().numpy(), crop)
            return torch.from_numpy(out)

        @staticmethod
        def backward(ctx, g):
            boxes, box_ind = ctx.saved_tensors
            gi = O.crop_and_resize_backward(g.contiguous().numpy(), boxes.detach().numpy(), box_ind.detach().numpy(), ctx.im_size)
            return torch.from_numpy(gi).reshape(ctx.in_shape), None, None, None

    class CropAndResizeFunction(object):
        def __init__(self, *args):
            n = dim
            self.crop = tuple(int(a) for a in args[:n])
            self.extrapolation_value = args[n] if len(args) > n else 0

        def __call__(self, image, boxes, box_ind):
            return _Fn.apply(image, boxes, box_ind, self.crop)

    return CropAndResizeFunction


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []
    sys.modules[name] = m
    return m


def install_import_shims(nms2d=None, nms3d=None, ra2d=None, ra3d=None):
    """shims 1 + 2: module stubs so that `import models.*` of the reference resolves"""
    class _Any(types.ModuleType):
        def __getattr__(self, k):
            if k.startswith("__"):
                raise AttributeError(k)
            return _Any(self.__name__ + "." + k)

        def __call__(self, *a, **k):
            return None

    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.gridspec", "matplotlib.patches", "matplotlib.colors", "matplotlib.cm"):
        if name not in sys.modules:
            m = _Any(name)
            m.__path__ = []
            m.use = lambda *a, **k: None
            sys.modules[name] = m
    _mod("cuda_functions")
    for d, nms, ra in ((2, nms2d, ra2d), (3, nms3d, ra3d)):
        _mod("cuda_functions.nms_%dD" % d)
        _mod("cuda_functions.nms_%dD.pth_nms" % d, nms_gpu=nms or oracle_nms(d))
        _mod("cuda_functions.roi_align_%dD" % d)
        _mod("cuda_functions.roi_align_%dD.roi_align" % d)
        _mod("cuda_functions.roi_align_%dD.roi_align.crop_and_resize" % d, CropAndResizeFunction=ra or oracle_roi_align(d))
    if REF not in sys.path:
        sys.path.insert(0, REF)


@contextlib.contextmanager
def torch04_semantics(cpu=True):
    """shims 3 + 4 + byte-mask indexing, active only inside the `with` block"""
    T = torch.Tensor
    saved = dict(cuda_t=T.cuda, cuda_m=torch.nn.Module.cuda, div=T.__truediv__, rdiv=T.__rtruediv__, getitem=T.__getitem__,
                 setitem=T.__setitem__)

    def _is_int(x):
        return (torch.is_tensor(x) and not x.is_floating_point() and x.dtype != torch.bool) or (isinstance(x, (int, np.integer)) and not isinstance(x, bool))

    def truediv(self, other):
        if _is_int(self) and _is_int(other):
            return torch.div(self, other, rounding_mode='trunc')     # C integer division of torch 0.4
        return saved['div'](self, other)

    def fix_index(ix):
        if torch.is_tensor(ix) and ix.dtype == torch.uint8:
            return ix.bool()
        if isinstance(ix, tuple):
            return tuple(fix_index(i) for i in ix)
        return ix

    def getitem(self, ix):
        return saved['getitem'](self, fix_index(ix))

    def setitem(self, ix, v):
        return saved['setitem'](self, fix_index(ix), v)

    if cpu:
        T.cuda = lambda self, *a, **k: self
        torch.nn.Module.cuda = lambda self, *a, **k: self
    T.__truediv__ = truediv
    T.__getitem__ = getitem
    T.__setitem__ = setitem
    try:
        yield
    finally:
        T.cuda, torch.nn.Module.cuda = saved['cuda_t'], saved['cuda_m']
        T.__truediv__, T.__getitem__, T.__setitem__ = saved['div'], saved['getitem'], saved['setitem']


def load_ref_module(name):
    """import models/<name>.py of the reference under the module name ref_<name> (unmodified source)"""
    spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(REF, "models", name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def ref_cf(cf):
    """shim 5 + the attributes the reference reads that our attribute bag does not carry"""
    c = types.SimpleNamespace(**vars(cf))
    c.backbone_path = os.path.join(REF, "models", "backbone.py")
    c.scale = np.asarray(c.scale)
    return c


def drop_cuda_functions():
    """forget the injected / drop-in `cuda_functions` modules"""
    for k in [k for k in sys.modules if k == "cuda_functions" or k.startswith("cuda_functions.")]:
        del sys.modules[k]


def dropin_setup(model, patch=(64, 64, 32)):
    """the reference's graph on this package (INTEGRATION.md §1): `install_dropin()` + the two `mutils` attribute patches + `cf.backbone_path`
    pointing at this package's backbone.py.  Returns (mutils, saved, cf); undo with dropin_teardown(mutils, saved)."""
    import medicaldetectiontoolkit_b200 as mdt
    from medicaldetectiontoolkit_b200 import conv as b200_conv
    from medicaldetectiontoolkit_b200 import model_utils as b200_mutils
    from medicaldetectiontoolkit_b200.configs import make_cf
    install_import_shims()          # matplotlib stubs + sys.path (its oracle-backed cuda_functions are replaced on the next line)
    mdt.install_dropin()
    import utils.model_utils as mutils
    saved = (mutils.NDConvGenerator, mutils.gt_anchor_matching)
    mutils.NDConvGenerator = b200_conv.NDConvGenerator
    mutils.gt_anchor_matching = b200_mutils.gt_anchor_matching
    cf = ref_cf(make_cf(model, 3, patch))
    cf.backbone_path = os.path.join(ROOT, "medicaldetectiontoolkit_b200", "backbone.py")
    return mutils, saved, cf


def dropin_teardown(mutils, saved):
    mutils.NDConvGenerator, mutils.gt_anchor_matching = saved
    drop_cuda_functions()
