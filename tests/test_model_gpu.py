"""Backbone / model level parity (GPU).  The FPN mirror is compared with fixtures produced by the REFERENCE's models/backbone.py
(stock nn.Conv3d, CPU fp32; tests/golden/make_golden.py) under identical, name-keyed deterministic weights — this also proves the
state-dict keys and shapes are the reference's.  The Retina U-Net mirror is exercised end to end (train_forward + backward)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import detweights  # noqa: E402

from medicaldetectiontoolkit_b200 import conv as C  # noqa: E402
from medicaldetectiontoolkit_b200.backbone import FPN  # noqa: E402
from medicaldetectiontoolkit_b200.configs import make_cf, synthetic_batch  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _rel_l2(a, b):
    """relative L2 error — the norm used for GRADIENTS that passed through ReLUs: a rounding-level change of a pre-activation near zero flips its
    mask and changes that single gradient element by O(1) (seen on B200: max-norm 1e-1 on one element of one block while every kernel is exact to
    6e-6 on the same tensors, tools/debug_fpn_backward.py), which the max norm reports as a gross error and the L2 norm correctly as noise."""
    a, b = np.asarray(a, dtype=np.float64).ravel(), np.asarray(b, dtype=np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _fpn_run(golden_dir, tag, op1, algo):
    g = np.load(os.path.join(golden_dir, "backbone3d_%s.npz" % tag))
    cf = make_cf('retina_unet' if op1 else 'mrcnn', 3, (32, 32, 16))
    old = C.DEFAULT_ALGO
    C.DEFAULT_ALGO = algo
    try:
        fpn = FPN(cf, C.NDConvGenerator(3), operate_stride1=op1)
        keys = [k for k, _ in fpn.named_parameters()]
        assert keys == list(g["keys"])                                             # same parameter names, same order
        shapes = {k: tuple(v.shape) for k, v in fpn.state_dict().items()}
        assert [str(shapes[k]) for k in keys] == list(g["key_shapes"])
        detweights.fill_(fpn)
        fpn = fpn.to(DEV)
        x = torch.from_numpy(np.random.RandomState(3).rand(1, 1, 32, 32, 16).astype(np.float32)).to(DEV).requires_grad_(True)
        outs = fpn(x)
        errs = {}
        for i, o in enumerate(outs):
            assert tuple(o.shape) == tuple(g["outshape%d" % i])
            errs["out%d" % i] = _rel(detweights.subsample(o.detach().cpu().numpy()), g["out%d" % i])
        loss = sum((o * o).mean() for o in outs)
        errs["loss"] = abs(loss.item() - float(g["loss"])) / abs(float(g["loss"]))
        loss.backward()
        errs["x_grad"] = _rel_l2(detweights.subsample(x.grad.cpu().numpy()), g["x_grad"])
        params = dict(fpn.named_parameters())
        for k in g.files:
            if k.startswith("grad__"):
                errs[k] = _rel_l2(detweights.subsample(params[k[6:]].grad.cpu().numpy()), g[k])
        nograd = sorted(k for k, p in params.items() if p.grad is None)
        assert nograd == sorted(g["nograd"])                                       # P1_conv2.* never used (backbone.py:175)
        return errs
    finally:
        C.DEFAULT_ALGO = old


@pytest.mark.parametrize("tag,op1", [("unet", True), ("mrcnn", False)])
def test_fpn_vs_reference_fixture(golden_dir, tag, op1):
    """FPN forward + all gradients vs the fixture produced by the reference's models/backbone.py on CPU fp32, for the exact fp32 SIMT kernels
    and for the default (tcgen05 split-bf16) path.  Forward: 1e-4 of max|ref| (north_star).  Gradients after the ~60-conv backward chain: relative L2 (see _rel_l2) 1e-3 for the fp32 kernels,
    5e-3 for the split-bf16 path (per-conv 1e-4 bars are in tests/test_conv_gpu.py)."""
    simt = _fpn_run(golden_dir, tag, op1, 1)
    auto = _fpn_run(golden_dir, tag, op1, 0)
    print("fpn parity", tag, "simt", {k: "%.1e" % v for k, v in simt.items()}, "auto", {k: "%.1e" % v for k, v in auto.items()})
    for k, v in simt.items():
        assert v < (1e-4 if k.startswith("out") or k == "loss" else 1e-3), ("simt", k, v)
    for k, v in auto.items():
        assert v < (1e-4 if k.startswith("out") or k == "loss" else 5e-3), ("auto", k, v)


def test_retina_unet_train_step_small():
    from medicaldetectiontoolkit_b200 import retina_unet
    cf = make_cf('retina_unet', 3, (64, 64, 32))
    torch.manual_seed(0)
    np.random.seed(0)
    net = retina_unet.net(cf, None).to(DEV)
    batch = synthetic_batch(cf, 2, seed=1)
    res = net.train_forward(batch)
    assert set(['boxes', 'seg_preds', 'torch_loss', 'monitor_values', 'logger_string']) <= set(res)
    assert res['seg_preds'].shape == (2, 1, 64, 64, 32) and res['seg_preds'].dtype == np.uint8
    assert len(res['boxes']) == 2 and any(b['box_type'] == 'gt' for b in res['boxes'][0])
    loss = res['torch_loss']
    assert torch.isfinite(loss).all()
    loss.backward()
    grads = [(k, p.grad) for k, p in net.named_parameters()]
    missing = sorted(k for k, g_ in grads if g_ is None)
    assert missing == ['Fpn.P1_conv2.bias', 'Fpn.P1_conv2.weight']             # 154 of 156 parameters receive gradients (SURVEY §5)
    assert all(torch.isfinite(g_).all() for _, g_ in grads if g_ is not None)
    n_params = sum(p.numel() for p in net.parameters())
    assert n_params == 4_950_000 or abs(n_params - 4.95e6) < 0.05e6            # SURVEY: 4.95 M parameters
    out = net.test_forward({'data': batch['data']})
    assert 'boxes' in out and out['seg_preds'].shape == (2, 1, 64, 64, 32)


def test_retina_losses_match_reference_formulas():
    """fixed-shape loss formulation == the reference's nonzero()-based one (retina_unet.py:126-187) on a case with known sampling"""
    from medicaldetectiontoolkit_b200.retina_unet import compute_bbox_loss, compute_class_loss
    import torch.nn.functional as F
    torch.manual_seed(3)
    A = 5000
    logits = torch.randn(A, 3, device=DEV)
    match = torch.full((A,), -1, dtype=torch.int32, device=DEV)
    match[torch.randperm(A, device=DEV)[:1500]] = 0
    pos = torch.tensor([17, 901, 4000], device=DEV)
    match[pos] = torch.tensor([1, 2, 1], dtype=torch.int32, device=DEV)
    loss, neg_ix = compute_class_loss(match, logits, shem_poolsize=20, max_pos=3)
    pos_loss = F.cross_entropy(logits[pos], match[pos].long())
    neg_all = torch.nonzero(match == -1).squeeze(1)
    picked = neg_all[neg_ix[neg_ix >= 0]]
    assert picked.numel() == 3
    probs = F.softmax(logits[neg_all], 1)[:, 1:].max(1)[0]
    pool = neg_all[probs.sort(descending=True)[1][:60]]
    assert set(picked.tolist()) <= set(pool.tolist())                          # sampled from the top shem_poolsize * n_neg pool
    neg_loss = F.cross_entropy(logits[picked], torch.zeros(3, dtype=torch.long, device=DEV))
    assert abs(loss.item() - ((pos_loss + neg_loss) / 2).item()) < 1e-5
    deltas = torch.randn(A, 6, device=DEV)
    tgt = torch.zeros(6, 6, dtype=torch.float64, device=DEV)
    tgt[:3] = torch.randn(3, 6, dtype=torch.float64, device=DEV)
    bl = compute_bbox_loss(tgt, deltas, match, max_pos=3)
    want = F.smooth_l1_loss(deltas[pos], tgt[:3].float())
    assert abs(bl.item() - want.item()) < 1e-6
    none = torch.full((A,), -1, dtype=torch.int32, device=DEV)
    assert compute_bbox_loss(tgt, deltas, none, max_pos=3).item() == 0.0


def test_mrcnn_train_step_small():
    """cfg3-style two-stage model end to end: proposals (NMS 0.7) -> RoIAlign (7,7,3)/(14,14,5) -> heads -> detection targets incl. RoIAlign
    (28,28,10) on GT masks -> 5 losses -> backward through RoIAlign into the FPN"""
    from medicaldetectiontoolkit_b200 import mrcnn
    cf = make_cf('mrcnn', 3, (64, 64, 32))
    cf.post_nms_rois_training = 64
    cf.post_nms_rois_inference = 64
    cf.pre_nms_limit = 1000
    torch.manual_seed(0)
    np.random.seed(0)
    net = mrcnn.net(cf, None).to(DEV)
    keys = set(net.state_dict().keys())
    for k in ['fpn.C1.0.weight', 'fpn.C2.1.conv1.0.weight', 'fpn.P5_conv1.bias', 'rpn.conv_shared.0.weight', 'rpn.conv_class.weight', 'rpn.conv_bbox.bias',
              'classifier.conv1.0.weight', 'classifier.linear_class.weight', 'classifier.linear_bbox.bias', 'mask.conv4.0.bias',
              'mask.deconv.weight', 'mask.deconv.bias', 'mask.conv5.weight']:
        assert k in keys, k
    assert tuple(net.mask.deconv.weight.shape) == (36, 36, 2, 2, 2) and tuple(net.classifier.conv1[0].weight.shape) == (144, 36, 7, 7, 3)
    batch = synthetic_batch(cf, 2, seed=2, with_masks=True)
    res = net.train_forward(batch)
    assert res['seg_preds'].shape == (2, 1, 64, 64, 32)
    loss = res['torch_loss']
    assert torch.isfinite(loss).all()
    loss.backward()
    g = {k: p.grad for k, p in net.named_parameters()}
    assert g['rpn.conv_shared.0.weight'] is not None and torch.isfinite(g['rpn.conv_shared.0.weight']).all()
    assert g['classifier.conv1.0.weight'] is not None and g['mask.deconv.weight'] is not None
    assert g['fpn.C1.0.weight'].abs().sum() > 0          # gradients reach the stem through RoIAlign backward
    out = net.test_forward({'data': batch['data']}, return_masks=True)
    assert out['seg_preds'].shape == (2, 1, 64, 64, 32)


def test_deconv2x_matches_conv_transpose():
    from medicaldetectiontoolkit_b200.mrcnn import _Deconv2x
    torch.manual_seed(1)
    m = _Deconv2x(36, 36, 3).to(DEV)
    x = torch.randn(3, 36, 5, 6, 4, device=DEV, requires_grad=True)
    y = m(x)
    xr = x.detach().double().requires_grad_(True)
    yr = torch.nn.functional.conv_transpose3d(xr, m.weight.double(), m.bias.double(), stride=2)
    assert _rel(y.detach().cpu().numpy(), yr.detach().cpu().numpy()) < 1e-4
    g = torch.randn_like(y)
    y.backward(g)
    yr.backward(g.double())
    assert _rel(x.grad.cpu().numpy(), xr.grad.cpu().numpy()) < 1e-4

    assert m.weight.grad is not None and torch.isfinite(m.weight.grad).all()


def test_upsample221_matches_torch():
    """csrc/resample.cu vs F.interpolate(scale (2,2,1), trilinear, align_corners=False), forward and backward (incl. edge clamping)"""
    from medicaldetectiontoolkit_b200.backbone import Interpolate
    torch.manual_seed(0)
    for shape in [(2, 36, 5, 7, 6), (1, 8, 1, 1, 3), (1, 36, 16, 16, 16)]:
        x = torch.randn(*shape, device=DEV).contiguous(memory_format=torch.channels_last_3d).requires_grad_(True)
        y = Interpolate((2, 2, 1), 'trilinear')(x)
        xr = x.detach().double().requires_grad_(True)
        yr = torch.nn.functional.interpolate(xr, scale_factor=(2, 2, 1), mode='trilinear', align_corners=False)
        assert y.shape == yr.shape and _rel(y.detach().cpu().numpy(), yr.detach().cpu().numpy()) < 1e-6
        g = torch.randn_like(y)
        y.backward(g)
        yr.backward(g.double())
        assert _rel(x.grad.cpu().numpy(), xr.grad.cpu().numpy()) < 1e-6


def _copy_state(dst, src):
    """load the CPU port's stock-torch weights into our modules: identical key sets are part of the check"""
    sd_src = {k: v for k, v in src.state_dict().items()}
    sd_dst = dst.state_dict()
    assert sorted(sd_src) == sorted(sd_dst), (sorted(set(sd_src) ^ set(sd_dst)))
    dst.load_state_dict(sd_src)


@pytest.mark.parametrize("dim,patch", [(3, (64, 64, 32)), (2, (128, 128))])
def test_retina_forward_matches_cpu_port(dim, patch):
    """Model-level parity: our Retina U-Net (3D) / RetinaNet-style heads (2D, the toy_exp plumbing config) on the GPU kernels vs the same graph
    built from stock torch.nn.Conv{2,3}d on the CPU (oracle/cpu_step.py), identical weights: class logits, box deltas, seg logits to 1e-4."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_step
    from medicaldetectiontoolkit_b200 import retina_unet
    cf = make_cf('retina_unet', dim, patch, exp='toy_exp' if dim == 2 else 'lidc_exp')
    torch.manual_seed(5)
    ref = cpu_step.build_cpu_net(cf).float()
    net = retina_unet.net(cf, None)
    _copy_state(net, ref)
    net = net.to(DEV)
    x = torch.from_numpy(np.random.RandomState(1).rand(2, 1, *patch).astype(np.float32))
    with torch.no_grad():
        cl_r, bb_r, seg_r = ref(x)
        det, cl, bb, seg = net(x.to(DEV))
    assert cl.shape == cl_r.shape and bb.shape == bb_r.shape and seg.shape == seg_r.shape
    assert _rel(cl.cpu().numpy(), cl_r.numpy()) < 1e-4
    assert _rel(bb.cpu().numpy(), bb_r.numpy()) < 1e-4
    assert _rel(seg.cpu().numpy(), seg_r.numpy()) < 1e-4
    assert det.shape[1] == 2 * dim + 3 and det.shape[0] <= 2 * cf.model_max_instances_per_batch_element
    # detections of the GPU path == the host restatement of refine_detections (retina_unet.py:194-271) on the reference logits
    import torch.nn.functional as F
    B, A = cl_r.shape[0], cl_r.shape[1]
    batch_ixs = torch.arange(B).unsqueeze(1).repeat(1, A).view(-1)
    det_r = cpu_step.refine_detections_cpu(cf, ref.anchors, F.softmax(cl.cpu().view(-1, cl.shape[-1]), 1), bb.cpu().view(-1, bb.shape[-1]), batch_ixs)
    got = det.cpu()
    assert got.shape == det_r.shape
    order_g = np.lexsort((got[:, -1].numpy(), got[:, 2 * dim].numpy()))
    order_r = np.lexsort((det_r[:, -1].numpy(), det_r[:, 2 * dim].numpy()))
    assert np.allclose(got.numpy()[order_g], det_r.numpy()[order_r], atol=1e-5)


def test_train_steps_are_bitwise_reproducible():
    """two independent runs of two Retina U-Net train steps (forward, matching, losses, detections, backward, Adam) from the same seeds
    compute the same bits: losses, detections, segmentation and the updated parameters"""
    from medicaldetectiontoolkit_b200 import retina_unet
    cf = make_cf('retina_unet', 3, (64, 64, 32))

    def run():
        torch.manual_seed(0)
        np.random.seed(0)
        net = retina_unet.net(cf, None).to(DEV)
        opt = torch.optim.Adam(net.parameters(), lr=1e-4)
        out = []
        for i in range(2):
            res = net.train_forward(synthetic_batch(cf, 2, seed=i))
            opt.zero_grad()
            res['torch_loss'].backward()
            opt.step()
            dets = [[b] + [float(c) for c in bx['box_coords']] + [float(bx['box_score'])]
                    for b, boxes in enumerate(res['boxes']) for bx in boxes if bx['box_type'] == 'det']
            out.append((float(res['torch_loss']), dets, np.array(res['seg_preds'], copy=True)))
        params = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).cpu()
        return out, params

    (a, pa), (b, pb) = run(), run()
    for (la, da, sa), (lb, db, sb) in zip(a, b):
        assert la == lb and da == db and np.array_equal(sa, sb)
    assert torch.equal(pa, pb)
