"""GPU parity tests (run on the B200 with -m gpu): every call goes through the C-ABI of libmdt_b200.so and is compared with
 (a) the CPU oracle (oracle/mdt_oracle.c, oracle/matching_oracle.py), (b) the committed golden fixtures, and
 (c) the reference's own unmodified kernels compiled for sm_100a (oracle/_ref), through their stored outputs (tests/golden/ref_*.npz).
Tolerances: NMS keep indices and anchor labels bit-exact; RoIAlign 1e-4 relative to max|ref| (north_star)."""
import os
import sys

import numpy as np
import pytest
import torch

import _oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_kernel_golden as RK  # noqa: E402
import matching_oracle as MO  # noqa: E402
from golden_cfg import cf2d, cf3d  # noqa: E402

from medicaldetectiontoolkit_b200 import model_utils as MU  # noqa: E402
from medicaldetectiontoolkit_b200 import native_ops as NO  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _keep(boxes, thr, dim):
    t = torch.from_numpy(boxes).to(DEV)
    keep, num = NO.nms_sorted(t, thr, dim)
    return keep[: int(num.item())].cpu().numpy()


# ----------------------------------------------------------------------------------------------------------------------------------- NMS
@pytest.mark.parametrize("dim", [2, 3])
def test_nms_vs_oracle_small_and_edges(dim):
    for n in [0, 1, 2, 63, 64, 65, 129, 1000, 1024, 1025, 2049, 2112]:   # incl. the 16-block chunk / first-worker boundaries of the grid scan
        for thr in [0.7, 0.5, 1e-5]:
            for rounded in (True, False):
                boxes = O.synth_boxes(n, dim, seed=17 * n + dim, rounded=rounded, extent=48.0 if n > 100 else 24.0)
                assert _keep(boxes, thr, dim).tolist() == O.nms(boxes, thr, dim).tolist(), (n, thr, rounded)
    # all boxes identical: only the first survives; disjoint boxes: all survive
    same = np.tile(np.array([[2, 2, 10, 10] + ([1, 5] if dim == 3 else []) + [0.5]], dtype=np.float32), (200, 1))
    same[:, -1] = np.linspace(1, 0, 200)
    assert _keep(same, 0.5, dim).tolist() == [0]
    dis = same.copy()
    dis[:, 0] += 20 * np.arange(200)
    dis[:, 2] += 20 * np.arange(200)
    assert _keep(dis, 0.5, dim).tolist() == list(range(200))


def test_nms_rpn_and_retina_shapes_vs_oracle():
    """cfg3 RPN shape (6000 unrounded boxes, 0.7) and a Retina-style set (rounded, 1e-5)"""
    b = O.synth_boxes(6000, 3, seed=5, rounded=False)
    assert _keep(b, 0.7, 3).tolist() == O.nms(b, 0.7, 3).tolist()
    b = O.synth_boxes(8000, 3, seed=6, rounded=True)   # CPU oracle is O(N^2): keep it to ~1 s even on a loaded host
    assert _keep(b, 1e-5, 3).tolist() == O.nms(b, 1e-5, 3).tolist()
    b = O.synth_boxes(6000, 2, seed=7, rounded=False)
    assert _keep(b, 0.7, 2).tolist() == O.nms(b, 0.7, 2).tolist()


def test_nms_negative_threshold_takes_slow_path():
    b = O.synth_boxes(500, 3, seed=9, rounded=True, extent=32.0)
    assert _keep(b, -1.0, 3).tolist() == O.nms(b, -1.0, 3).tolist() == [0]


def test_nms_dropin_api_and_mask():
    from medicaldetectiontoolkit_b200 import install_dropin
    install_dropin()
    from cuda_functions.nms_3D.pth_nms import nms_gpu as nms_3D
    from cuda_functions.nms_2D.pth_nms import nms_gpu as nms_2D
    for dim, fn in ((3, nms_3D), (2, nms_2D)):
        srt = O.synth_boxes(3000, dim, seed=21, rounded=False)
        perm = np.random.RandomState(0).permutation(3000)
        dets = torch.from_numpy(srt[perm]).to(DEV)
        got = fn(dets, 0.5)
        assert got.dtype == torch.int64 and got.is_cuda
        want = np.argsort(perm)[O.nms(srt, 0.5, dim)]  # dets[i] = srt[perm[i]] -> index of sorted row j in dets is perm^-1[j]
        assert got.cpu().numpy().tolist() == want.tolist()
        assert fn(dets[:0], 0.5).numel() == 0
        m = NO.nms_mask(torch.from_numpy(srt[:777]).to(DEV), 0.5, dim).cpu().numpy().view(np.uint64)
        assert np.array_equal(m, O.nms_mask(srt[:777], 0.5, dim))
    with pytest.raises(Exception):
        NO.nms_sorted(torch.zeros(4, 7), 0.5, 3)  # CPU tensor: no fallback


def test_nms_full_size_cfg4_properties_and_reference_kernel(golden_dir):
    """BASELINE cfg4: 100 k boxes, IoU 0.5.  Size-independent properties + equality with the reference's own kernel + host scan
    (its keep lists on the same inputs, tests/golden/ref_nms.npz from make_ref_kernel_golden.py)."""
    g = np.load(os.path.join(golden_dir, "ref_nms.npz"))
    for n, thr, rounded in RK.NMS_3D_CASES:
        b = O.synth_boxes(n, 3, seed=n, rounded=rounded)
        keep = _keep(b, thr, 3)
        assert keep[0] == 0 and np.all(np.diff(keep) > 0)          # sorted, first box always kept
        again = _keep(b[keep], thr, 3)
        assert again.tolist() == list(range(len(keep)))            # idempotence: survivors do not suppress each other
        assert keep.tolist() == RK.kept(g["nms3d_%d" % n], n).tolist()   # bit-identical to the reference kernel
    n, thr, rounded, seed = RK.NMS_2D_CASE
    b = O.synth_boxes(n, 2, seed=seed, rounded=rounded)
    assert _keep(b, thr, 2).tolist() == RK.kept(g["nms2d_%d" % n], n).tolist()


# ----------------------------------------------------------------------------------------------------------------------------------- RoIAlign
def _rel(a, b):
    return float(np.abs(a.astype(np.float64) - b).max() / max(1e-12, np.abs(b).max()))


@pytest.mark.parametrize("dim,shape,crop", [(3, (2, 36, 16, 16, 32), (7, 7, 3)), (3, (2, 5, 9, 8, 7), (4, 1, 2)), (3, (3, 8, 8, 8, 8), (1, 1, 1)),
                                            (2, (2, 36, 24, 24), (7, 7)), (2, (1, 3, 10, 9), (1, 5))])
def test_roi_align_forward_backward_vs_oracle(dim, shape, crop):
    rs = np.random.RandomState(1)
    img = rs.randn(*shape).astype(np.float32)
    boxes, ind = O.synth_rois(50, dim, shape[0], seed=2)
    ind[7] = shape[0] + 3   # out-of-range -> zero crop (crop_and_resize_kernel.cu:43-47)
    ind[9] = -1
    boxes[3, :] = [0.9, 0.9, 1.3, 1.2] + ([0.8, 1.5] if dim == 3 else [])   # partly outside: clamped sampling
    want = O.crop_and_resize_forward(img, boxes, ind, crop)
    gy = rs.randn(*want.shape).astype(np.float32)
    want_gx = O.crop_and_resize_backward(gy, boxes, ind, shape)
    fn = (NO.CropAndResizeFunction if dim == 3 else NO.CropAndResizeFunction2D)(*crop, 0)
    mf = torch.channels_last_3d if dim == 3 else torch.channels_last
    for layout in ("nc_first", "channels_last"):
        x = torch.from_numpy(img).to(DEV)
        if layout == "channels_last":
            x = x.contiguous(memory_format=mf)
        x.requires_grad_(True)
        y = fn(x, torch.from_numpy(boxes).to(DEV), torch.from_numpy(ind).to(DEV))
        assert tuple(y.shape) == want.shape
        assert _rel(y.detach().cpu().numpy(), want) < 1e-4, layout
        assert float(y[7].abs().max()) == 0.0 and float(y[9].abs().max()) == 0.0
        g = torch.from_numpy(gy).to(DEV)
        if layout == "channels_last":
            g = g.contiguous(memory_format=mf)
        y.backward(g)
        assert _rel(x.grad.cpu().numpy(), want_gx) < 1e-4, layout


def test_roi_align_vs_reference_kernels_cfg3(golden_dir):
    """cfg3 shapes: 36-channel FPN maps, 512 boxes per image x 2, pools (7,7,3) and (14,14,5); compared with the reference's own kernels
    (seeded samples of their outputs on the same inputs, tests/golden/ref_roi_align.npz from make_ref_kernel_golden.py; where oracle/_ref is
    built, also whole arrays against the kernels themselves)"""
    g = np.load(os.path.join(golden_dir, "ref_roi_align.npz"))
    live = O.ref_lib("roi3d") is not None and O.ref_lib("roi2d") is not None
    full = {}

    def check(tag, got, tol):
        assert list(got.shape) == g[tag + "__shape"].tolist(), tag
        err = np.abs(got.reshape(-1)[RK.sample_ix(got.size, tag)].astype(np.float64) - g[tag + "__sample"]).max() / g[tag + "__maxabs"][0]
        assert err < tol, (tag, err)
        if live:
            assert _rel(got, full[tag]) < tol, tag

    for tag, kind, args in RK.roi_inputs():
        if live:
            full[tag] = RK.ref_output(kind, args)
        if kind == "fwd3":
            img, boxes, ind, crop = args
            fn, fwd_tag = NO.CropAndResizeFunction(*crop, 0), tag
        elif kind == "bwd3":
            gy, boxes, ind, shape, layout = args
            x = torch.from_numpy(img).to(DEV)
            x = x.contiguous(memory_format=torch.channels_last_3d) if layout == "channels_last" else x
            x.requires_grad_(True)
            y = fn(x, torch.from_numpy(boxes).to(DEV), torch.from_numpy(ind).to(DEV))
            check(fwd_tag, y.detach().cpu().numpy(), 1e-5)
            y.backward(torch.from_numpy(gy).to(DEV))
            check(tag, x.grad.cpu().numpy(), 1e-4)  # fp32 atomics reorder on both sides
        else:
            img2, boxes, ind, crop = args
            y = NO.CropAndResizeFunction2D(*crop, 0)(torch.from_numpy(img2).to(DEV), torch.from_numpy(boxes).to(DEV), torch.from_numpy(ind).to(DEV))
            check(tag, y.cpu().numpy(), 1e-5)


def test_roi_align_gt_mask_call_shape():
    """mrcnn.py:558: ra3D(28,28,10) on GT masks [n_pos, 1, Y, X, Z] with box_ind = arange"""
    rs = np.random.RandomState(5)
    masks = (rs.rand(4, 1, 32, 32, 16) > 0.5).astype(np.float32)
    boxes, _ = O.synth_rois(4, 3, 4, seed=3)
    ind = np.arange(4, dtype=np.int32)
    want = O.crop_and_resize_forward(masks, boxes, ind, (28, 28, 10))
    y = NO.CropAndResizeFunction(28, 28, 10, 0)(torch.from_numpy(masks).to(DEV), torch.from_numpy(boxes).to(DEV), torch.from_numpy(ind).to(DEV))
    assert _rel(y.cpu().numpy(), want) < 1e-4


# ----------------------------------------------------------------------------------------------------------------------------------- matching
def test_matching_vs_golden_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "matching.npz"))
    anc = np.load(os.path.join(golden_dir, "anchors.npz"))
    for name in ["m3_sub", "m3_nosub", "m3_g1", "m2_nosub", "m2_sub"]:
        dim, tpi, seed, iou = g[name + "_cfg"]
        cf = cf3d() if int(dim) == 3 else cf2d()
        cf.rpn_train_anchors_per_image = int(tpi)
        cf.anchor_matching_iou = float(iou)
        anchors = anc["a3" if int(dim) == 3 else "a2"]
        np.random.seed(int(seed))
        m, t = MU.gt_anchor_matching(cf, anchors, g[name + "_gt"], g[name + "_cls"])
        assert m.dtype == np.int32 and np.array_equal(m, g[name + "_matches"]), name       # labels bit-exact incl. seeded sub-sampling
        want_t = g[name + "_targets"]
        assert np.allclose(t[: want_t.shape[0]], want_t, rtol=1e-12, atol=1e-12), name       # fp64 log may differ in the last ulp
    cf = cf3d()
    cf.rpn_train_anchors_per_image = 100000
    m, _ = MU.gt_anchor_matching(cf, anc["a3"], g["m3_rpn_gt"])
    assert np.array_equal(m, g["m3_rpn_matches"])
    m, t = MU.gt_anchor_matching(cf, anc["a3"], None)
    assert np.all(m == -1) and np.all(t == 0)


def test_matching_cfg4_and_full_grid_vs_oracle():
    """cfg4: 50 000 shuffled anchors of the cfg2 grid x G in {8, 64}; plus the full 1 347 840-anchor grid x 8 (cfg2 per-step call)"""
    full = MU.generate_pyramid_anchors(None, cf3d((128, 128, 128)))
    rs = np.random.RandomState(0)
    sub = full[rs.permutation(full.shape[0])[:50000]]
    from golden_cfg import rand_gt
    for anchors, G in [(sub, 8), (sub, 64), (full, 8), (sub[:8000], 600)]:   # the numpy oracle materialises A x G fp64
        gt = rand_gt(rs, G, (128, 128, 128), 3, 4, 48).astype(np.float64)
        gt[0] = anchors[2345 % anchors.shape[0]]           # exact IoU 1.0 hit
        if G >= 8:
            gt[5] = gt[2]                                   # duplicate GT: tie in the row argmax, later GT wins the column step
        cls = rs.randint(1, 3, size=G).astype(np.int32)
        a_dev = torch.from_numpy(anchors).to(DEV)
        m, arg, npos = MU.anchor_match_device(a_dev, torch.from_numpy(gt).to(DEV), torch.from_numpy(cls).to(DEV), 3, 0.01, 0.5)
        want_m, want_arg = MO.match_labels(anchors, gt, cls, 0.5, 3)
        assert np.array_equal(m.cpu().numpy(), want_m), G
        assert np.array_equal(arg.cpu().numpy(), want_arg), G
        assert int(npos.item()) == int((want_m > 0).sum())


def test_matching_touching_nested_and_flat_boxes_vs_oracle():
    """the comparison-only reject of separated pairs must reproduce numpy for touching faces, nested boxes, zero-extent (flat) GT
    boxes and a GT that overlaps nothing (its column maximum stays 0 -> np.argmax picks anchor 0)"""
    for dim in (2, 3):
        B = 2 * dim
        rs = np.random.RandomState(dim)
        lo = rs.randint(0, 40, size=(3000, dim)).astype(np.float64)
        ext = rs.randint(1, 24, size=(3000, dim)).astype(np.float64)
        anchors = np.zeros((3000, B))
        gt = np.zeros((7, B))
        def put(dst, i, l, e):
            dst[i, 0], dst[i, 1], dst[i, 2], dst[i, 3] = l[0], l[1], l[0] + e[0], l[1] + e[1]
            if dim == 3:
                dst[i, 4], dst[i, 5] = l[2], l[2] + e[2]
        for i in range(3000):
            put(anchors, i, lo[i], ext[i])
        put(gt, 0, lo[10] + np.array([ext[10][0]] + [0] * (dim - 1)), ext[10])      # shares a face with anchor 10
        put(gt, 1, lo[20] + 1, np.maximum(ext[20] - 2, 1))                            # nested in anchor 20
        put(gt, 2, lo[30], ext[30])                                                  # identical to anchor 30
        put(gt, 3, lo[40], ext[40] * np.array([0] + [1] * (dim - 1)))                # flat: zero extent along y
        put(gt, 4, np.full(dim, 500.0), np.full(dim, 4.0))                           # far away from every anchor
        put(gt, 5, lo[50] - 0.5, ext[50] + 1.0)                                      # contains anchor 50
        put(gt, 6, lo[60] + 0.25, ext[60])                                           # shifted copy
        cls = np.arange(1, 8).astype(np.int32)
        m, arg, npos = MU.anchor_match_device(torch.from_numpy(anchors).to(DEV), torch.from_numpy(gt).to(DEV), torch.from_numpy(cls).to(DEV),
                                              dim, 0.1 if dim == 2 else 0.01, 0.5)
        want_m, want_arg = MO.match_labels(anchors, gt, cls, 0.5, dim)
        assert np.array_equal(arg.cpu().numpy(), want_arg), dim
        assert np.array_equal(m.cpu().numpy(), want_m), dim
        assert int(npos.item()) == int((want_m > 0).sum())


def test_nms_at_the_exact_threshold():
    """pairs whose IoU equals the threshold exactly (`>` is strict, nms_kernel.cu:72): a lattice of equal 10x10x10 boxes shifted by 5 along y
    (neighbours overlap by exactly half: IoU = 500 / 1500) at the threshold, one ulp below and one ulp above, vs the C oracle"""
    n = 4096
    lat = np.zeros((n, 7), dtype=np.float32)
    lat[:, 0] = 5.0 * np.arange(n); lat[:, 2] = lat[:, 0] + 9.0
    lat[:, 3] = 9.0; lat[:, 5] = 9.0
    lat[:, 6] = np.linspace(1.0, 0.0, n, dtype=np.float32)
    third = np.float32(500.0) / np.float32(1500.0)
    kept = []
    for thr in (float(third), float(np.nextafter(third, np.float32(0))), float(np.nextafter(third, np.float32(1))), 1.0, 0.0):
        k = _keep(lat, thr, 3).tolist()
        assert k == O.nms(lat, thr, 3).tolist(), thr
        kept.append(len(k))
    assert kept[0] == n and kept[1] == n // 2 and kept[2] == n          # IoU == thr keeps both boxes; one ulp below suppresses every second box


@pytest.mark.parametrize("dim,thr", [(3, 1e-5), (3, 0.5), (2, 0.3)])
def test_nms_skips_separated_tiles_bit_exactly(dim, thr):
    """boxes of independent groups translated apart along y and ordered group by group (what retina_unet.refine_detections feeds): the mask
    kernel skips (row block, column tile) pairs with separated y extents — the keep list must still be the greedy oracle's, including tiles
    that straddle a group boundary, touching bands (gap of exactly one pixel = IoU 0) and a ragged last tile"""
    parts = []
    for g, n in enumerate((3000, 1777, 64, 2500)):
        b = O.synth_boxes(n, dim, seed=40 + g, rounded=True)
        b = b[np.argsort(-b[:, -1], kind="stable")]
        b[:, 0] += 129.0 * g                                  # extent 128 + 1: neighbouring bands touch without overlapping
        b[:, 2] += 129.0 * g
        parts.append(b)
    boxes = np.concatenate(parts).astype(np.float32)
    assert _keep(boxes, thr, dim).tolist() == O.nms(boxes, thr, dim).tolist()
    # negative threshold: disjoint pairs DO suppress (0 > thr), so nothing may be skipped
    small = boxes[::37].copy()
    assert _keep(small, -1.0, dim).tolist() == O.nms(small, -1.0, dim).tolist()
