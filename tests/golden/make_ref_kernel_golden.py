#!/usr/bin/env python
"""Golden vectors of the reference's own CUDA kernels (NMS 2D/3D, crop-and-resize 3D/2D), compiled unmodified for sm_100a into
oracle/_ref by oracle/build_ref.sh.  The inputs are the seeded ones of tests/test_ops_gpu.py (test_nms_full_size_cfg4_properties_and_reference_kernel,
test_roi_align_vs_reference_kernels_cfg3), drawn in the same order, so the tests compare against these files without the reference build.
Needs a GPU and oracle/_ref:  python tests/golden/make_ref_kernel_golden.py OUT_DIR  ->  OUT_DIR/ref_nms.npz, OUT_DIR/ref_roi_align.npz

NMS keep lists are stored whole, as bit masks over the sorted boxes (keep_bits / kept).  The RoIAlign outputs are up to 36 M values each,
so only SAMPLE_N values at seeded flat positions (sample_ix) are stored, together with max|value| of the whole array (the denominator of
the tests' relative error)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import _oracle as O  # noqa: E402

NMS_3D_CASES = [(100000, 0.5, True), (50000, 1e-5, True), (6000, 0.7, False)]   # (n, threshold, rounded); boxes seeded with n
NMS_2D_CASE = (30000, 0.5, False, 3)                                               # (n, threshold, rounded, seed)
ROI_3D_CASES = [((2, 36, 32, 32, 128), (7, 7, 3)), ((2, 36, 16, 16, 64), (14, 14, 5)), ((2, 36, 4, 4, 16), (7, 7, 3))]
SAMPLE_N = 2048


def keep_bits(keep, n):
    """keep list (ascending indices into n boxes) -> packed bit mask"""
    mask = np.zeros(n, dtype=bool)
    mask[keep] = True
    return np.packbits(mask)


def kept(bits, n):
    """inverse of keep_bits"""
    return np.flatnonzero(np.unpackbits(bits, count=n))


def sample_ix(size, tag):
    """SAMPLE_N seeded flat positions into an array of `size` elements (the seed is derived from the array's name)"""
    return np.random.RandomState(sum(map(ord, tag))).randint(0, size, size=SAMPLE_N)


def roi_inputs():
    """yields (tag, kind, args) in the order tests/test_ops_gpu.py::test_roi_align_vs_reference_kernels_cfg3 draws them from one RandomState(4):
    kind "fwd3" -> (img, boxes, ind, crop); "bwd3" -> (gy, boxes, ind, image_shape, layout); "fwd2" -> (img, boxes, ind, crop).
    The gradient gy is drawn once per layout (nc_first, channels_last) after the forward."""
    rs = np.random.RandomState(4)
    for i, (shape, crop) in enumerate(ROI_3D_CASES):
        img = rs.randn(*shape).astype(np.float32)
        boxes, ind = O.synth_rois(1024, 3, 2, seed=8)
        out_shape = (boxes.shape[0], shape[1]) + crop
        yield "roi3d_%d_fwd" % i, "fwd3", (img, boxes, ind, crop)
        for layout in ("nc_first", "channels_last"):
            gy = rs.randn(*out_shape).astype(np.float32)
            yield "roi3d_%d_bwd_%s" % (i, layout), "bwd3", (gy, boxes, ind, shape, layout)
    img = rs.randn(2, 36, 64, 64).astype(np.float32)
    boxes, ind = O.synth_rois(300, 2, 2, seed=9)
    yield "roi2d_fwd", "fwd2", (img, boxes, ind, (7, 7))


def ref_output(kind, args):
    """the reference kernel's whole output for one item of roi_inputs() (needs oracle/_ref and a GPU)"""
    if kind == "bwd3":
        gy, boxes, ind, shape, _ = args
        return O.ref_crop_and_resize_backward(gy, boxes, ind, shape)
    return O.ref_crop_and_resize_forward(*args)


def main():
    out_dir = sys.argv[1]
    for name in ("nms3d", "nms2d", "roi3d", "roi2d"):
        if O.ref_lib(name) is None:
            raise SystemExit("oracle/_ref/libref_%s.so is missing: run oracle/build_ref.sh where the reference tree is present" % name)
    nms = {}
    for n, thr, rounded in NMS_3D_CASES:
        nms["nms3d_%d" % n] = keep_bits(O.ref_nms(O.synth_boxes(n, 3, seed=n, rounded=rounded), thr, 3), n)
    n, thr, rounded, seed = NMS_2D_CASE
    nms["nms2d_%d" % n] = keep_bits(O.ref_nms(O.synth_boxes(n, 2, seed=seed, rounded=rounded), thr, 2), n)
    for k, v in nms.items():
        print(k, "keeps", int(np.unpackbits(v).sum()))
    np.savez_compressed(os.path.join(out_dir, "ref_nms.npz"), **nms)

    roi = {}
    for tag, kind, args in roi_inputs():
        ref = ref_output(kind, args)
        roi[tag + "__sample"] = ref.reshape(-1)[sample_ix(ref.size, tag)]
        roi[tag + "__maxabs"] = np.array([np.abs(ref).max()], dtype=np.float64)
        roi[tag + "__shape"] = np.array(ref.shape, dtype=np.int64)
        print(tag, ref.shape, "max|ref|", float(np.abs(ref).max()))
    np.savez_compressed(os.path.join(out_dir, "ref_roi_align.npz"), **roi)


if __name__ == "__main__":
    main()
