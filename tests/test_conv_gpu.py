"""conv3d parity (GPU): libmdt_b200 conv kernels through the C-ABI vs a plain PyTorch reference of the same op (fp64 on the GPU, i.e.
the exact result up to rounding; tolerance 1e-4 relative to max|ref|, the north_star bar for conv).  Covers every (kernel, stride,
padding, channel) combination the reference's backbone and heads use (models/backbone.py:27-206, models/retina_unet.py:40-119,
models/mrcnn.py:40-169) for both algorithms (fp32 SIMT and, where the shape is supported, the tcgen05 implicit GEMM)."""
import os
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from medicaldetectiontoolkit_b200 import _lib as L
from medicaldetectiontoolkit_b200 import conv as C

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-4

# (cin, cout, k, stride, pad, spatial)
SHAPES = [
    (1, 18, 3, 1, 1, (12, 10, 16)),            # C0 first conv (Cin = 1)
    (1, 18, 3, 1, 1, (3, 5, 128)),             # stem at the full line length; 30 lines = 7.5 groups of the 4-line wgrad kernel
    (1, 24, 3, 1, 1, (3, 3, 20)),              # stem with 24 output channels (the 32-wide weight padding of the specialised fprop)
    (1, 7, 3, 1, 1, (2, 3, 9)),                # odd channel count: partial co tiles in the stem wgrad
    (2, 18, 3, 1, 1, (4, 4, 16)),              # Cin = 2: the generic stem kernels
    (18, 18, 3, 1, 1, (8, 8, 32)),             # C0 second conv / ResBlock conv2
    (18, 18, 7, (2, 2, 1), 3, (16, 16, 12)),   # C1 k7 s(2,2,1)
    (18, 72, 1, 1, 0, (6, 6, 8)),              # bottleneck expand / downsample
    (72, 36, 1, (2, 2, 2), 0, (8, 8, 8)),      # strided 1x1x1 (ResBlock conv1 with stride)
    (36, 36, 3, 1, 1, (8, 8, 128)),            # P*_conv2
    (36, 64, 3, 1, 1, (4, 4, 128)),            # head conv_1
    (64, 64, 3, 1, 1, (4, 8, 128)),            # head tower
    (64, 27, 3, 1, 1, (4, 4, 128)),            # classifier conv_final
    (64, 54, 3, 1, 1, (4, 4, 16)),             # regressor conv_final on a small level
    (36, 144, (7, 7, 3), 1, 0, (7, 7, 3)),     # mrcnn Classifier conv1 with ks = pool_size
    (144, 288, 3, 1, 1, (4, 4, 8)),            # deep encoder conv2
    (36, 2, 1, 1, 0, (8, 8, 16)),              # final_conv (seg logits)
    # lines of 65..128 voxels: the tap-stacked tcgen05 kernel (conv3d_tcw.cu) for fprop / dgrad
    (36, 36, 3, 1, 1, (5, 7, 128)),            # P0_conv2: odd line count (half-empty last tile), K = 48 as 32 + 16 channel chunks
    (18, 18, 3, 1, 1, (3, 6, 128)),            # C0 second conv: 2 CTAs per SM
    (18, 18, 7, (2, 2, 1), 3, (8, 12, 128)),   # C1 k7 s(2,2,1): 9 source lines per kd, 7 shifts, dgrad with line parity
    (64, 54, 3, 1, 1, (3, 4, 128)),            # regressor conv_final: 3 unstacked MMAs per K step
    (36, 36, 3, 1, 1, (4, 4, 96)),             # line shorter than the 128-row tile
    (72, 72, 3, 1, 1, (3, 4, 128)),            # K = 80 as 64 + 16
    (36, 96, 3, 1, 1, (2, 3, 128)),            # N tiling: 3 x 96 columns > 256 -> two tiles of 84 / 12 channels
    (36, 36, 1, 1, 0, (4, 4, 128)),            # 1x1x1: no shifts
    (18, 36, 3, (2, 2, 1), 1, (6, 8, 128)),    # strided k3
    (36, 36, 3, 1, 0, (5, 6, 128)),            # valid conv: output lines of 126 voxels
    (36, 18, 3, 1, 1, (3, 5, 72)),             # 18 output channels (float2 stores), 72-voxel lines
    # pointwise fp32 streaming kernels (conv3d_pw.cu, algo 4)
    (18, 36, 1, 1, 0, (5, 7, 128)),            # P0_conv1 lateral; voxel count not a multiple of the 256-voxel tile
    (36, 144, 1, 1, 0, (4, 4, 16)),            # ResBlock conv3: 36 output quads = 3 chunks of 12
    (144, 36, 1, 1, 0, (4, 4, 16)),            # ResBlock conv1 of the next block: one voxel per thread
    (72, 18, 1, 1, 0, (4, 4, 32)),
    (64, 96, 1, 1, 0, (3, 3, 16)),             # the largest cin * cout that stays off the tensor cores; two chunks of 12 quads
    (5, 7, 1, 1, 0, (3, 5, 9)),                # odd channel counts: scalar global accesses, padded quads
]


def _ref(x, w, b, stride, pad, relu, res):
    y = F.conv3d(x.double(), w.double(), None if b is None else b.double(), stride=stride, padding=pad)
    if res is not None:
        y = y + res.double()
    return torch.relu(y) if relu else y


def _rel(a, ref):
    return float((a.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _tc_passes(desc_args):
    """passes (0 fprop, 1 dgrad, 2 wgrad) for which `auto` resolves to the tcgen05 path"""
    lib = L.load()
    d = C._desc(*desc_args, False, 0, 0)
    return [ps for ps in (0, 1, 2) if lib.mdt_conv3d_algo(d, ps) == 2]


@pytest.mark.parametrize("cin,cout,k,stride,pad,sp", SHAPES)
def test_conv3d_fprop_dgrad_wgrad(cin, cout, k, stride, pad, sp):
    torch.manual_seed(cin * 131 + cout)
    k3, s3, p3 = C._triple(k), C._triple(stride), C._triple(pad)
    x = torch.randn(2, cin, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d)
    w = torch.randn(cout, cin, *k3, device=DEV) / np.sqrt(cin * np.prod(k3))
    b = torch.randn(cout, device=DEV)
    yref = _ref(x, w, b, s3, p3, True, None)
    res = torch.randn_like(yref.float()).contiguous(memory_format=torch.channels_last_3d)
    gy = torch.randn_like(yref.float()).contiguous(memory_format=torch.channels_last_3d)
    xd = x.double().requires_grad_(True)
    wd = w.double().requires_grad_(True)
    F.conv3d(xd, wd, None, stride=s3, padding=p3).backward(gy.double())
    tc = _tc_passes((tuple(x.shape), tuple(w.shape), s3, p3))
    if cin <= 4:   # stem: `auto` resolves to the direct SIMT kernels; still exercise the tensor-core kernels explicitly
        tc = [0, 1, 2]
    lib = L.load()
    pw = [ps for ps in (0, 1, 2) if lib.mdt_conv3d_algo(C._desc(tuple(x.shape), tuple(w.shape), s3, p3, False, 0, 4), ps) == 4]
    assert bool(pw) == (k3 == (1, 1, 1) and s3 == (1, 1, 1) and cin * cout <= 6144)
    for algo in (1, 2, 4):
        if algo == 4:
            tc = pw
        for prec in ([0] if algo != 2 else [0, 1]):
            tol = TOL if prec == 0 else 2e-2   # precision 1 = single-pass bf16 throughput mode
            if algo == 1 or 0 in tc:
                y = C.conv3d_forward(x, w, b, s3, p3, relu=True, precision=prec, algo=algo)
                assert y.shape == yref.shape and y.is_contiguous(memory_format=torch.channels_last_3d)
                assert _rel(y, yref) < tol, ("fprop", algo, prec)
                y2 = C.conv3d_forward(x, w, None, s3, p3, relu=False, residual=res, precision=prec, algo=algo)
                assert _rel(y2, _ref(x, w, None, s3, p3, False, res)) < tol, ("fprop+res", algo, prec)
            if algo == 1 or 1 in tc:
                dx = C.conv3d_dgrad(gy, w, tuple(x.shape), s3, p3, precision=prec, algo=algo)
                assert _rel(dx, xd.grad) < tol, ("dgrad", algo, prec)
            if algo == 1 or 2 in tc:
                dw, db = C.conv3d_wgrad(x, gy, tuple(w.shape), s3, p3, True, precision=prec, algo=algo)
                assert _rel(dw, wd.grad) < tol, ("wgrad", algo, prec)
                assert _rel(db, gy.double().sum(dim=(0, 2, 3, 4))) < tol, ("bgrad", algo, prec)


def test_tap_stacked_kernel_is_selected_for_long_lines():
    """fprop / dgrad of the long-line layers with >= 112 stacked columns (36 -> 36/64, 64 -> 64 k3, 18 -> 18 k7: where it measured faster,
    profiles/r02_tcw_vs_halo.txt) run on conv3d_tcw.cu, the others on conv3d_tc.cu"""
    lib = L.load()
    for cin, cout, k, stride, pad, sp, want in [(36, 36, 3, 1, 1, (128, 128, 128), [3, 3]), (18, 18, 7, (2, 2, 1), 3, (128, 128, 128), [3, 3]),
                                                (36, 64, 3, 1, 1, (32, 32, 128), [3, 3]), (64, 64, 3, 1, 1, (32, 32, 128), [3, 3]),
                                                (18, 18, 3, 1, 1, (128, 128, 128), [2, 2]), (64, 64, 3, 1, 1, (16, 16, 64), [2, 2]),
                                                (144, 144, 3, 1, 1, (8, 8, 32), [2, 2])]:
        d = C._desc((2, cin) + sp, (cout, cin) + C._triple(k), C._triple(stride), C._triple(pad), False, 0, 0)
        assert [lib.mdt_conv3d_variant(d, ps) for ps in (0, 1)] == want, (cin, cout, k, sp)
        assert lib.mdt_conv3d_variant(d, 2) == 2


def test_pointwise_layers_run_on_the_streaming_kernels():
    """1x1x1 stride-1 convs with cin * cout <= 2592 (laterals, the narrow bottleneck 1x1x1s, final_conv: where tools/pw_bench.py measured them
    faster) resolve to conv3d_pw.cu for all passes and for the fused backward; wider ones and strided ones stay where they were"""
    lib = L.load()
    for cin, cout, stride, sp, want in [(18, 36, 1, (128, 128, 128), 4), (36, 2, 1, (128, 128, 128), 4), (18, 72, 1, (32, 32, 128), 4),
                                        (72, 18, 1, (32, 32, 128), 4), (144, 36, 1, (16, 16, 64), 2), (36, 144, 1, (16, 16, 64), 2), (288, 72, 1, (8, 8, 32), 2), (72, 144, 2, (32, 32, 128), None)]:
        d = C._desc((2, cin) + sp, (cout, cin, 1, 1, 1), C._triple(stride), (0, 0, 0), False, 0, 0)
        got = [lib.mdt_conv3d_variant(d, ps) for ps in (0, 1, 2)]
        if want is None:
            assert 4 not in got
        else:
            assert got == [want] * 3, (cin, cout, got)
            assert lib.mdt_conv3d_backward_fused(d, 1) == 1


def test_tc_path_covers_the_hot_layers():
    """the layers that carry the FLOPs of cfg2 (SURVEY §8d breakdown) must resolve to the tcgen05 kernels for all three passes"""
    lib = L.load()
    for cin, cout, k, stride, pad, sp in [(64, 64, 3, 1, 1, (32, 32, 128)), (36, 36, 3, 1, 1, (128, 128, 128)), (18, 18, 7, (2, 2, 1), 3, (128, 128, 128)),
                                          (18, 18, 3, 1, 1, (128, 128, 128)), (36, 64, 3, 1, 1, (32, 32, 128)), (64, 54, 3, 1, 1, (32, 32, 128)),
                                          (64, 64, 3, 1, 1, (16, 16, 64))]:
        d = C._desc((2, cin) + sp, (cout, cin) + C._triple(k), C._triple(stride), C._triple(pad), False, 0, 0)
        assert [lib.mdt_conv3d_algo(d, ps) for ps in (0, 1, 2)] == [2, 2, 2], (cin, cout, k)


def test_conv_module_autograd_and_state_dict_keys():
    """NDConvGenerator nesting / keys (probe in SURVEY §5: `C0.0.0.weight`) and autograd through the fused bias+ReLU epilogue"""
    gen = C.NDConvGenerator(3)
    m = torch.nn.Sequential(gen(1, 18, ks=3, pad=1, relu='relu'), gen(18, 18, ks=3, pad=1, relu='relu')).to(DEV)
    assert sorted(m.state_dict().keys()) == ['0.0.bias', '0.0.weight', '1.0.bias', '1.0.weight']
    bare = gen(18, 36, ks=1, relu=None).to(DEV)
    assert sorted(bare.state_dict().keys()) == ['bias', 'weight'] and tuple(bare.weight.shape) == (36, 18, 1, 1, 1)
    ref = torch.nn.Sequential(torch.nn.Conv3d(1, 18, 3, padding=1), torch.nn.ReLU(), torch.nn.Conv3d(18, 18, 3, padding=1), torch.nn.ReLU()).to(DEV).double()
    ref[0].load_state_dict({k[2:]: v.double() for k, v in m[0].state_dict().items()})
    ref[2].load_state_dict({k[2:]: v.double() for k, v in m[1].state_dict().items()})
    x = torch.randn(2, 1, 8, 8, 16, device=DEV, requires_grad=True)
    xr = x.detach().double().requires_grad_(True)
    y = m(x)
    yr = ref(xr)
    assert _rel(y, yr) < TOL
    g = torch.randn_like(y)
    y.backward(g)
    yr.backward(g.double())
    assert _rel(x.grad, xr.grad) < TOL
    assert _rel(m[1][0].weight.grad, ref[2].weight.grad) < TOL and _rel(m[0][0].bias.grad, ref[0].bias.grad) < TOL


def test_conv2d_module_matches_torch():
    gen = C.NDConvGenerator(2)
    m = gen(3, 8, ks=3, pad=1, stride=2, relu='relu').to(DEV)
    x = torch.randn(2, 3, 16, 16, device=DEV, requires_grad=True)
    y = m(x)
    yr = torch.relu(F.conv2d(x.double(), m[0].weight.double(), m[0].bias.double(), stride=2, padding=1))
    assert _rel(y, yr) < TOL
    y.sum().backward()
    assert x.grad is not None and m[0].weight.grad.shape == m[0].weight.shape


@pytest.mark.parametrize("cin,cout,sp", [(18, 72, (8, 8, 32)), (64, 64, (4, 8, 128)), (36, 36, (8, 8, 128)), (1, 18, (8, 8, 128)), (36, 144, (5, 5, 9)),
                                         (144, 36, (4, 4, 16))])
def test_fused_backward_relu_residual_bias(cin, cout, sp):
    """mdt_conv3d_backward: one pass over dy feeds dgrad + wgrad, with the ReLU mask, the bias gradient and the residual gradient folded in"""
    torch.manual_seed(cin + cout)
    k = 1 if (cin, cout) in ((18, 72), (36, 144), (144, 36)) else 3
    pad = k // 2
    x = torch.randn(2, cin, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d).requires_grad_(cin > 1)
    w = (torch.randn(cout, cin, k, k, k, device=DEV) / np.sqrt(cin * k ** 3)).requires_grad_(True)
    b = torch.randn(cout, device=DEV).requires_grad_(True)
    res = torch.randn(2, cout, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d).requires_grad_(True)
    y = C._Conv3dFn.apply(x, w, b, res, (1, 1, 1), (pad,) * 3, True, 0, 0)
    g = torch.randn_like(y)
    y.backward(g)
    xd, wd, bd, rd = (t.detach().double().requires_grad_(True) for t in (x, w, b, res))
    pre = F.conv3d(xd, wd, bd, padding=pad) + rd
    assert _rel(y, torch.relu(pre)) < TOL
    # the reference backward uses OUR forward's ReLU mask: a pre-activation within rounding distance of zero may legitimately fall on either
    # side, and one flipped element would dominate a max-norm comparison of the gradients (see tests/test_model_gpu.py::_rel_l2)
    pre.backward(g.double() * (y.detach() > 0))
    assert _rel(w.grad, wd.grad) < TOL and _rel(b.grad, bd.grad) < TOL and _rel(res.grad, rd.grad) < TOL
    if cin > 1:
        assert _rel(x.grad, xd.grad) < TOL
    d = C._desc(tuple(x.shape), tuple(w.shape), (1, 1, 1), (pad,) * 3, False, 0, 0)
    assert L.load().mdt_conv3d_backward_fused(d, int(cin > 1)) == (1 if cin > 4 else 0)    # fused tcgen05 path; the Cin<=4 stem uses the direct kernels


@pytest.mark.parametrize("cin,cout,k,stride,sp", [(36, 36, 3, 1, (3, 5, 128)), (36, 64, 3, 1, (2, 4, 128)), (64, 64, 3, 1, (2, 4, 128)), (64, 54, 3, 1, (4, 8, 32)),
                                                    (18, 18, 7, (2, 2, 1), (8, 8, 128)), (72, 18, 1, 1, (4, 4, 32)), (18, 72, 1, 1, (3, 4, 128)),
                                                    (18, 36, 1, 1, (3, 5, 128)), (36, 144, 1, 1, (2, 3, 40)), (144, 288, 1, 1, (2, 2, 16))])
def test_epilogue_emits_the_split_planes_of_the_result(cin, cout, k, stride, sp):
    """mdt_conv3d_fprop_presplit_out: the (hi, lo) bf16 planes written by the conv epilogue are byte-identical to mdt_conv3d_split applied to
    the fp32 result (incl. zero padding channels), for both tcgen05 fprop kernels; a consumer conv fed from them gives identical output"""
    torch.manual_seed(cin * 7 + cout)
    lib = L.load()
    k3, s3 = C._triple(k), C._triple(stride)
    p3 = tuple(kk // 2 for kk in k3)
    x = torch.randn(2, cin, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d)
    w = torch.randn(cout, cin, *k3, device=DEV) / np.sqrt(cin * np.prod(k3))
    b = torch.randn(cout, device=DEV)
    d = C._desc(tuple(x.shape), tuple(w.shape), s3, p3, True, 0, 0)
    if lib.mdt_conv3d_algo(d, 0) not in (2, 4):
        pytest.skip("shape on neither the tcgen05 nor the pointwise path")
    y0 = C.conv3d_forward(x, w, b, s3, p3, relu=True)
    y1 = C.conv3d_forward(x, w, b, s3, p3, relu=True, emit_split=True)
    assert torch.equal(y0, y1)
    ys, ver, prec = y1._mdt_split
    w2 = torch.randn(8, cout, 1, 1, 1, device=DEV)
    d2 = C._desc(tuple(y1.shape), tuple(w2.shape), (1, 1, 1), (0, 0, 0), False, 0, 0)
    want = torch.empty(lib.mdt_conv3d_split_bytes(d2), dtype=torch.uint8, device=DEV)
    assert want.numel() == ys.numel()
    L.check(lib.mdt_conv3d_split(d2, L.ptr(y0), L.ptr(want), L.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(ys, want), (int((ys != want).sum()), ys.numel())


@pytest.mark.parametrize("cin,cout,sp", [(72, 288, (8, 8, 32)), (144, 576, (4, 4, 16)), (36, 36, (4, 4, 16)), (18, 72, (32, 32, 64))])
def test_bias_gradient_of_the_unfused_wgrad(cin, cout, sp):
    """db = column sums of dy from mdt_conv3d_wgrad (the wide cout > 256 layers of C4/C5 take the row-serial branch of bias_grad_kernel)"""
    torch.manual_seed(7)
    x = torch.randn(2, cin, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d)
    gy = torch.randn(2, cout, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d)
    dw, db = C.conv3d_wgrad(x, gy, (cout, cin, 1, 1, 1), (1, 1, 1), (0, 0, 0), True)
    ref = gy.double().sum((0, 2, 3, 4))
    assert float((db.double() - ref).abs().max() / ref.abs().max()) < 1e-5
    ref_w = torch.einsum('ncdhw,nkdhw->ck', gy.double(), x.double()).reshape(cout, cin, 1, 1, 1)
    assert float((dw.double() - ref_w).abs().max() / ref_w.abs().max()) < 1e-4


@pytest.mark.parametrize("cin,cout,k,stride,pad", [(36, 36, 3, (1, 1, 1), 1), (18, 18, 7, (2, 2, 1), 3)])
def test_full_resolution_layers_vs_fp64(cin, cout, k, stride, pad):
    """the two heaviest layers of cfg2 at their BASELINE size (2 x C x 128^3) against fp64 F.conv3d: forward, input gradient and weight gradient.
    Weight gradients at this size sum 4.2 M products per element: the bound below (3e-5 of max|ref|, measured 9e-6) is what the accumulator
    chain limit of the wgrad kernel (<= 512 MMAs per TMEM accumulator, partial sums combined in IEEE fp32) guarantees; 1e-4 is the parity bar."""
    torch.manual_seed(11)
    sp = (128, 128, 128)
    k3, p3 = C._triple(k), C._triple(pad)
    x = torch.randn(2, cin, *sp, device=DEV).contiguous(memory_format=torch.channels_last_3d)
    w = torch.randn(cout, cin, *k3, device=DEV) / float(np.sqrt(cin * np.prod(k3)))
    b = torch.randn(cout, device=DEV) * 0.1
    y = C.conv3d_forward(x, w, b, stride, p3)
    gy = torch.randn_like(y)
    dx = C.conv3d_dgrad(gy, w, tuple(x.shape), stride, p3)
    dw, db = C.conv3d_wgrad(x, gy, tuple(w.shape), stride, p3, True)
    xd = x.double().contiguous().requires_grad_(True)          # NCDHW fp64 reference
    wd, bd = w.double().requires_grad_(True), b.double().requires_grad_(True)
    ref = F.conv3d(xd, wd, bd, stride=stride, padding=p3)
    ref.backward(gy.double().contiguous())
    errs = {"fprop": _rel(y, ref.detach()), "dgrad": _rel(dx, xd.grad), "wgrad": _rel(dw, wd.grad), "bias": _rel(db, bd.grad)}
    assert errs["fprop"] < 3e-5 and errs["dgrad"] < 3e-5 and errs["wgrad"] < 3e-5 and errs["bias"] < 3e-5, errs


@pytest.mark.parametrize("cin,cout,k,sp,algo", [(1, 18, 3, (8, 8, 128), 0),     # stem, c1k3 weight-gradient kernel
                                                (2, 18, 3, (4, 4, 16), 0),      # stem, generic kernel
                                                (18, 18, 3, (8, 8, 32), 1),     # fp32 SIMT split-M weight gradient
                                                (36, 36, 3, (8, 16, 128), 2),   # tcgen05 weight gradient + bias_grad_kernel
                                                (288, 576, 1, (4, 4, 8), 0)])   # wide bias gradient (cout > 256)
def test_weight_and_bias_gradients_are_bitwise_reproducible(cin, cout, k, sp, algo):
    """the cross-block reductions of the weight / bias gradients combine per-block partials in a fixed order (no float atomics): the same
    inputs give the same bits on every call, through both the unfused wgrad and the fused backward"""
    g = torch.Generator(device=DEV).manual_seed(cin * 1000 + cout)
    x = torch.randn((2, cin) + sp, device=DEV, generator=g).contiguous(memory_format=torch.channels_last_3d)
    w = torch.randn(cout, cin, k, k, k, device=DEV, generator=g) * 0.05
    gy = torch.randn((2, cout) + sp, device=DEV, generator=g).contiguous(memory_format=torch.channels_last_3d)
    p3 = (k // 2,) * 3
    first = C.conv3d_wgrad(x, gy, tuple(w.shape), (1, 1, 1), p3, True, algo=algo)
    for _ in range(3):
        again = C.conv3d_wgrad(x, gy, tuple(w.shape), (1, 1, 1), p3, True, algo=algo)
        assert torch.equal(first[0], again[0]) and torch.equal(first[1], again[1])
    fused = C.conv3d_backward(x, gy, None, w, (1, 1, 1), p3, True, True, False, algo=algo)
    if fused is not None:
        for _ in range(3):
            again = C.conv3d_backward(x, gy, None, w, (1, 1, 1), p3, True, True, False, algo=algo)
            assert all(torch.equal(a, b) for a, b in zip(fused[:3], again[:3]))
        ref_db = gy.double().sum(dim=(0, 2, 3, 4))
        assert float((fused[2].double() - ref_db).abs().max() / ref_db.abs().max()) < TOL
