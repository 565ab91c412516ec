"""bench.py host-side pieces that do not need a GPU: the roofline object of the JSON line."""
import json

import bench


def test_roofline_object_has_the_contract_keys():
    tag = (0, (2, 36, 128, 128, 128), (36, 36, 3, 3, 3), (1, 1, 1), 0)
    dom = (2.0 * 2 * 128 ** 3 * 36 * 36 * 27, 2.5, tag, 1.0)
    btag = (3, (2, 36, 128, 128, 128), (36, 36, 3, 3, 3), (1, 1, 1), 2)
    slow = (2 * dom[0], 6.3, btag, 1.0)
    traffic = {"input_shape": [2, 36, 128, 128, 128], "dram_bytes": 1.378e9, "source": "profiles/r02_ncu_conv_tcw_p0_36.txt"}
    r = bench.make_roofline(3.6e12, 52.0, 229, 66.7, dom, 1444.3, True, slow, traffic)
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "slowest_launch"):
        assert k in r
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and r["traffic"] == 1.378e9 and "r02" in r["traffic_source"]
    assert r["slowest_launch"]["ms"] == 6.3 and "fused backward" in r["slowest_launch"]["kernel"]
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0 < r["frac"] < 1
    assert abs(r["achieved"] - dom[0] / 2.5 / 1e9) < 1e-9
    agg = r["all_conv_launches"]
    assert abs(agg["achieved"] - 3.6e12 / 52e-3 / 1e12) < 1e-9 and abs(agg["conv_share_of_step"] - 52.0 / 66.7) < 1e-12
    json.dumps(r)
    # no per-launch tag (e.g. SIMT-only run): the aggregate is reported at the top level; no conv time at all: no roofline
    r2 = bench.make_roofline(3.6e12, 52.0, 229, 66.7, None, 1400.0, False)
    assert r2["traffic"] is None and "fallback" in r2["peak_source"] and r2["frac"] == r2["all_conv_launches"]["frac"]
    assert bench.make_roofline(3.6e12, None, 0, 66.7, None, 1400.0, False) is None


def test_step_outputs_are_float_copies_and_large_arrays_are_sampled(monkeypatch):
    import numpy as np
    import torch
    net = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 2))
    seg = np.zeros((2, 1, 4, 4, 2), dtype=np.uint8)
    seg[1, 0, 2] = 1
    res = {'torch_loss': torch.tensor([1.5]), 'monitor_values': {'loss': 1.5, 'class_loss': 0.25}, 'seg_preds': seg,
           'boxes': [[{'box_coords': np.array([1, 2, 3, 4, 0, 1]), 'box_label': 1, 'box_type': 'gt'}],
                     [{'box_coords': np.array([5, 6, 9, 9, 1, 2], dtype=np.int32), 'box_score': np.float32(0.75), 'box_type': 'det',
                       'box_pred_class_id': np.int32(1)}]]}
    out = bench.step_outputs(res, net, 3)
    assert sorted(out) == ["detections", "loss", "monitor_class_loss", "monitor_loss", "parameters", "seg_preds"]
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert out["detections"].tolist() == [[1, 5, 6, 9, 9, 1, 2, 1, 0.75]]
    assert out["loss"].tolist() == [1.5] and out["monitor_class_loss"].tolist() == [0.25]
    seg[:] = 7                                                    # the step's host buffer is reused by the next step
    assert out["seg_preds"].shape == (2, 1, 4, 4, 2) and out["seg_preds"].sum() == 8
    flat = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).numpy()
    assert np.array_equal(out["parameters"], flat)
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 10)
    a, b = bench.step_outputs(res, net, 3), bench.step_outputs(res, net, 3)
    assert a["parameters"].shape == (10,) and np.array_equal(a["parameters"], b["parameters"])   # fixed sample
    assert np.all(np.isin(a["parameters"], flat)) and a["seg_preds"].shape == (10,)
    empty = dict(res, boxes=[[], []])
    assert bench.step_outputs(empty, net, 3)["detections"].shape == (0, 9)
