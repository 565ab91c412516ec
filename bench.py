#!/usr/bin/env python
"""bench.py — BASELINE metric: 3D patches/sec (128^3) of the Retina U-Net train step (lidc_exp config, synthetic 1-channel patches,
batch 2 per GPU), on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--patch 128 128 128] [--batch 2] [--dump-outputs DIR]

A step = train_forward (H2D of the batch, FPN + heads on the tcgen05/SIMT conv kernels, on-device anchor matching, losses, batched NMS,
results D2H) + backward + (N > 1: one NCCL all-reduce of the flat fp32 gradient buffer) + Adam.
Prints ONE JSON line (rank 0).  `value` = device-timed throughput with the batch already resident in HBM; `e2e` = same metric through
the public API with host (pinned) buffers, H2D/D2H inside the timed region.  `--impl reference` times the CPU port of the same step
(oracle/cpu_step.py) on the host cores — see DESIGN.md for why it is a port and not the reference install.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "patches_per_sec_128cubed_retina_unet_train_step"


def conv_flops_per_step(net, cf, batch_size):
    """algorithmic conv FLOPs of one train step (fprop + dgrad + wgrad = 3 x forward; SURVEY.md §8d) from a meta-shape walk"""
    import torch
    from medicaldetectiontoolkit_b200.conv import Conv3d
    total = [0]

    def hook(m, inp, out):
        k = m.kernel_size
        total[0] += 2 * out.numel() * m.in_channels * k[0] * k[1] * k[2]
    hooks = [m.register_forward_hook(hook) for m in net.modules() if isinstance(m, Conv3d)]
    return hooks, total


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons with nvidia-smi while the timed region runs (B200_PROFILING.md clocks line)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.samples = []
        self.reasons = set()
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    """CPU arm: the port of the step on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import cpu_step
    from medicaldetectiontoolkit_b200.configs import make_cf, synthetic_batch
    cores = cpu_step.calibrate_threads(os.cpu_count() or 1)
    torch.set_num_threads(cores)
    patch = tuple(args.patch)
    cf = make_cf('retina_unet', 3, patch)
    # same config as the GPU arm: batch, warm-up and timed step count exactly as requested (a CPU step of 2 x 128^3 patches takes ~14 s)
    b = args.batch
    batch = synthetic_batch(cf, b, seed=0)
    warm = args.warmup
    times, used = cpu_step.time_cpu_steps(cf, batch, steps=args.steps, warmup=warm, threads=cores)
    ms = 1e3 * sum(times) / len(times)
    val = b / (ms / 1e3)
    sample = "%d full train step(s) of %d patch(es) %s (forward+detections+matching+losses+backward+Adam), fp32, torch CPU" % (len(times), b, "x".join(map(str, patch)))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "patches/s", "n_gpus": args.gpus, "steps": len(times),
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "configs[1]: lidc_exp 3D Retina U-Net, synthetic 1-ch %s patches, batch %d per GPU" % ("x".join(map(str, patch)), args.batch),
                       "global_batch": b, "parallelism": "host cores (%d threads)" % used, "optimizer": "Adam lr 1e-4",
                       "sample": "each step = one full train step of %d patch(es) on the CPU" % b},
            "cpu_baseline": {"value": val, "unit": "patches/s", "cores": used, "host_cpus": os.cpu_count(), "cpu_model": cpu_model(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": val, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def load_traffic(shape):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture of THIS round (profiles/r02_traffic.json, written from
    `ncu --set full`: dram__bytes_read.sum + dram__bytes_write.sum), or None when there is no capture for this shape"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        for e in t.get("entries", []):
            if tuple(e["input_shape"]) == tuple(shape):
                return e
    except Exception:
        pass
    return None


def make_roofline(step_flops, conv_ms, n_conv_calls, ms_step, dom, peak_tf, peaks_measured, slowest=None, traffic=None):
    """roofline object of the JSON line.  Top level = the dominant kernel launch (the heaviest forward conv: flops of that launch / its
    CUDA-event duration measured live in a separate instrumented pass, DRAM traffic from its committed ncu capture); `slowest_launch` = the conv
    call with the longest average duration (a fused backward: dy split + dgrad + wgrad); `all_conv_launches` = the same ratio over every
    conv call of the step.  dom / slowest = (flops, ms, tag, calls_per_step) or None; pure function (tests/test_bench_cpu.py)."""
    if not conv_ms:
        return None
    src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks_measured else "fallback 1.4 PF sustained (of fallback)"
    ach = step_flops / (conv_ms / 1e3) / 1e12
    agg = {"kernel": "conv3d fprop+dgrad+wgrad (all layers, %d launches/step)" % round(n_conv_calls), "achieved": ach, "unit": "TFLOP/s",
           "frac": ach / peak_tf, "algorithmic_flops_per_step": step_flops, "conv_ms_per_step": conv_ms, "conv_share_of_step": conv_ms / ms_step}

    def describe(tag):
        names = ("fprop", "dgrad", "wgrad", "fused backward (dy split + dgrad + wgrad)")
        return "%s %d->%d k%s on %s" % (names[tag[0]], tag[1][1], tag[2][0], "x".join(map(str, tag[2][2:])), "x".join(map(str, tag[1])))
    if dom is None:
        roof = {"bound": "tensor", "kernel": agg["kernel"], "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": None}
    else:
        fl, ms_k, tag, _ = dom
        roof = {"bound": "tensor", "kernel": "conv " + describe(tag) + " (kernel + its weight pack launch; operand planes come from the producer's epilogue)",
                "achieved": fl / ms_k / 1e9, "peak": peak_tf, "unit": "TFLOP/s", "frac": fl / ms_k / 1e9 / peak_tf,
                "traffic": traffic["dram_bytes"] if traffic else None,
                "traffic_source": traffic["source"] if traffic else None,
                "algorithmic_flops": fl, "ms": ms_k,
                "note": "fp32-faithful split-bf16 arithmetic issues 3 bf16 MMAs per algorithmic MAC: at most 1/3 of the bf16 peak by construction"}
    if slowest is not None:
        fl, ms_k, tag, n = slowest
        roof["slowest_launch"] = {"kernel": "conv " + describe(tag), "ms": ms_k, "algorithmic_flops": fl, "achieved": fl / ms_k / 1e9, "unit": "TFLOP/s",
                                  "frac": fl / ms_k / 1e9 / peak_tf, "calls_per_step": n}
    roof["peak_source"] = src
    roof["all_conv_launches"] = agg
    return roof


DUMP_MAX_ELEMS = 1 << 22    # per array (16 MB in float32): segmentation + parameters + the small arrays stay under 64 MB in all


def step_outputs(res, net, dim):
    """What a caller of one train step receives, as float32 / float64 numpy arrays: the loss, the monitor values, the detections (rows
    [batch index, 2 * dim box coordinates, class id, score]), the segmentation and the parameters after the optimizer step (flattened in
    net.parameters() order).  An array of more than DUMP_MAX_ELEMS values is replaced by a fixed, seeded sample of its flattened values.
    Copies everything: train_forward's host buffers are reused by the next step."""
    import numpy as np
    import torch
    out = {"loss": np.array([float(res['torch_loss'])], dtype=np.float64)}
    for k, v in res['monitor_values'].items():
        out["monitor_" + k] = np.array([float(v)], dtype=np.float64)
    dets = [[b] + [float(c) for c in bx['box_coords']] + [float(bx['box_pred_class_id']), float(bx['box_score'])]
            for b, boxes in enumerate(res['boxes']) for bx in boxes if bx['box_type'] == 'det']
    out["detections"] = np.array(dets, dtype=np.float64).reshape(len(dets), 2 * dim + 3)
    out["seg_preds"] = np.asarray(res['seg_preds'], dtype=np.float32).copy()
    out["parameters"] = torch.cat([p.detach().reshape(-1).float() for p in net.parameters()]).cpu().numpy()
    for k, a in out.items():
        if a.size > DUMP_MAX_ELEMS:
            ix = np.sort(np.random.RandomState(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            out[k] = a.reshape(-1)[ix]
    return out


def capture_logits_graph(net, batch, lib, eager_logits, reducer):
    """torch.cuda.make_graphed_callables over net._forward_logits (backbone + heads): one graph for the forward, one for the backward.  Returns
    {"enabled", "kernels_per_step", ...}; on success net._forward_logits is the graphed callable."""
    import torch
    info = {"enabled": False, "kernels_per_step": 0}

    class _Logits(torch.nn.Module):
        def __init__(self, n):
            super().__init__()
            self.n = n

        def forward(self, img):
            return eager_logits(img)

    try:
        img = batch['data'].float()
        warm = 2
        c0 = lib.mdt_launch_count()
        graphed = torch.cuda.make_graphed_callables(_Logits(net), (img,), num_warmup_iters=warm, allow_unused_input=True)
        torch.cuda.synchronize()
        info["kernels_per_step"] = int((lib.mdt_launch_count() - c0) // (warm + 1))   # warm-up iterations + the captured one, forward + backward each

        def probe(fn):
            reducer.zero_grad()
            outs = fn(img)
            loss = sum((o.float() ** 2).mean() for o in outs if o is not None)
            loss.backward()
            return [o.detach().clone() for o in outs if o is not None], reducer.flat.clone()

        outs_e, grads_e = probe(eager_logits)
        outs_g, grads_g = probe(graphed)
        same = all(torch.equal(a, b) for a, b in zip(outs_e, outs_g))
        gerr = float((grads_e - grads_g).abs().max() / grads_e.abs().max().clamp_min(1e-30))
        reducer.zero_grad()
        info["forward_bit_identical"] = bool(same)
        info["grad_rel_err"] = gerr
        if same and gerr < 1e-6:
            net._forward_logits = lambda x, _g=graphed: _g(x)   # a plain function: assigning the module itself would register it as a child of net
            info["enabled"] = True
        else:
            info["note"] = "graphed results differ from eager: running eagerly"
            info["kernels_per_step"] = 0
    except Exception as ex:   # capture is an optimisation only
        info["note"] = "capture failed: " + repr(ex)[:200]
        info["kernels_per_step"] = 0
        try:
            torch.cuda.synchronize()
        except Exception:
            pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--patch", type=int, nargs=3, default=[128, 128, 128])
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--precision", type=int, default=0, help="0 = fp32-faithful conv (default, parity mode); 1 = single-pass bf16")
    ap.add_argument("--algo", type=int, default=0, help="0 auto, 1 force SIMT conv, 2 force tcgen05 conv")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graphs", action="store_true",
                    help="capture backbone + heads (forward and backward) in CUDA graphs; measured SLOWER than eager launches on this step "
                         "(53.9 vs 51.8 ms: the conv part is not launch-bound, the replay adds node-to-node latency), hence opt-in")
    ap.add_argument("--model", default="retina_unet", choices=["retina_unet", "mrcnn"],
                    help="retina_unet = BASELINE configs[1] (the metric's config); mrcnn = configs[2]: 3D Mask R-CNN, 512 proposals, RoIAlign 7x7x3")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (bench.step_outputs) to DIR/<name>.npy; the inputs "
                         "are seeded, so two builds can be compared output for output.  Inside the tree, bench_outputs/ is ignored by git")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from medicaldetectiontoolkit_b200 import _lib as L
    from medicaldetectiontoolkit_b200 import conv as C
    from medicaldetectiontoolkit_b200 import mrcnn, retina_unet
    from medicaldetectiontoolkit_b200.configs import make_cf, synthetic_batch
    from medicaldetectiontoolkit_b200.parallel import FlatGradAllReduce

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl ours) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version / debug lines must not mix with the one JSON line on stdout
        dist.init_process_group("nccl", device_id=dev)
    lib = L.load()
    C.DEFAULT_PRECISION = args.precision
    C.DEFAULT_ALGO = args.algo

    patch = tuple(args.patch)
    cf = make_cf(args.model, 3, patch, batch_size=args.batch)
    is_mrcnn = args.model == 'mrcnn'
    if is_mrcnn:   # BASELINE configs[2]: 512 proposals per element, one second-stage chunk
        cf.post_nms_rois_training = cf.post_nms_rois_inference = 512
        cf.roi_chunk_size = 1024
    torch.manual_seed(0)          # identical replicas on every rank
    np.random.seed(1000 + rank)   # disjoint data streams / sub-sampling streams
    net = (mrcnn if is_mrcnn else retina_unet).net(cf, None).to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=cf.learning_rate[0], weight_decay=cf.weight_decay, fused=True)
    reducer = FlatGradAllReduce(net, world)

    host_batches = [synthetic_batch(cf, args.batch, seed=100 * rank + i, with_masks=is_mrcnn) for i in range(2)]
    for hb in host_batches:  # pinned host staging, as a loader would provide
        hb['data'] = torch.from_numpy(hb['data']).pin_memory()
        hb['seg'] = torch.from_numpy(hb['seg']).pin_memory()
    dev_batches = []
    for hb in host_batches:
        db = dict(hb)
        db['data'] = hb['data'].to(dev)
        db['seg'] = hb['seg'].to(dev)
        dev_batches.append(db)

    hooks, flop_counter = conv_flops_per_step(net, cf, args.batch)

    def step(batch):
        res = net.train_forward(batch, monitor_anchors=False)
        reducer.zero_grad()
        res['torch_loss'].backward()
        reducer.all_reduce()
        opt.step()
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(batches, n):
        """(ms for n steps, the last step's result)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n - 1):
            step(batches[i % len(batches)])
        res = step(batches[(n - 1) % len(batches)])
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, res

    for i in range(max(args.warmup, 1)):
        step(dev_batches[i % 2])
    fwd_flops = flop_counter[0] / max(args.warmup, 1)
    for h in hooks:
        h.remove()

    # --- optional CUDA graphs for the static part of the step: backbone + heads, forward and backward (~900 kernel nodes).  Matching, losses,
    # NMS, Adam and the all-reduce stay eager.  Falls back to eager execution if capture fails or the graphed results differ from the eager ones.
    graph = {"enabled": False, "kernels_per_step": 0}
    eager_logits = getattr(net, "_forward_logits", None)
    if args.graphs and not is_mrcnn and eager_logits is not None:
        graph = capture_logits_graph(net, dev_batches[0], lib, eager_logits, reducer)
        if world > 1:   # all ranks must take the same path (the step's collective count does not depend on it, but keep the replicas identical)
            flag = torch.tensor([1.0 if graph["enabled"] else 0.0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() < 1.0 and graph["enabled"]:
                net._forward_logits = eager_logits
                graph = {"enabled": False, "kernels_per_step": 0, "note": "another rank fell back"}

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # --- kernel-resident throughput (inputs already in HBM), uninstrumented
    launches0 = lib.mdt_launch_count()
    torch.cuda.profiler.start()     # no-op unless run under `ncu --profile-from-start off`: the launch list then covers exactly the timed steps
    ms_dev, last = timed(dev_batches, args.steps)
    torch.cuda.profiler.stop()
    dumped = step_outputs(last, net, cf.dim) if args.dump_outputs and rank == 0 else None
    del last
    launches = lib.mdt_launch_count() - launches0 + graph["kernels_per_step"] * args.steps   # eager launches + kernel nodes replayed from the graphs
    # --- separate instrumented pass: every conv call bracketed by CUDA events on the launching stream (roofline object only)
    conv_ms = None
    if rank == 0:
        n_inst = min(args.steps, 4)
        graphed_logits = getattr(net, "_forward_logits", None)
        if graph["enabled"]:
            net._forward_logits = eager_logits        # events cannot be recorded from inside a replayed graph: the instrumented pass runs eagerly
        C.EVENT_LOG = []
        for i in range(n_inst):
            step(dev_batches[i % 2])
        torch.cuda.synchronize()
        log, C.EVENT_LOG = C.EVENT_LOG, None
        if graph["enabled"]:
            net._forward_logits = graphed_logits
        conv_ms = sum(a.elapsed_time(b) for a, b, _ in log) / n_inst
        n_conv_calls = len(log) / n_inst
        per_tag = {}
        for a, b, tag in log:
            if tag is not None:
                per_tag.setdefault(tag, []).append(a.elapsed_time(b))
        dom = slowest = None
        for tag, ts in per_tag.items():
            ps, xs, ws, st, which = tag
            fl = 2.0 * xs[0] * (xs[2] // st[0]) * (xs[3] // st[1]) * (xs[4] // st[2]) * ws[0] * ws[1] * ws[2] * ws[3] * ws[4] * (2.0 if ps == 3 else 1.0)
            ent = (fl, sum(ts) / len(ts), tag, len(ts) / n_inst)
            if ps == 0 and (dom is None or fl > dom[0]):      # the single heaviest forward launch (P0_conv2 36->36 k3 at full resolution for cfg2)
                dom = ent
            if slowest is None or ent[1] > slowest[1]:
                slowest = ent
    elif world > 1:
        for i in range(min(args.steps, 4)):                   # keep the ranks in step (the all-reduce is collective)
            step(dev_batches[i % 2])
    # --- end to end through the public API with host buffers
    ms_e2e, _ = timed(host_batches, args.steps)
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join(timeout=3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    n_patches = args.batch * world * args.steps
    value = n_patches / (ms_dev / 1e3)
    e2e = n_patches / (ms_e2e / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    step_flops = 3.0 * fwd_flops
    traffic = load_traffic(dom[2][1]) if (conv_ms and dom) else None
    roof = make_roofline(step_flops, conv_ms, n_conv_calls if conv_ms else 0, ms_dev / args.steps, dom if conv_ms else None, peak_tf, bool(peaks),
                         slowest if conv_ms else None, traffic)
    h2d = sum(int(hb['data'].numel() * hb['data'].element_size() + hb['seg'].numel() * hb['seg'].element_size()) for hb in host_batches[:1])
    if is_mrcnn:
        h2d = int(host_batches[0]['data'].numel() * 4 + sum(int(np.asarray(m).size) for m in host_batches[0]['roi_masks']))   # image + GT masks (uint8)
    d2h = int(args.batch * np.prod(patch)) + 60 * 9 * 4 + 5 * 4  # seg_preds uint8 + detections + loss scalars
    if is_mrcnn:
        d2h = 60 * 9 * 4 + 6 * 4 + args.batch * 512 * 7 * 4       # detections + loss scalars + proposals for the monitoring boxes
    workload = ("configs[1]: lidc_exp 3D Retina U-Net, synthetic 1-ch %s patches, batch %d per GPU" if not is_mrcnn else
                "configs[2]: lidc_exp 3D Mask R-CNN (mrcnn.py), %s patches, 512 proposals, RoIAlign 7x7x3, batch %d per GPU") % ("x".join(map(str, patch)), args.batch)
    line = {"metric": METRIC if not is_mrcnn else "patches_per_sec_128cubed_mask_rcnn_train_step", "value": value, "unit": "patches/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (conv: split-bf16 x3 on tcgen05, fp32 accumulate)" if args.precision == 0 else "bf16",
            "data": "synthetic",
            "config": {"workload": workload,
                       "global_batch": args.batch * world, "parallelism": "dp%d" % world, "optimizer": "Adam lr 1e-4",
                       "l2": "no flush needed: per-step activation working set (>5 GB) far exceeds the 126 MB L2",
                       "conv_precision": args.precision, "conv_algo": args.algo},
            "e2e": {"value": e2e, "unit": "patches/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "cuda_graph": graph, "clocks": sampler.summary(), "roofline": roof}
    if world == 1 and not args.no_cpu_baseline and not is_mrcnn:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import cpu_step
        cores = cpu_step.calibrate_threads(os.cpu_count() or 1)
        cb = synthetic_batch(cf, args.batch, seed=0)
        times, used = cpu_step.time_cpu_steps(cf, cb, steps=1, warmup=0, threads=cores)
        line["cpu_baseline"] = {"value": args.batch / times[0], "unit": "patches/s", "cores": used, "host_cpus": os.cpu_count(), "cpu_model": cpu_model(),
                                "kind": "port",
                                "sample": "1 full train step of %d patches %s on the host cores (oracle/cpu_step.py: torch CPU fp32 convs, numpy fp64 matching, C NMS)" % (args.batch, "x".join(map(str, patch)))}
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), a)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
