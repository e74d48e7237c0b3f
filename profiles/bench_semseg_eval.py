"""Cost of semantic-segmentation evaluation on the C4 scenes (S3DIS-shaped rooms, 107,750 voxels for seed 0, Res16UNet34C 3 -> 13):

  (a) forward-only scenes/s (the loop of bench.py's c4 workload: forward + argmax)
  (b) forward + SegmentationMeter.update scenes/s, alternated with (a) in the same run
  (c) pcb_seg_eval alone on one scene's logits: CUDA events over many calls, and the split between its kernels (torch.profiler,
      after the timed windows)
  (d) the original project's host path on the same logits: softmax to the host, np.bincount histogram, scikit-learn's
      average_precision_score (the numpy restatement of it when scikit-learn is absent)

    python profiles/bench_semseg_eval.py [--rounds 6 --scenes-per-round 10 --calls 300]

Prints one JSON line, with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

NUM_LABELS, IGNORE = 13, 255


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                                   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def host_path(prob_dev, target):
    """`lib/test.py:119-145` on the host: softmax copied back, fast_hist, average precision per class."""
    prob = prob_dev.cpu().numpy()
    pred = prob.argmax(1)
    k = (target >= 0) & (target < NUM_LABELS)
    np.bincount(NUM_LABELS * target[k] + pred[k], minlength=NUM_LABELS ** 2).reshape(NUM_LABELS, NUM_LABELS)
    try:
        from sklearn.metrics import average_precision_score
        from sklearn.preprocessing import label_binarize
        label = label_binarize(target, classes=list(range(NUM_LABELS)))
        with np.errstate(divide="ignore", invalid="ignore"):
            average_precision_score(label, prob, average=None)
        return "scikit-learn"
    except ImportError:
        from oracle import seg_metrics_cpu
        seg_metrics_cpu.average_precision(prob, target, IGNORE)
        return "numpy restatement (oracle/seg_metrics_cpu.py)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--scenes-per-round", type=int, default=10)
    ap.add_argument("--calls", type=int, default=300)
    ap.add_argument("--host-scenes", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    from pointcontrast_b200 import _lib, me, semseg, synth
    from pointcontrast_b200.config import default_config
    from pointcontrast_b200.model import load_model
    torch.cuda.set_device(0)
    info = card()
    cfg = default_config(["net.normalize_feature=False"])
    torch.manual_seed(0)
    net = load_model("Res16UNet34C")(3, NUM_LABELS, cfg, D=3).cuda().eval()
    scenes = [synth.synth_scene(s) for s in range(3)]
    rng = np.random.default_rng(0)
    targets = []
    for s in scenes:
        t = rng.integers(0, NUM_LABELS, len(s["coords"]))
        t[rng.random(len(t)) < 0.1] = IGNORE
        targets.append(t)
    devb = [(torch.from_numpy(s["feats"]).cuda(), torch.from_numpy(s["coords"]).cuda(), torch.from_numpy(t).cuda())
            for s, t in zip(scenes, targets)]
    meter = semseg.SegmentationMeter(NUM_LABELS, IGNORE)

    def run(n, with_eval):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for i in range(n):
            f, c, t = devb[i % len(devb)]
            with torch.no_grad():
                logits = net(me.SparseTensor(f, coords=c).to("cuda")).F
                if with_eval:
                    meter.update(logits, t)
                else:
                    logits.argmax(1)
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    run(2 * len(devb), False)                                    # warm-up: every scene shape on both paths
    run(2 * len(devb), True)
    ms_a, ms_b = [], []
    for _ in range(args.rounds):
        ms_a.append(run(args.scenes_per_round, False))
        ms_b.append(run(args.scenes_per_round, True))
    n_ab = args.rounds * args.scenes_per_round
    a_sps, b_sps = n_ab * 1e3 / sum(ms_a), n_ab * 1e3 / sum(ms_b)

    # (c) the op alone on scene 0's logits
    f, c, t = devb[0]
    with torch.no_grad():
        logits = net(me.SparseTensor(f, coords=c).to("cuda")).F.contiguous()
    n = logits.shape[0]
    pred = torch.empty(n, dtype=torch.int32, device="cuda")
    hist = torch.zeros(NUM_LABELS, NUM_LABELS, dtype=torch.int64, device="cuda")
    stats = torch.empty(4, dtype=torch.float64, device="cuda")
    apd = torch.empty(NUM_LABELS, dtype=torch.float64, device="cuda")
    ws = torch.empty(int(_lib.lib.pcb_seg_eval_ws_bytes(n, NUM_LABELS)), dtype=torch.uint8, device="cuda")
    st = _lib.stream()

    def op():
        _lib.check(_lib.lib.pcb_seg_eval(logits.data_ptr(), t.data_ptr(), n, NUM_LABELS, IGNORE, pred.data_ptr(), hist.data_ptr(),
                                         stats.data_ptr(), apd.data_ptr(), None, ws.data_ptr(), ws.numel(), st))
    for _ in range(20):
        op()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(args.calls):
        op()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / args.calls
    io_bytes = n * NUM_LABELS * 4 + n * 8

    # kernel split of the op (profiled after the timed windows)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(50):
            op()
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        name = ev.key
        dev_us = getattr(ev, "device_time_total", None)
        if dev_us is None:
            dev_us = getattr(ev, "cuda_time_total", 0)
        if not dev_us:
            continue
        if "seg_rows_kernel" in name:
            part = "row_pass"
        elif "RadixSort" in name or "Onesweep" in name or "radix" in name.lower():
            part = "sort"
        elif "ap_flags" in name or "Scan" in name or "ap_terms" in name or "seg_final" in name:
            part = "ap_pass"
        else:
            part = "other"
        split[part] = split.get(part, 0.0) + dev_us / 50.0
    split = {k: round(v, 2) for k, v in split.items()}

    # (d) the host path on the same logits
    prob = torch.softmax(logits, 1)
    torch.cuda.synchronize()
    host_path(prob, targets[0])                                  # warm-up (imports)
    t0 = time.perf_counter()
    for _ in range(args.host_scenes):
        how = host_path(prob, targets[0])
    host_s = (time.perf_counter() - t0) / args.host_scenes

    print(json.dumps({
        "metric": "semseg_eval", "card": info, "voxels_scene0": n, "classes": NUM_LABELS,
        "forward_only_scenes_per_s": round(a_sps, 2), "forward_plus_meter_scenes_per_s": round(b_sps, 2),
        "ratio_b_over_a": round(b_sps / a_sps, 4), "scenes_each": n_ab, "round_ms_a": [round(x, 2) for x in ms_a],
        "round_ms_b": [round(x, 2) for x in ms_b],
        "seg_eval_us_per_scene": round(us, 2), "seg_eval_calls": args.calls,
        "seg_eval_op_rate_GBps": round(io_bytes / (us * 1e-6) / 1e9, 2),
        "seg_eval_op_rate_note": "logits + target bytes over the op's time: an op rate, not a kernel's share of peak",
        "seg_eval_split_us": split,
        "host_path_s_per_scene": round(host_s, 4), "host_path": how, "host_torch_threads": torch.get_num_threads(),
        "host_cpus": os.cpu_count(),
    }), flush=True)


if __name__ == "__main__":
    main()
