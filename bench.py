#!/usr/bin/env python
"""bench.py -- scene-pairs/sec of the PointContrast hot path (Res16UNet34C + PointInfoNCE, 2.5 cm voxels).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--loss nce|hardest] [--workload c1|c0|c4]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one full training iteration on one batch of synthetic scene pairs per rank: coordinate-manager build for
both views (stacked in one pass by default; PCB_PAIR=0: two forward calls), loss, backward, gradient all-reduce (N > 1,
overlapped with the backward pass), fused SGD step.  Prints ONE JSON line (rank 0).

  value    : pairs/s with the batches already resident in HBM, through the trainer's own loop (`Trainer.iter_losses`, what
             `Trainer.train()` runs: the next batch staged and enqueued while the current one runs, every loss read back), CUDA-event
             timed over all K steps, max over ranks.
  e2e      : the same loop with the batches in pinned HOST memory: host->device copies and the loss read-back inside the timed region.
  roofline : the dominant kernel (conv_tcgen05_split_kernel: sparse-conv forward / data-gradient) -- algorithmic bytes
             (BASELINE.md section 2) of all its launches in one step / their CUDA-event time (events recorded by the library
             around every launch, `pcb_profile_enable`), vs the measured HBM peak.
  cpu_baseline : the oracle (ME-0.4.3-algorithm CPU restatement) timed on this box's host cores: full training steps on
             ONE full-size scene pair of the workload (a quarter of the per-rank batch).

--impl reference times that CPU restatement as the whole measurement (the reference's own arithmetic layer,
MinkowskiEngine 0.4.3, is not in the reference tree and not installable offline -- DESIGN.md): the reference's own
`model/res16unet.py` (when /root/reference or its staged copy oracle/_ref is present) on the oracle operators, the thread
count chosen by a measured sweep; it never loads libpcb200.so.

--workload c4: BASELINE configs[4], S3DIS-shaped full-scene inference (5 cm voxels, eval-mode BatchNorm, 13 classes, forward only,
`downstream/semseg/lib/test.py:95-117`); metric scenes/sec.

--dump-outputs DIR: after the timed steps, what the last of them computed goes to DIR/<name>.npy, so that two builds can be compared
output for output (inputs, weights and sampling draws are seeded: the same arguments give the same inputs).  Training workloads:
loss (float64, the step's loss or (loss, pos, neg)), params and grads (the flat parameters after the step's SGD update and the
step's gradients), bn_running_stats; c4: logits and pred of the last scene.  An array of more than 2^19 rows is a fixed seeded
sample of 2^19 rows in ascending order (`host_rows`).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np   # noqa: E402
import torch         # noqa: E402

METRIC = "scene-pairs/sec Res16UNet34C PointInfoNCE @2.5cm voxel"
METRIC_C4 = "scenes/sec Res16UNet34C S3DIS-shape full-scene inference @5cm voxel"
WORKLOADS = {   # per-rank batch, synthetic scale -> ~voxels/view
    "c1": dict(batch=4, scale=0.9, desc="BASELINE configs[1]: ~40k voxels/view synthetic ScanNet-shape, batch=4 per GPU"),
    "c0": dict(batch=1, scale=0.24, desc="BASELINE configs[0]: ~4k voxels/view, batch=1"),
    "c4": dict(batch=1, scale=2.5, desc="BASELINE configs[4]: S3DIS-shape full scene, 5cm voxels, eval BatchNorm, 13 classes, forward only"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--loss", default="nce", choices=["nce", "hardest"])
    ap.add_argument("--workload", default="c1", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-json", default=None, help="write the per-launch conv profile of one step here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64, a fixed sample of large arrays)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_ROWS = 1 << 19     # rows kept of a larger output: <= 64 MB in all for every workload


def host_rows(x, seed=0):
    """`x` as a host array; with more than DUMP_ROWS rows, a fixed seeded sample of DUMP_ROWS of them in ascending order (the same
    rows for any array of the same length)."""
    if len(x) > DUMP_ROWS:
        idx = np.sort(np.random.default_rng(seed).choice(len(x), DUMP_ROWS, replace=False))
        x = x[torch.from_numpy(idx).to(x.device)]
    return x.detach().cpu().numpy()


def dump_outputs(dirname, arrays):
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(dirname, name + ".npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def static_config(args, world):
    """The part of `config` both arms print identically."""
    wl = WORKLOADS[args.workload]
    return {"workload": wl["desc"], "loss": args.loss if args.workload != "c4" else "none", "pairs_per_gpu": wl["batch"],
            "global_batch": wl["batch"] * world, "parallelism": f"dp{world}"}


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------- clocks sampler
class Clocks:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except Exception:
                continue
            for nm, v in zip(names, f[2:]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores():
    """Host cores this process may really use: affinity mask, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


# ----------------------------------------------------------------------------------------------- CPU oracle leg
def _oracle_model_ctor():
    """Res16UNet34C on the oracle operators: the REFERENCE's own model file when it is present (/root/reference in the build
    container, the staged copy under oracle/_ref on the GPU box) -- nothing of this package's CUDA side is imported then --
    else this package's model file (same graph, checked module by module in tests/test_host.py)."""
    from oracle import me_cpu as OR
    from tests import refload
    if refload.available():
        pkg = refload.load_reference_model_module(OR.install)
        return pkg.load_model("Res16UNet34C"), refload.default_config(), "reference model file (model/res16unet.py, unmodified)"
    from pointcontrast_b200.model import res16unet          # imports the CUDA binding as a side effect
    res16unet.ME = OR
    return res16unet.Res16UNet34C, refload.default_config(), "this package's model file (reference tree absent)"


def cpu_oracle_steps(workload, steps, warmup, loss_kind, sweep=True):
    """ME-0.4.3-algorithm CPU restatement (the oracle), fp32.  Every step is a full training step (2x forward, loss, backward,
    SGD) on ONE full-size scene pair of the workload -- a quarter of a 'c1' per-rank batch, no shrinking, no extrapolation.
    The torch thread count is chosen by timing one step at each of {8, 16, 32, all usable} (more threads are slower on big hosts)."""
    from oracle import loss_cpu, me_cpu as OR
    from pointcontrast_b200 import synth
    ctor, cfg, model_src = _oracle_model_ctor()
    cores = usable_cores()
    scale = WORKLOADS[workload]["scale"]
    batch = synth.collate_pairs([synth.synth_pair(0, scale=scale)])
    n_vox = len(batch["sinput0_C"]) + len(batch["sinput1_C"])
    net = ctor(3, 32, cfg, D=3).train()
    opt = torch.optim.SGD(net.parameters(), lr=0.1, momentum=0.8, weight_decay=1e-4)
    rng = np.random.default_rng(0)

    def one_step():
        t0 = time.perf_counter()
        opt.zero_grad()
        F = [net(OR.SparseTensor(torch.from_numpy(batch[f"sinput{v}_F"]), coords=torch.from_numpy(batch[f"sinput{v}_C"]))).F for v in "01"]
        pairs = batch["correspondences"]
        if loss_kind == "nce":
            nq = len(np.unique(pairs[:, 0]))
            q, k = loss_cpu.select_positives(pairs, rng.random(nq).astype(np.float32), 4096,
                                             rng.choice(nq, 4096, replace=False) if nq > 4096 else None)
            loss = loss_cpu.point_nce_loss(F[0], F[1], q, k, 0.4)
        else:
            sel0 = rng.choice(len(F[0]), min(256, len(F[0])), replace=False)
            sel1 = rng.choice(len(F[1]), min(256, len(F[1])), replace=False)
            ps = rng.choice(len(pairs), 1024, replace=False) if len(pairs) > 1024 else None
            a, b = loss_cpu.hardest_contrastive_loss(F[0], F[1], pairs, sel0, sel1, ps)
            loss = a + b
        loss.backward()
        opt.step()
        return time.perf_counter() - t0

    torch.set_num_threads(min(cores, 16))
    one_step()                                              # thread pools, allocator, kernel maps are NOT cached across steps
    cand = sorted({c for c in (8, 16, 32, cores) if c <= cores}) if sweep else [min(cores, 16)]
    sweep_t = {}
    for c in cand:
        torch.set_num_threads(c)
        sweep_t[c] = one_step()
    best = min(sweep_t, key=sweep_t.get)
    torch.set_num_threads(best)
    times = [one_step() for _ in range(warmup + steps)][warmup:]
    t_s = float(np.mean(times))
    return dict(value=1.0 / t_s, unit="pairs/s", cores=best, kind="port",
                sample=f"{len(times)} full training steps (2x fwd, loss, bwd, SGD), each on ONE full-size synthetic scene pair of the "
                       f"'{workload}' workload ({n_vox} voxels, i.e. 1 of the {WORKLOADS[workload]['batch']} pairs of a per-rank batch); fp32; "
                       f"{model_src}; {best} torch threads (sweep s/step: {({c: round(t, 3) for c, t in sweep_t.items()})}, "
                       f"{cores} usable cores)"), t_s * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = "c1" if args.workload == "c4" else args.workload
    cb, ms = cpu_oracle_steps(wl, args.steps, args.warmup, args.loss)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": static_config(args, int(os.environ.get("WORLD_SIZE", "1"))),
            "details": {"note": "ME-0.4.3-algorithm CPU restatement (oracle); MinkowskiEngine itself is not in the reference tree; "
                                "one step = one full-size scene pair", "libpcb200_loaded": "pointcontrast_b200._lib" in sys.modules},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
def conv_alg_bytes(rec):
    M = sum(rec["plan"].pair_counts())
    return M * (rec["Cin"] + rec["Cout"]) * 4 + M * 8 + rec["K"] * rec["Cin"] * rec["Cout"] * 4, 2 * M * rec["Cin"] * rec["Cout"]


def profiled_step(step_fn, lib):
    """Runs `step_fn` once with the library bracketing every convolution / weight-gradient launch by CUDA events; returns the
    records (description from the host side, elapsed ms from the library), matched by issue order."""
    import ctypes
    from pointcontrast_b200 import me
    me.PROFILE = []
    lib.pcb_profile_enable(1)
    try:
        step_fn()
        torch.cuda.synchronize()
    finally:
        lib.pcb_profile_enable(0)
        prof, me.PROFILE = me.PROFILE, None
    n = 4 * len(prof) + 64
    ms = (ctypes.c_float * n)(); kinds = (ctypes.c_int32 * n)(); cnt = ctypes.c_int(0)
    rc = lib.pcb_profile_read(ms, kinds, n, ctypes.byref(cnt))
    assert rc == 0 and cnt.value <= n
    recs = list(zip(ms[:cnt.value], kinds[:cnt.value]))
    conv = [(t, kd) for t, kd in recs if kd in (0, 1)]
    assert len(conv) == len(prof), f"profile records {len(conv)} != host records {len(prof)}"
    for r, (t, kd) in zip(prof, conv):
        assert (kd == 1) == (r["kind"] == "wgrad"), "profile record order mismatch"
        r["ms"] = float(t)
    names = {2: "BatchNorm forward passes (statistics not fused into a split reduction + normalise/residual/ReLU/planes)",
             3: "BatchNorm backward passes (column sums + finalize + apply)", 4: "PointInfoNCE forward + backward",
             5: "SGD step", 6: "weight re-tiling (one launch)"}
    other = {}
    for t, kd in recs:
        if kd >= 2:
            o = other.setdefault(names.get(kd, str(kd)), {"ms": 0.0, "calls": 0})
            o["ms"] += float(t); o["calls"] += 1
    profiled_step.other = other
    return prof


def run_ours(args):
    import torch.distributed as dist
    from pointcontrast_b200 import _lib, fused, me
    from pointcontrast_b200.config import default_config
    from pointcontrast_b200.data import SyntheticPairLoader
    from pointcontrast_b200.trainer import get_trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = WORKLOADS[args.workload]
    cfg = default_config([f"trainer.batch_size={wl['batch'] * world}", f"misc.num_gpus={world}", "misc.nceT=0.4"])
    loader = SyntheticPairLoader(wl["batch"], scale=wl["scale"], num_batches=2, rank=rank, pin=True)
    torch.manual_seed(0)
    name = "PointNCELossTrainer" if args.loss == "nce" else "HardestContrastiveLossTrainer"
    trainer = get_trainer(name)(cfg, loader)
    host_batches = loader.batches
    keys = ("sinput0_C", "sinput0_F", "sinput1_C", "sinput1_F", "correspondences")
    dev_batches = [{k: (v.to(dev) if k in keys else v) for k, v in b.items()} for b in host_batches]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def gather_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing: one event per step boundary (no host sync inside the timed region)
    # (the nvidia-smi sampler is started BEFORE the warm-up: its start-up -- process spawn, NVML / driver initialisation -- otherwise opens
    #  an idle gap right before the timed region, the SM clocks drop, and the first timed steps take 60-90 ms while they ramp up again)
    clocks = Clocks(local) if rank == 0 else None
    # The timed loop is the trainer's own loop (`Trainer.iter_losses`: batch i+1 staged and enqueued while batch i runs, every loss read
    # back) over DEVICE-resident batches.  Calling `train_step(batch)` back to back instead builds each batch's coordinate manager inline
    # and never reads a loss: at 8 ranks that loop showed 3-4 steps of 45-80 ms among the first ten (all ranks wait in the all-reduce
    # for one late rank), the trainer's loop none in 60 (profiles/r2_results.md, runs 17 / 23).
    import itertools
    it_dev = itertools.cycle(dev_batches)
    for _ in trainer.iter_losses(it_dev, args.warmup):
        pass
    sync_all()
    from pointcontrast_b200.trainer import quiesce_gc
    quiesce_gc()                       # what Trainer.train() does after its first iteration
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record()
    trainer.step_end_events = []                     # the trainer records one CUDA event at the end of every iteration
    for loss in trainer.iter_losses(it_dev, args.steps):
        pass
    ev1.record()
    sync_all()
    step_evs, trainer.step_end_events = [ev0] + trainer.step_end_events, None
    t_wall1 = time.time()
    launches = _lib.launch_count() - l0
    ms_total = gather_max(ev0.elapsed_time(ev1))
    per_step = [a.elapsed_time(b) for a, b in zip(step_evs[:-1], step_evs[1:])]
    host_ms_per_step = (t_wall1 - t_wall0) * 1e3 / args.steps
    clk = clocks.stop(t_wall0, t_wall1) if clocks else None
    pairs_per_step = wl["batch"] * world
    value = pairs_per_step * args.steps / (ms_total / 1e3)
    outputs = None
    if args.dump_outputs and rank == 0:    # the last timed step: its loss(es), the parameters it left, its gradients, BatchNorm statistics
        opt = trainer.optimizer
        outputs = {"loss": np.asarray(loss, dtype=np.float64).reshape(-1), "params": host_rows(opt.flat_param),
                   "grads": host_rows(opt.flat_grad),
                   "bn_running_stats": torch.cat([b.reshape(-1) for b in trainer.model.buffers() if b.dtype.is_floating_point]).cpu().numpy()}

    # ---- end-to-end through the public trainer call, host (pinned) batches
    it = iter(loader)
    for _ in trainer.iter_losses(it, 2):
        pass
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_losses = list(trainer.iter_losses(it, args.steps))       # what Trainer.train() runs between two LR / checkpoint boundaries
    e1.record()
    sync_all()
    assert len(e2e_losses) == args.steps and all(np.isfinite(np.asarray(e2e_losses, dtype=np.float64).ravel()))
    e2e_value = pairs_per_step * args.steps / (gather_max(e0.elapsed_time(e1)) / 1e3)
    h2d = int(np.mean([sum(b[k].numel() * b[k].element_size() for k in keys) for b in host_batches]))

    # ---- per-rank breakdown of one step (N > 1): own compute vs waiting in / for the gradient all-reduce
    ranks = None
    if world > 1:
        staged = trainer.prepare(dev_batches[0])
        torch.cuda.synchronize()
        trainer.timing = {}
        trainer.train_step(staged)
        torch.cuda.synchronize()
        tm = trainer.timing
        mine = torch.tensor([tm["total"][0].elapsed_time(tm["total"][1]),
                             sum(a.elapsed_time(b) for a, b in tm.get("allreduce", [])),
                             tm["tail"][0].elapsed_time(tm["tail"][1]) if "tail" in tm else 0.0,
                             float(sum(len(b[k]) for b in host_batches[:1] for k in ("sinput0_C", "sinput1_C")))], device=dev, dtype=torch.float64)
        trainer.timing = None
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        ranks = {"step_ms": [round(float(a[0]), 2) for a in allr], "allreduce_stream_ms": [round(float(a[1]), 2) for a in allr],
                 "exposed_wait_plus_sgd_ms": [round(float(a[2]), 2) for a in allr], "voxels": [int(a[3]) for a in allr],
                 "note": "allreduce_stream_ms = time the chunked NCCL all-reduces occupy the side stream (includes waiting for the slowest "
                         "rank); exposed_wait_plus_sgd_ms = end of this rank's backward -> end of its SGD kernel"}

    # ---- roofline of the dominant kernel: one instrumented step
    roof = None
    if rank == 0:                      # every rank runs the instrumented step (it contains the all-reduce); rank 0 records
        prof = profiled_step(lambda: trainer.train_step(dev_batches[0]), _lib.lib)
    else:
        trainer.train_step(dev_batches[0])
    sync_all()
    if rank == 0:
        peak, peak_src = peaks()
        agg = {}
        for r in prof:
            b, f = conv_alg_bytes(r)
            key = ("conv_tcgen05_split_kernel" if r["kind"] in ("fwd", "dgrad") else "wgrad_tcgen05_kernel") if r["tc"] \
                else "fp32 SIMT (3-channel stem conv / wgrad)"
            a = agg.setdefault(key, dict(bytes=0, flops=0, ms=0.0, launches=0))
            a["bytes"] += b; a["flops"] += f; a["ms"] += r["ms"]; a["launches"] += 1
            r["bytes"], r["flops"] = b, f
        dom = max(agg, key=lambda k: agg[k]["ms"])
        a = agg[dom]
        traffic, traffic_note = None, "no ncu pass of this schedule committed"
        try:        # dram__bytes_read+write per launch of this kernel, from the committed ncu pass of THIS schedule (profiles/traffic.json)
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            traffic = tj["kernels"][dom]["dram_bytes_per_launch"]
            traffic_note = tj.get("note", "")
        except Exception:
            pass
        conv_ms = sum(v["ms"] for v in agg.values())
        conv_bytes = sum(v["bytes"] for v in agg.values())
        step_ms = ms_total / args.steps
        roof = {"kernel": dom, "bound": "hbm", "achieved": a["bytes"] / (a["ms"] / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": a["bytes"] / (a["ms"] / 1e3) / 1e9 / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "launches_per_step": a["launches"], "avg_launch_ms": a["ms"] / a["launches"],
                "alg_bytes_per_launch": a["bytes"] / a["launches"], "tensor_tflops": a["flops"] / (a["ms"] / 1e3) / 1e12,
                "share_of_step": a["ms"] / step_ms,
                "other": {k: {"ms": v["ms"], "GB/s": v["bytes"] / (v["ms"] / 1e3) / 1e9, "launches": v["launches"]}
                          for k, v in agg.items() if k != dom},
                "non_conv_ms": {k: {"ms": round(v["ms"], 4), "calls": v["calls"]} for k, v in getattr(profiled_step, "other", {}).items()},
                "step_level": {"conv_alg_bytes_per_step": conv_bytes, "all_conv_kernels_ms": conv_ms,
                               "frac_of_peak_over_conv_kernel_time": conv_bytes / (conv_ms / 1e3) / 1e9 / peak,
                               "frac_of_peak_over_whole_step": conv_bytes / (step_ms / 1e3) / 1e9 / peak}}
        if args.profile_json:
            slim = [{k: v for k, v in r.items() if k != "plan"} for r in prof]
            json.dump({"per_launch": slim, "agg": agg, "ms_per_step": step_ms}, open(args.profile_json, "w"), indent=1)

    if rank == 0:
        cb = None
        if not args.no_cpu_baseline and world == 1:
            cb, _ = cpu_oracle_steps(args.workload, 3, 1, args.loss, sweep=False)
        n0 = int(np.mean([len(b["sinput0_C"]) for b in host_batches])); n1 = int(np.mean([len(b["sinput1_C"]) for b in host_batches]))
        line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 (hi+lo split 16-bit operands: 3 tensor-core products per fp32 product; fp16 planes forward, bf16 planes for gradients; fp32 accumulate)", "data": "synthetic",
                "config": static_config(args, world),
                "details": {"voxels_per_view_per_rank": [n0, n1],
                            "schedule": "both views stacked in one pass (per-view BatchNorm statistics)" if fused.PAIR else "two forward calls",
                            "l2": "per-step working set (activations + kernel maps, GBs) far exceeds the 126 MB L2; 2 distinct batches cycled",
                            "final_loss": float(loss[0] if isinstance(loss, tuple) else loss),
                            "per_step_ms": {"median": float(np.median(per_step)), "min": float(np.min(per_step)), "max": float(np.max(per_step)),
                                            "p90": float(np.percentile(per_step, 90))},
                            "per_step_ms_list": [round(t, 2) for t in per_step],
                            "host_ms_per_step": host_ms_per_step, "launches_per_step": launches / args.steps, "ranks": ranks},
                "clocks": clk, "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
                "roofline": roof, "cpu_baseline": cb}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------- configs[4]: S3DIS-shape inference
def run_c4(args):
    """Full-scene eval-mode forward (`downstream/semseg/lib/test.py:95-117`): SparseTensor build + Res16UNet34C(3 -> 13) + argmax."""
    from pointcontrast_b200 import _lib, me, synth
    from pointcontrast_b200.config import default_config
    from pointcontrast_b200.model import load_model
    torch.cuda.set_device(0)
    cfg = default_config(["net.normalize_feature=False"])
    torch.manual_seed(0)
    net = load_model("Res16UNet34C")(3, 13, cfg, D=3).cuda().eval()
    scenes = [synth.synth_scene(s) for s in range(3)]
    devb = [(torch.from_numpy(s["feats"]).cuda(), torch.from_numpy(s["coords"]).cuda()) for s in scenes]
    host = [(torch.from_numpy(s["feats"]).pin_memory(), torch.from_numpy(s["coords"]).pin_memory()) for s in scenes]

    last = {}

    def run(batches, n, to_host):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for i in range(n):
            f, c = batches[i % len(batches)]
            with torch.no_grad():
                logits = net(me.SparseTensor(f, coords=c).to("cuda")).F
                pred = logits.argmax(1)
            if to_host:
                pred = pred.cpu()
        e1.record(); torch.cuda.synchronize()
        last.update(logits=logits, pred=pred)
        return e0.elapsed_time(e1) / n
    if args.warmup:
        run(devb, args.warmup, False)
    clocks = Clocks(0)
    t0 = time.time(); l0 = _lib.launch_count()
    ms = run(devb, args.steps, False)
    launches = _lib.launch_count() - l0
    t1 = time.time()
    clk = clocks.stop(t0, t1)
    if args.dump_outputs:                  # the last timed scene: per-voxel class scores and the predicted class
        dump_outputs(args.dump_outputs, {"logits": host_rows(last["logits"]), "pred": host_rows(last["pred"])})
    ms_e2e = run(host, args.steps, True)
    nvox = sum(len(s["coords"]) for s in scenes) / len(scenes)
    h2d = int(np.mean([f.numel() * 4 + c.numel() * 4 for f, c in host]))
    print(json.dumps({"metric": METRIC_C4, "value": 1e3 / ms, "unit": "scenes/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "f32 (hi+lo split 16-bit operands: 3 tensor-core products per fp32 product; fp16 planes forward, bf16 planes for gradients; fp32 accumulate)", "data": "synthetic",
                      "config": static_config(args, 1), "details": {"voxels_per_scene": nvox, "voxels_per_s": nvox * 1e3 / ms},
                      "clocks": clk, "gpu_launches": int(launches),
                      "e2e": {"value": 1e3 / ms_e2e, "unit": "scenes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(nvox * 8)}}), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "c4":
        run_c4(a)
    else:
        run_ours(a)
