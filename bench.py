#!/usr/bin/env python
"""Benchmark of the B200 OCT metric suite on the BASELINE.json configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--config cfg4|cfg1|cfg2|cfg3|cfg5] [--items M] [--noise f] [--uniform-random] [--dump-outputs DIR]

Default = cfg4 AS STATED in BASELINE.json: the full metric suite (fused label pass + contour metrics + float64
epilogue) over 100,000 synthetic 496x512 8-class B-scans, sharded over the N ranks (ceil(100000 / N) per GPU:
total work fixed => "scaling": "strong"; --items M fixes the per-GPU batch instead => "weak").  One process per GPU
(torchrun for N > 1), no data-path collective, ONE small NCCL all-reduce of the dataset totals per step, inside
the timed region.  A "step" is one pass of the suite over this rank's batch with the inputs resident in HBM; steps
are enqueued asynchronously and timed with CUDA events, max over ranks.  "e2e" is the same suite through the
host-array API (pinned host buffers, H2D inside the timed region, metrics read back).  Rank 0 prints ONE JSON line.

--config cfg1 / cfg2 / cfg3 / cfg5: the other BASELINE configurations (single volumes; their committed lines live
under profiles/).  cfg5 shards its 2 K (class, direction) distance transforms over the ranks.

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float64): the per-item
metrics (``item_*``; a fixed, seeded sample of DUMP_ITEMS items of larger batches, ``item_index`` names them) and the
dataset totals (``dataset_*``); cfg5: the per-class surface integers and metrics.  The inputs depend only on the
arguments, so two builds of the project can be compared output for output.  With N > 1, rank 0 writes its own shard.

--impl reference times the reference's own CPU path on the box's host cores: the UNMODIFIED Metrics/*.py modules
(baseline/_ref/Metrics, importable for 4 of the 5 modules) called the only way the reference can be called -- per
class, per function -- with the contour functions on the restated find_contours (scikit-image is not installable
here); all host cores, bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark leaves the tree as it found it (it may be read-only)

CFG4_ITEMS = 100_000
DUMP_ITEMS = 8192                     # per-item rows written by --dump-outputs
CONFIGS = {
    # name: H, W, K, items of the configuration as BASELINE.json states it, generator, what a step computes
    "cfg1": dict(H=496, W=768, K=8, items=61, gen="layered", noise=0.01, seed=1001, contours=False,
                 workload="cfg1: confusion matrix + Dice/IoU/... per class, synthetic Duke-DME-sized volume (61x496x768, 8 classes)"),
    "cfg2": dict(H=496, W=1024, K=10, items=49, gen="layered", noise=0.0, seed=2002, contours=False,
                 workload="cfg2: layer boundary pixel error + thickness biomarkers, synthetic HC-MS-shaped volume (49x496x1024, 9 boundaries)"),
    "cfg3": dict(H=512, W=512, K=4, items=128, gen="lesions", noise=0.0, seed=3003, contours=True,
                 workload="cfg3: contour metrics (Hausdorff, HD95, ASSD) + counts, synthetic RETOUCH-style fluid lesion masks (128x512x512)"),
    "cfg4": dict(H=496, W=512, K=8, items=CFG4_ITEMS, gen="layered", noise=0.0, seed=4004, contours=True,
                 workload="cfg4: full metric suite, 100k synthetic layered 496x512 B-scans, 8 classes"),
    "cfg5": dict(H=1024, W=1024, K=11, items=1, gen="volume", D=128, seed=5005, contours=True,
                 workload="cfg5: 3-D surface-distance metrics, synthetic OCT volume 1024x1024x128, 11 classes (22 exact EDT units)"),
}
KERNEL_NOTES = {
    # bound + the counter that shows it (ncu summaries under profiles/)
    "label_pass_fast": ("hbm", "dram read = algorithmic bytes (ratio 1.01); issue-active 70.5 %, 109 k warp-instructions per B-scan: in-order issue at 4 warps/scheduler, 128 registers (r2)"),
    "label_pass_generic": ("latency", "thread-per-column run-length scan (any shape, small batches of K > 8); 1.46 TB/s at scale (r2), latency-bound on one volume"),
    "layered_distance_kernel_rows": ("issue", "PASS 1's code for a lightly noisy stream: sides of rejected maps are re-centred rows from the pixel verification, measured table x table like certified ones"),
    "walk_report_kernel": ("latency", "one thread: contours walked / contours -> a host-mapped word that picks the next call's step order (noisy streams only)"),
    "seed_feedback_kernel": ("latency", "one CTA: maps the certificate rejected / maps seen -> a host-mapped word that picks the next call's seed source"),
    "label_pass_wide": ("latency", "warp per 128-column strip, run queues drained in lockstep (K <= 16, W % 4 == 0): 2.6 TB/s at 2048 x 496x1024 K=10; issue-active 39 %, 10-14 warps per SM by shared memory (r2)"),
    "first_pos_fix_kernel": ("hbm", "rescans only the maps the layering certificate rejected (nothing on clean data): 3.9 TB/s of those maps"),
    "layered_distance_kernel": ("issue", "boundary-row verification + shared-memory column tables + fused distances; issue-active 75 %, DRAM 2 % of peak: 16.4 k warp-instructions per (B-scan, class) pair (r2)"),
    "layered_distance_kernel_pass2": ("issue", "pairs handed on (noisy predictions): tables x short vertex lists, wide counting; barrier-bound; returns at once on clean data"),
    "trace_layered_kernel": ("latency", "verification against label pixels with re-centred rows, only for contours the boundary-row check rejects; returns at once on clean layered data"),
    "trace_kernel": ("latency", "serial walk, first-touch label loads; only what is not a height function"),
    "distance_column_kernel": ("issue", "vertex-list search, only long x long lists (lesions); DRAM 6.5 % of peak, issue-active 68 % (r1_v10)"),
    "distance_select_kernel": ("latency", "only units the counters cannot hold"),
    "derive_kernel": ("hbm", "streams the integer outputs once"),
    "totals_kernel": ("latency", "one CTA per output element"),
    "near_surface_kernel": ("hbm", "surface bits: 16 voxels per thread, five label lines (L2 reuse between neighbouring lines)"),
    "near_pass1_kernel": ("issue", "distance to the nearest surface bit within +-10 from three 16-bit words (BREV / FFS)"),
    "near_pass2_kernel": ("issue", "windowed min-plus along D1, VIADDMNMX.U16x2: 672 per thread for 64 voxels"),
    "near_pass3_kernel": ("latency", "windowed min-plus along D0 at the query-surface voxels only (tiles without a query bit are skipped)"),
    "edt3_pass1_vec_kernel": ("latency", "general (Meijster) path: only units with a distance >= 11 voxels; returns at once otherwise"),
    "edt3_pass2_kernel": ("latency", "general path, see above"),
    "edt3_pass3_kernel": ("latency", "general path, see above"),
}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured copy bandwidth (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_traffic():
    """DRAM bytes per unit of work of the dominant kernel from the committed ncu --set full capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler:
    """SM clock and throttle reasons sampled WHILE the timed region runs.

    In-process NVML (nvidia_ml_py) from a thread, one cheap query every 20 ms: an `nvidia-smi -lms` child
    process holds the driver for milliseconds per query and was measured to stretch a 17 ms step to 18-27 ms.
    Falls back to that child process only if NVML cannot be imported."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.rows, self.proc, self.index, self.thread, self.stop_flag = [], None, index, None, False
        self.max_mhz, self.source = None, None

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def start(self):
        if os.environ.get("OCTM_BENCH_NOCLOCKS") == "1":      # diagnosis only: is the sampler disturbing the run?
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = [getattr(pynvml, n, 0) for n in ("nvmlClocksEventReasonHwSlowdown", "nvmlClocksEventReasonHwThermalSlowdown",
                                                    "nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksEventReasonSwPowerCap")]
            if not all(bits):
                bits = [0x8, 0x40, 0x20, 0x4]            # NVML ABI values of the four reasons above

            def loop():
                while not self.stop_flag:
                    try:
                        mhz = int(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        try:
                            r = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                        except Exception:
                            r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                        self.rows.append((time.perf_counter(), mhz, [bool(r & b) for b in bits]))
                    except Exception:
                        pass
                    time.sleep(0.02)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.source = "nvml"
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            self.source = "nvidia-smi"
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            if c and c[0].isdigit():
                if len(c) > 1 and c[1].isdigit():
                    self.max_mhz = max(self.max_mhz or 0, int(c[1]))
                self.rows.append((time.perf_counter(), int(c[0]), [len(c) > 2 + i and c[2 + i] == "Active" for i in range(4)]))

    def stop(self, t0=None, t1=None):
        """Summary of the samples taken inside [t0, t1] (perf_counter; all samples if none fall inside).
        Sampling starts BEFORE the warm-up so that its own initialisation is not in the timed region."""
        if self.thread is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        time.sleep(0.05)
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for r in self.rows if t0 is None or t0 <= r[0] <= t1 + 0.05] or list(self.rows)
        sm = sorted(r[1] for r in rows)
        reasons = [n for i, n in enumerate(self.NAMES) if any(r[2][i] for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm), "source": self.source}


# ------------------------------------------------------------------------------------ synthetic inputs
def host_pair(cfg, n, seed):
    """numpy (y_true, y_pred) [n, H, W] of a 2-D configuration (seeded)."""
    from retinal_oct_image_segmentation_via_deep_learning_b200 import synth
    if cfg["gen"] == "lesions":
        return synth.lesion_pair(n, cfg["H"], cfg["W"], cfg["K"], seed=seed, single_blob_interior=False)
    return synth.layered_pair(n, cfg["H"], cfg["W"], cfg["K"], seed=seed, noise=cfg.get("noise", 0.0))


# ------------------------------------------------------------------------------------ CPU arm
_REF = None


def _ref_functions():
    """The unmodified reference modules (baseline/_ref/Metrics, installed by __graft_entry__.build()) + restated contours,
    or None -> the oracle port."""
    global _REF
    if _REF is None:
        from oracle import ref_loader
        _REF = ref_loader.load() or False
    return _REF or None


def _cpu_one(job):
    """One unit of CPU work of a configuration, timed (runs in a worker process)."""
    name, seed = job
    cfg = CONFIGS[name]
    from oracle import labelmap_oracle as lo
    if name == "cfg5":
        from oracle import surface3d_oracle as so
        from retinal_oct_image_segmentation_via_deep_learning_b200 import synth
        vt, vp = synth.layered_volume_pair(128, 128, 32, 3, seed=seed)       # bounded sub-volume, one class per job
        t0 = time.perf_counter()
        so.class_metrics(vt, vp, 1)
        return time.perf_counter() - t0
    yt, yp = host_pair(cfg, 1, seed)
    f = _ref_functions()
    t0 = time.perf_counter()
    lo.score_bscan(yt[0], yp[0], cfg["K"], contours=cfg["contours"], functions=f)
    return time.perf_counter() - t0


def cpu_baseline(name, n_units, cores):
    """(units/s over `cores` worker processes, mean seconds per unit per core)."""
    import multiprocessing as mp
    jobs = [(name, 5000 + i) for i in range(n_units)]
    t0 = time.perf_counter()
    if cores == 1:
        per = [_cpu_one(j) for j in jobs]
    else:
        with mp.get_context("fork").Pool(cores) as pool:
            per = pool.map(_cpu_one, jobs)
    wall = time.perf_counter() - t0
    return n_units / wall, sum(per) / len(per)


def _cpu_kind():
    f = _ref_functions()
    return ("reference+restated-contours" if f is not None else "port"), (f.root if f is not None else "oracle/metrics_oracle.py")


def _cpu_unit_scale(name):
    """cfg5's CPU unit is one class of a 128x128x32 sub-volume: scale to full volumes (22 units of 1024x1024x128)."""
    if name != "cfg5":
        return 1.0
    cfg = CONFIGS[name]
    return (128 * 128 * 32) / (cfg["H"] * cfg["W"] * cfg["D"]) / cfg["K"]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.config
    cfg = CONFIGS[name]
    cores = os.cpu_count() or 1
    n_units = max(cores, 1)                      # one unit per core per step (~1-2 s of CPU work each)
    for _ in range(min(args.warmup, 1)):
        cpu_baseline(name, n_units, cores)
    t0 = time.perf_counter()
    rates = [cpu_baseline(name, n_units, cores)[0] for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    scale = _cpu_unit_scale(name)
    value = n_units * args.steps / wall * scale
    kind, root = _cpu_kind()
    unit = "volumes/s" if name == "cfg5" else "B-scans/s"
    sample = (f"{n_units} units per step (one per core), {args.steps} steps; unit = "
              + ("one class of a 128x128x32 sub-volume through scipy's exact EDT, scaled by voxels x classes to full volumes"
                 if name == "cfg5" else "one B-scan, every reference function called per class"
                 + (" incl. contour metrics (restated find_contours)" if cfg["contours"] else ""))
              + f"; functions from {root}")
    print(json.dumps({
        "impl": "reference", "metric": "bscans_per_sec_full_metric_suite", "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "strong" if (name == "cfg4" and not args.items) or name == "cfg5" else "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": cfg["workload"], "height": cfg["H"], "width": cfg["W"], "num_classes": cfg["K"]},
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "per_step_rates": [r * scale for r in rates],
    }))


# ------------------------------------------------------------------------------------ outputs of the timed path
def step_outputs(name, pend, out):
    """Host float64 copies of what the last timed step returned: ``pend`` is what ``step()`` returned, ``out`` what
    ``settle()`` made of it."""
    import numpy as np
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    f64 = lambda v: np.asarray(v, dtype=np.float64)          # noqa: E731
    if name == "cfg5":
        ints = {k: v.cpu().numpy() for k, v in out.items()}
        arrays = {"surface_" + k: f64(v.view(np.uint32) if v.dtype == np.int32 else v) for k, v in ints.items()}
        arrays.update({k: f64(v) for k, v in suite.surface_metrics_3d(out).items()})
        return arrays
    res = pend.res
    n = res.num_items
    idx = np.arange(n) if n <= DUMP_ITEMS else np.sort(np.random.default_rng(0).choice(n, DUMP_ITEMS, replace=False))
    arrays = {"item_index": f64(idx)}
    arrays.update({"item_" + k: f64(v[idx]) for k, v in res.metrics().items()})
    arrays.update({"dataset_" + k: f64(v) for k, v in out.items()})
    return arrays


def write_outputs(directory, arrays):
    import numpy as np
    total = sum(v.nbytes for v in arrays.values())
    assert total <= 64 << 20, f"{total} bytes of outputs: lower DUMP_ITEMS"
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), v)


# ------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite, synth
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    name = args.config
    cfg = CONFIGS[name]
    H, W, K = cfg["H"], cfg["W"], cfg["K"]
    contours = cfg["contours"] and not args.no_contours
    peak, peak_src = _peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- workload
    if name == "cfg5":
        D = cfg["D"]
        vt_h, vp_h = synth.layered_volume_pair(H, W, D, K, seed=cfg["seed"])
        vt, vp = torch.from_numpy(vt_h).to(dev), torch.from_numpy(vp_h).to(dev)
        units_per_step = 1.0 / world                     # the volume's 2 K units are split over the ranks
        bytes_per_unit = 2 * H * W * D
        unit = "volumes/s"
        scaling = "strong"
        n = 1

        def step():
            return odist.surface_distance_3d_sharded(vt, vp, K, rank, world)

        def settle(out):
            return out

        l2_note = f"one unit's planes ({H * W * D * 6 / 1e6:.0f} MB of g/h2) exceed the 126 MB L2"
        cfg_extra = {"depth": D, "sharding": f"{2 * K} (class, direction) units over {world} rank(s), one small all-reduce"}
    else:
        unit = "B-scans/s"
        if name == "cfg4":
            n = args.items if args.items else math.ceil(CFG4_ITEMS / world)
            scaling = "weak" if args.items else "strong"
            if args.uniform_random:
                g = torch.Generator(device=dev)
                g.manual_seed(cfg["seed"] + rank)
                yt = torch.randint(0, K, (n, H, W), generator=g, device=dev, dtype=torch.uint8)
                yp = torch.randint(0, K, (n, H, W), generator=g, device=dev, dtype=torch.uint8)
            else:
                yt, yp = synth.layered_pair_device(n, H, W, K, seed=cfg["seed"] + rank, device=dev, noise=args.noise)
            ring = [(yt, yp)]
            l2_note = "inputs (%.1f GB per GPU) exceed the 126 MB L2" % (n * 2 * H * W / 1e9)
        else:
            # single small volumes: every rank scores the same configuration (replicas) on a ring of distinct copies,
            # so that a step never finds its inputs in L2
            n = cfg["items"]
            scaling = "weak"
            copies = max(2, math.ceil(3 * 126e6 / (n * 2 * H * W)))
            ring = []
            for c in range(copies):
                a, b = host_pair(cfg, n, cfg["seed"] + 17 * c + 1000 * rank)
                ring.append((torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev)))
            l2_note = f"{copies} distinct volumes cycled ({copies * n * 2 * H * W / 1e6:.0f} MB > 126 MB L2)"
        units_per_step = float(n)
        bytes_per_unit = 2 * H * W
        timers = {}
        state = {"i": 0}

        def step():
            a, b = ring[state["i"] % len(ring)]
            state["i"] += 1
            res = suite.evaluate(a, b, K, contours=contours, boundaries=(name == "cfg2"), timers=timers)
            return odist.dataset_totals_async(res, world)     # one small all-reduce on the device vector

        def settle(pend):
            return pend.result()

        cfg_extra = {"items_per_gpu": n, "contours": contours,
                     "sharding": (f"{CFG4_ITEMS if not args.items else n * world} items over {world} rank(s), one NCCL all-reduce of totals"
                                  if name == "cfg4" else f"{world} replica(s) of the volume")}
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)                      # let the sampler finish initialising before anything is timed
    prev = None
    for _ in range(args.warmup):          # two evaluations in flight, like the timed loop: primes torch's allocator
        cur = step()
        if prev is not None:
            settle(prev)
        prev = cur
    if prev is not None:
        settle(prev)
    prev = cur = None
    barrier()
    if name != "cfg5":
        timers.clear()
    gc.collect()
    gc.disable()          # a generational collection inside a ~15 ms step is a 10 ms host stall
    keep = None
    if name != "cfg5":
        keep = torch.zeros((args.steps, int(_lib.load().octm_totals_len(K))), dtype=torch.float64, device=dev)
    launches0 = _lib.launch_count()
    t_begin = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    pend = None
    for i in range(args.steps):
        pend = step()                     # the previous step's outputs go back to torch's caching allocator here:
        if keep is not None:              # no cudaMalloc in the timed region (one can stall the host for 50+ ms)
            keep[i].copy_(pend.reduced)
    ev1.record()
    barrier()
    out = settle(pend)
    dumped = step_outputs(name, pend, out) if args.dump_outputs and rank == 0 else None
    if keep is not None and len(ring) == 1:
        kh = keep.cpu().numpy()
        assert all((kh[i] == kh[0]).all() for i in range(args.steps)), "steps disagree on the dataset totals"
    ms = ev0.elapsed_time(ev1)
    gc.enable()
    launches = _lib.launch_count() - launches0
    families = None
    if name != "cfg5":
        families = {k: sum(a.elapsed_time(b) for a, b in v) / args.steps for k, v in timers.items()}
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * units_per_step * args.steps / (ms / 1e3)

    # ---------------------------------------------------------------- per-kernel device times: two extra, UNTIMED steps
    # bracketed kernel by kernel with CUDA events on the launch stream (octm_profile_*)
    with _lib.kernel_profile() as prof:
        for _ in range(2):
            settle(step())
        torch.cuda.synchronize()
    step_ms = ms / args.steps
    ksum = sum(v[1] for v in prof.kernels.values()) / 2
    traffic = _ncu_traffic()
    kernels = []
    for kname, (cnt, tot) in sorted(prof.kernels.items(), key=lambda kv: -kv[1][1]):
        bound, counter = KERNEL_NOTES.get(kname, ("latency", ""))
        kernels.append({"kernel": kname, "launches_per_step": cnt // 2, "ms_per_step": tot / 2,
                        "share_of_kernel_time": (tot / 2) / ksum if ksum else None, "bound": bound, "evidence": counter,
                        "algorithmic_gbs": units_per_step * bytes_per_unit / (tot / 2 / 1e3) / 1e9 if bound == "hbm" else None})
    achieved = units_per_step * bytes_per_unit * args.steps / (ms / 1e3) / 1e9
    dominant = kernels[0]["kernel"] if kernels else None
    tr = traffic.get(name, {}).get(dominant) if dominant else None
    roofline = {"bound": "hbm", "level": "suite: compulsory label bytes (each byte of y_true and y_pred once) over the whole step",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (tr["dram_bytes_per_unit"] * units_per_step) if tr else None,
                "traffic_source": tr["source"] if tr else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": units_per_step * bytes_per_unit, "ms_per_launch": step_ms,
                "dominant_kernel": dominant, "kernel_time_over_step_time": ksum / step_ms if step_ms else None,
                "kernels": kernels}

    # ---------------------------------------------------------------- end to end through the public host-array API
    e2e = None
    if not args.no_e2e:
        if name == "cfg5":
            ht, hp = torch.from_numpy(vt_h).pin_memory(), torch.from_numpy(vp_h).pin_memory()
            m = 1

            def e2e_step():
                a, b = ht.to(dev, non_blocking=True), hp.to(dev, non_blocking=True)
                ints = odist.surface_distance_3d_sharded(a, b, K, rank, world)
                mm = suite.surface_metrics_3d(ints)
                return sum(np.asarray(v).nbytes for v in mm.values())
            h2d_bytes = 2 * H * W * D
            e2e_units = 1.0 / world
        else:
            m = min(n, args.e2e_items)
            ht, hp = ring[0][0][:m].cpu().pin_memory(), ring[0][1][:m].cpu().pin_memory()

            def e2e_step():
                r = suite.evaluate_host(ht, hp, K, contours=contours, device=dev)
                return sum(v.nbytes for v in r.metrics().values()) + r.totals_host().nbytes
            h2d_bytes = m * 2 * H * W
            e2e_units = float(m)
        # pinned host->device copy rate with ALL ranks copying at once: the ceiling of the end-to-end number
        probe_h = ht if name != "cfg5" else ht
        probe_d = torch.empty_like(probe_h, device=dev)
        probe_d.copy_(probe_h, non_blocking=True)
        barrier()
        tp = time.perf_counter()
        for _ in range(3):
            probe_d.copy_(probe_h, non_blocking=True)
        torch.cuda.synchronize()
        dt_probe = time.perf_counter() - tp
        tpr = torch.tensor([dt_probe], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tpr, op=dist.ReduceOp.MAX)
        h2d_gbs_contended = 3 * probe_h.numel() / float(tpr.item()) / 1e9          # per GPU, all ranks busy
        del probe_d
        for _ in range(max(1, min(args.warmup, 2))):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        e2e_steps = max(1, min(args.steps, 6))
        d2h = 0
        for _ in range(e2e_steps):
            d2h = e2e_step()
        barrier()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": world * e2e_units * e2e_steps / float(t.item()), "unit": unit,
               "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h),
               "items_per_step_per_gpu": m, "steps": e2e_steps,
               "pinned_h2d_gbs_per_gpu_all_ranks_copying": round(h2d_gbs_contended, 1),
               "h2d_gbs_achieved_per_gpu": round(e2e_units * e2e_steps * (h2d_bytes / e2e_units if e2e_units else 0) / float(t.item()) / 1e9, 1)}
        if args.e2e_pack and name != "cfg5" and K <= 16:
            # the same call with pack=True: two labels per byte across PCIe, packed by the host's cores (half the bytes on the
            # link; pays where the link, not the host's memory, is the limit)
            def e2e_packed_step():
                r = suite.evaluate_host(ht, hp, K, contours=contours, device=dev, pack=True)
                return sum(v.nbytes for v in r.metrics().values()) + r.totals_host().nbytes
            for _ in range(2):
                e2e_packed_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_packed_step()
            barrier()
            tpk = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tpk, op=dist.ReduceOp.MAX)
            e2e["packed"] = {"value": world * e2e_units * e2e_steps / float(tpk.item()), "unit": unit,
                             "h2d_bytes_per_step": int(h2d_bytes // 2), "note": "evaluate_host(pack=True)"}

    # ---------------------------------------------------------------- secondary rates (cfg4): harder inputs, smaller batch
    secondary = {}
    if name == "cfg4" and not args.no_secondary and not args.noise and not args.uniform_random:
        m = min(n, 4096)
        g = torch.Generator(device=dev)
        g.manual_seed(99 + rank)
        variants = {
            "noise_2e-5": synth.layered_pair_device(m, H, W, K, seed=7001 + rank, device=dev, noise=2e-5),
            "noise_2e-3": synth.layered_pair_device(m, H, W, K, seed=7002 + rank, device=dev, noise=2e-3),
            "uniform_random": (torch.randint(0, K, (m, H, W), generator=g, device=dev, dtype=torch.uint8),
                               torch.randint(0, K, (m, H, W), generator=g, device=dev, dtype=torch.uint8)),
        }
        # ragged predicted boundaries (one-pixel teeth and overhangs along every layer): most predicted contours are walked
        variants["ragged_boundaries"] = synth.ragged_pair_device(m, H, W, K, seed=7004 + rank, device=dev)
        # a 10-class label set at HC-MS geometry (496 x 1024): the K <= 16 label pass (label_pass_wide) + the same contour stage
        kk = {vname: K for vname in variants}
        variants["k10_496x1024"] = synth.layered_pair_device(min(n, 2048), 496, 1024, 10, seed=7003 + rank, device=dev, noise=0.0)
        kk["k10_496x1024"] = 10
        for vname, (a, b) in variants.items():
            K2, m = kk[vname], a.shape[0]
            for _ in range(2):
                odist.dataset_totals_async(suite.evaluate(a, b, K2, contours=contours), world).result()
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            reps = 3
            for _ in range(reps):
                p2 = odist.dataset_totals_async(suite.evaluate(a, b, K2, contours=contours), world)
            s1.record()
            barrier()
            p2.result()
            tv = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tv, op=dist.ReduceOp.MAX)
            secondary[vname] = {"value": world * m * reps / (float(tv.item()) / 1e3), "unit": unit, "items_per_gpu": m,
                                "shape": [int(a.shape[1]), int(a.shape[2])], "num_classes": K2}
        del variants

    clocks = sampler.stop(t_begin, time.perf_counter()) if rank == 0 else None   # device-timed + e2e regions
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            ns = max(1, min(cores, 64))
            rate, per = cpu_baseline(name, ns, min(cores, ns))
            rate1, per1 = cpu_baseline(name, 2, 1)
            kind, root = _cpu_kind()
            scale = _cpu_unit_scale(name)
            cpu = {"value": rate * scale, "unit": unit, "cores": min(cores, ns), "kind": kind,
                   "one_core_value": rate1 * scale,
                   "sample": f"{ns} units of the same workload on {min(cores, ns)} processes (+ 2 on one core); "
                             + ("unit = one class of a 128x128x32 sub-volume (scipy EDT), scaled to full volumes"
                                if name == "cfg5" else "unit = one B-scan, the reference's functions called per class per function"
                                + (", contour functions on the restated find_contours" if contours else ""))
                             + f"; {per:.2f} s per unit per core; functions from {root}"}
        line = {
            "metric": "bscans_per_sec_full_metric_suite", "value": value, "unit": unit, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": dict({"workload": cfg["workload"]
                            + (f", {args.noise:g} of the predicted pixels randomised" if args.noise else "")
                            + (", uniform random labels (adversarial variant)" if args.uniform_random else ""),
                            "height": H, "width": W, "num_classes": K, "l2": l2_note,
                            "results": "left in HBM during the timed region; every step's dataset totals are read back and compared after it"},
                           **cfg_extra),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu, "secondary": secondary or None,
        }
        if name != "cfg5":
            line["kernel_family_ms_per_step"] = families
            line["dataset_dice"] = [float(x) for x in out["dice_coefficient"]] if out else None
        else:
            mm = suite.surface_metrics_3d(out)
            line["hausdorff_distance"] = [float(x) for x in mm["hausdorff_distance"]]
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg4", choices=sorted(CONFIGS))
    ap.add_argument("--items", type=int, default=0,
                    help="cfg4: B-scans per GPU per step (weak scaling); default ceil(100000 / world) = the configuration as stated")
    ap.add_argument("--e2e-pack", action="store_true", help="also time evaluate_host(pack=True) (two labels per byte across PCIe)")
    ap.add_argument("--noise", type=float, default=0.0,
                    help="cfg4: fraction of predicted pixels replaced by a random class (default 0: the contract's clean layered maps)")
    ap.add_argument("--uniform-random", action="store_true", help="cfg4: every pixel of both maps a random class")
    ap.add_argument("--e2e-items", type=int, default=4096)
    ap.add_argument("--no-contours", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (float64, seeded sample of large batches)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
