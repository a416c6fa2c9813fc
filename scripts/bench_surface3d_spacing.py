#!/usr/bin/env python
"""3-D surface distances with a physical voxel spacing (BASELINE config 5 volume: 1024 x 1024 x 128, 11 classes).

    python scripts/bench_surface3d_spacing.py                      # one GPU, all 22 (class, direction) units
    torchrun --nproc-per-node N scripts/bench_surface3d_spacing.py # units sharded over N GPUs, one small all-reduce

Three legs in the same run, alternating, each repeated: the voxel-unit integer path, spacing = (0.0039, 0.0117, 0.047)
mm (axial, lateral, between B-scans, Spectralis-like), and the same spacing with tolerances (0.01, 0.02) mm.  Each
timed sample is CUDA events around STEPS calls after a barrier, max over ranks.  The per-kernel times come from a
separate, untimed call per leg with the library's kernel profiler (rank 0's kernels).  With N > 1 every leg's sharded
outputs are compared with an unsharded call on rank 0.  Prints one JSON line, with the card's name and power limit.
Ranks beyond the visible GPUs share them (gloo instead of NCCL; ``n_gpus`` < ``n_ranks`` in the JSON line): that checks
the sharded path, but its times are not those of N GPUs.
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np      # noqa: E402
import torch            # noqa: E402

SPACING = (0.0039, 0.0117, 0.047)
LEGS = {"integer": {}, "spacing": {"spacing": SPACING},
        "spacing_tolerances": {"spacing": SPACING, "tolerances": (0.01, 0.02)}}
STEPS, REPEATS = 3, 5


def card(local):
    """Name and power limit of this rank's GPU (read-only query)."""
    name = torch.cuda.get_device_name(local)
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return name, r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        return name, f"unavailable: {e}"


def main():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite, synth
    from retinal_oct_image_segmentation_via_deep_learning_b200 import dist as odist
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")))
    d0, d1, d2, k = 1024, 1024, 128, 11
    # one GPU per rank (NCCL); with more ranks than GPUs the ranks share them round-robin, which NCCL does not allow,
    # so gloo carries the all-reduces (of CUDA tensors): a run of the sharded code path, not a scaling measurement
    gpus = torch.cuda.device_count()
    backend = "nccl" if world <= gpus else "gloo"
    local = local % gpus
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        torch.distributed.init_process_group(backend, device_id=dev if backend == "nccl" else None)
    vt, vp = synth.layered_volume_pair(d0, d1, d2, k, seed=5005)
    vt, vp = torch.from_numpy(vt).to(dev), torch.from_numpy(vp).to(dev)

    def run(kw):
        return odist.surface_distance_3d_sharded(vt, vp, k, rank, world, **kw)

    outs = {name: run(kw) for name, kw in LEGS.items()}           # warm-up, and the outputs
    torch.cuda.synchronize()
    samples = {name: [] for name in LEGS}
    for _ in range(REPEATS):
        for name, kw in LEGS.items():
            if world > 1:
                torch.distributed.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(STEPS):
                run(kw)
            b.record()
            torch.cuda.synchronize()
            ms = torch.tensor([a.elapsed_time(b) / STEPS], dtype=torch.float64, device=dev)
            if world > 1:
                torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
            samples[name].append(float(ms.item()))
    kernels = {}
    for name, kw in LEGS.items():
        with _lib.kernel_profile() as prof:
            run(kw)
            torch.cuda.synchronize()
        kernels[name] = {kn: {"launches": n, "ms": round(ms, 4)} for kn, (n, ms) in sorted(prof.kernels.items())}
    same = None
    if world > 1 and rank == 0:
        same = {}
        for name, kw in LEGS.items():
            single = suite.surface_distance_3d(vt, vp, k, **kw)
            same[name] = all(torch.equal(single[key], outs[name][key]) for key in single) and \
                set(single) == set(outs[name])
    if rank == 0:
        name, power = card(local)
        res = {"workload": f"cfg5 volume {d0}x{d1}x{d2}, {k} classes, {2 * k} (class, direction) units",
               "n_ranks": world, "n_gpus": min(world, gpus), "backend": backend if world > 1 else None,
               "card": name, "power_limit_and_max_sm_clock": power,
               "spacing_mm": SPACING, "tolerances_mm": LEGS["spacing_tolerances"]["tolerances"],
               "ms_per_volume_pair": {n: {"median": float(np.median(s)), "min": min(s), "samples": s}
                                      for n, s in samples.items()},
               "kernels_rank0": kernels}
        if same is not None:
            res["sharded_equals_single_gpu"] = same
        m = suite.surface_metrics_3d(outs["spacing_tolerances"])
        res["hausdorff_distance_mm"] = [round(float(x), 6) for x in m["hausdorff_distance"]]
        res["assd_mm"] = [round(float(x), 6) for x in m["assd"]]
        res["surface_dice"] = [[round(float(x), 6) for x in row] for row in m["surface_dice"]]
        print(json.dumps(res))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
