#!/usr/bin/env python
"""Connected-component metrics on 16,384-item batches: the full suite without ``components``, with ``components=4``
and with ``components=8``, timed alternately; then components_kernel alone at each connectivity with its achieved
bandwidth over the label bytes (2 * H * W per item); then per-kernel times from a separate profiled pass.  One JSON
line per workload; the card's name and power limit first.

    python scripts/bench_components.py [--items 16384] [--reps 5]

The workloads are those of bench_surface_dice.py.  The kernel's cost follows the number of runs of equal labels per
row: a few on layers, scattered extra ones on noisy and ragged predictions and lesions, two 512-column passes per row
at W = 1024, and about seven of every eight pixels starting a run on uniform-random labels (the worst case).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch      # noqa: E402

CONNS = (4, 8)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def workloads(n, dev):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import synth
    yield "cfg4 layered 496x512 K=8 clean", 8, synth.layered_pair_device(n, 496, 512, 8, seed=4004, device=dev)
    yield ("cfg4 layered 496x512 K=8 noise 0.002", 8,
           synth.layered_pair_device(n, 496, 512, 8, seed=4004, device=dev, noise=0.002))
    yield "ragged 496x512 K=8", 8, synth.ragged_pair_device(n, 496, 512, 8, seed=4005, device=dev)
    yt, yp = synth.lesion_pair(256, 512, 512, 4, seed=3003, single_blob_interior=False)
    reps = (n + 255) // 256
    yield ("lesion 512x512 K=4 (256 distinct items tiled)", 4,
           (torch.from_numpy(yt).to(dev).repeat(reps, 1, 1)[:n].contiguous(),
            torch.from_numpy(yp).to(dev).repeat(reps, 1, 1)[:n].contiguous()))
    yield "layered 496x1024 K=10 noise 0.002", 10, synth.layered_pair_device(n, 496, 1024, 10, seed=4007, device=dev,
                                                                             noise=0.002)
    g = torch.Generator(device=dev).manual_seed(4008)
    yield ("uniform random 496x512 K=8", 8,
           tuple(torch.randint(0, 8, (n, 496, 512), generator=g, device=dev, dtype=torch.uint8) for _ in range(2)))


def timed(fn, reps):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return out


def median(v):
    return sorted(v)[len(v) // 2]


def main():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required")
    dev = torch.device("cuda", 0)
    print(json.dumps(card()), flush=True)
    n = args.items
    for name, k, (yt, yp) in workloads(n, dev):
        h, w = yt.shape[1:]
        runs = {"evaluate": lambda: suite.evaluate(yt, yp, k).totals_host()}
        for conn in CONNS:
            runs[f"evaluate+components={conn}"] = lambda conn=conn: suite.evaluate(yt, yp, k, components=conn).metrics()
        for f in runs.values():          # warm-up: modules, allocator, contour scratch
            f()
            f()
        ms = {m: [] for m in runs}
        for _ in range(args.reps):       # alternate so that all see the same machine state
            for m, f in runs.items():
                ms[m] += timed(f, 1)
        kernel = {}
        for conn in CONNS:
            def cc():
                suite.components(yt, yp, k, conn)
            cc()
            t = median(timed(cc, max(args.reps, 5)))
            kernel[str(conn)] = {"ms": round(t, 3), "gb_per_s": round(2 * n * h * w / (t / 1e3) / 1e9, 1)}
        prof = {}
        for m, f in runs.items():
            with _lib.kernel_profile() as p:
                f()
                torch.cuda.synchronize()
            prof[m] = {kname: round(t, 3) for kname, (_, t) in p.kernels.items()}
        print(json.dumps({
            "workload": name, "items": n,
            "bscans_per_s": {m: round(n / (median(v) / 1e3)) for m, v in ms.items()},
            "ms_per_batch": {m: [round(x, 2) for x in v] for m, v in ms.items()},
            "components_kernel_alone": kernel,
            "kernel_ms": prof,
        }), flush=True)
        del yt, yp
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
