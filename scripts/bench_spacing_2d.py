#!/usr/bin/env python
"""B-scan metrics with a physical pixel spacing against pixel units on 16,384-item batches: B-scans/s of the full suite
for contours="all", contours=True and surface_dice=(1, 2) axial pixels, each without and with the Spectralis-like
spacing (0.0039, 0.0117) mm, the two legs timed alternately; then per-kernel times from a separate profiled pass.  One
JSON line per workload; the card's name and power limit first.

    python scripts/bench_spacing_2d.py [--items 16384] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch      # noqa: E402

OCT = (0.0039, 0.0117)          # mm: axial (rows), lateral (columns)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def workloads(n, dev):
    from retinal_oct_image_segmentation_via_deep_learning_b200 import synth
    yield "cfg4 layered 496x512 K=8 clean", 8, synth.layered_pair_device(n, 496, 512, 8, seed=4004, device=dev)
    yield ("cfg4 layered 496x512 K=8 noise 0.002", 8,
           synth.layered_pair_device(n, 496, 512, 8, seed=4004, device=dev, noise=0.002))
    yt, yp = synth.lesion_pair(256, 512, 512, 4, seed=3003, single_blob_interior=False)
    reps = (n + 255) // 256
    yield ("lesion 512x512 K=4 (256 distinct items tiled)", 4,
           (torch.from_numpy(yt).to(dev).repeat(reps, 1, 1)[:n].contiguous(),
            torch.from_numpy(yp).to(dev).repeat(reps, 1, 1)[:n].contiguous()))


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required")
    dev = torch.device("cuda", 0)
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    n = args.items
    for name, k, (yt, yp) in workloads(n, dev):
        # surface Dice at 1 and 2 axial pixels: the same physical tolerances in both legs
        legs = {}
        for mode, kw in (("all", dict(contours="all")), ("first", dict(contours=True)),
                         ("surface_dice", dict(contours=False, surface_dice=(1.0, 2.0)))):
            legs[f"{mode} px"] = lambda kw=kw: suite.evaluate(yt, yp, k, **kw).totals_host()
            kws = dict(kw)
            if "surface_dice" in kws:
                kws["surface_dice"] = (1.0 * OCT[0], 2.0 * OCT[0])
            legs[f"{mode} spacing"] = lambda kw=kws: suite.evaluate(yt, yp, k, spacing=OCT, **kw).totals_host()
        for f in legs.values():           # warm-up: modules, allocator, scratch of every leg
            f()
            f()
        ms = {leg: [] for leg in legs}
        for _ in range(args.reps):        # alternate the legs so that all see the same machine state
            for leg, f in legs.items():
                ms[leg].append(timed(f))
        rate = {leg: n / (sorted(v)[len(v) // 2] / 1e3) for leg, v in ms.items()}
        prof = {}
        for leg, f in legs.items():       # per-kernel times in separate, profiled passes
            with _lib.kernel_profile() as p:
                f()
                torch.cuda.synchronize()
            prof[leg] = {kname: round(t, 3) for kname, (_, t) in p.kernels.items()}
        line = {"workload": name, "items": n, "spacing": OCT,
                "bscans_per_s": {leg: round(r) for leg, r in rate.items()},
                "ms_per_batch": {leg: [round(x, 2) for x in v] for leg, v in ms.items()},
                "kernel_ms": prof}
        lines.append(line)
        print(json.dumps(line), flush=True)
        del yt, yp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
