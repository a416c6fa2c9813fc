#!/usr/bin/env python
"""ETDRS-sector layer thickness on batches of whole OCT volumes: Duke DME (61 x 496 x 768, K = 8) and HC-MS
(49 x 496 x 1024, K = 10), 64 volumes each by default (3 GB of label bytes per pair at HC-MS shape, far beyond the
126 MB L2).  Per shape, alternating over several repetitions after a warm-up, CUDA events time:

- ``label_pass``: ``suite.label_pass(counts, columns, boundaries)`` alone;
- ``sector_kernel``: ``octm_sector_thickness_i32`` alone on those boundary rows (one group per class);
- ``sector_kernel_maps``: the same with the per-A-scan thickness maps written;
- ``call``: the whole ``suite.sector_thickness`` call (label pass, host grid, region upload, kernel).

Reported: medians, volumes/s of the whole call, the label bytes over the label-pass time and the boundary-row bytes
over the sector-kernel time, and the card's name and power limit, read in the same run.  One JSON line per shape.

    python scripts/bench_sector_thickness.py [--volumes 64] [--reps 7] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch        # noqa: E402

SHAPES = (("duke_dme", 61, 496, 768, 8, (0.1185, 0.00387, 0.00772)),
          ("hc_ms", 49, 496, 1024, 10, (0.1229, 0.00387, 0.00583)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, derive, suite, synth
    ap = argparse.ArgumentParser()
    ap.add_argument("--volumes", type=int, default=64)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required")
    dev = torch.device("cuda", 0)
    lines = [card()]
    print(json.dumps(lines[0]), flush=True)
    v = args.volumes
    for name, b, h, w, k, sp in SHAPES:
        yt, yp = synth.layered_pair_device(v * b, h, w, k, seed=61, device=dev, noise=0.002)
        yt4, yp4 = yt.view(v, b, h, w), yp.view(v, b, h, w)
        lp = suite.label_pass(yt, yp, k, counts=True, columns=True, boundaries=True)
        reg = derive.etdrs_regions(b, w, sp, ((b - 1) / 2, (w - 1) / 2))
        region = torch.from_numpy(reg).to(dev).expand(v, b, w).contiguous()
        groups = (ctypes.c_int32 * (2 * k))(*[c for c in range(k) for _ in range(2)])
        sums = torch.empty((v, k, 9, 5), dtype=torch.int64, device=dev)
        thick = torch.empty((v, b, 2, k, w), dtype=torch.int32, device=dev)

        def kernel(maps):
            _lib.call("octm_sector_thickness_i32", suite._ptr(lp.bnd_true), suite._ptr(lp.bnd_pred), v * b, k, h, w, b,
                      suite._ptr(region), 9, groups, k, suite._ptr(sums), suite._ptr(thick) if maps else None,
                      suite._stream())
        legs = {"label_pass": lambda: suite.label_pass(yt, yp, k, counts=True, columns=True, boundaries=True),
                "sector_kernel": lambda: kernel(False),
                "sector_kernel_maps": lambda: kernel(True),
                "call": lambda: suite.sector_thickness(yt4, yp4, k, sp)}
        for f in legs.values():           # warm-up: modules, allocator
            f()
            f()
        torch.cuda.synchronize()
        ms = {leg: [] for leg in legs}
        for _ in range(args.reps):        # alternate the legs so that all see the same machine state
            for leg, f in legs.items():
                ms[leg].append(timed(f))
        med = {leg: float(np.median(x)) for leg, x in ms.items()}
        # the whole call equals the sums of the kernel leg (same rows, same regions)
        out = suite.sector_thickness(yt4, yp4, k, sp)
        kernel(False)
        torch.cuda.synchronize()
        assert torch.equal(out.sums, sums), "the call and the kernel leg disagree"
        with _lib.kernel_profile() as p:  # per-kernel times in a separate, profiled pass
            suite.sector_thickness(yt4, yp4, k, sp)
            torch.cuda.synchronize()
        n = v * b
        label_bytes = 2 * n * h * w
        row_bytes = 2 * n * (k - 1) * w * 4 + n * w            # both maps' boundary rows and the region codes
        maps_bytes = n * 2 * k * w * 4
        line = {"workload": f"{name} {b}x{h}x{w} K={k} layered noise 0.002", "volumes": v, "spacing_mm": sp,
                "ms_median": {leg: round(x, 4) for leg, x in med.items()},
                "ms": {leg: [round(t, 4) for t in x] for leg, x in ms.items()},
                "volumes_per_s_call": round(v / (med["call"] / 1e3), 1),
                "label_pass_GBps": round(label_bytes / (med["label_pass"] / 1e3) / 1e9, 1),
                "sector_kernel_GBps": round(row_bytes / (med["sector_kernel"] / 1e3) / 1e9, 1),
                "sector_kernel_maps_GBps": round((row_bytes + maps_bytes) / (med["sector_kernel_maps"] / 1e3) / 1e9, 1),
                "row_bytes_over_label_bytes": round(row_bytes / label_bytes, 4),
                "sector_over_label_pass": round(med["sector_kernel"] / med["label_pass"], 4),
                "kernel_ms_profiled_call": {kn: round(t, 4) for kn, (_, t) in p.kernels.items()}}
        lines.append(line)
        print(json.dumps(line), flush=True)
        del yt, yp, yt4, yp4, lp, region, sums, thick, out
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
