#!/usr/bin/env python
"""All-contour distances (contours="all") against contour [0] (contours=True) on 16,384-item batches: B-scans/s of
the full suite in both modes, timed alternately, then per-kernel times from a separate profiled pass, and the
achieved bandwidth of contour_all_vertices_kernel.  One JSON line per workload; the card's name and power limit first.

    python scripts/bench_all_contours.py [--items 16384] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch      # noqa: E402


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
        modes = {"first": lambda: suite.evaluate(yt, yp, k, contours=True).totals_host(),
                 "all": lambda: suite.evaluate(yt, yp, k, contours="all").totals_host()}
        for f in modes.values():          # warm-up: modules, allocator, scratch of both modes
            f()
            f()
        ms = {m: [] for m in modes}
        for _ in range(args.reps):        # alternate the modes so that both see the same machine state
            for m, f in modes.items():
                ms[m] += timed(f, 1)
        rate = {m: n / (sorted(v)[len(v) // 2] / 1e3) for m, v in ms.items()}
        # the emission kernel alone, on a bound no item exceeds
        cap = suite.default_max_pts_all(w)
        verts = torch.empty((n, k, 2, cap), dtype=torch.int32, device=dev)
        n_pts = torch.empty((n, k, 2), dtype=torch.int32, device=dev)
        flags = torch.empty((n, k), dtype=torch.int32, device=dev)

        def emit():
            _lib.call("octm_contour2d_all_vertices_u8", suite._ptr(yt), suite._ptr(yp), n, h, w, k, cap,
                      suite._ptr(verts), suite._ptr(n_pts), suite._ptr(flags), suite._stream())
        emit()
        torch.cuda.synchronize()
        emit_ms = sorted(timed(emit, 10))[5]
        total_pts = int(n_pts.to(torch.int64).sum())
        stored = int(n_pts.to(torch.int64).clamp(max=cap).sum())
        overflow = int((flags != 0).any(dim=1).sum())
        del verts
        # per-kernel times in separate, profiled passes
        prof = {}
        for m, f in modes.items():
            with _lib.kernel_profile() as p:
                f()
                torch.cuda.synchronize()
            prof[m] = {kname: round(t, 3) for kname, (_, t) in p.kernels.items()}
        print(json.dumps({
            "workload": name, "items": n,
            "bscans_per_s": {m: round(r) for m, r in rate.items()},
            "ms_per_batch": {m: [round(x, 2) for x in v] for m, v in ms.items()},
            "kernel_ms": prof,
            "emission": {"ms": round(emit_ms, 3), "vertices": total_pts, "vertices_stored": stored,
                         "items_over_first_bound": overflow, "first_bound": cap,
                         "gb_per_s": round((2 * n * h * w + 4 * stored) / (emit_ms / 1e3) / 1e9, 1),
                         "gb_per_s_all_counted": round((2 * n * h * w + 4 * total_pts) / (emit_ms / 1e3) / 1e9, 1)},
        }), flush=True)
        del yt, yp
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
