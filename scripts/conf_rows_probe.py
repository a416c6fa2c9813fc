#!/usr/bin/env python
"""Certified label pass (the suite's call) per 16,384 cfg4 items, by count source and data: one JSON line per case.

policy 1: counts from the boundary rows (+ a per-pixel histogram of the rejected items); policy 2: the strip kernel's
per-pixel histogram.  Prints the call time (CUDA events, mean of 5 calls after 2 warm-up calls) and, from one separate
profiled call, every kernel's time.  OCTM_TREE=<another checkout, built> times that tree's library instead."""
import ctypes
import json
import os
import sys

sys.path.insert(0, os.environ.get("OCTM_TREE") or os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, synth  # noqa: E402

dev = torch.device("cuda", 0)
n, h, w, k = 16384, 496, 512, 8
lib = _lib.load()
P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
i64 = dict(dtype=torch.int64, device=dev)
i32 = dict(dtype=torch.int32, device=dev)
counts, thick = torch.empty((n, k, k), **i64), torch.empty((n, k), **i64)
bsq, bab = torch.empty((n, k - 1), **i64), torch.empty((n, k - 1), **i64)
bt, bp = torch.empty((n, k - 1, w), **i32), torch.empty((n, k - 1, w), **i32)
fp, uns = torch.empty((n, 2, k), **i32), torch.empty((n,), **i32)
st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
tree = os.path.dirname(os.path.dirname(os.path.abspath(_lib.__file__)))
for data, noise in (("clean", 0.0), ("noise_2e-3", 2e-3)):
    yt, yp = synth.layered_pair_device(n, h, w, k, seed=1, device=dev, noise=noise)
    for policy in (1, 2):
        before = lib.octm_label_pass_seed_policy(policy)
        call = lambda: _lib.call("octm_label_pass_sorted_u8", P(yt), P(yp), n, h, w, k, P(counts), P(thick), P(bsq), P(bab),
                                 P(bt), P(bp), P(fp), P(uns), st)
        for _ in range(2):
            call()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(5):
            call()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 5
        with _lib.kernel_profile() as prof:
            call()
            torch.cuda.synchronize()
        lib.octm_label_pass_seed_policy(before)
        print(json.dumps({"tree": tree, "data": data, "policy": policy, "items": n, "ms_per_call": round(ms, 4),
                          "rejected_items": int((uns != 0).sum()),
                          "kernels_ms": {kn: round(v[1], 4) for kn, v in sorted(prof.kernels.items())}}), flush=True)
    del yt, yp
