#!/usr/bin/env python
"""Device time of svrs_ssim (ssim_kernel + ssim_finalize_kernel) at the sizes evaluate() sees, printed as one JSON line.

    python tools/ssim_bench.py [--iters 50]

Workloads: the config-3 validation batch (128 pairs at 4x64^2 for SSIM_HR / SSIM_SR and 128 at 4x32^2 for SSIM_LR), a batch larger
than the 126 MB L2 (1024 pairs at 4x64^2, 134 MB read: every pass comes from HBM) and config 4's HR crops (16 pairs at 4x256^2).
Algorithmic bytes = the two input batches read once (2*N*C*H*W*4); bandwidth is compared with the measured HBM copy rate
6549.8 GB/s.  Time per call = CUDA events around --iters back-to-back calls (both launches each) after warm-up, median of five such
windows; the 128-pair batches (17 / 4 MB) fit in L2 across calls, the 1024-pair batch does not.  The numpy fp64 oracle's host
time on the same pairs is reported as `oracle_host_ms` (the oracle of the tests, not scikit-image)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "simple-vae-rs_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ssim_oracle  # noqa: E402
from svrs_native.lib import lib  # noqa: E402

HBM_GBS = 6549.8
WORKLOADS = [("cfg3_val_hr_128x4x64", (128, 4, 64, 64)), ("cfg3_val_lr_128x4x32", (128, 4, 32, 32)),
             ("beyond_l2_1024x4x64", (1024, 4, 64, 64)), ("cfg4_hr_16x4x256", (16, 4, 256, 256))]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in q.split(","))
    except Exception as e:  # still report the device name from torch
        name, power = torch.cuda.get_device_name(0), f"unknown ({e})"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ssim_bench needs a CUDA device")
    name, power = gpu_info()
    res = {"gpu": name, "power_limit": power, "hbm_ref_GBps": HBM_GBS, "iters": args.iters, "workloads": {}}
    rng = np.random.default_rng(0)
    for label, shape in WORKLOADS:
        a_np = rng.random(shape, dtype=np.float32)
        b_np = np.clip(a_np + 0.1 * rng.standard_normal(shape, dtype=np.float32), 0, 1)
        a, b = torch.from_numpy(a_np).cuda(), torch.from_numpy(b_np).cuda()
        N, C, H, W = shape
        ws = torch.empty(lib.ssim_workspace_doubles(N, C, H, W, 11), device="cuda", dtype=torch.float64)
        out = torch.empty(N, device="cuda", dtype=torch.float64)
        call = lambda: lib.ssim(a.data_ptr(), b.data_ptr(), N, C, H, W, 11, 1.0, ws.data_ptr(), out.data_ptr(),
                                torch.cuda.current_stream().cuda_stream)
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        times = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(5_000_000)        # device-side spin: the calls below are enqueued before e0 starts the clock
            e0.record()
            for _ in range(args.iters):
                call()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) * 1e3 / args.iters)
        us = float(np.median(times))
        nbytes = 2 * a.numel() * 4
        t0 = time.perf_counter()
        ref = ssim_oracle.ssim(a_np, b_np)
        oracle_ms = (time.perf_counter() - t0) * 1e3
        res["workloads"][label] = {
            "shape": list(shape), "ssim_us": round(us, 2), "ssim_us_min": round(min(times), 2),
            "bytes": nbytes, "GBps": round(nbytes / us / 1e3, 1), "of_hbm_peak": round(nbytes / us / 1e3 / HBM_GBS, 3),
            "max_abs_err_vs_oracle": float(np.abs(out.cpu().numpy() - ref).max()), "oracle_host_ms": round(oracle_ms, 1)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
