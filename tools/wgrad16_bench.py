"""Per-launch timing of the 3x3 weight gradients that produce 16 channels (64 -> 16 and 16 -> 16) at the benchmarked steps'
shapes: the tcgen05 halo kernel (wgrad_halo.cu, the default route) against the route taken when the halo kernels are switched
off with svrs_set_halo_mode(0) (wgrad_tc.cu; before the halo kernel took these layers, the mma.sync kernel wgrad16.cuh).

Each variant's launches are captured in a CUDA graph with their own inputs; the graphs are replayed alternately (A B A B ...)
and timed with CUDA events.  Consecutive launches rotate over enough input copies (> 2 x the 126 MB L2) that every launch
reads its X and dy from HBM.  Achieved bytes/s counts the bytes the weight gradient must read (X + dy, bf16) and is set
against the HBM bound (6.55 TB/s, the copy rate measured on B200 in DESIGN.md §3.1).
    python tools/wgrad16_bench.py [--reps 20] [--rounds 7] [--quick]"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "simple-vae-rs_b200")]
import torch  # noqa: E402
from svrs_native.lib import BF16, lib  # noqa: E402

HBM_TBS = 6.55
L2_BYTES = 126e6
# name, N (patches), H = W, Cin ; Cout = 16.  The layers of cond_grid (128) / cond_grid1024 (1024), vae and cond256
CASES = [
    ("dec_x 64->16 @64", 128, 64, 64), ("dec_x 16->16 @64", 128, 64, 16),
    ("dec_y 64->16 @32", 128, 32, 64), ("dec_y 16->16 @32", 128, 32, 16),
    ("down  16->16 @16", 128, 16, 16), ("down  16->16 @32", 128, 32, 16),
    ("dec_x 64->16 @64", 1024, 64, 64), ("dec_x 16->16 @64", 1024, 64, 16),
    ("dec_y 64->16 @32", 1024, 32, 64), ("dec_y 16->16 @32", 1024, 32, 16),
    ("down  16->16 @16", 1024, 16, 16),
]


def st():
    return torch.cuda.current_stream().cuda_stream


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def make_graph(mode, N, H, Cin, reps, copies):
    """reps launches of the layer's weight gradient (+ folded bias gradient) under halo mode `mode`, in one CUDA graph."""
    Cout = 16
    xs = [torch.randn(N, H, H, Cin, device="cuda").to(torch.bfloat16) for _ in range(copies)]
    dys = [torch.randn(N, H, H, Cout, device="cuda").to(torch.bfloat16) for _ in range(copies)]
    dw = torch.zeros(Cout * Cin * 9, device="cuda")
    dwp = torch.zeros(Cout * Cin * 9, device="cuda")
    db = torch.zeros(Cout, device="cuda")
    lib.set_halo_mode(mode)
    try:
        layout = lib.conv2d_wgrad_layout(BF16, N, H, H, Cin, Cout, 3)

        def one(i):
            lib.conv2d_wgrad(xs[i % copies].data_ptr(), dys[i % copies].data_ptr(), dw.data_ptr(), dwp.data_ptr(), db.data_ptr(),
                             BF16, N, H, H, Cin, Cout, 3, 0, st())
        for i in range(3):
            one(i)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(reps):
                one(i)
    finally:
        lib.set_halo_mode(1)
    g.replay()
    torch.cuda.synchronize()
    return g, layout, (xs, dys, dw, dwp, db)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="launches per graph")
    ap.add_argument("--rounds", type=int, default=7, help="alternating replays of each graph")
    ap.add_argument("--quick", action="store_true", help="128-patch cases only")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wgrad16_bench: no CUDA device")
    lib.load()
    print(f"# {gpu_info()}")
    print(f"# per launch, median of {a.rounds} alternating replays of {a.reps}-launch graphs; bytes = X + dy (bf16)")
    print(f"{'layer':18s} {'N':>5s} {'MB':>7s} | {'variant':9s} {'us':>8s} {'TB/s':>6s} {'of HBM':>7s}")
    for name, N, H, Cin in CASES:
        if a.quick and N != 128:
            continue
        nbytes = N * H * H * (Cin + 16) * 2
        copies = max(1, min(64, int(2 * L2_BYTES / nbytes) + 1))
        variants = [("halo", 1), ("halo off", 0)]
        graphs = [make_graph(m, N, H, Cin, a.reps, copies) for _, m in variants]
        times = [[] for _ in variants]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(a.rounds):
            for v, (g, _, _) in enumerate(graphs):
                e0.record()
                g.replay()
                e1.record()
                torch.cuda.synchronize()
                times[v].append(e0.elapsed_time(e1) * 1e3 / a.reps)
        bound_us = nbytes / (HBM_TBS * 1e12) * 1e6
        for (vname, _), (g, layout, _), ts in zip(variants, graphs, times):
            t = sorted(ts)[len(ts) // 2]
            print(f"{name:18s} {N:5d} {nbytes / 1e6:7.1f} | {vname:9s} {t:8.1f} {nbytes / t / 1e6:6.2f} {bound_us / t:7.1%}"
                  f"   (layout {layout}, spread {min(ts):.1f}-{max(ts):.1f})")
        del graphs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
