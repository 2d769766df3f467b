"""Training-step time of Cond_SRVAE at the compression ratios the reference trains at (cr 1.5: train.py's default and test.sh;
cr 1.2: the CondVAE production run) next to the benchmarked cr 2, and per-launch times of the layers whose channel counts
(168 / 336 / 424 / 672 / 848 / 1344 / 1696: multiples of 8, not of 16 or 64) run on tcgen05 with a zero-filled last chunk.

Step: FusedCondTrainer, bf16, 128 seeded patches of P = 64, graph-replayed; median of --rounds timed windows of --steps
steps each, the ratios interleaved (2, 1.5, 1.2, 2, 1.5, 1.2, ...).

Per launch: each pass of a layer that left the CUDA-core kernels (f = fprop, d = dgrad, w = wgrad with its bias gradient,
into the per-tap packed layout the fused optimiser reads) is captured --reps times in a CUDA graph on tcgen05 and again with
svrs_set_tc_enabled(0), which routes exactly these passes to the CUDA-core kernels (conv_simt.cu) the parent commit ran;
the two graphs are replayed alternately.  The inputs of one launch fit in L2 (at most 27 MB), as in the step.
    python tools/cr_bench.py [--steps 20] [--rounds 5] [--reps 20] [--no-layers] [--no-steps]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "simple-vae-rs_b200")]
import torch  # noqa: E402
from svrs_native.lib import BF16, lib  # noqa: E402

B, P = 128, 64
RATIOS = (2, 1.5, 1.2)
# (layer, cr, form, H = W of the input, Cin, Cout, passes that moved to tcgen05): the layers of MOVED in
# tests/test_cpu_ragged_dispatch.py, which derives them from the models
LAYERS = [
    ("mu/logvar_u_y_to_z.1", 1.5, "c3", 4, 1344, 672, "w"),
    ("mu/logvar_u_y_to_z.2", 1.5, "c3", 4, 672, 672, "w"),
    ("decoder_x.1.upsample", 1.5, "ct", 8, 336, 256, "w"),
    ("decoder_x.1.conv", 1.5, "c3", 8, 336, 336, "w"),
    ("encoder_x.6", 1.5, "c3", 8, 128, 336, "w"),
    ("y_to_z.4", 1.5, "c3", 4, 128, 672, "w"),
    ("u_to_z.2", 1.5, "c3", 4, 168, 672, "fw"),
    ("u_to_z.1", 1.5, "c3", 4, 168, 168, "fdw"),
    ("mu/logvar_u_y_to_z.1", 1.2, "c3", 4, 1696, 848, "w"),
    ("mu/logvar_u_y_to_z.2", 1.2, "c3", 4, 848, 848, "w"),
    ("decoder_x.1.upsample", 1.2, "ct", 8, 424, 256, "fw"),
    ("decoder_x.1.conv", 1.2, "c3", 8, 424, 424, "fdw"),
    ("encoder_x.6", 1.2, "c3", 8, 128, 424, "dw"),
    ("y_to_z.4", 1.2, "c3", 4, 128, 848, "w"),
]


def st():
    return torch.cuda.current_stream().cuda_stream


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def _median(v):
    return sorted(v)[len(v) // 2]


def time_steps(steps, rounds):
    import models
    from svrs_native.trainer import FusedCondTrainer
    runs = {}
    g = torch.Generator().manual_seed(11)
    x = torch.rand(B, 4, P, P, generator=g).cuda()
    y = torch.nn.functional.avg_pool2d(x, 2)
    for cr in RATIOS:
        torch.manual_seed(0)
        m = models.Cond_SRVAE(cr, P).cuda().train()
        m.set_compute_dtype(torch.bfloat16)
        tr = FusedCondTrainer(m)
        tr.eng.rng.seed = 5
        for _ in range(5):
            tr.step(x, y, use_graph=True)
        torch.cuda.synchronize()
        fl = sum(2 * B * oh * oh * k * ci * co for oh, k, ci, co in _conv_shapes(m)) * 3
        runs[cr] = dict(tr=tr, ms=[], gflop=fl / 1e9)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for cr in RATIOS:
            tr = runs[cr]["tr"]
            e0.record()
            for _ in range(steps):
                loss = tr.step(x, y, use_graph=True)
            e1.record()
            torch.cuda.synchronize()
            runs[cr]["ms"].append(e0.elapsed_time(e1) / steps)
            assert torch.isfinite(loss).all(), f"cr {cr}: non-finite loss"
    out = {}
    for cr in RATIOS:
        t = _median(runs[cr]["ms"])
        out[cr] = dict(ms_per_step=round(t, 4), patches_per_s=round(B / t * 1e3, 1), train_gflop_per_step=round(runs[cr]["gflop"], 1),
                       spread_ms=[round(min(runs[cr]["ms"]), 4), round(max(runs[cr]["ms"]), 4)])
    base = out[2]
    for cr in RATIOS:
        out[cr]["time_ratio_vs_cr2"] = round(out[cr]["ms_per_step"] / base["ms_per_step"], 3)
        out[cr]["flop_ratio_vs_cr2"] = round(out[cr]["train_gflop_per_step"] / base["train_gflop_per_step"], 3)
    return out


def _conv_shapes(model):
    """(output H, taps, Cin, Cout) of every conv of the model at patch size P."""
    from svrs_native.engine import ConvOp
    eng = model._engine()
    shapes = eng.conv_input_shapes(1)
    res = []
    for net in eng.nets.values():
        for op in net.ops:
            if isinstance(op, ConvOp):
                _, h, _ = shapes[id(op)]
                oh, taps = (h, 9) if op.kind == "c3" else ((h // 2, 16) if op.kind == "c4" else (2 * h, 4))
                res.append((oh, taps, op.cin, op.cout))
    return res


def _layer_graph(form, H, Cin, Cout, passes, tc, reps):
    g = torch.Generator().manual_seed(H + Cin + Cout)
    OH = 2 * H if form == "ct" else H
    x = torch.randn(B, H, H, Cin, generator=g).to(torch.bfloat16).cuda()
    dy = torch.randn(B, OH, OH, Cout, generator=g).to(torch.bfloat16).cuda()
    wshape = (Cin, Cout, 4, 4) if form == "ct" else (Cout, Cin, 3, 3)
    w = (torch.randn(wshape, generator=g) * 0.05).cuda()
    kk = wshape[2] * wshape[3]
    p01 = torch.empty(w.numel(), device="cuda", dtype=torch.bfloat16)
    p10 = torch.empty_like(p01)
    lib.pack_weights(w.data_ptr(), wshape[0], wshape[1], kk, p01.data_ptr(), p10.data_ptr(), BF16, st())
    pf, pb = (p01, p10) if form == "ct" else (p10, p01)
    bias = torch.zeros(Cout, device="cuda")
    y = torch.empty(B, OH, OH, Cout, device="cuda", dtype=torch.bfloat16)
    dx = torch.empty_like(x)
    dw = torch.zeros(w.numel(), device="cuda")
    db = torch.zeros(Cout, device="cuda")
    ops = []
    if form == "ct":
        if "f" in passes:
            ops.append(lambda: lib.convT2d_fprop(x.data_ptr(), pf.data_ptr(), pb.data_ptr(), bias.data_ptr(), y.data_ptr(), BF16, B, H, H, Cin, Cout, 0, st()))
        if "d" in passes:
            ops.append(lambda: lib.convT2d_dgrad(dy.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), BF16, B, H, H, Cin, Cout, st()))
        if "w" in passes:
            ops.append(lambda: lib.convT2d_wgrad(x.data_ptr(), dy.data_ptr(), dw.data_ptr(), dw.data_ptr(), db.data_ptr(), BF16, B, H, H, Cin, Cout, 0, st()))
    else:
        if "f" in passes:
            ops.append(lambda: lib.conv2d_fprop(x.data_ptr(), pf.data_ptr(), pb.data_ptr(), bias.data_ptr(), y.data_ptr(), BF16, B, H, H, Cin, Cout, 3, 0, st()))
        if "d" in passes:
            ops.append(lambda: lib.conv2d_dgrad(dy.data_ptr(), pb.data_ptr(), pf.data_ptr(), dx.data_ptr(), BF16, B, H, H, Cin, Cout, 3, st()))
        if "w" in passes:
            ops.append(lambda: lib.conv2d_wgrad(x.data_ptr(), dy.data_ptr(), dw.data_ptr(), dw.data_ptr(), db.data_ptr(), BF16, B, H, H, Cin, Cout, 3, 0, st()))
    graphs = []
    lib.set_tc_enabled(tc)
    try:
        for op in ops:
            for _ in range(2):
                op()
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                for _ in range(reps):
                    op()
            gr.replay()
            graphs.append(gr)
        torch.cuda.synchronize()
    finally:
        lib.set_tc_enabled(1)
    return graphs, (x, dy, w, p01, p10, bias, y, dx, dw, db)


def time_layers(reps, rounds):
    rows = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, cr, form, H, Cin, Cout, passes in LAYERS:
        variants = [_layer_graph(form, H, Cin, Cout, passes, tc, reps) for tc in (1, 0)]
        OH = 2 * H if form == "ct" else H
        fl = 2 * B * OH * OH * (4 if form == "ct" else 9) * Cin * Cout
        for i, ps in enumerate(passes):
            ts = [[], []]
            for _ in range(rounds):
                for v in (0, 1):
                    e0.record()
                    variants[v][0][i].replay()
                    e1.record()
                    torch.cuda.synchronize()
                    ts[v].append(e0.elapsed_time(e1) * 1e3 / reps)
            t_tc, t_core = _median(ts[0]), _median(ts[1])
            rows.append(dict(layer=name, cr=cr, form=form, map=H, cin=Cin, cout=Cout, pass_=ps, gflop=round(fl / 1e9, 2),
                             us_tcgen05=round(t_tc, 1), us_cuda_cores=round(t_core, 1), speedup=round(t_core / t_tc, 2),
                             tflops_tcgen05=round(fl / t_tc / 1e6, 1)))
            r = rows[-1]
            print(f"{name:22s} cr {cr:<3} {form} {H}x{H} {Cin:5d}->{Cout:<5d} {ps} {r['gflop']:6.2f} GF | tcgen05 {t_tc:8.1f} us "
                  f"({r['tflops_tcgen05']:6.1f} TF/s) | CUDA cores {t_core:9.1f} us | x{r['speedup']:.2f}", flush=True)
        del variants
        torch.cuda.empty_cache()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="graph-replayed steps per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="timed windows per ratio (interleaved), or alternating replays per layer")
    ap.add_argument("--reps", type=int, default=20, help="launches per per-layer graph")
    ap.add_argument("--no-layers", action="store_true")
    ap.add_argument("--no-steps", action="store_true")
    ap.add_argument("--json", type=str, default=None, help="also write the results to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cr_bench: no CUDA device")
    lib.load()
    res = dict(gpu=gpu_info())
    print(f"# {res['gpu']}")
    if not a.no_steps:
        res["steps"] = time_steps(a.steps, a.rounds)
        for cr, r in res["steps"].items():
            print(f"cr {cr:<3}: {r['ms_per_step']:.3f} ms/step  {r['patches_per_s']:.0f} patches/s  "
                  f"({r['train_gflop_per_step']:.0f} GFLOP, time x{r['time_ratio_vs_cr2']:.3f} / FLOP x{r['flop_ratio_vs_cr2']:.3f} "
                  f"of cr 2, spread {r['spread_ms'][0]:.3f}-{r['spread_ms'][1]:.3f})", flush=True)
    if not a.no_layers:
        res["layers"] = time_layers(a.reps, a.rounds)
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
