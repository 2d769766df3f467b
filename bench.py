#!/usr/bin/env python
"""bench.py - headline benchmark: train patches/sec of the 64x64 SR CondVAE step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--workload cond_grid|cond_grid1024|vae|cond256|sample] [--dump-outputs DIR]

Default workload at every N (weak scaling): BASELINE.json config 3 - CondVAE cr=2, P=64, grid mode: 8 synthetic 256x256
multispectral tiles per GPU -> 128 patches per GPU (64 tiles / 1024 patches at N=8), bf16 compute, fp32 master
weights, gradients SUM-all-reduced over NCCL.  One "step" = grid-patch gather + normalise, forward, ELBO, backward,
clip, Adam (the reference's models/base.py:103-107 body preceded by its dataset.py grid mode).
Other BASELINE configs are selectable with --workload (config 2 `vae`, config 3 on ONE GPU `cond_grid1024`, config 4
`cond256` = P=256 cr=16, config 5 `sample` = 32 posterior samples per LR patch).

Prints ONE JSON line (rank 0).  `value` = device-timed whole-job units/s with tiles resident in HBM;
`e2e` = the same through the public API with HOST (pinned) tile buffers: H2D copy of every step's tiles and a D2H read
of the loss inside the timed region.  `--impl reference` times the CPU restatement of the reference (oracle/) on the
host cores on a bounded sample of the same workload (same per-step batch).  Outside the timed regions the default line
also carries `roofline` (dominant kernel), `roofline_hbm` (the bandwidth-bound kernels at the bench batch),
`cpu_baseline`, `gpu_reference` (the reference's torch ops under cuDNN on the same GPU) and, for N > 1, `ddp_check`.

`--dump-outputs DIR` writes what the last step of the device-timed region computed, as DIR/<name>.npy (rank 0):
`loss_terms` (the tensor the step returns), `gammas` and `params_sample` (the updated weights: a fixed PCG64 sample of
the fp32 parameter store) for the training workloads, `std` (the posterior std maps) for `sample`.  Inputs, weights and
noise are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "simple-vae-rs_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# ---- workloads (BASELINE.json configs 2-5).  flop = algorithmic FLOPs per unit of one optimisation step / sample
# (SURVEY 8.4 row d, BASELINE.md section 4)
WORKLOADS = {
    "cond_grid": dict(model="cond", cr=2, P=64, tiles=8, S=256, flop=8.13e9, unit="patches/s",
                      metric="train patches/sec (64x64 SR CondVAE, device-timed)",
                      name="CondVAE cr=2 P=64 grid mode: 8 tiles (256x256x4) -> 128 patches per GPU"),
    "cond_grid1024": dict(model="cond", cr=2, P=64, tiles=64, S=256, flop=8.13e9, unit="patches/s",
                          metric="train patches/sec (64x64 SR CondVAE, device-timed)",
                          name="CondVAE cr=2 P=64 grid mode: 64 tiles (256x256x4) -> 1024 patches per GPU (config 3 on one GPU)"),
    "vae": dict(model="vae", cr=2, P=64, tiles=16, S=256, flop=4.44e9, unit="patches/s",
                metric="train patches/sec (64x64 VAE, device-timed)",
                name="VAE cr=2 P=64, 16 tiles -> 256 patches per GPU (config 2)"),
    "cond256": dict(model="cond", cr=16, P=256, tiles=16, S=256, flop=222e9, unit="crops/s",
                    metric="train crops/sec (256x256 SR CondVAE cr=16, device-timed)",
                    name="CondVAE cr=16 P=256 full 256x256 crops, 16 crops per GPU (config 4: 128 crops at 8 GPUs)"),
    "sample": dict(model="cond", cr=2, P=64, tiles=1, S=256, flop=1.752e9, unit="samples/s",
                   metric="posterior samples/sec (CondVAE sample(), 32 per LR patch, device-timed)",
                   name="CondVAE cr=2 P=64 inference: 1 LR tile -> 16 patches x 32 posterior samples per step (config 5)"),
}
SAMPLES_PER_PATCH = 32
DUMP_PARAMS = 1 << 22       # weights written by --dump-outputs: 16 MB of fp32, well inside the dump's 64 MB


def timed_step_outputs(out, tr):
    """Host copies of what the last timed step computed: the step's return value and, for a training step (`tr` given),
    the loss weights and a fixed sample of the updated fp32 parameter store."""
    def host(t):
        a = t.detach().cpu()
        return (a if a.dtype in (torch.float32, torch.float64) else a.float()).numpy()

    if tr is None:
        return {"std": host(out)}
    flat = tr.rt.store.flat
    if flat.numel() > DUMP_PARAMS:
        # numpy's PCG64 draws the same indices on every host
        idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_PARAMS, replace=False))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    return {"loss_terms": host(out), "gammas": host(tr.gam[:tr.n_gammas]), "params_sample": host(flat)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# reference arms (the oracle's restatement of the reference's call sequence; same ATen kernels as the reference)
# ------------------------------------------------------------------------------------------------------------------
def _oracle_problem(wl, batch, device="cpu"):
    """Weights (reference constructor under torch.manual_seed(0)), inputs and a step closure factory for the oracle."""
    from oracle import ref_oracle as O
    import models
    cr, P = wl["cr"], wl["P"]
    torch.manual_seed(0)
    m = models.VAE(cr, P) if wl["model"] == "vae" else models.Cond_SRVAE(cr, P)
    sd = {k: v.detach().clone().to(device) for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(1)
    x = torch.rand(batch, 4, P, P, generator=g).to(device)
    y = torch.rand(batch, 4, P // 2, P // 2, generator=g).to(device)
    if wl["model"] == "vae":
        Wd = (m.latent_size // 64) * (P // 4) ** 2
        widths = (Wd,)
    else:
        widths = ((m.latent_size_y // 64) * (P // 8) ** 2, (m.latent_size // 64) * (P // 8) ** 2)
    return O, sd, x, y, widths


def cpu_reference_arm(args, wl, batch, steps, warmup):
    """The reference's CPU implementation of the step (oracle restatement, fp32), all host threads, on `batch` patches
    per step - the SAME per-step batch as one GPU of the b200 arm."""
    torch.set_num_threads(os.cpu_count())
    O, sd, x, y, widths = _oracle_problem(wl, batch)
    opt = O.AdamState()
    cr, P = wl["cr"], wl["P"]
    if wl["model"] == "vae":
        gam = {"gamma": torch.tensor(1.0)}
        fn = lambda: O.vae_train_step(sd, gam, opt, cr, P, x, torch.randn(batch, widths[0]))
    elif args.workload == "sample":
        S = SAMPLES_PER_PATCH
        fn = lambda: [O.cond_sample(sd, cr, P, y[i:i + 1], torch.randn(1, widths[0]), torch.randn(S, widths[1]))
                      for i in range(batch)]
    else:
        gam = {"gammax": torch.tensor(1.0), "gammay": torch.tensor(1.0)}
        fn = lambda: O.cond_train_step(sd, gam, opt, cr, P, x, y, torch.randn(batch, widths[0]), torch.randn(batch, widths[1]))
    with torch.no_grad() if args.workload == "sample" else torch.enable_grad():
        for _ in range(warmup):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        dt = (time.perf_counter() - t0) / steps
    units = batch * (SAMPLES_PER_PATCH if args.workload == "sample" else 1)
    return dict(value=units / dt, ms=dt * 1e3, cores=os.cpu_count(), steps=steps,
                sample=f"{steps} steps x batch {batch} per step (= one GPU's share of the workload), fp32, torch CPU ops, "
                       f"{os.cpu_count()} threads")


def gpu_reference_arm(wl, batch, dev, steps=10):
    """THE BAR (SURVEY 2.1 / BASELINE.md section 5): the reference's own torch call sequence (oracle restatement ->
    F.conv2d / F.conv_transpose2d / F.batch_norm / autograd / clip_grad_norm_ / torch.optim.Adam) on the same B200,
    i.e. cuDNN/cuBLAS kernels: fp32 with TF32 convs (torch default) and autocast(bf16) + channels_last, each eager and
    as a whole-step CUDA graph.  Device-timed with CUDA events; not part of the timed regions of this repo's arm."""
    from oracle import ref_oracle as O
    cr, P = wl["cr"], wl["P"]
    _, sd0, x, y, widths = _oracle_problem(wl, batch, dev)
    out = {}

    def build(bf16):
        sd = {k: v.clone() for k, v in sd0.items()}
        pk = O.param_keys(sd)
        params = {k: torch.nn.Parameter(sd[k].to(memory_format=torch.channels_last) if (bf16 and sd[k].dim() == 4) else sd[k])
                  for k in pk}
        work = dict(sd)
        work.update(params)
        gam = [torch.nn.Parameter(torch.tensor(1.0, device=dev)) for _ in range(1 if wl["model"] == "vae" else 2)]
        opt = torch.optim.Adam([{"params": list(params.values())}, {"params": gam}], lr=1e-4, capturable=True)
        xi = x.to(memory_format=torch.channels_last) if bf16 else x
        yi = y.to(memory_format=torch.channels_last) if bf16 else y
        eps = [torch.randn(batch, w, device=dev) for w in widths]

        def step():
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
                if wl["model"] == "vae":
                    x_hat, mu, lv = O.vae_forward(work, cr, P, xi, eps[0], training=True)
                    terms = O.base_loss(x_hat.float(), x, mu.float(), lv.float(), gam[0])
                else:
                    o = O.cond_forward(work, cr, P, xi, yi, eps[0], eps[1], training=True)
                    x_hat, y_hat, mu_z, lv_z, mu_u, lv_u, mu3, lv3 = [t.float() for t in o]
                    terms = O.cond_loss(x_hat, x, y_hat, y, mu_u, lv_u, mu_z, lv_z, mu3, lv3, gam[0], gam[1])
            loss = sum(terms)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(list(params.values()), 1.0)
            opt.step()
            return loss
        return step

    def timeit(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    for name, bf16 in (("fp32_tf32", False), ("bf16_autocast_channels_last", True)):
        try:
            step = build(bf16)
            for _ in range(3):
                step()
            ms = timeit(step, steps)
            out[name + "_eager"] = {"ms_per_step": ms, "value": batch / (ms * 1e-3)}
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(3):
                    step()
            torch.cuda.current_stream().wait_stream(s)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step()
            g.replay()
            ms = timeit(g.replay, steps)
            out[name + "_cuda_graph"] = {"ms_per_step": ms, "value": batch / (ms * 1e-3)}
            del g
        except Exception as ex:  # keep whatever was measured
            out[name + "_error"] = repr(ex)[:300]
    best = max((v["value"] for v in out.values() if isinstance(v, dict)), default=None)
    return {"what": "reference call sequence as torch CUDA ops (cuDNN %s, torch %s) on this GPU, batch %d, device-timed over "
                    "%d steps" % (torch.backends.cudnn.version(), torch.__version__, batch, steps),
            "unit": wl["unit"], "variants": out, "best": best}


def patch_gather_bandwidth(dev, pk, tiles=64, reps=10):
    """The TMA patch gather + normalise (dataset.py:220-247,265-274 + utils.py:4-23) at BASELINE config 3's full tile batch
    (64 HR tiles 256x256x4 fp32 -> 1024 patches, fp32 NHWC + bf16 NHWC emitted): algorithmic bytes = tiles read once + both
    outputs written once; `reps` launches captured in one CUDA graph (no host launch gaps), CUDA-event timed."""
    from dataset import grid_patch_pair, synthetic_tiles
    _, hr = synthetic_tiles(tiles, 256, seed=7)
    hr = hr.to(dev)
    for _ in range(2):
        grid_patch_pair(hr, 64, torch.bfloat16)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            out = grid_patch_pair(hr, 64, torch.bfloat16)
    g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / reps * 1e3
    nbytes = hr.numel() * (4 + 4 + 2)
    return {"us_per_launch": round(us, 2), "launches": 1.0, "MB_per_launch": round(nbytes / 1e6, 3),
            "achieved": round(nbytes / us / 1e3, 1), "frac": round(nbytes / us / 1e3 / pk["hbm"], 3),
            "note": "64 tiles (config 3's whole tile batch), tiles larger than L2 together with the outputs: 168 MB per launch"}


def ddp_check(dev, rank, world, pg=None):
    """Hardware parity of the data-parallel step (printed by rank 0 under `ddp_check`): every rank runs ONE fp32 fused
    step on its own shard of a small global batch (sync_bn on, so BatchNorm sees the global batch); rank 0 then repeats
    the step single-process on the gathered global batch.  grad_rel_err = |g_ddp - g_single|_2 / |g_single|_2 on the
    all-reduced flat gradient; param_spread = max |p_rank - p_rank0| after the update."""
    import models
    from svrs_native.trainer import FusedCondTrainer
    B = 4
    res = {}
    g = torch.Generator().manual_seed(77)
    X = torch.rand(B * world, 4, 64, 64, generator=g).to(dev)
    Y = torch.rand(B * world, 4, 32, 32, generator=g).to(dev)
    eu_all, ez_all = None, None

    def fresh(sync_bn, w):
        torch.manual_seed(0)
        m = models.Cond_SRVAE(2, 64).to(dev).train()
        tr = FusedCondTrainer(m, sync_bn=sync_bn, process_group=pg if w > 1 else None, world_override=w)
        tr.eng.rng.seed = 99
        return m, tr

    m, tr = fresh(True, world)
    tr.eng.rng.sample_offset = rank * B
    tr.keep_grad = True
    tr.step(X[rank * B:(rank + 1) * B], Y[rank * B:(rank + 1) * B])
    g_ddp = tr.last_grad.clone()
    p_ddp = tr.rt.store.flat.clone()
    p0 = p_ddp.clone()
    torch.distributed.broadcast(p0, 0, group=pg)
    spread = (p_ddp - p0).abs().max()
    torch.distributed.all_reduce(spread, op=torch.distributed.ReduceOp.MAX, group=pg)
    res["param_spread"] = float(spread)
    # the overlapped exchange (early all-reduce of the decoders' range on the bounded, high-priority communicator) against
    # the single all-reduce after the backward pass: same shard, per-rank BatchNorm statistics, fp32
    g_ov = []
    for overlap in (True, False):
        mo, tro = fresh(False, world)
        tro.eng.rng.sample_offset = rank * B
        tro.keep_grad = True
        tro._ensure_state()
        tro._ar_overlap = overlap
        tro.step(X[rank * B:(rank + 1) * B], Y[rank * B:(rank + 1) * B])
        g_ov.append(tro.last_grad.clone())
    res["overlap_vs_plain_allreduce_grad_rel_err"] = float((g_ov[0] - g_ov[1]).norm() / g_ov[1].norm())
    if rank == 0:
        m1, tr1 = fresh(False, 1)
        tr1.keep_grad = True
        tr1.step(X, Y)
        g1 = tr1.last_grad
        res["grad_rel_err"] = float((g_ddp - g1).norm() / g1.norm())
        res["param_max_abs_diff_vs_single_process"] = float((p_ddp - tr1.rt.store.flat).abs().max())
        res["what"] = (f"fp32, {B} patches per rank x {world} ranks vs one process on the {B * world}-patch global batch; sync_bn; "
                       "SUM all-reduce with KL upstream gradients scaled 1/world")
    torch.distributed.barrier(group=pg)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", type=str, default="cond_grid", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", type=str, default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]
    P, S = wl["P"], wl["S"]
    per_tile = (S // P) ** 2
    per_gpu = wl["tiles"] * per_tile                     # patches (crops) per GPU and step
    units_per_gpu = per_gpu * (SAMPLES_PER_PATCH if args.workload == "sample" else 1)
    metric, unit = wl["metric"], wl["unit"]

    if args.impl == "reference":
        if rank != 0:
            return
        steps = max(1, min(args.steps, 20))
        warm = max(1, min(args.warmup, 2))
        if per_gpu >= 512 or args.workload == "cond256":   # keep the CPU arm within minutes
            steps, warm = min(steps, 3), 1
        r = cpu_reference_arm(args, wl, per_gpu, steps, warm)
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": r["value"], "unit": unit, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": wl["name"], "note": f"CPU arm: one GPU's share of the workload ({per_gpu} per step) on the host cores"},
            "cpu_baseline": {"value": r["value"], "unit": unit, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    import models
    from dataset import TilePrefetcher, grid_patch_pair, synthetic_tiles
    from svrs_native.trainer import FusedCondTrainer, FusedVaeTrainer

    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    torch.manual_seed(0)
    is_vae = wl["model"] == "vae"
    model = (models.VAE(wl["cr"], P) if is_vae else models.Cond_SRVAE(wl["cr"], P)).to(dev)
    model.set_compute_dtype(dtype)
    use_graph = not args.no_graph
    is_sample = args.workload == "sample"
    if is_sample:
        model.eval()
        eng = model._engine()
        eng.rng.seed = 2026
        rt = eng.rt
    else:
        model.train()
        tr = (FusedVaeTrainer if is_vae else FusedCondTrainer)(model)
        tr.eng.rng.seed = 2026
        tr.eng.rng.sample_offset = rank * per_gpu           # partition-invariant eps (SURVEY 8.4 row e iii)
        rt = tr.rt

    # synthetic tiles: a few distinct tile sets rotated across steps; pinned host copies for the e2e leg
    n_sets = 4 if wl["tiles"] <= 16 else 2
    host_sets = []
    for s in range(n_sets):
        lr, hr = synthetic_tiles(wl["tiles"], S, seed=100 + 17 * rank + s)
        host_sets.append((lr.pin_memory(), hr.pin_memory()))
    dev_sets = [(lr.to(dev), hr.to(dev)) for lr, hr in host_sets]
    h2d_bytes = sum(t.numel() * 4 for t in dev_sets[0])

    def step_from_device(lr, hr):
        """One step from device-resident tiles: grid-patch gather + normalise (dual emit: fp32 targets and the
        compute-dtype NHWC operands of the first conv layers), then the fused step / the sample decode."""
        if is_sample:
            if use_graph and sample_graph:
                sg = sample_graph[0]
                if sg["lr"].data_ptr() != lr.data_ptr():
                    sg["lr"].copy_(lr, non_blocking=True)
                rt.add_replayed(sg["launches"])
                sg["graph"].replay()
                return sg["out"]
            yb = grid_patch_pair(lr, P // 2, dtype, rt=rt)
            return eng.sample_stats_batch(yb, SAMPLES_PER_PATCH)
        if is_vae:
            return tr.step_tiles(hr, patch_size=P, use_graph=use_graph)
        return tr.step_tiles(hr, lr, patch_size=P, use_graph=use_graph)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---------------- warm-up
    sample_graph = []
    for i in range(args.warmup):
        step_from_device(*dev_sets[i % n_sets])
    if is_sample and use_graph:
        # the inference step (patch gather -> encoders -> prior -> S draws -> decoder -> streaming statistics) as one CUDA
        # graph, like the training step; the engine's device-side noise counter advances on every replay
        torch.cuda.synchronize()
        sg = {"lr": dev_sets[0][0].clone(), "graph": torch.cuda.CUDAGraph()}
        l0g = rt.launches
        with torch.cuda.graph(sg["graph"]):
            sg["out"] = eng.sample_stats_batch(grid_patch_pair(sg["lr"], P // 2, dtype, rt=rt), SAMPLES_PER_PATCH)
        sg["launches"] = rt.launches - l0g
        sample_graph.append(sg)
        for i in range(2):
            step_from_device(*dev_sets[i % n_sets])
    barrier()

    # ---------------- timed region 1: device-resident inputs (value)
    l0 = rt.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record()
        for i in range(args.steps):
            out = step_from_device(*dev_sets[i % n_sets])
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches = rt.launches - l0
    # taken before the e2e region steps the model on
    dump = timed_step_outputs(out, None if is_sample else tr) if args.dump_outputs and rank == 0 else None
    out_small = out if out.numel() <= 8 else out.flatten()[:5]
    last_loss = float(out_small.flatten()[-1])

    # ---------------- timed region 2: host buffers through the public API (e2e)
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d2h_elems = out.numel()
    loss_host = torch.empty(out.shape, dtype=out.dtype).pin_memory()
    # untimed warm-up of the host-fed path itself (copy stream, staging buffers, first asynchronous H2D / D2H): one fresh
    # box showed a ~40 ms one-off inside the first pass through the prefetcher
    for lr_d, hr_d in TilePrefetcher((host_sets[i % n_sets] for i in range(max(3, args.warmup))), dev):
        loss_host.copy_(step_from_device(lr_d, hr_d), non_blocking=True)
    barrier()
    e2.record()
    # the package's own feed (dataset.TilePrefetcher): pinned host tiles -> device on a copy stream, double-buffered, so the
    # H2D copy of step i+1 overlaps step i; every step's copy and the D2H of its result are inside the timed region
    feed = TilePrefetcher((host_sets[i % n_sets] for i in range(args.steps)), dev)
    for lr_d, hr_d in feed:
        out = step_from_device(lr_d, hr_d)
        loss_host.copy_(out, non_blocking=True)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    total_units = units_per_gpu * world * args.steps
    value = total_units / (ms * 1e-3)
    e2e_value = total_units / (ms_e2e * 1e-3)

    # ---------------- roofline of the dominant kernel family (eager, per-launch CUDA events; not in the timed region)
    pk = peaks()
    roof, roof_hbm = None, None
    if not args.no_profile:
        try:
            from svrs_native import profile as prof
            if is_sample:
                roof, roof_hbm = prof.dominant_kernel_roofline(None, None, pk, steps=2, rt=rt,
                                                               eager=lambda: step_from_device(*dev_sets[0]))
            else:
                roof, roof_hbm = prof.dominant_kernel_roofline(tr, dev_sets[0], pk, steps=2, dtype=dtype)
            roof_hbm["kernels"]["patch_gather_normalize_64_tiles"] = patch_gather_bandwidth(dev, pk)
            # DRAM bytes per launch of the same kernel from the committed `ncu --set full` capture (tools/ncu_traffic.py)
            for tname in ("traffic_r02.json", "traffic_r01.json"):
                tpath = os.path.join(ROOT, "profiles", tname)
                if os.path.exists(tpath):
                    tj = json.load(open(tpath))
                    if tj.get("kernel") and tj["kernel"] in roof.get("kernel", ""):
                        roof["traffic"] = tj["dram_bytes_per_launch"]
                        roof["traffic_source"] = f"profiles/{tname} (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)"
                        break
        except Exception as ex:  # keep the headline number even if the profiling pass fails
            roof = {"error": repr(ex)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_reference_arm(args, wl, min(per_gpu, 128) if args.workload != "cond256" else 2, 2, 1)
            cpu = {"value": r["value"], "unit": unit, "cores": r["cores"], "kind": "port", "sample": r["sample"]}
        except Exception as ex:
            cpu = {"error": repr(ex)}

    gref = None
    if rank == 0 and world == 1 and not args.no_gpu_reference and not is_sample:
        try:
            gref = gpu_reference_arm(wl, per_gpu, dev)
            if gref.get("best"):
                gref["this_repo_over_best_reference_variant"] = value / gref["best"]
        except Exception as ex:
            gref = {"error": repr(ex)[:300]}

    ddp = None
    if world > 1 and not is_sample and not is_vae and P == 64:
        try:
            ddp = ddp_check(dev, rank, world)
        except Exception as ex:
            ddp = {"error": repr(ex)[:300]}

    if rank == 0:
        line = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": wl["name"], "global_units_per_step": units_per_gpu * world, "parallelism": f"dp{world}",
                       "cuda_graph": use_graph,
                       "l2": f"inputs + activations + weights + Adam state per step far exceed the 126 MB L2 "
                             f"(~{6.24 * 3 * per_gpu * (P // 64) ** 2:.0f} MB of activations); {n_sets} tile sets rotated",
                       "tensor_roofline_units_per_s_per_gpu": pk["tf_sus"] * 1e12 / wl["flop"],
                       "frac_of_step_roofline": (value / world) / (pk["tf_sus"] * 1e12 / wl["flop"]),
                       "last_loss": last_loss},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_elems * out.element_size(), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "roofline": roof,
            "roofline_hbm": roof_hbm,
            "cpu_baseline": cpu,
            "gpu_reference": gref,
        }
        if ddp is not None:
            line["ddp_check"] = ddp
        if dump is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without tearing NCCL down: communicators captured inside CUDA graphs make destroy_process_group() hang
        # (observed at N=2).  Everything is synchronised and flushed, so a hard exit is safe.
        torch.cuda.synchronize()
        torch.distributed.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
