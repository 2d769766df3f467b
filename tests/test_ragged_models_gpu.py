"""Cond_SRVAE at the reference's own compression ratios (cr 1.5: train.py's default and test.sh; cr 1.2: the CondVAE
production run) in bf16, now that their 168 / 336 / 424 / 672 / 848 / 1344 / 1696-channel layers run on tcgen05 (-m gpu).

Against the CPU oracle on the same weights, inputs and eps, with the bounds tests/test_parity_configs_gpu.py asserts for
config 3: NLL terms and loss 1e-4, KL terms 1e-3, gradient norm 2e-3, decoder images 4e-3 / 1e-3 and heads 3e-2 / 3e-2
(relative to the maximum / relative L2).

Parameter gradients are read from the flat buffer the fused optimiser reads, in the layout the weight-gradient kernel left
them (per-tap packed for the tcgen05 layers), and bounded at 0.3 relative L2: twice the worst figure measured on a B200
(0.158, the BatchNorm of y_to_z.0; the decoders' 0.08-0.10 is the same on layers whose kernels did not change, e.g.
decoder_x.2 and the CUDA-core decoder_y.1).  bf16 operands through the whole backward chain at a batch of 2 put these
gradients 1e-2 to 1.6e-1 away from fp32; a gradient read in the wrong layout or with a lost channel chunk is off by O(1).
The kernels themselves are checked against fp64 in tests/test_conv_ragged_channels_gpu.py."""
import pytest
import torch

import fixtures as FX
from helpers import BF16, lib
from oracle import ref_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
NAMES8 = ["x_hat", "y_hat", "mu_z", "logvar_z", "mu_u", "logvar_u", "mu_z_uy", "logvar_z_uy"]
ACT_TOL = {"image": (4e-3, 1e-3), "latent": (3e-2, 3e-2)}
TERM_TOL = dict(nll=1e-4, kl=1e-3, gn=2e-3)
GRAD_TOL = (float("inf"), 0.3)      # (rel-to-max: printed only, rel-L2)
ZERO_GRAD_BIAS = ("downsample.bias", "upsample.bias")     # true gradient 0 (conv bias feeding BatchNorm)
CUDA_CORE_CONV = ("conv_taps_kernel", "wgrad_taps_kernel", "wgrad_direct_kernel")


def _gam2():
    return {"gammax": torch.tensor(1.0), "gammay": torch.tensor(1.0)}


def _errs(name, got, ref, tol):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    assert torch.isfinite(got).all(), name
    e = got - ref
    rmax = float(e.abs().max() / (ref.abs().max() + 1e-30))
    rl2 = float(e.norm() / (ref.norm() + 1e-30))
    print(f"[ragged-bf16] {name}: rel-to-max {rmax:.3e} (tol {tol[0]:.1e})  rel-L2 {rl2:.3e} (tol {tol[1]:.1e})")
    return [] if (rmax <= tol[0] and rl2 <= tol[1]) else [(name, rmax, rl2)]


def _term(name, got, ref, tol):
    got, ref = float(got), float(ref)
    rel = abs(got - ref) / max(abs(ref), 1e-30)
    print(f"[ragged-bf16] {name}: cuda {got:.6f} oracle {ref:.6f} rel {rel:.3e} (tol {tol:.1e})")
    return [] if (got == got and rel <= tol) else [(name, got, ref, rel)]


def _problem(which, golden_dir):
    """-> (model, sd, cr, P, x, y, eu, ez): the cr 1.5 golden fixture, or a cr 1.2 model and inputs from seeds."""
    if which == "cr1p5":
        fx = FX.load(golden_dir, "cond_cr1p5_p64_b2")
        model, sd = FX.build(fx, device=DEV, dtype=torch.bfloat16)
        x, y = FX.inputs(fx)
        eu, ez = fx["eps"]
        return model, sd, fx["cr"], fx["P"], x, y, eu, ez
    cr, P, B = 1.2, 64, 2
    model, sd = FX.build("cond", cr, P, seed=14, device=DEV, dtype=torch.bfloat16)
    eng = model._engine()
    r = O.PortableRng(24)
    x = r.rand(B, 4, P, P)
    y = torch.nn.functional.avg_pool2d(x, 2)
    eu, ez = r.randn(B, eng.Wu), r.randn(B, eng.Wz)
    return model, sd, cr, P, x, y, eu, ez


def _torch_layout_grads(tr, model, batch):
    """Per-parameter gradients of the last fused step, read from the flat gradient the optimiser read: conv / convT weights
    whose weight-gradient kernel reports layout 1 hold the per-tap packed [tap][d1][d0] there."""
    from svrs_native.engine import ConvOp
    rt = tr.eng.rt
    store = rt.store
    flat = tr.last_grad
    shapes = tr.eng.conv_input_shapes(batch)
    layout = {}
    for net in rt.nets:
        for op in net.ops:
            if isinstance(op, ConvOp):
                n, h, w = shapes[id(op)]
                if op.kind == "ct":
                    layout[id(op.mod.weight)] = lib.convT2d_wgrad_layout(BF16, n, h, w, op.cin, op.cout)
                else:
                    layout[id(op.mod.weight)] = lib.conv2d_wgrad_layout(BF16, n, h, w, op.cin, op.cout, 3 if op.kind == "c3" else 4)
    out = {}
    for k, p in model.named_parameters():
        if id(p) not in store._index:
            continue
        off = store.offsets[store._index[id(p)]]
        g = flat[off:off + p.numel()]
        if layout.get(id(p), 0) == 1:
            d0, d1, kk = p.shape[0], p.shape[1], p.shape[2] * p.shape[3]
            g = g.view(kk, d1, d0).permute(2, 1, 0).reshape(p.shape)
        out[k] = g.view(p.shape).detach().cpu()
    return out


@pytest.mark.parametrize("which", ["cr1p5", "cr1p2"])
def test_bf16_forward_elbo_gradients_vs_oracle(golden_dir, which):
    from svrs_native.trainer import FusedCondTrainer
    model, sd, cr, P, x, y, eu, ez = _problem(which, golden_dir)
    B = x.shape[0]
    osd = {k: v.clone() for k, v in sd.items()}
    terms_o, outs_o, grads_o = O.cond_train_step(osd, _gam2(), O.AdamState(), cr, P, x, y, eu, ez, return_grads=True)
    bad = []
    model.train()
    with torch.no_grad():
        outs = model(x.to(DEV), y.to(DEV), eu.to(DEV), ez.to(DEV))
    for n, got, ref in zip(NAMES8, outs, outs_o):
        bad += _errs(f"{which} fwd {n}", got, ref, ACT_TOL["image" if n in ("x_hat", "y_hat") else "latent"])
    model2, _ = _problem(which, golden_dir)[:2]
    model2.train()
    tr = FusedCondTrainer(model2)
    tr.keep_grad = True
    t = tr.step(x.to(DEV), y.to(DEV), eu.to(DEV), ez.to(DEV)).cpu()
    for i, k in enumerate(["mse_x", "kld_u", "mse_y", "kld_z", "loss"]):
        bad += _term(f"{which} {k}", t[i], terms_o[k], TERM_TOL["kl"] if k.startswith("kld") else TERM_TOL["nll"])
    bad += _term(f"{which} grad norm", tr.grad_norm(), terms_o["grad_norm"], TERM_TOL["gn"])
    grads = _torch_layout_grads(tr, model2, B)
    n = 0
    for k, g in grads.items():
        if k.endswith(ZERO_GRAD_BIAS) or k not in grads_o:
            continue
        bad += _errs(f"{which} grad {k}", g, grads_o[k], GRAD_TOL)
        n += 1
    assert n > 50
    assert not bad, bad


def test_fused_steps_cr1p5_vs_oracle(golden_dir):
    """Three FusedCondTrainer steps (fused clip + Adam reading the packed gradients of the ragged layers) against the
    oracle's Adam steps on the same eps: ELBO terms and gradient norm of every step, which depend on the updated weights."""
    from svrs_native.trainer import FusedCondTrainer
    model, sd, cr, P, x, y, eu, ez = _problem("cr1p5", golden_dir)
    B = x.shape[0]
    eng = model._engine()
    r = O.PortableRng(31)
    eps = [(eu, ez)] + [(r.randn(B, eng.Wu), r.randn(B, eng.Wz)) for _ in range(2)]
    osd = {k: v.clone() for k, v in sd.items()}
    ogam, oopt = _gam2(), O.AdamState()
    model.train()
    tr = FusedCondTrainer(model)
    bad = []
    for it, (u, z) in enumerate(eps):
        t = tr.step(x.to(DEV), y.to(DEV), u.to(DEV), z.to(DEV)).cpu()
        to = O.cond_train_step(osd, ogam, oopt, cr, P, x, y, u, z)
        for i, k in enumerate(["mse_x", "kld_u", "mse_y", "kld_z", "loss"]):
            bad += _term(f"step {it} {k}", t[i], to[k], TERM_TOL["kl"] if k.startswith("kld") else TERM_TOL["nll"])
        bad += _term(f"step {it} grad norm", tr.grad_norm(), to["grad_norm"], TERM_TOL["gn"])
    assert not bad, bad


def _conv_calls(model, B, seed):
    """Run one eager fused training step with every C-ABI call recorded -> [(entry point, (H, W, Cin, Cout), kernels)]."""
    from svrs_native.trainer import FusedCondTrainer
    P = model.patch_size
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 4, P, P, generator=g).to(DEV)
    y = torch.nn.functional.avg_pool2d(x, 2)
    model.train()
    tr = FusedCondTrainer(model)
    tr.step(x, y)                       # first step: plans, packs, job tables
    torch.cuda.synchronize()
    lib.timing = []
    try:
        tr.step(x, y)
        torch.cuda.synchronize()
        rec = lib.timing
    finally:
        lib.timing = None
    out = []
    for name, args, _e0, _e1, kernels in rec:
        if "conv" not in name:
            continue
        names = [a for _t, a in lib.protos[name][1]]
        a = dict(zip(names, args))
        out.append((name, (a["H"], a["W"], a["Cin"], a["Cout"]), tuple(k for k in kernels.split(",") if k)))
    return out


def test_cr1p5_step_trace_cuda_core_convs():
    """In a fused bf16 cr 1.5 step the CUDA-core conv kernels serve only encoder_y's 128 -> 84 conv and decoder_y's 42 ->
    42 / 42 -> 128 block (channel counts without 16-byte rows), plus the launches a cr 2 step also makes."""
    import models
    B = 128
    calls = {}
    for cr in (2, 1.5):
        m = models.Cond_SRVAE(cr, 64).to(DEV)
        m.set_compute_dtype(torch.bfloat16)
        calls[cr] = _conv_calls(m, B, 5)
    core = {cr: {(n, shp) for n, shp, ks in c if any(k in CUDA_CORE_CONV for k in ks)} for cr, c in calls.items()}
    for cr in (2, 1.5):
        print(f"[trace] cr {cr}: {len(calls[cr])} conv calls, on CUDA cores: {sorted(core[cr])}")
    assert any(k == "conv_tc_kernel" for _n, _s, ks in calls[1.5] for k in ks)
    extra = {(n, shp) for n, shp in core[1.5] - core[2] if not ({42, 84} & {shp[2], shp[3]})}
    assert not extra, f"CUDA-core conv kernels for layers with 16-byte rows: {sorted(extra)}"
    narrow = {(n, shp) for n, shp in core[1.5] if {42, 84} & {shp[2], shp[3]}}
    assert narrow, "expected the 42 / 84-channel layers on the CUDA-core kernels"
