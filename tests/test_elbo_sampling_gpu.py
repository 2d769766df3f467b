"""Direct C-ABI tests (-m gpu) of the kernels between the conv stacks against fp64 references on the CPU:
svrs_elbo_fwd / _finalize / _bwd (csrc/elbo.cu) at the fused training step's own calls, and svrs_sample_latents /
svrs_sample_tail_stats (csrc/sample_stats.cu) of the `sample` workload.

Every reference is computed from exactly the values the kernel reads: inputs rounded to bf16 first where the kernel reads
bf16, and the fp32 recon r itself where the backward chains through r(1 - r).  Every output buffer sits inside a sentinel
guard band (helpers.Guarded), so a write outside it fails the test.

Bounds are derived next to each assert; u = 2^-24 is the fp32 unit roundoff, and CUDA's expf and logf are within 2 and
1 ulp (one ulp is at most 2u relative).  The bounds of the sample_tail_stats maps (TAIL_TOL) are not derived: each is at
most 2x the worst error measured.

Measured on an NVIDIA B200 (power limit 1000 W), worst error as a fraction of its derived bound:
  ELBO sums (acc) 0.045; finalize from the kernel's acc 0.46, end to end 0.20;
  d_recon fp32 0.45; d_mu1 below 0.001; d_lv1 0.30; d_mu2 / d_mu3 0.32; d_lv2 0.55; d_lv3 0.44; d_gammas 0.13;
  d_recon bf16: never more than 1 ulp from bf16(ref), bit-equal on at least 99.9989 % of the elements;
  sample_latents z half 0.49.
sample_tail_stats, worst error relative to the map's maximum (both dtypes): mean 3.9e-7, std 2.3e-7, mae 6.0e-7,
mse 5.9e-7, bias 5.0e-6, sample0 3.4e-7."""
import functools
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import BF16, F32, Guarded, lib, pack, st, task_stats
from oracle import ref_oracle as O
from svrs_native.lib import ACT_NONE, ACT_SIGMOID, SvrsError, SvrsUnsupported

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24
TORCH_DT = {F32: torch.float32, BF16: torch.bfloat16}


@functools.lru_cache(maxsize=None)
def _widths():
    """(Wz, Wu) of Cond_SRVAE(2, 64) and Wd of VAE(2, 64): the latent widths of the benchmarked models."""
    import models
    cond = models.Cond_SRVAE(2, 64)._engine()
    return cond.Wz, cond.Wu, models.VAE(2, 64)._engine().Wd


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _within(name, got, ref, bound):
    """|got - ref| <= bound element by element (bound: fp64 tensor of ref's shape)."""
    got = got.detach().double().cpu().reshape(ref.shape)
    err = (got - ref).abs()
    ratio = float((err / bound.clamp_min(1e-300)).max()) if err.numel() else 0.0
    print(f"[elbo/sample] {name}: max|err| {float(err.max()):.3e}  worst err/bound {ratio:.3f}")
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    assert ratio <= 1.0, f"{name}: error exceeds its bound by {ratio:.3f}x (max|err| {float(err.max()):.3e})"


def _bf16_ulp_check(name, got, ref):
    """bf16 output: at most one bf16 ulp from bf16(ref) everywhere and bit-equal to it on >= 99.9 % of the elements.
    The fp32 value before the final rounding is within 8u of ref, so the rounding can only differ from bf16(ref) where ref
    lies within 8u of a rounding boundary: a fraction of about 2 * 8u / 2^-8 = 2^-12 of the elements."""
    got = got.detach().cpu().reshape(ref.shape)
    rb = ref.float().to(torch.bfloat16)
    diff = (got.double() - rb.double()).abs()
    mag = torch.maximum(got.double().abs(), rb.double().abs()).clamp_min(1e-30)
    ulp = torch.exp2(torch.floor(torch.log2(mag)) - 7)
    equal = float((got == rb).double().mean())
    print(f"[elbo/sample] {name}: bit-equal to bf16(ref) {100 * equal:.4f} %, max diff/ulp {float((diff / ulp).max()):.2f}")
    assert bool((diff <= ulp).all()), f"{name}: more than one bf16 ulp from bf16(ref)"
    assert equal >= 0.999, f"{name}: only {100 * equal:.3f} % bit-equal"


# ------------------------------------------------------------------------------------------------ ELBO: inputs
def _latent(g, B, W, regime):
    """(mu, logvar) fp32 [B, W].  'init': both ~ N(0, 0.1^2), where exp(l) - 1 - l cancels in fp32; 'wide': mu ~ N(0, 1) and
    logvar uniform over the Hardtanh range [-7, 7]."""
    if regime == "init":
        return 0.1 * torch.randn(B, W, generator=g), 0.1 * torch.randn(B, W, generator=g)
    return torch.randn(B, W, generator=g), 14 * torch.rand(B, W, generator=g) - 7


class _Elbo:
    """The operands of one svrs_elbo_fwd / _bwd call on the device, and the fp64 values the kernels read.
    halves=True lays the latents out as the fused step does: mu1 / lv1 and mu2 / lv2 are the two halves of enc_u [B, 2 W1]
    and enc_z [B, 2 W2] (row stride 2W), mu3 / lv3 contiguous.  Otherwise every latent has its own buffer with row stride
    W + pad (W + pad + 4 for mu3 / lv3), and the padding columns hold NaN, which poisons any sum that reads them."""

    def __init__(self, seed, B, nx=0, ny=0, dts=(F32, F32, F32, F32), W1=0, W2=0, halves=False, pad=0, regime="init"):
        g = torch.Generator().manual_seed(seed)
        self.B, self.nx, self.ny, self.W1, self.W2 = B, nx, ny, W1, W2
        self.dtx, self.dttx, self.dty, self.dtty = dts
        self.keep = []
        self.img = {}
        for k, n, dr, dtt in (("x", nx, self.dtx, self.dttx), ("y", ny, self.dty, self.dtty)):
            if n:
                r = torch.rand(n, generator=g).to(TORCH_DT[dr])
                t = torch.rand(n, generator=g).to(TORCH_DT[dtt])
                rd, td = r.to(DEV), t.to(DEV)
                self.keep += [rd, td]
                self.img[k] = (rd.data_ptr(), td.data_ptr(), r.double(), t.double())
        self.lat = {}       # name -> (device pointer, row stride, fp64 [B, W] values)
        if W1:
            self._pair(g, "1", W1, regime, halves, W1 + pad)
        if W2:
            self._pair(g, "2", W2, regime, halves, W2 + pad)
            self._pair(g, "3", W2, regime, False, W2 if halves else W2 + pad + 4)

    def _pair(self, g, k, W, regime, halves, ld):
        mu, lv = _latent(g, self.B, W, regime)
        if halves:
            enc = torch.cat([mu, lv], dim=1).to(DEV)
            self.keep.append(enc)
            self.lat["mu" + k] = (enc.data_ptr(), 2 * W, mu.double())
            self.lat["lv" + k] = (enc.data_ptr() + 4 * W, 2 * W, lv.double())
            return
        for name, v in (("mu" + k, mu), ("lv" + k, lv)):
            buf = torch.full((self.B, ld), float("nan"))
            buf[:, :W] = v
            buf = buf.to(DEV)
            self.keep.append(buf)
            self.lat[name] = (buf.data_ptr(), ld, v.double())

    def _ptr(self, name):
        return self.lat[name][0] if name in self.lat else None

    def _ld(self, name):
        return self.lat[name][1] if name in self.lat else 0

    def _img_args(self, k, n, dr, dtt):
        if not n:
            return [None, None, F32, F32, 0]
        return [self.img[k][0], self.img[k][1], dr, dtt, n]

    def _lat_args(self):
        return [self._ptr("mu1"), self._ptr("lv1"), self._ld("mu1"), self.W1,
                self._ptr("mu2"), self._ptr("lv2"), self._ld("mu2"),
                self._ptr("mu3"), self._ptr("lv3"), self._ld("mu3"), self.W2]

    def fwd(self, acc_ptr):
        lib.elbo_fwd(*self._img_args("x", self.nx, self.dtx, self.dttx), *self._img_args("y", self.ny, self.dty, self.dtty),
                     *self._lat_args(), self.B, acc_ptr, st())

    def per_thread(self, n):
        """Values one thread sums from a segment of n elements: the grid of elbo.cu's ew_grid2 (256 threads per block, at
        most 8 blocks per SM, sized by the larger of the image and latent work), vector trips plus the scalar tail."""
        work = max(max(self.nx, self.ny) // 4, self.B * max(self.W1, self.W2) // 4)
        gsize = 256 * min(max((work + 255) // 256, 1), 8 * _sms())
        return 4 * -(-(n // 4) // gsize) + 3

    def ref_sums(self):
        """fp64 {ssq_x, ssq_y, kl1, kl23}, and per sum the magnitude sum its rounding error is bounded by."""
        ref, mag = [0.0] * 4, [0.0] * 4
        for i, k in ((0, "x"), (1, "y")):
            if k in self.img:
                ref[i] = mag[i] = float(((self.img[k][2] - self.img[k][3]) ** 2).sum())
        if self.W1:
            m, l = self.lat["mu1"][2], self.lat["lv1"][2]
            ref[2] = float((m * m + l.exp() - 1 - l).sum())
            mag[2] = float((m * m + l.exp() + 1 + l.abs()).sum())
        if self.W2:
            m2, l2, m3, l3 = (self.lat[k][2] for k in ("mu2", "lv2", "mu3", "lv3"))
            d2e = (m2 - m3) ** 2 * (-l3).exp()
            ref[3] = float((l3 - l2 - 1 + (l2 - l3).exp() + d2e).sum())
            # exp's argument l2 - l3 is rounded in fp32: a relative error of |l2 - l3| u in exp(l2 - l3)
            mag[3] = float((l3.abs() + l2.abs() + 1 + (1 + (l2 - l3).abs()) * (l2 - l3).exp() + d2e).sum())
        return ref, mag

    def acc_bounds(self):
        """|acc - ref| per sum.  Each term is within 10u of its magnitude (a subtraction, squares, expf at 4u, up to three
        additions); one thread then adds up k terms in fp32 (recursive summation: (k - 1) u of the magnitude sum); warps,
        blocks and the atomics add in fp64 (negligible).  Asserted at (k + 12) u of the magnitude sum."""
        _, mag = self.ref_sums()
        ks = [self.per_thread(self.nx), self.per_thread(self.ny), self.per_thread(self.B * self.W1), self.per_thread(self.B * self.W2)]
        return [(k + 12) * U * m for k, m in zip(ks, mag)]


def _finalize_ref(acc, nx, ny, B, gam):
    """fp64 of svrs_elbo_finalize from sums acc: {mse_x, kld_u, mse_y, kld_z, loss} (oracle cond_loss / base_loss)."""
    gx, gy = (float(v) for v in gam)
    mse = lambda s, n, g_: n * (s / n / (2 * g_ * g_) + math.log(g_)) if n else 0.0
    t = [mse(acc[0], nx, gx), 0.5 * acc[2] / B, mse(acc[1], ny, gy), 0.5 * acc[3] / B]
    return t + [sum(t)]


def _finalize_bounds(acc, nx, ny, B, gam, ref5):
    """finalize in fp32: mse = (float)n * ((float)(s / n) / (2 g g) + logf(g)) has six roundings, each at most u of
    n (|s/n| / (2 g^2) + |log g|) (logf: 1 ulp); kld = 0.5 (float)(s / B) one; the loss adds four terms in three steps."""
    gx, gy = (float(v) for v in gam)
    mb = lambda s, n, g_: 8 * U * (abs(s) / (2 * g_ * g_) + n * abs(math.log(g_))) if n else 0.0
    b = [mb(acc[0], nx, gx), 2 * U * abs(ref5[1]), mb(acc[1], ny, gy), 2 * U * abs(ref5[3])]
    return b + [sum(b) + 4 * U * sum(abs(v) for v in ref5[:4])]


GAMMAS = [(1.0, 1.0), (0.05, 3.0), (3.0, 0.05)]

FWD_CASES = {
    # the fused cond step at the cond_grid bench shape: x [128,64,64,4], y [128,32,32,4] fp32 NHWC, enc halves (ld = 2W)
    "cond_grid": dict(B=128, nx=128 * 64 * 64 * 4, ny=128 * 32 * 32 * 4, W1="Wu", W2="Wz", halves=True),
    "cond_grid_wide": dict(B=128, nx=128 * 64 * 64 * 4, ny=128 * 32 * 32 * 4, W1="Wu", W2="Wz", halves=True, regime="wide"),
    # the VAE step: x and kl1 only
    "vae": dict(B=256, nx=256 * 64 * 64 * 4, W1="Wd", halves=True),
    # cond_grid1024: n_x = 16.8 M, about 14 grid-stride trips per thread at 148 SMs
    "cond_grid1024": dict(B=1024, nx=1024 * 64 * 64 * 4, ny=1024 * 32 * 32 * 4, W1="Wu", W2="Wz", halves=True, regime="wide"),
    # recon / target dtype pairs, with ragged n (4k + 3) and n_x != n_y
    "bf16_bf16": dict(B=8, nx=4099, ny=1027, dts=(BF16, BF16, BF16, BF16), W1=16, W2=32),
    "bf16_f32": dict(B=8, nx=4099, ny=1027, dts=(BF16, F32, BF16, F32), W1=16, W2=32),
    "f32_bf16": dict(B=8, nx=4099, ny=1027, dts=(F32, BF16, F32, BF16), W1=16, W2=32),
    "n1_2": dict(B=2, nx=1, ny=2, W1=4, W2=4),
    "n3_5": dict(B=2, nx=3, ny=5, W1=4, W2=4),
    "n5_3": dict(B=2, nx=5, ny=3, W1=4, W2=4),
    # each piece absent in turn
    "no_x": dict(B=4, ny=1027, W1=8, W2=8),
    "no_y": dict(B=4, nx=4099, W1=8, W2=8),
    "no_kl1": dict(B=4, nx=4099, ny=1027, W2=8),
    "no_kl23": dict(B=4, nx=4099, ny=1027, W1=8),
    # W1 != W2, every row stride larger than its width (padding holds NaN)
    "w1_ne_w2_padded": dict(B=6, nx=4096, ny=1024, W1=12, W2=20, pad=8, regime="wide"),
    # B * W, not n, sizes the grid
    "latent_grid": dict(B=2048, nx=8, ny=12, W1=64, W2=64, pad=4),
}


def _case(name, seed):
    spec = dict(FWD_CASES[name])
    wz, wu, wd = _widths()
    for k in ("W1", "W2"):
        if isinstance(spec.get(k), str):
            spec[k] = {"Wz": wz, "Wu": wu, "Wd": wd}[spec[k]]
    return _Elbo(seed, **spec)


@pytest.mark.parametrize("name", list(FWD_CASES))
def test_elbo_fwd_finalize_against_fp64(name):
    """acc against fp64 sums (bounded by the magnitude sums, not the results, which cancel); finalize once from the
    kernel's own acc (isolates it) and once end to end, for gammas 1, 0.05 and 3."""
    c = _case(name, seed=sum(map(ord, name)))
    acc = Guarded((4,), torch.float64, fill=0.0)
    c.fwd(acc.t.data_ptr())
    torch.cuda.synchronize()
    got = acc.t.cpu()
    ref, _ = c.ref_sums()
    bnd = c.acc_bounds()
    for i, k in enumerate(("ssq_x", "ssq_y", "kl1", "kl23")):
        _within(f"{name} acc {k}", got[i:i + 1], torch.tensor([ref[i]], dtype=torch.float64), torch.tensor([bnd[i]], dtype=torch.float64))
    got_acc = [float(v) for v in got]
    for gam in GAMMAS:
        gd = torch.tensor(gam, dtype=torch.float32, device=DEV)
        out = Guarded((5,), torch.float32)
        lib.elbo_finalize(acc.t.data_ptr(), c.nx, c.ny, c.B, gd.data_ptr(), out.t.data_ptr(), st())
        torch.cuda.synchronize()
        gam32 = [float(v) for v in gd.cpu()]
        iso = _finalize_ref(got_acc, c.nx, c.ny, c.B, gam32)
        ib = _finalize_bounds(got_acc, c.nx, c.ny, c.B, gam32, iso)
        _within(f"{name} finalize{gam} from kernel acc", out.t.cpu(), torch.tensor(iso, dtype=torch.float64), torch.tensor(ib, dtype=torch.float64))
        e2e = _finalize_ref(ref, c.nx, c.ny, c.B, gam32)
        eb = _finalize_bounds(ref, c.nx, c.ny, c.B, gam32, e2e)
        # the sums' errors enter through 1 / (2 g^2) (NLL) and 0.5 / B (KL)
        prop = [bnd[0] / (2 * gam32[0] ** 2), 0.5 * bnd[2] / c.B, bnd[1] / (2 * gam32[1] ** 2), 0.5 * bnd[3] / c.B]
        eb = [b + p for b, p in zip(eb, prop + [sum(prop)])]
        _within(f"{name} finalize{gam} end to end", out.t.cpu(), torch.tensor(e2e, dtype=torch.float64), torch.tensor(eb, dtype=torch.float64))
        if not c.nx:
            assert float(out.t[0]) == 0.0
        if not c.ny:
            assert float(out.t[2]) == 0.0
        assert out.intact(), "finalize wrote outside out5"
    assert acc.intact(), "elbo_fwd wrote outside acc"


# ------------------------------------------------------------------------------------------------ ELBO backward
_OUTS = ("d_rx", "d_ry", "d_mu1", "d_lv1", "d_mu2", "d_lv2", "d_mu3", "d_lv3")


class _BwdOut:
    """Guarded gradient buffers.  halves=True: d_mu1 / d_lv1 and d_mu2 / d_lv2 are the halves of d_enc_u / d_enc_z
    [B, 2W] (dld = 2W), d_mu3 / d_lv3 contiguous: the fused step's layout.  Otherwise each has its own [B, W] buffer."""

    def __init__(self, c, ddt, halves, null=None):
        self.c, self.ddt, self.null = c, ddt, null
        self.g = {}         # guarded buffers
        self.view = {}      # output name -> its device view (a half of d_enc when halves=True)
        self.ld = {}
        if c.nx:
            self.g["d_rx"] = Guarded((c.nx,), TORCH_DT[ddt])
        if c.ny:
            self.g["d_ry"] = Guarded((c.ny,), TORCH_DT[ddt])
        self.g["d_gammas"] = Guarded((2,), torch.float32)
        for n in ("d_rx", "d_ry", "d_gammas"):
            if n in self.g:
                self.view[n] = self.g[n].t
        for k, W in (("1", c.W1), ("2", c.W2), ("3", c.W2)):
            if not W:
                continue
            if halves and k != "3":
                enc = self.g["d_enc" + k] = Guarded((c.B, 2 * W), torch.float32)
                self.view["d_mu" + k], self.view["d_lv" + k] = enc.t[:, :W], enc.t[:, W:]
                self.ld["d_mu" + k] = 2 * W
            else:
                for n in ("d_mu" + k, "d_lv" + k):
                    self.g[n] = Guarded((c.B, W), torch.float32)
                    self.view[n] = self.g[n].t
                self.ld["d_mu" + k] = W

    def p(self, n):
        return None if n == self.null or n not in self.view else self.view[n].data_ptr()

    def values(self, n):
        return self.view[n].cpu()

    def intact(self):
        return all(gb.intact() for gb in self.g.values())


def _bwd_call(c, o, acc_ptr, gam_ptr, gout_ptr, act):
    lib.elbo_bwd(*c._img_args("x", c.nx, c.dtx, c.dttx), o.p("d_rx"), o.ddt,
                 *c._img_args("y", c.ny, c.dty, c.dtty), o.p("d_ry"), o.ddt,
                 c._ptr("mu1"), c._ptr("lv1"), c._ld("mu1"), c.W1, o.p("d_mu1"), o.p("d_lv1"), o.ld.get("d_mu1", 0),
                 c._ptr("mu2"), c._ptr("lv2"), c._ld("mu2"), o.p("d_mu2"), o.p("d_lv2"), o.ld.get("d_mu2", 0),
                 c._ptr("mu3"), c._ptr("lv3"), c._ld("mu3"), c.W2, o.p("d_mu3"), o.p("d_lv3"), o.ld.get("d_mu3", 0),
                 c.B, acc_ptr, gam_ptr, gout_ptr, o.p("d_gammas"), act, st())


def _ref_grads(c, gam, gout, act):
    """fp64 autograd of the oracle loss (cond_loss with both NLL pairs, else base_loss) with upstream gradients gout."""
    leaf = lambda t: t.clone().requires_grad_(True)
    L = {k: leaf(v[2]) for k, v in c.lat.items()}
    gx, gy = (torch.tensor(float(v), dtype=torch.float64, requires_grad=True) for v in gam)
    rx = leaf(c.img["x"][2])
    if c.ny:
        ry = leaf(c.img["y"][2])
        terms = O.cond_loss(rx, c.img["x"][3], ry, c.img["y"][3], L["mu1"], L["lv1"], L["mu2"], L["lv2"], L["mu3"], L["lv3"], gx, gy)
        leaves = dict(d_rx=rx, d_ry=ry, d_mu1=L["mu1"], d_lv1=L["lv1"], d_mu2=L["mu2"], d_lv2=L["lv2"], d_mu3=L["mu3"], d_lv3=L["lv3"])
    else:
        shape = (c.B, -1, 1, 1)          # base_loss takes the element count from a 4-d shape
        terms = O.base_loss(rx.view(shape), c.img["x"][3].view(shape), L["mu1"], L["lv1"], gx)
        terms = (terms[0], terms[1], None, None)
        leaves = dict(d_rx=rx, d_mu1=L["mu1"], d_lv1=L["lv1"])
    tot = sum(float(gout[i]) * t for i, t in enumerate(terms) if t is not None)
    names = list(leaves)
    gs = torch.autograd.grad(tot, [leaves[n] for n in names] + [gx, gy], allow_unused=True)
    ref = dict(zip(names, gs[:len(names)]))
    ref["d_gammas"] = torch.stack([gs[-2] if gs[-2] is not None else torch.zeros((), dtype=torch.float64),
                                   gs[-1] if gs[-1] is not None else torch.zeros((), dtype=torch.float64)])
    if act == ACT_SIGMOID:
        for n, k in (("d_rx", "x"), ("d_ry", "y")):
            if n in ref:
                r = c.img[k][2]
                ref[n] = ref[n] * r * (1 - r)
    return ref


def _grad_bounds(c, gam, gout, ref, acc):
    """Per-element bounds of the fp32 gradients (k = g / B, two roundings; expf 4u relative):
    d_recon: (r - t) * (g / gam^2) [* r * (1 - r)]: at most seven roundings, all relative -> 8u |ref|;
    d_mu1 = k mu: 4u |ref|;  d_lv1 = k/2 (expf(l) - 1): 8u |k|/2 (e^l + 1);
    d_mu2 = -d_mu3 = k (mu2 - mu3) expf(-l3): nine roundings -> 12u |ref|;
    d_lv2 = k/2 (e23 - 1), e23 = expf(l2 - l3) with a rounded argument (relative error |l2 - l3| u + 4u):
        (|l2 - l3| + 10) u |k|/2 (e23 + 1);
    d_lv3 = k/2 (1 - e23 - d^2 expf(-l3)): (|l2 - l3| + 16) u |k|/2 (1 + e23 + d^2 e^-l3);
    d_gammas = g (-acc / gam^3 + n / gam): five roundings of the two terms, which cancel near the optimum, so the bound
    is 8u (|acc / gam^3| + n / gam) |g|, plus |g| |acc - ssq| / gam^3 for the sum's own error against the exact ssq."""
    B = c.B
    b = {n: 8 * U * ref[n].abs() for n in ("d_rx", "d_ry") if n in ref}
    if c.W1:
        k = abs(float(gout[1])) / B
        b["d_mu1"] = 4 * U * ref["d_mu1"].abs()
        b["d_lv1"] = 8 * U * k / 2 * (c.lat["lv1"][2].exp() + 1)
    if c.W2:
        k = abs(float(gout[3])) / B
        m2, l2, m3, l3 = (c.lat[n][2] for n in ("mu2", "lv2", "mu3", "lv3"))
        e23, d2e = (l2 - l3).exp(), (m2 - m3) ** 2 * (-l3).exp()
        b["d_mu2"] = 12 * U * ref["d_mu2"].abs()
        b["d_mu3"] = 12 * U * ref["d_mu3"].abs()
        b["d_lv2"] = ((l2 - l3).abs() + 10) * U * k / 2 * (e23 + 1)
        b["d_lv3"] = ((l2 - l3).abs() + 16) * U * k / 2 * (1 + e23 + d2e)
    ref_s, _ = c.ref_sums()
    dg = []
    for i, n, gi in ((0, c.nx, 0), (1, c.ny, 2)):
        g_, gm = abs(float(gout[gi])), float(gam[i])
        dg.append(8 * U * (abs(acc[i]) / gm ** 3 + n / gm) * g_ + g_ * abs(acc[i] - ref_s[i]) / gm ** 3 if n else 0.0)
    b["d_gammas"] = torch.tensor(dg, dtype=torch.float64)
    return b


def _check_bwd(tag, c, o, ref, bnd):
    for n in _OUTS + ("d_gammas",):
        if n not in ref or o.p(n) is None:
            continue
        got = o.values(n)
        if n in ("d_rx", "d_ry") and o.ddt == BF16:
            _bf16_ulp_check(f"{tag} {n}", got, ref[n])
        else:
            _within(f"{tag} {n}", got, ref[n].detach(), bnd[n])
    assert o.intact(), f"{tag}: elbo_bwd wrote outside an output buffer"


def _run_bwd(c, ddt, halves, gam, gout, act, null=None):
    acc = Guarded((4,), torch.float64, fill=0.0)
    c.fwd(acc.t.data_ptr())
    gd = torch.tensor(gam, dtype=torch.float32, device=DEV)
    god = torch.tensor(gout, dtype=torch.float32, device=DEV)
    o = _BwdOut(c, ddt, halves, null)
    _bwd_call(c, o, acc.t.data_ptr(), gd.data_ptr(), god.data_ptr(), act)
    torch.cuda.synchronize()
    accv = [float(v) for v in acc.t.cpu()]
    gam32 = [float(v) for v in gd.cpu()]
    ref = _ref_grads(c, gam32, gout, act)
    return o, ref, _grad_bounds(c, gam32, gout, ref, accv)


GOUTS = [(1.0, 1.0, 1.0, 1.0), (0.5, 0.25, 2.0, 0.0)]


@pytest.mark.parametrize("gout", GOUTS, ids=["gout1", "gout_mixed"])
@pytest.mark.parametrize("ddt", [F32, BF16], ids=["drecon_f32", "drecon_bf16"])
@pytest.mark.parametrize("model", ["cond", "vae"])
def test_elbo_bwd_fused_step_call(model, ddt, gout):
    """The fused training step's call (trainer.py, FusedCondTrainer / FusedVaeTrainer): fp32 NHWC recon and target,
    ACT_SIGMOID folded into d_recon (compute dtype), latent gradients into the halves of d_enc [B, 2W]; gout covers the
    1/world scaling and a zero upstream gradient (kld_z)."""
    wz, wu, wd = _widths()
    if model == "cond":
        c = _Elbo(11, 128, nx=128 * 64 * 64 * 4, ny=128 * 32 * 32 * 4, W1=wu, W2=wz, halves=True, regime="wide")
    else:
        c = _Elbo(12, 256, nx=256 * 64 * 64 * 4, W1=wd, halves=True, regime="wide")
    gam = (0.7, 1.3)
    o, ref, bnd = _run_bwd(c, ddt, True, gam, gout, ACT_SIGMOID)
    _check_bwd(f"bwd[{model}, ddt={ddt}, gout={gout}]", c, o, ref, bnd)


def test_elbo_bwd_autograd_path_call():
    """svrs_native.elbo's autograd Function: ACT_NONE, fp32 everything, contiguous latents (dld = W)."""
    c = _Elbo(13, 16, nx=16 * 32 * 32 * 4, ny=16 * 16 * 16 * 4, W1=256, W2=512, regime="init")
    o, ref, bnd = _run_bwd(c, F32, False, (1.0, 0.05), GOUTS[0], ACT_NONE)
    _check_bwd("bwd[autograd path]", c, o, ref, bnd)


@pytest.mark.parametrize("null", list(_OUTS) + ["d_gammas"])
def test_elbo_bwd_each_output_may_be_null(null):
    """Any output may be NULL (include/svrs_b200.h): with each of the nine left out in turn, every other one is written
    and correct."""
    c = _Elbo(14, 8, nx=4099, ny=1027, W1=16, W2=24, pad=4, regime="wide")
    o, ref, bnd = _run_bwd(c, F32, False, (0.9, 1.1), GOUTS[1], ACT_SIGMOID, null=null)
    _check_bwd(f"bwd[{null} = NULL]", c, o, ref, bnd)
    if null in o.g:
        assert torch.isnan(o.g[null].t).all(), f"{null} was NULL but its buffer changed"


# ------------------------------------------------------------------------------------------------ svrs_sample_latents
def _latents_inputs(B, Wz, ld, seed):
    """mu3 / lv3 / yflat fp32 with row stride ld (the padding holds NaN), as (device buffer, fp32 CPU [B, Wz])."""
    g = torch.Generator().manual_seed(seed)
    vals = [torch.randn(B, Wz, generator=g), 14 * torch.rand(B, Wz, generator=g) - 7, torch.randn(B, Wz, generator=g)]
    out = []
    for v in vals:
        buf = torch.full((B, ld), float("nan"))
        buf[:, :Wz] = v
        out.append((buf.to(DEV), v))
    return out


def _check_draws(tag, stack, mu, lv, yflat, eps, S):
    """y half bit-equal to yflat[b]; z half against fp64 mu + eps exp(lv / 2): expf (4u, exact argument lv / 2) and
    one fmaf rounding give |err| <= 5u (|mu| + |eps exp(lv / 2)|); asserted at 6u."""
    Wz = mu.shape[1]
    st_ = stack.cpu()
    assert torch.equal(st_[:, :Wz], yflat.repeat_interleave(S, 0)), f"{tag}: y half differs from yflat"
    m, s = mu.double().repeat_interleave(S, 0), (0.5 * lv.double()).exp().repeat_interleave(S, 0)
    es = eps.double() * s
    _within(f"{tag} z half", st_[:, Wz:], m + es, 6 * U * (m.abs() + es.abs()))


@pytest.mark.parametrize("pad", [0, 12], ids=["ld_eq_Wz", "ld_gt_Wz"])
def test_sample_latents_injected_eps(pad):
    """Config 5 (16 patches x 32 draws, Wz of cr = 2 / P = 64): stack[b*S + s] = [yflat[b] | mu3[b] + eps exp(lv3[b] / 2)]."""
    Wz = _widths()[0]
    B, S = 16, 32
    (mu, muc), (lv, lvc), (yf, yfc) = _latents_inputs(B, Wz, Wz + pad, 21)
    eps = torch.randn(B * S, Wz, generator=torch.Generator().manual_seed(22))
    stack = Guarded((B * S, 2 * Wz), torch.float32)
    lib.sample_latents(mu.data_ptr(), lv.data_ptr(), Wz + pad, yf.data_ptr(), Wz + pad, eps.to(DEV).data_ptr(), stack.t.data_ptr(),
                       B, S, Wz, 0, 0, 0, None, st())
    torch.cuda.synchronize()
    _check_draws(f"sample_latents[pad {pad}]", stack.t, muc, lvc, yfc, eps, S)
    assert stack.intact(), "sample_latents wrote outside the stack"


def test_sample_latents_philox_addressing():
    """On-device draws: eps(row) is svrs_philox_normal's row sample_offset + b*S + s of the same (seed, stream, step);
    patch b drawn alone at sample_offset + b*S reproduces rows [b*S, (b+1)*S) of the full call; step_ptr changes the
    draws and the same step repeats them."""
    Wz = _widths()[0]
    B, S, seed, sid, off = 16, 32, 0x9E3779B97F4A7C15, 2, 1000
    ld = Wz + 4
    (mu, muc), (lv, lvc), (yf, yfc) = _latents_inputs(B, Wz, ld, 23)
    step = torch.tensor([5], dtype=torch.int64, device=DEV)

    def draw(b0, nb, off_, step_):
        out = Guarded((nb * S, 2 * Wz), torch.float32)
        lib.sample_latents(mu.data_ptr() + 4 * b0 * ld, lv.data_ptr() + 4 * b0 * ld, ld, yf.data_ptr() + 4 * b0 * ld, ld, None,
                           out.t.data_ptr(), nb, S, Wz, seed, sid, off_, step_.data_ptr(), st())
        return out

    full = draw(0, B, off, step)
    eps = torch.empty(B * S, Wz, device=DEV)
    lib.philox_normal(eps.data_ptr(), B * S, Wz, seed, sid, off, step.data_ptr(), st())
    torch.cuda.synchronize()
    _check_draws("sample_latents[philox]", full.t, muc, lvc, yfc, eps.cpu(), S)
    for b in (0, 7, 15):
        one = draw(b, 1, off + b * S, step)
        torch.cuda.synchronize()
        assert torch.equal(one.t, full.t[b * S:(b + 1) * S]), f"patch {b} drawn alone differs from the full call"
        assert one.intact()
    again = draw(0, B, off, step)
    step6 = torch.tensor([6], dtype=torch.int64, device=DEV)
    other = draw(0, B, off, step6)
    torch.cuda.synchronize()
    assert torch.equal(again.t, full.t), "the same step gave different draws"
    same = (other.t[:, Wz:] == full.t[:, Wz:]).double().mean().item()
    assert same < 1e-3, f"a different step repeated {100 * same:.2f} % of the draws"
    assert full.intact() and again.intact() and other.intact()


# ------------------------------------------------------------------------------------------------ svrs_sample_tail_stats
MAPS = ("mean", "std", "mae", "mse", "bias", "sample0")
REF_KEY = dict(mean="mean", std="std", mae="mae", mse="mse", bias="mean_bias", sample0="sample0")
# fp32 arithmetic on identical inputs in both dtypes: 144 fmas per output, the sigmoid and the Welford / Chan updates.
# Relative to each map's maximum, at most 2x the worst error measured on a B200 at 1000 W (module docstring).  The kernels
# use no atomics, so these seeded inputs give the same errors on every run.  The bias map is smaller than the mean it is
# computed from, which makes its error relative to its own maximum larger.
TAIL_TOL = dict(mean=7e-7, std=4e-7, mae=1.2e-6, mse=1.1e-6, bias=9e-6, sample0=6e-7)


def _tail_inputs(B, S, H, W, dtype, seed):
    """Independent draws x [B*S, H, W, 16] and weights scaled so that the sigmoid outputs spread over about (0.1, 0.9)
    (pre-activations ~ N(0, 1)): the std map is O(0.1).  Values as the kernel reads them (rounded to bf16 for bf16)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B * S, H, W, 16, generator=g).to(dtype)
    w = (torch.randn(4, 16, 3, 3, generator=g) / 12).to(dtype).float()
    bias = 0.1 * torch.randn(4, generator=g)
    target = torch.rand(B, H, W, 4, generator=g)
    return x, w, bias, target


def _tail_ref(x, w, bias, target, B, S):
    """fp64 conv2d(16 -> 4, k3, p1) + sigmoid per draw, then the statistics of task() per patch."""
    H, W = x.shape[1:3]
    pre = F.conv2d(x.double().permute(0, 3, 1, 2), w.double(), bias.double(), padding=1)
    draws = torch.sigmoid(pre).view(B, S, 4, H, W)
    tg = target.double().permute(0, 3, 1, 2)
    per = [task_stats(draws[b], tg[b:b + 1]) for b in range(B)]
    return {k: torch.stack([p[k] for p in per]) for k in per[0]}


class _TailOut:
    def __init__(self, B, H, W, scratch_floats, null=None):
        self.g = dict(mean=Guarded((B, 4, H, W), torch.float32), std=Guarded((B, H, W), torch.float32),
                      mae=Guarded((B, H, W), torch.float32), mse=Guarded((B, H, W), torch.float32),
                      bias=Guarded((B, H, W), torch.float32), sample0=Guarded((B, 4, H, W), torch.float32))
        self.scratch = Guarded((scratch_floats,), torch.float32)
        self.null = null

    def p(self, k):
        return None if k == self.null else self.g[k].t.data_ptr()

    def intact(self):
        return self.scratch.intact() and all(gb.intact() for gb in self.g.values())


def _tail_call(xd, dt_, wpack, bd, td, B, S, H, W, splits, o, cin=16):
    lib.sample_tail_stats(xd.data_ptr(), dt_, wpack.data_ptr(), bd.data_ptr(), None if td is None else td.data_ptr(), B, S, H, W, cin, 4,
                          splits, o.scratch.t.data_ptr(), *(o.p(k) for k in MAPS), st())


def _tail_setup(B, S, H, W, dtype, splits, seed=31):
    x, w, bias, target = _tail_inputs(B, S, H, W, dtype, seed)
    dt_ = F32 if dtype == torch.float32 else BF16
    xd, td, bd = x.to(DEV), target.to(DEV), bias.to(DEV)
    wpack = pack(w.to(DEV), dtype)[0]          # the p10 pack [9][16][4] the engine hands to the kernel
    if splits is None:
        splits = int(lib.sample_tail_splits(B, S, H, W))
    nscr = int(lib.sample_tail_scratch_floats(B, H, W, splits))
    return x, w, bias, target, dt_, xd, td, bd, wpack, splits, nscr


TAIL_CASES = [((16, 32, 64, 64), None),       # the sample bench shape; default split (1 on 148 SMs)
              ((1, 32, 64, 64), None),        # default split 4
              ((3, 37, 12, 20), 1), ((3, 37, 12, 20), 2), ((3, 37, 12, 20), 5), ((3, 37, 12, 20), 37),   # 240 pixels: a partial CTA
              ((1, 8, 3, 130), None),
              ((2, 9, 1, 1), None),           # only the centre tap lies inside the map
              ((2, 2, 64, 64), None),
              ((1, 1, 8, 8), None)]           # S = 1: std is NaN like torch.std of one sample


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("shape,splits", TAIL_CASES, ids=[f"{'x'.join(map(str, s))}-splits{p}" for s, p in TAIL_CASES])
def test_sample_tail_stats_against_fp64(shape, splits, dtype):
    """All six maps against fp64 statistics of the materialised draws.  A biased std (x sqrt((S-1)/S), 1.6 % at S = 32),
    a missing Chan term (every split > 1) or a lost draw would exceed TAIL_TOL (below 1e-5) by orders of magnitude."""
    B, S, H, W = shape
    x, w, bias, target, dt_, xd, td, bd, wpack, splits, nscr = _tail_setup(B, S, H, W, dtype, splits)
    o = _TailOut(B, H, W, nscr)
    _tail_call(xd, dt_, wpack, bd, td, B, S, H, W, splits, o)
    torch.cuda.synchronize()
    ref = _tail_ref(x, w, bias, target, B, S)
    for k in MAPS:
        got = o.g[k].t.cpu()
        if k == "std" and S == 1:
            assert torch.isnan(got).all(), "std of one draw must be NaN (torch.std, unbiased)"
            continue
        _rel_to_max(f"tail[{shape}, splits={splits}, {dtype}] {k}", got, ref[REF_KEY[k]], TAIL_TOL[k])
    assert o.intact(), "sample_tail_stats wrote outside an output or the scratch"


def _rel_to_max(name, got, ref, tol):
    got, ref = got.double(), ref.double().reshape(got.shape)
    scale = float(ref.abs().max())
    err = float((got - ref).abs().max())
    print(f"[elbo/sample] {name}: max|err| {err:.3e}  rel-to-max {err / scale:.3e}")
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    assert err <= tol * scale, f"{name}: max|err| {err:.3e} > {tol} * {scale:.3e}"


@pytest.mark.parametrize("null", list(MAPS) + ["target"])
def test_sample_tail_stats_null_outputs(null):
    """Each map NULL in turn leaves the others correct; with target = NULL the mae / mse / bias buffers stay untouched."""
    B, S, H, W, splits = 3, 37, 12, 20, 5
    x, w, bias, target, dt_, xd, td, bd, wpack, splits, nscr = _tail_setup(B, S, H, W, torch.float32, splits, seed=32)
    o = _TailOut(B, H, W, nscr, null=None if null == "target" else null)
    _tail_call(xd, dt_, wpack, bd, None if null == "target" else td, B, S, H, W, splits, o)
    torch.cuda.synchronize()
    ref = _tail_ref(x, w, bias, target, B, S)
    for k in MAPS:
        got = o.g[k].t.cpu()
        if k == null or (null == "target" and k in ("mae", "mse", "bias")):
            assert torch.isnan(got).all(), f"{k} was not to be written"
            continue
        _rel_to_max(f"tail[{null} NULL] {k}", got, ref[REF_KEY[k]], TAIL_TOL[k])
    assert o.intact()


def test_sample_tail_stats_rejects_bad_splits_and_channels():
    B, S, H, W = 1, 8, 8, 8
    x, w, bias, target, dt_, xd, td, bd, wpack, _, _ = _tail_setup(B, S, H, W, torch.float32, 1)
    o = _TailOut(B, H, W, int(lib.sample_tail_scratch_floats(B, H, W, S + 1)))
    for splits in (0, S + 1):
        with pytest.raises(SvrsError, match="splits"):
            _tail_call(xd, dt_, wpack, bd, td, B, S, H, W, splits, o)
    with pytest.raises(SvrsUnsupported):
        _tail_call(xd, dt_, wpack, bd, td, B, S, H, W, 1, o, cin=8)
    torch.cuda.synchronize()
    assert all(torch.isnan(gb.t).all() for gb in o.g.values()) and o.intact(), "a rejected call wrote something"
