"""VAE - the unconditional patch VAE of the reference (models/vae.py:11-262) behind the same Python API,
executed by the sm_100a kernel library.  `forward(x) -> (x_hat, mu, logvar)` (vae.py:103-107); batches are
(x, _); `gamma` is a plain CPU tensor with requires_grad (vae.py:34, SURVEY Q3); 52-key state_dict.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from loss import base_loss

from .base import BaseVAE, wandb
from .layers import conv3, down_block, up_block


class VAE(BaseVAE):
    def __init__(self, cr, patch_size=64, callbacks=None, slurm_job_id="local"):
        super().__init__(patch_size, [] if callbacks is None else callbacks, slurm_job_id)
        self.cr = cr
        L = int((patch_size * patch_size * 4 // cr) // 16) * 16          # vae.py:29-31
        self.latent_size, self.patch_size = L, patch_size
        self.gamma = torch.tensor(1.0, requires_grad=True)
        self.encoder = nn.Sequential(                                     # vae.py:36-58
            down_block(4, 16), down_block(16, 64), conv3(64, 64), conv3(64, 128), conv3(128, 128),
            conv3(128, (L // 64) * 2), nn.Flatten(start_dim=1))
        self.decoder = nn.Sequential(                                     # vae.py:60-85
            nn.Unflatten(1, (L // 64, patch_size // 4, patch_size // 4)), up_block(L // 64, 128), up_block(128, 64),
            conv3(64, 64), conv3(64, 16), conv3(16, 16), conv3(16, 4), nn.Sigmoid())
        self.num_params = sum(p.numel() for p in self.parameters() if p.requires_grad)

    # ------------------------------------------------------------------ engine
    def _make_engine(self, dtype):
        from svrs_native.engine import VaeEngine
        return VaeEngine(self, dtype)

    def _fused_trainer(self, optimizer):
        from svrs_native.trainer import FusedVaeTrainer
        if self._trainer is None or self._trainer.optimizer is not optimizer:
            self._trainer = FusedVaeTrainer(self, optimizer, sync_bn=getattr(self, "sync_bn", False))
        return self._trainer

    # ------------------------------------------------------------------ reference API
    def forward(self, x, eps=None):
        from svrs_native.autograd import VaeForwardFn
        x_hat, enc = VaeForwardFn.apply(self._grad_anchor(x.device), self._engine(), x, eps, self.training,
                                        torch.is_grad_enabled())
        mu, logvar = enc.chunk(2, dim=1)                                   # vae.py:89-92
        return x_hat, mu, logvar

    def _subnet(self, name, t, chw):
        eng = self._engine()
        rt = eng.rt
        rt.ensure()
        rt.packs_dirty = True
        rt.pack_weights()
        B = t.shape[0]
        c, h, w = chw
        flat = t.reshape(B, -1).contiguous().float()
        xin = rt.to_nhwc(flat, c * h * w, B, c, h, w)
        out, _ = rt.net_forward(eng.nets[name], xin, self.training, save=False)
        n, oh, ow, oc = out.shape
        res = torch.empty((B, oc * oh * ow), device=t.device, dtype=torch.float32)
        rt.to_nchw(out, res, oc * oh * ow)
        return res, (oc, oh, ow)

    def encode(self, x):
        P = self.patch_size
        with torch.no_grad():
            enc, _ = self._subnet("encoder", x, (4, P, P))
        return enc.chunk(2, dim=1)

    def reparameterize(self, mu, logvar):
        from svrs_native.engine import RngState, reparam_fwd
        eng = self._engine()
        eng.rt.ensure()
        B, Wd = mu.shape
        enc = torch.cat((mu.float(), logvar.float()), dim=1).contiguous()
        z = torch.empty((B, Wd), device=mu.device, dtype=torch.float32)
        self._free_draws = getattr(self, "_free_draws", 0) + 1
        reparam_fwd(eng.rt, enc, None, z, Wd, B, Wd, RngState(seed=eng.rng.key() + 7919 * self._free_draws), 3)
        return z

    def decode(self, z):
        P, L = self.patch_size, self.latent_size
        with torch.no_grad():
            out, (c, h, w) = self._subnet("decoder", z, (L // 64, P // 4, P // 4))
        return out.view(-1, c, h, w)

    def train_step(self, batch, device):
        """vae.py:109-120 (autograd-compatible path)."""
        x, _ = batch
        x = x.to(device)
        x_hat, mu, logvar = self.forward(x)
        mse, kld = base_loss(x_hat, x, mu, logvar, self.gamma)
        loss = mse + kld
        return loss, {"Loss/loss": loss.detach(), "Loss/mse": mse.detach(), "Loss/kld": kld.detach()}

    def fused_train_step(self, batch, device, fused):
        x, _ = batch
        x = x.to(device, non_blocking=True)
        t = fused.step(x, use_graph=self.use_cuda_graph).clone()
        return t[4], {"Loss/loss": t[4], "Loss/mse": t[0], "Loss/kld": t[1]}

    def val_step(self, batch, device):
        """vae.py:122-140."""
        x, _ = batch
        x = x.to(device)
        with torch.no_grad():
            x_hat, mu, logvar = self.forward(x)
            mse, kld = base_loss(x_hat, x, mu, logvar, self.gamma)
            loss = mse + kld
        return loss, {"Loss/val_loss": loss, "Loss/val_mse": mse, "Loss/val_kld": kld}

    def evaluate(self, val_loader, wandb_run, epoch, full_val=False):
        """vae.py:142-216: on full-validation epochs Metrics/SSIM (skimage's structural_similarity with win_size=11,
        data_range=1.0, averaged over the validation images) is computed on the device (svrs_native.metrics); it is not
        logged for patches smaller than the window.  Image logging kept."""
        from svrs_native import metrics
        device = next(self.parameters()).device
        x, _ = next(iter(val_loader))
        x = x.to(device)
        with torch.no_grad():
            x_hat, _, _ = self.forward(x)
        if full_val and min(x.shape[-2:]) >= 11:
            tot, cnt = torch.zeros((), device=device, dtype=torch.float64), 0
            for b, _ in val_loader:
                b = b.to(device)
                with torch.no_grad():
                    r, _, _ = self.forward(b)
                tot += metrics.ssim(b, r).sum()
                cnt += b.size(0)
            wandb_run.log({"Metrics/SSIM": float(tot) / cnt}, step=epoch)
        if epoch % 5 == 0 or epoch == 1:
            try:
                wandb_run.log({"Images/Input": [wandb.Image(i.permute(1, 2, 0).cpu().numpy()) for i in x[:4]]}, step=epoch)
                wandb_run.log({"Images/Reconstruction": [wandb.Image(i.permute(1, 2, 0).cpu().numpy()) for i in x_hat[:4]]},
                              step=epoch)
            except Exception:
                pass

    def on_train_epoch_end(self, **kwargs):
        self.wandb_run.log({"HyperParameters/Gamma": self.gamma.item(),
                            "HyperParameters/Learning Rate": self.scheduler.get_last_lr()[0]}, step=self.current_epoch)

    def on_train_start(self, **kwargs):
        """vae.py:227-231."""
        self.gamma.requires_grad = True
        have = {id(p) for g in self.optimizer.param_groups for p in g["params"]}
        if id(self.gamma) not in have:
            self.optimizer.add_param_group({"params": [self.gamma]})

    def get_task_data(self, val_loader):
        x, _ = next(iter(val_loader))
        x = x.to(next(self.parameters()).device)[0:1]
        return x, x

    def sample(self, y, samples=1000):
        """vae.py:240-252: `samples` decodes around the posterior of one patch.  (The reference draws noise of
        width `latent_size`, which only matches the true latent width at P=32 - SURVEY Q10; here the true width
        is used.)"""
        mu, logvar = self.encode(y)
        eng = self._engine()
        mu = mu.expand(samples, -1).contiguous()
        logvar = logvar.expand(samples, -1).contiguous()
        z = self.reparameterize(mu, logvar)
        return self.decode(z).view(samples, 4, self.patch_size, self.patch_size)
