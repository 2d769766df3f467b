"""Cond_SRVAE - the conditional super-resolution VAE of the reference (models/cond_vae.py:15-625) behind the
same Python API, executed by the sm_100a kernel library.

API parity (SURVEY 8.4 row b): `Cond_SRVAE(cr, patch_size=64, callbacks=None, slurm_job_id="local")`;
attributes cr / latent_size / latent_size_y / patch_size / gammax / gammay / num_params; the eight
sub-networks under the reference's names (so `state_dict()` has the reference's 165 keys and NCHW shapes);
`forward(x, y)` returns the 8-tuple (x_hat, y_hat, mu_z, logvar_z, mu_u, logvar_u, mu_z_uy, logvar_z_uy) with
mu/logvar being chunk views; batches are (y, x).  gammax / gammay are plain CPU tensors with requires_grad,
exactly as in the reference (cond_vae.py:24-25, SURVEY Q3).
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from loss import cond_loss

from .base import BaseVAE, wandb
from .layers import conv3, down_block, up_block


class Cond_SRVAE(BaseVAE):
    def __init__(self, cr, patch_size=64, callbacks=None, slurm_job_id="local"):
        super().__init__(patch_size, [] if callbacks is None else callbacks, slurm_job_id)
        self.cr = cr
        L = int((patch_size * patch_size * 4 / cr) // 256) * 256          # cond_vae.py:21
        Lu = L // 4                                                       # cond_vae.py:22
        self.latent_size, self.latent_size_y, self.patch_size = L, Lu, patch_size
        self.gammax = torch.tensor(1.0, requires_grad=True)
        self.gammay = torch.tensor(1.0, requires_grad=True)
        P = patch_size
        tail = lambda: [conv3(64, 64), conv3(64, 16), conv3(16, 16), conv3(16, 4), nn.Sigmoid()]

        # construction order == the reference's, so torch.manual_seed(s) yields identical initial weights
        self.encoder_y = nn.Sequential(                                   # cond_vae.py:27-49
            down_block(4, 16), down_block(16, 64), conv3(64, 64), conv3(64, 128), conv3(128, 128),
            conv3(128, (Lu // 64) * 2), nn.Flatten(start_dim=1))
        self.decoder_y = nn.Sequential(                                   # cond_vae.py:51-81
            nn.Unflatten(1, (Lu // 64, P // 8, P // 8)), up_block(Lu // 64, 128), up_block(128, 64), *tail())
        self.encoder_x = nn.Sequential(                                   # cond_vae.py:83-108
            down_block(4, 16), down_block(16, 64), down_block(64, 128), conv3(128, 128), conv3(128, 128),
            conv3(128, 128), conv3(128, (L // 64) * 2), nn.Flatten(1))
        self.decoder_x = nn.Sequential(                                   # cond_vae.py:110-144
            nn.Unflatten(1, (L * 2 // 64, P // 8, P // 8)), up_block(L * 2 // 64, 256), up_block(256, 128),
            up_block(128, 64), *tail())
        self.y_to_z = nn.Sequential(                                      # cond_vae.py:146-165
            down_block(4, 16), down_block(16, 64), down_block(64, 128), conv3(128, 128), conv3(128, L // 16),
            nn.Flatten(start_dim=1))
        self.u_to_z = nn.Sequential(                                      # cond_vae.py:167-189
            nn.Unflatten(1, (Lu // 16, P // 16, P // 16)), conv3(Lu // 16, Lu // 16), conv3(Lu // 16, L // 16),
            nn.Flatten(1))
        self.mu_u_y_to_z = nn.Sequential(                                 # cond_vae.py:191-210
            nn.Unflatten(1, (L * 2 // 16, P // 16, P // 16)), conv3(L * 2 // 16, L // 16), conv3(L // 16, L // 16),
            nn.Flatten(1))
        self.logvar_u_y_to_z = nn.Sequential(                             # cond_vae.py:211-231
            nn.Unflatten(1, (L * 2 // 16, P // 16, P // 16)), conv3(L * 2 // 16, L // 16), conv3(L // 16, L // 16),
            nn.Flatten(1), nn.Hardtanh(-7, 7))
        self.num_params = sum(p.numel() for p in self.parameters() if p.requires_grad)
        print(f"Cond_SRVAE initialized with {self.num_params} trainable parameters.")

    # ------------------------------------------------------------------ engine
    def _make_engine(self, dtype):
        from svrs_native.engine import CondEngine
        return CondEngine(self, dtype)

    def _fused_trainer(self, optimizer):
        from svrs_native.trainer import FusedCondTrainer
        if self._trainer is None or self._trainer.optimizer is not optimizer:
            self._trainer = FusedCondTrainer(self, optimizer, sync_bn=getattr(self, "sync_bn", False))
        return self._trainer

    def _run(self, x, y, eps_u=None, eps_z=None):
        from svrs_native.autograd import CondForwardFn
        eng = self._engine()
        return CondForwardFn.apply(self._grad_anchor(x.device), eng, x, y, eps_u, eps_z, self.training,
                                   torch.is_grad_enabled())

    # ------------------------------------------------------------------ reference API
    def forward(self, x, y, eps_u=None, eps_z=None):
        """cond_vae.py:275-286.  eps_u / eps_z (optional) inject the reparameterisation noise; by default it
        is drawn on the device with Philox (u first, then z - the reference's draw order, SURVEY Q5)."""
        x_hat, y_hat, enc_z, enc_u, mu_z_uy, logvar_z_uy = self._run(x, y, eps_u, eps_z)
        mu_z, logvar_z = torch.chunk(enc_z, 2, dim=1)
        mu_u, logvar_u = torch.chunk(enc_u, 2, dim=1)
        return x_hat, y_hat, mu_z, logvar_z, mu_u, logvar_u, mu_z_uy, logvar_z_uy

    def reparameterize(self, mu, logvar):
        """cond_vae.py:261-265 on free-standing tensors (inference helper; device Philox noise)."""
        from svrs_native.engine import RngState, reparam_fwd
        eng = self._engine()
        eng.rt.ensure()
        B, Wd = mu.shape
        enc = torch.cat((mu.float(), logvar.float()), dim=1).contiguous()
        z = torch.empty((B, Wd), device=mu.device, dtype=torch.float32)
        self._free_draws = getattr(self, "_free_draws", 0) + 1
        reparam_fwd(eng.rt, enc, None, z, Wd, B, Wd, RngState(seed=eng.rng.key() + 7919 * self._free_draws), 3)
        return z

    def _subnet(self, name, t, chw):
        """Run one sub-network stand-alone (inference): NCHW-flat in -> NCHW-flat fp32 out."""
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

    def encode_y(self, y):
        P = self.patch_size
        with torch.no_grad():
            enc, _ = self._subnet("encoder_y", y, (4, P // 2, P // 2))
        return torch.chunk(enc, 2, dim=1)

    def encode_x(self, x):
        P = self.patch_size
        with torch.no_grad():
            enc, _ = self._subnet("encoder_x", x, (4, P, P))
        return torch.chunk(enc, 2, dim=1)

    def z_cond(self, y, u):
        """cond_vae.py:237-249."""
        P, L, Lu = self.patch_size, self.latent_size, self.latent_size_y
        with torch.no_grad():
            yz, _ = self._subnet("y_to_z", y, (4, P // 2, P // 2))
            uz, _ = self._subnet("u_to_z", u, (Lu // 16, P // 16, P // 16))
            joint = torch.cat((yz, uz), dim=1)
            mu, _ = self._subnet("mu_u_y_to_z", joint, (2 * L // 16, P // 16, P // 16))
            lv, _ = self._subnet("logvar_u_y_to_z", joint, (2 * L // 16, P // 16, P // 16))
        return mu, lv

    def decode_y(self, u):
        P, Lu = self.patch_size, self.latent_size_y
        with torch.no_grad():
            out, (c, h, w) = self._subnet("decoder_y", u, (Lu // 64, P // 8, P // 8))
        return out.view(-1, c, h, w)

    def decode_x(self, z, y):
        """cond_vae.py:270-273."""
        P, L = self.patch_size, self.latent_size
        with torch.no_grad():
            yz, _ = self._subnet("y_to_z", y, (4, P // 2, P // 2))
            out, (c, h, w) = self._subnet("decoder_x", torch.cat((yz, z.float()), dim=1), (2 * L // 64, P // 8, P // 8))
        return out.view(-1, c, h, w)

    def conditional_generation(self, y):
        """cond_vae.py:288-297."""
        mu_u, logvar_u = self.encode_y(y)
        u = self.reparameterize(mu_u, logvar_u)
        mu_z_uy, logvar_z_uy = self.z_cond(y, u)
        z = self.reparameterize(mu_z_uy, logvar_z_uy)
        return self.decode_x(z, y)

    def sample(self, y, samples=1000, eps_u=None, eps_s=None) -> torch.Tensor:
        """cond_vae.py:299-318: `samples` decodes of one LR patch; y_to_z is computed once, eps on device."""
        return self._engine().sample(y, samples, eps_u, eps_s, training=self.training)

    def sample_stats(self, y, samples=1000, target=None, eps_u=None, eps_s=None, splits=0):
        """The per-pixel uncertainty statistics task() derives from `samples` posterior draws (models/base.py:305-313, 341)
        for a batch of LR patches, accumulated in the decoder tail kernel (streaming Welford): the [S,4,P,P] draws are never
        written to memory.  -> dict(mean [B,4,P,P], std, mae, mse, mean_bias [B,P,P], sample0 [B,4,P,P])."""
        return self._engine().sample_stats(y, samples, target, eps_u, eps_s, training=self.training, splits=splits)

    def generation(self):
        """cond_vae.py:320-324."""
        dev = next(self.parameters()).device
        u = self.reparameterize(torch.zeros(1, self._engine().Wu, device=dev), torch.zeros(1, self._engine().Wu, device=dev))
        y = self.decode_y(u)
        return y, self.conditional_generation(y)

    # ------------------------------------------------------------------ steps
    def _terms(self, x_hat, x, y_hat, y, mu_z, logvar_z, mu_u, logvar_u, mu_z_uy, logvar_z_uy):
        return cond_loss(x_hat, x, y_hat, y, mu_u, logvar_u, mu_z, logvar_z, mu_z_uy, logvar_z_uy,
                         self.gammax, self.gammay)

    def train_step(self, batch, device):
        """cond_vae.py:326-354 (autograd-compatible path; fit() prefers fused_train_step).  Log values are
        0-dim device tensors (they accumulate in fit() without a host sync)."""
        y, x = batch
        y, x = y.to(device), x.to(device)
        x_hat, y_hat, mu_z, logvar_z, mu_u, logvar_u, mu_z_uy, logvar_z_uy = self.forward(x, y)
        mse_x, kld_u, mse_y, kld_z = self._terms(x_hat, x, y_hat, y, mu_z, logvar_z, mu_u, logvar_u, mu_z_uy, logvar_z_uy)
        loss = mse_x + kld_u + mse_y + kld_z
        logs = {"Loss/loss": loss.detach(), "Loss/mse_x": mse_x.detach(), "Loss/kld_u": kld_u.detach(),
                "Loss/mse_y": mse_y.detach(), "Loss/kld_z": kld_z.detach()}
        return loss, logs

    def fused_train_step(self, batch, device, fused):
        """zero_grad + train_step + backward + clip + Adam as one kernel chain (models/base.py:103-107)."""
        y, x = batch
        y = y.to(device, non_blocking=True)
        x = x.to(device, non_blocking=True)
        t = fused.step(x, y, use_graph=self.use_cuda_graph)
        t = t.clone()
        logs = {"Loss/loss": t[4], "Loss/mse_x": t[0], "Loss/kld_u": t[1], "Loss/mse_y": t[2], "Loss/kld_z": t[3]}
        return t[4], logs

    def val_step(self, batch, device):
        """cond_vae.py:356-385."""
        y, x = batch
        y, x = y.to(device), x.to(device)
        with torch.no_grad():
            outs = self(x, y)
            mse_x, kld_u, mse_y, kld_z = self._terms(outs[0], x, outs[1], y, *outs[2:])
            loss = mse_x + kld_u + mse_y + kld_z
        logs = {"Loss/val_loss": loss, "Loss/val_mse_x": mse_x, "Loss/val_kld_u": kld_u,
                "Loss/val_mse_y": mse_y, "Loss/val_kld_z": kld_z}
        return loss, logs

    # ------------------------------------------------------------------ epoch-rate hooks
    def evaluate(self, val_loader, wandb_run, epoch, full_val=False):
        """cond_vae.py:387-525.  On full-validation epochs the SSIM metrics (skimage's structural_similarity with
        win_size=11, data_range=1.0, averaged over the validation images) are computed on the device (svrs_native.metrics);
        SSIM_LR is not logged when the LR patches are smaller than the window (patch_size < 22).  LPIPS needs pretrained
        AlexNet weights and is not computed.  Image logging keeps the reference's keys."""
        from svrs_native import metrics
        device = next(self.parameters()).device
        batch = next(iter(val_loader))
        y, x = [t.to(device) for t in batch]
        with torch.no_grad():
            x_hat, y_hat, *_ = self.forward(x, y)
            x_sr = self.conditional_generation(y)
        keys = [k for k, img in (("Metrics/SSIM_LR", y), ("Metrics/SSIM_HR", x), ("Metrics/SSIM_SR", x))
                if min(img.shape[-2:]) >= 11]
        if full_val and keys:
            tot = {k: torch.zeros((), device=device, dtype=torch.float64) for k in keys}
            cnt = 0
            for b in val_loader:
                yy, xx = [t.to(device) for t in b]
                with torch.no_grad():
                    xh, yh, *_ = self.forward(xx, yy)
                    sr = self.conditional_generation(yy)
                pairs = {"Metrics/SSIM_LR": (yy, yh), "Metrics/SSIM_HR": (xx, xh), "Metrics/SSIM_SR": (xx, sr)}
                for k in keys:
                    tot[k] += metrics.ssim(*pairs[k]).sum()
                cnt += yy.size(0)
            vals = torch.stack([tot[k] for k in keys]).tolist()         # one host read for all metrics
            wandb_run.log({k: v / cnt for k, v in zip(keys, vals)}, step=epoch)
        if epoch % 10 == 0 or epoch == 1:
            imgs = {"Images/LR_Input": y[:4], "Images/HR_Input": x[:4], "Images/LR_Recon": y_hat[:4],
                    "Images/HR_Recon": x_hat[:4], "Images/SR_Output": x_sr[:4]}
            try:
                wandb_run.log({k: [wandb.Image(i.permute(1, 2, 0).cpu().numpy()) for i in v] for k, v in imgs.items()},
                              step=epoch)
            except Exception:
                pass

    def on_train_start(self, **kwargs):
        """cond_vae.py:527-582: the gammas join the optimizer as a second param group (same lr, unclipped).
        The bicubic SSIM/LPIPS baseline of the reference is not computed (LPIPS needs pretrained AlexNet weights); a cached
        baseline_ckpt.pth is loaded."""
        self.gammax.requires_grad = True
        self.gammay.requires_grad = True
        have = {id(p) for g in self.optimizer.param_groups for p in g["params"]}
        if id(self.gammax) not in have:
            self.optimizer.add_param_group({"params": [self.gammax, self.gammay]})
        if self.val_loader is None:
            raise ValueError("Validation loader must be provided for baseline evaluation.")
        self.ssim_base, self.lpips_base = float("nan"), float("nan")
        if os.path.exists("baseline_ckpt.pth"):
            try:
                baseline = torch.load("baseline_ckpt.pth")
                self.ssim_base, self.lpips_base = baseline["ssim_base"], baseline["lpips_base"]
            except Exception:
                pass

    def on_train_epoch_end(self, **kwargs):
        """cond_vae.py:584-592."""
        self.wandb_run.log({"HyperParameters/Gamma_X": self.gammax.item(), "HyperParameters/Gamma_Y": self.gammay.item(),
                            "HyperParameters/Learning Rate": self.scheduler.get_last_lr()[0]}, step=self.current_epoch)

    def get_task_data(self, val_loader):
        """cond_vae.py:594-603: second sample of the first validation batch."""
        y, x = next(iter(val_loader))
        dev = next(self.parameters()).device
        return y.to(dev)[1:2], x.to(dev)[1:2]
