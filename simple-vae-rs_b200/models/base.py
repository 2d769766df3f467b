"""BaseVAE: the reference's Keras-style training interface (models/base.py:16-348), re-hosted on the
sm_100a kernel path.

Kept from the reference: constructor signature, attributes (`callbacks`, `optimizer`, `scheduler`,
`val_loader`, `current_epoch`, `wandb_run`, `num_params`, `latent_size`, `patch_size`), `fit()` kwargs and
control flow (ReduceLROnPlateau(min, 0.5, patience=500) :51-53; callbacks :86-93,167-178; NaN guard :125-128),
`log`, `task`, and the abstract method set.  Changed: the per-batch body (:103-116) runs as ONE fused kernel
chain (svrs_native.trainer) when the optimizer is Adam on a CUDA device, and loss terms stay on the device
until the epoch ends (the reference pays six `.item()` syncs per step).
"""
from __future__ import annotations

import abc
import os
from math import isnan
from typing import List, Optional

import torch
import torch.nn as nn

try:  # logging backend of the reference (models/base.py:62-79); tests monkeypatch wandb.init
    import wandb
except Exception:  # pragma: no cover - wandb is optional for the hot path
    class _NoWandb:
        @staticmethod
        def init(*a, **k):
            return None

        @staticmethod
        def Image(x):
            return x

    wandb = _NoWandb()

from callbacks import Callback


class _NullRun:
    def log(self, *a, **k):
        pass

    def finish(self):
        pass


def _as_float(v):
    return float(v.item()) if isinstance(v, torch.Tensor) else float(v)


class BaseVAE(nn.Module, metaclass=abc.ABCMeta):
    """Common training / validation interface of VAE and Cond_SRVAE."""

    #: compute dtype of the kernel path: torch.float32 (parity mode) or torch.bfloat16 (throughput mode)
    compute_dtype = torch.float32

    def __init__(self, patch_size: int = 64, callbacks: Optional[List[Callback]] = None, slurm_job_id: str = "local"):
        super().__init__()
        self.latent_size: int = 0
        self.slurm_job_id: str = slurm_job_id
        self.patch_size: int = patch_size
        self.callbacks: List[Callback] = [] if callbacks is None else callbacks
        self.num_params: int = 0
        self.lpips_fn = None
        self._eng = None
        self._trainer = None
        self._anchor = None
        self.use_cuda_graph = os.environ.get("SVRS_CUDA_GRAPH", "1") == "1"
        # data parallel only: BatchNorm statistics of the GLOBAL batch (per-layer all-reduce of the 2C sums) - exact parity with
        # a single process on the global batch; default = per-rank statistics (standard DDP)
        self.sync_bn = os.environ.get("SVRS_SYNC_BN", "0") == "1"

    # ------------------------------------------------------------------ kernel engine plumbing
    def set_compute_dtype(self, dtype: torch.dtype):
        """fp32 = bit-faithful parity mode; bf16 = tensor-core throughput mode."""
        self.compute_dtype = dtype
        if self._eng is not None:
            self._eng.rt.set_dtype(dtype)
        return self

    def _make_engine(self, dtype):
        raise NotImplementedError

    def _engine(self, dtype=None):
        if dtype is not None and dtype != self.compute_dtype:
            self.set_compute_dtype(dtype)
        if self._eng is None:
            self._eng = self._make_engine(self.compute_dtype)
        return self._eng

    def _grad_anchor(self, device):
        if self._anchor is None or self._anchor.device != device:
            self._anchor = torch.zeros((), device=device, requires_grad=True)
        return self._anchor

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Reference checkpoints written with the real `lpips` package carry `lpips_fn.*` entries
        (callbacks.py:140-153 saves model.state_dict()); they are not part of this model."""
        sd = {k: v for k, v in state_dict.items() if not k.startswith("lpips_fn.")}
        out = super().load_state_dict(sd, strict=strict, assign=assign)
        if self._eng is not None:
            self._eng.rt.packs_dirty = True
        if self._trainer is not None:
            self._trainer.rt.packs_dirty = True
        return out

    def _fused_trainer(self, optimizer):
        raise NotImplementedError

    def _can_fuse(self, optimizer, device) -> bool:
        return (torch.device(device).type == "cuda" and type(optimizer) is torch.optim.Adam
                and not optimizer.param_groups[0].get("amsgrad", False)
                and optimizer.param_groups[0].get("weight_decay", 0) == 0
                and os.environ.get("SVRS_FUSED_STEP", "1") == "1")

    # ------------------------------------------------------------------ fit
    def fit(self, train_loader, val_loader, device, optimizer, epochs=1000, **kwargs):
        """Same contract as the reference's BaseVAE.fit (models/base.py:40-185)."""
        self.val_loader = val_loader
        self.optimizer = optimizer
        self.scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(self.optimizer, mode="min", factor=0.5, patience=500)
        self.current_epoch: int = 0
        start_epoch = kwargs.get("start_epoch", 1)
        val_metrics_every = kwargs.get("val_metrics_every", float("inf"))
        first, _ = next(iter(train_loader))
        # data parallel (torchrun, one process per GPU): the loaders shard every global batch by rank (dataset.py), the fused
        # trainer SUM-all-reduces the gradients; logging / checkpoint files belong to rank 0, stop decisions are agreed on
        dist_on = torch.distributed.is_available() and torch.distributed.is_initialized()
        rank = torch.distributed.get_rank() if dist_on else 0
        world = torch.distributed.get_world_size() if dist_on else 1
        self.rank, self.world = rank, world
        try:
            self.wandb_run = _NullRun() if rank != 0 else wandb.init(
                project=self.__class__.__name__,
                name=f"Latent-{self.latent_size}-Patch-{self.patch_size}-SLURM-{kwargs.get('slurm_job_id', 'local')}",
                entity="ebardet-isae-supaero",
                config=kwargs.get("config", {
                    "latent_size": self.latent_size, "patch_size": self.patch_size, "epochs": epochs,
                    "batch_size": first.size(0), "val_metrics_every": val_metrics_every,
                    "slurm_job_id": kwargs.get("slurm_job_id", "local"), "Parameter_number": self.num_params,
                    "cr": self.cr}),
            ) or _NullRun()
        except Exception as e:  # no network on the box: keep training, drop logging
            print(f"wandb.init failed ({e}); continuing without a wandb run")
            self.wandb_run = _NullRun()

        if torch.device(device).type != "cuda":
            raise RuntimeError(
                f"fit(device={device!r}): this build runs the training step on hand-written sm_100a kernels only; "
                "there is no CPU path. Use the reference implementation for CPU runs.")
        self.on_train_start()
        fused = self._fused_trainer(optimizer) if self._can_fuse(optimizer, device) else None

        for epoch in range(start_epoch, epochs + 1):
            self.current_epoch = epoch
            for cb in self.callbacks:
                if self._agree(cb.on_epoch_begin(epoch=epoch, optimizer=optimizer, device=device, model=self), device):
                    print(f"Stopping training before epoch {epoch} due to {cb.__class__.__name__} condition.")
                    return
            self.train()
            terms_dict = {}
            train_loss = 0.0
            for batch in train_loader:
                if fused is not None:
                    # Philox eps is keyed by the GLOBAL sample index: this rank's first sample inside the global batch
                    fused.eng.rng.sample_offset = getattr(train_loader, "sample_offset", rank * batch[0].shape[0])
                    loss, terms = self.fused_train_step(batch, device, fused)
                else:
                    optimizer.zero_grad()
                    loss, terms = self.train_step(batch, device)
                    loss.backward()
                    torch.nn.utils.clip_grad_norm_(self.parameters(), 1.0)
                    optimizer.step()
                for key, value in terms.items():
                    terms_dict[key] = terms_dict[key] + value if key in terms_dict else value
                train_loss = train_loss + loss.detach()
            if fused is not None:
                fused.sync_to_model()
            nb = len(train_loader)
            terms_dict = {k: _as_float(v) / nb for k, v in terms_dict.items()}   # one sync per epoch
            self.terms_dict = terms_dict
            train_loss = _as_float(train_loss) / nb
            self.log(self.wandb_run, terms_dict, step=epoch)
            if isnan(train_loss):
                raise ValueError(f"NaN detected in training loss at epoch {epoch}. Check your model and data.")

            self.on_train_epoch_end()
            self.eval()
            val_terms_dict = {}
            val_loss = 0.0
            with torch.no_grad():
                for batch in val_loader:
                    loss, terms = self.val_step(batch, device)
                    for key, value in terms.items():
                        val_terms_dict[key] = val_terms_dict[key] + value if key in val_terms_dict else value
                    val_loss = val_loss + loss.detach()
                full_val = epoch % val_metrics_every == 0 or epoch in [1, epochs]
                self.evaluate(val_loader, self.wandb_run, epoch, full_val=full_val)
            nv = len(val_loader)
            val_terms_dict = {k: _as_float(v) / nv for k, v in val_terms_dict.items()}
            val_loss = _as_float(val_loss) / nv
            if self.scheduler:
                self.scheduler.step(val_loss)
            self.log(self.wandb_run, val_terms_dict, step=epoch)
            for cb in self.callbacks:
                if self._agree(cb.on_epoch_end(epoch=epoch, optimizer=optimizer, device=device, model=self, logs=val_terms_dict), device):
                    print(f"Stopping training after epoch {epoch} due to {cb.__class__.__name__} condition.")
                    return
            print(f"Epoch {epoch}/{epochs}, Train Loss: {train_loss:.4f}, Val Loss: {val_loss:.4f}")

        self.wandb_run.finish()
        return

    def fused_train_step(self, batch, device, fused):
        raise NotImplementedError

    def _agree(self, stop, device) -> bool:
        """A callback's stop decision, made identical on every rank (any rank that wants to stop stops all)."""
        stop = bool(stop)
        if getattr(self, "world", 1) > 1:
            t = torch.tensor([int(stop)], device=device)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            stop = bool(int(t))
        return stop

    # ------------------------------------------------------------------ abstract interface (base.py:187-291)
    @abc.abstractmethod
    def forward(self, *args, **kwargs):
        raise NotImplementedError("forward must be implemented in the derived class.")

    @abc.abstractmethod
    def train_step(self, batch, device):
        raise NotImplementedError("train_step must be implemented in the derived class.")

    @abc.abstractmethod
    def val_step(self, batch, device):
        raise NotImplementedError("val_step must be implemented in the derived class.")

    @abc.abstractmethod
    def evaluate(self, val_loader, wandb_run, epoch, full_val):
        raise NotImplementedError("evaluate must be implemented in the derived class.")

    def log(self, wandb_run, logs: dict, step=None):
        if not wandb_run:
            print("WandB run not initialized, skipping logging.")
            return
        if step is not None:
            wandb_run.log(logs, step=step)

    @abc.abstractmethod
    def on_train_start(self, **kwargs):
        pass

    @abc.abstractmethod
    def on_train_epoch_end(self, **kwargs):
        pass

    @abc.abstractmethod
    def sample(self, y, samples=1000):
        raise NotImplementedError("sample must be implemented in the derived class.")

    @abc.abstractmethod
    def get_task_data(self, val_loader):
        raise NotImplementedError("get_task_data must be implemented in the derived class.")

    # ------------------------------------------------------------------ task (base.py:293-348)
    def task(self, val_loader, samples: int = 1000):
        """Monte-Carlo uncertainty maps from `samples` posterior draws.  The per-pixel statistics of the
        reference are computed and saved as tensors; the matplotlib figure is drawn only if matplotlib is
        installed (plotting is outside the hot-path scope)."""
        results_dir = os.path.join("results", f"{self.slurm_job_id}_CRx{self.cr}")
        os.makedirs(results_dir, exist_ok=True)
        pred, target = self.get_task_data(val_loader)
        if hasattr(self, "sample_stats"):
            # fused path (SURVEY 8.4 row f4): the statistics are accumulated inside the decoder tail kernel while the draws
            # are produced; the [S,4,P,P] sample stack of base.py:303 is never materialised
            with torch.no_grad():
                st = self.sample_stats(pred, samples=samples, target=target)
            stats = {"mean": st["mean"][0].cpu(), "std": st["std"][0].cpu(), "mae": st["mae"][0].cpu(), "mse": st["mse"][0].cpu(),
                     "mean_bias": st["mean_bias"][0].cpu(), "target": target.cpu(), "sample0": st["sample0"][0].cpu()}
            mmse = stats["mse"].mean()          # == (samples - target).pow(2).mean()   (base.py:346)
        else:
            with torch.no_grad():
                draws = self.sample(pred, samples=samples)
            diff = draws - target
            stats = {
                "mean": draws.mean(dim=0).cpu(),
                "std": draws.std(dim=0).mean(dim=0).cpu(),
                "mae": diff.abs().mean(dim=(0, 1)).cpu(),
                "mse": diff.pow(2).mean(dim=(0, 1)).cpu(),
                "mean_bias": (target - draws.mean(dim=0)).mean(dim=0).mean(dim=0).cpu(),
                "target": target.cpu(),
                "sample0": draws[0].cpu(),
            }
            mmse = diff.pow(2).mean()
        torch.save(stats, os.path.join(results_dir, "error_mean_std_maps.pt"))
        try:
            import matplotlib
            matplotlib.use("Agg")
            import matplotlib.pyplot as plt

            panels = [("Input Image", stats["target"][0, [2, 1, 0]].permute(1, 2, 0), None),
                      ("Sampled Image", stats["sample0"][[2, 1, 0]].permute(1, 2, 0), None),
                      ("Mean of Samples", stats["mean"][[2, 1, 0]].permute(1, 2, 0), None),
                      ("MAE Map", stats["mae"], "hot"), ("MSE Map", stats["mse"], "hot"),
                      (f"STD of Samples, Mean: {stats['std'].mean():.2f}", stats["std"], "hot"),
                      (f"Mean Bias Map, Mean: {stats['mean_bias'].mean():.2f}", stats["mean_bias"], "hot")]
            plt.figure(figsize=(20, 10))
            for i, (title, img, cmap) in enumerate(panels):
                plt.subplot(2, 4, i + 1)
                plt.imshow(img.numpy(), cmap=cmap)
                plt.title(title)
            plt.savefig(f"{results_dir}/error_mean_std_maps.png", bbox_inches="tight")
            plt.close()
        except Exception:
            pass
        print(f"MMSE: {mmse:.4f}")
        return stats
