"""`HNN`: mirror of bayesrul.models.frequentist.HNN (frequentist.py:9-154) -- heteroscedastic NN /
MC-dropout wrapper.  `step` runs the fused CUDA forward (+ backward when training); `mc_sampling`
is ONE batched launch sequence over all S dropout masks instead of a Python loop of S net calls."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from ..engine import Noise
from .bayesian import _Base
from .nets import enable_dropout, weights_init


class _FusedStepLoss(torch.autograd.Function):
    """Autograd node of the fused step.  brl_hnn_step has already computed d loss / d theta (one flat vector); this node
    hands its per-site slices to autograd, so `loss.backward()` -- Lightning's automatic optimisation runs training_step,
    `optimizer.zero_grad()`, `loss.backward()`, `optimizer.step()` in that order -- fills `param.grad` like the reference's
    autograd graph does (frequentist.py:39-48)."""

    @staticmethod
    def forward(ctx, loss, grad_flat, sites, *params):
        ctx.grad_flat, ctx.sites = grad_flat, sites
        return loss.clone()

    @staticmethod
    def backward(ctx, g):
        grads = []
        for off, shape in ctx.sites:
            n = 1
            for d in shape:
                n *= d
            grads.append(g * ctx.grad_flat[off: off + n].view(shape))
        return (None, None, None, *grads)


class HNN(_Base):
    def __init__(self, net, optimizer, mc_samples: int, p_dropout, device=None, engine: str = "simt", train_backend: str = "auto"):
        super().__init__()
        self.save_hyperparameters(logger=False, ignore=["net", "device", "engine", "train_backend"])
        self.net = net
        self.net.apply(weights_init)
        self._engine_kind = engine
        # kernels of HNN.step: "auto" = the level-fused tcgen05 kernels for the Inception net (fp16 / bf16 operands: loss 5e-3,
        # gradient cosine > 0.999 of the fp32 oracle), the fp32 FFMA kernels for the other nets; "fused" also runs the level-fused
        # kernels on the Linear and Conv-D3 nets (same bound); "simt" forces the fp32 parity back-end
        self._train_backend = train_backend
        self._it = 0
        if device is not None:
            self._device = torch.device(device)
            self.net.to(self._device)

    def forward(self, x):
        return self.net(x)

    def get_device(self):
        return next(self.net.parameters()).device

    def to_device(self, device: torch.device):
        self.net.to(device)

    def _noise(self):
        self._it += 1
        return Noise(seed=(torch.initial_seed() + 0x9E3779B97F4A7C15 * self._it) & 0xFFFFFFFFFFFFFFFF)

    def step(self, batch, phase):  # frequentist.py:39-48
        (x, y) = batch
        if phase == "predict":
            output = self.net(x)
            return output[:, 0], output[:, 1]
        train = phase == "train"
        p = float(self.net.dropout) if (train or getattr(self.net, "mc_dropout", False)) else 0.0
        be = self._train_backend
        if be == "auto":
            be = "fused" if getattr(self.net, "kind", "") == "inception" else "simt"
        self.net.engine().set_gemm_backend(be)
        res = self.net.engine().hnn_step(x.contiguous(), y.contiguous(), self.net.flat(), p, self._noise(), compute_grads=train)
        loss = res["scalars"][0].float()
        if train:  # the returned loss carries a grad_fn whose backward writes the fused step's gradient into param.grad
            loss = _FusedStepLoss.apply(loss, res["grad"], tuple(self.net._sites), *self.net._params)
        self.log(f"nll/{phase}", loss, on_step=False, on_epoch=True)
        return loss, res["out"][:, 0], res["out"][:, 1]

    def training_step(self, batch, batch_idx):
        loss, loc, scale = self.step(batch, "train")
        m = self.net.engine().step_metrics(loc, scale, batch[1])  # mse, sharpness, rmsce in one fused pass (N3)
        self.log("mse/train", m[1].float(), on_step=False, on_epoch=True)
        self.log("rmsce/train", m[3].float(), on_step=False, on_epoch=True)
        self.log("sharp/train", m[2].float(), on_step=False, on_epoch=True)
        return loss

    def mc_sampling(self, batch, mc_samples: int, phase: str, agg: bool = True):  # frequentist.py:60-81
        (x, y) = batch
        eng = self.net.engine()
        out = eng.forward(x.contiguous(), "det", theta=self.net.flat(), S=mc_samples, p_dropout=float(self.net.dropout),
                          noise=self._noise(), engine=self._engine_kind)
        locs, scales = out[:, :, 0], out[:, :, 1]
        if phase == "predict":
            return locs, scales
        loss = F.gaussian_nll_loss(locs, y.expand_as(locs), scales**2, reduction="none").mean(1).mean(0)
        if agg:
            pred, std, _, _ = eng.moments(out)
            return loss, pred, std
        return loss, locs, scales

    def validation_step(self, batch, batch_idx):
        phase = "val"
        if self.net.dropout > 0:
            enable_dropout(self.net)
            loss, loc, scale = self.mc_sampling(batch, self.hparams.mc_samples, phase=phase)
        else:
            loss, loc, scale = self.step(batch, phase)
        return {"loss": loss, "label": batch[1], "pred": loc, "std": scale}

    def validation_epoch_end(self, outputs) -> None:
        preds = torch.cat([o["pred"].detach() for o in outputs])
        labels = torch.cat([o["label"].detach() for o in outputs])
        stds = torch.cat([o["std"].detach() for o in outputs])
        m = self.net.engine().step_metrics(preds.contiguous(), stds.contiguous(), labels.contiguous())
        self.log("mse/val", m[1].float())
        self.log("rmsce/val", m[3].float())
        self.log("sharp/val", m[2].float())

    def _mc_moments(self, batch):
        x = batch[0]
        return self.net.engine().predict_moments(x.contiguous(), self.net.flat(), None, S=self.hparams.mc_samples, guide=None,
                                                 p_dropout=float(self.net.dropout), noise=self._noise(),
                                                 engine=self._engine_kind)

    def test_step(self, batch, batch_idx):  # frequentist.py:112-130
        y = batch[1]
        if self.net.dropout > 0:
            enable_dropout(self.net)
            loss, locs, scales = self.mc_sampling(batch, self.hparams.mc_samples, phase="test", agg=False)
            loc, scale, _, _ = self.net.engine().moments(torch.stack([locs, scales], -1).contiguous())
        else:
            loss, loc, scale = self.step(batch, "test")
        m = self.net.engine().step_metrics(loc.contiguous(), scale.contiguous(), y.contiguous())
        self.log("nll/test", loss)
        self.log("mse/test", m[1].float())
        self.log("rmsce/test", m[3].float())
        self.log("sharp/test", m[2].float())

    def predict_step(self, batch, batch_idx, dataloader_idx=0):  # frequentist.py:132-151
        pred = dict()
        pred["labels"] = batch[1].cpu().numpy()
        if self.net.dropout > 0 and batch[0].device.type == "cpu" and batch[0].dtype == torch.float32:
            # MC-dropout on a host batch (the DataLoader's): brl_predict_moments_host -- chunked copy underneath the compute
            enable_dropout(self.net)
            out = self.net.engine().predict_moments_host(batch[0], self.net.flat(), None, S=self.hparams.mc_samples, guide=None,
                                                         p_dropout=float(self.net.dropout), noise=self._noise(),
                                                         engine=self._engine_kind)
            pred["ep_vars"], pred["al_vars"] = out[2].numpy(), out[3].numpy()
            pred["preds"], pred["stds"] = out[0].numpy(), out[1].numpy()
            return pred
        batch = (batch[0].to(self.get_device(), non_blocking=True), batch[1])
        if self.net.dropout > 0:
            enable_dropout(self.net)
            loc, scale, ep_var, al_var = self._mc_moments(batch)
            pred["ep_vars"] = ep_var.cpu().numpy()
            pred["al_vars"] = al_var.cpu().numpy()
        else:
            loc, scale = self.step(batch, "predict")
        pred["preds"] = loc.cpu().numpy()
        pred["stds"] = scale.cpu().numpy()
        return pred

    def configure_optimizers(self):
        return self.hparams.optimizer(params=self.parameters())
