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

    def _train_backend_of_net(self):
        """the back-end of the training step: "auto" is the level-fused kernels for the Inception net, the fp32 ones otherwise"""
        be = self._train_backend
        if be == "auto":
            be = "fused" if getattr(self.net, "kind", "") == "inception" else "simt"
        return be

    def _step(self, x, y, phase):
        """HNN.step without its log: (loss, loc, scale)"""
        train = phase == "train"
        p = float(self.net.dropout) if (train or getattr(self.net, "mc_dropout", False)) else 0.0
        self.net.engine().set_gemm_backend(self._train_backend_of_net())
        res = self.net.engine().hnn_step(x.contiguous(), y.contiguous(), self.net.flat(), p, self._noise(), compute_grads=train)
        loss = res["scalars"][0].float()
        if train:  # the returned loss carries a grad_fn whose backward writes the fused step's gradient into param.grad
            loss = _FusedStepLoss.apply(loss, res["grad"], tuple(self.net._sites), *self.net._params)
        return loss, res["out"][:, 0], res["out"][:, 1]

    def step(self, batch, phase):  # frequentist.py:39-48
        (x, y) = batch
        if phase == "predict":
            output = self.net(x)
            return output[:, 0], output[:, 1]
        loss, loc, scale = self._step(x, y, phase)
        self.log(f"nll/{phase}", loss, on_step=False, on_epoch=True)
        return loss, loc, scale

    def _train_batch(self, x, y):
        """the training step on one batch: (loss, the values training_step logs, in its order)"""
        loss, loc, scale = self._step(x, y, "train")
        m = self.net.engine().step_metrics(loc, scale, y)  # mse, sharpness, rmsce in one fused pass (N3)
        return loss, {"nll/train": loss, "mse/train": m[1].float(), "rmsce/train": m[3].float(), "sharp/train": m[2].float()}

    def training_step(self, batch, batch_idx):
        loss, vals = self._train_batch(batch[0], batch[1])
        for k, v in vals.items():
            self.log(k, v, on_step=False, on_epoch=True)
        return loss

    def _adam_group(self, optimizer):
        """the one param group of `optimizer` if it is a torch.optim.Adam over exactly the net's site parameters whose update
        Engine.adam computes (amsgrad, maximize, differentiable, capturable, fused and decoupled weight decay off); else raises"""
        why = None
        if type(optimizer) is not torch.optim.Adam:
            why = f"runs torch.optim.Adam, got {type(optimizer).__name__}"
        elif len(optimizer.param_groups) != 1:
            why = f"needs one param group, got {len(optimizer.param_groups)}"
        else:
            g = optimizer.param_groups[0]
            sites = self.net._params
            theta = self.net.flat()
            if len(g["params"]) != len(sites) or {id(p) for p in g["params"]} != {id(p) for p in sites}:
                why = "needs the param group to hold exactly the net's site parameters"
            elif any(p.data_ptr() != theta.data_ptr() + 4 * off for p, (off, _) in zip(sites, self.net._sites)):
                why = "needs the site parameters to be the views of net.flat()"
            else:
                on = [k for k in ("amsgrad", "maximize", "differentiable", "capturable", "fused", "decoupled_weight_decay") if g.get(k)]
                if on:
                    why = f"runs Adam without {', '.join(on)}"
        if why:
            raise RuntimeError(f"bayesrul_b200: HNN.fit_epoch {why}")
        return optimizer.param_groups[0]

    def fit_epoch(self, x, y, batch_size: int, optimizer, generator=None):
        """One training epoch over the DEVICE-resident split x [N,30,18], y [N]: what Lightning's fit does with training_step and
        the torch.optim.Adam `optimizer` that configure_optimizers() returned, over the shuffled batches of a DataLoader, without
        a host round trip per batch.  The permutation is torch.randperm(N, generator=generator, device=x.device); its
        floor(N / batch_size) full batches run as ONE Engine.hnn_train_steps(optimizer="adam") call with the dropout rate and
        back-end of training_step, continuing the seed sequence of the HNN's steps and the optimizer's step count.  The
        optimizer's per-site exp_avg / exp_avg_sq go in as flat [P] buffers and come back, and each state["step"] advances by
        the number of full batches.  The remainder batch goes through training_step, zero_grad, backward and optimizer.step, as
        Lightning's automatic optimisation runs it.  Logs the epoch means of the keys training_step logs, each batch weighted by
        its size as Lightning's epoch mean weighs it, and returns dict(scalars [K,1,2], metrics [K,1,5], perm) of the K full
        batches (Engine.hnn_train_steps)."""
        N, bs = int(x.shape[0]), int(batch_size)
        if bs <= 0 or y.numel() != N:
            raise RuntimeError("bayesrul_b200: fit_epoch needs batch_size > 0 and one target per window")
        group = self._adam_group(optimizer)
        net, theta = self.net, self.net.flat()
        perm = torch.randperm(N, generator=generator, device=x.device)
        K = N // bs
        x, y = x.contiguous(), y.reshape(-1).contiguous()
        res = None
        sums, weight = {}, 0
        if K > 0:
            states = [optimizer.state.get(p) for p in net._params]
            steps = {float(st["step"]) if st else 0.0 for st in states}
            if len(steps) != 1:
                raise RuntimeError("bayesrul_b200: HNN.fit_epoch needs every site parameter at the same Adam step")
            # exp_avg / exp_avg_sq in net.flat() order, in buffers kept from epoch to epoch: stable addresses let a later epoch
            # replay the step graph the first one captured
            if getattr(self, "_flat_moments", None) is None or self._flat_moments[0].shape != theta.shape or \
                    self._flat_moments[0].device != theta.device:
                self._flat_moments = (torch.empty_like(theta), torch.empty_like(theta))
            m, v = self._flat_moments
            m.zero_()
            v.zero_()
            for st, (off, _) in zip(states, net._sites):
                if st:
                    n = st["exp_avg"].numel()
                    m[off: off + n].copy_(st["exp_avg"].reshape(-1))
                    v[off: off + n].copy_(st["exp_avg_sq"].reshape(-1))
            eng = net.engine()
            eng.set_gemm_backend(self._train_backend_of_net())
            res = eng.hnn_train_steps(x, y, perm[: K * bs].view(K, bs), theta, (m, v), step0=int(steps.pop()), lr=float(group["lr"]),
                                      betas=tuple(float(b) for b in group["betas"]), eps=float(group["eps"]),
                                      weight_decay=float(group["weight_decay"]), p_dropout=float(net.dropout),
                                      seed=(torch.initial_seed() + 0x9E3779B97F4A7C15 * self._it) & 0xFFFFFFFFFFFFFFFF,
                                      optimizer="adam")
            self._it += K
            for p, st, (off, _) in zip(net._params, states, net._sites):
                if not st:  # Adam's lazy state: a CPU step counter of the default scalar dtype, moments shaped as the parameter
                    st = optimizer.state[p]
                    st["step"] = torch.tensor(0.0, dtype=torch.float64 if torch.get_default_dtype() == torch.float64 else torch.float32)
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                n = p.numel()
                st["exp_avg"].copy_(m[off: off + n].view_as(st["exp_avg"]))
                st["exp_avg_sq"].copy_(v[off: off + n].view_as(st["exp_avg_sq"]))
                st["step"] += K
            sc, mt = res["scalars"][:, 0], res["metrics"][:, 0]
            sums = {"nll/train": sc[:, 0], "mse/train": mt[:, 1], "rmsce/train": mt[:, 3], "sharp/train": mt[:, 2]}
            sums = {k: t.float().double().sum() * bs for k, t in sums.items()}  # each logged as float32
            weight = K * bs
        if K * bs < N:
            rest = perm[K * bs:]
            loss, vals = self._train_batch(x[rest], y[rest])
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            for k, val in vals.items():
                sums[k] = sums.get(k, 0.0) + val.detach().double() * rest.numel()
            weight += rest.numel()
        means = torch.stack([torch.as_tensor(val, dtype=torch.float64, device=x.device) for val in sums.values()]).div(weight).tolist()
        for k, val in zip(sums, means):
            self.log(k, val, on_step=False, on_epoch=True)
        return dict(scalars=res["scalars"] if res else None, metrics=res["metrics"] if res else None, perm=perm)

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
