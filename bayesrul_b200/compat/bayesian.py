"""`BNN`: mirror of bayesrul.models.bayesian.BNN (bayesian.py:20-260) on top of the CUDA engine.

Same constructor / hyper-parameters, same hook names, same logged keys, same return values and the
same checkpoint key ("param_store").  pytorch_lightning is optional: when it is not installed the class
derives from a small stand-in that provides `save_hyperparameters`, `hparams`, `log` and `device`.
Differences are confined to performance: `svi.step` is one fused CUDA ELBO step; the extra
`bnn.predict` + KL-only passes of training_step (bayesian.py:149-155) reuse that step's outputs
(same distribution, no second and third forward).
"""
from __future__ import annotations

import os
import contextlib
import copy
from functools import partial
from types import SimpleNamespace

import torch

from . import pyro_shim as pyro
from . import tyxe_shim as tyxe
from .nets import weights_init
from .radial import AutoRadial

try:  # pragma: no cover - optional dependency
    import pytorch_lightning as pl

    _Base = pl.LightningModule
except Exception:  # noqa: BLE001

    class _Base(torch.nn.Module):
        """Stand-in for pl.LightningModule (hooks are called by the user / tests / bench)."""

        def __init__(self):
            super().__init__()
            self.hparams = SimpleNamespace()
            self.logged = {}
            self.trainer = None
            self._device = None

        def save_hyperparameters(self, logger=False, ignore=()):
            import inspect

            frame = inspect.currentframe().f_back
            args = inspect.getargvalues(frame)
            for k in args.args:
                if k not in ("self",) and k not in ignore:
                    setattr(self.hparams, k, args.locals[k])

        def log(self, name, value, **kw):
            self.logged[name] = value

        @property
        def device(self):
            if self._device is not None:
                return self._device
            p = next(self.parameters(), None)
            return p.device if p is not None else torch.device("cpu")


class BNN(_Base):
    """Variational BNN wrapper (bayesian.py:20-43)."""

    def __init__(self, net, optimizer, pretrain_epochs, mc_samples_train: int, mc_samples_eval: int, dataset_size: int,
                 fit_context: str, prior_loc: float, prior_scale: float, guide: str, q_scale: float, device=None,
                 engine: str = "simt", train_backend: str = "auto"):
        super().__init__()
        pyro.clear_param_store()
        self.save_hyperparameters(logger=False, ignore=["net", "device", "engine", "train_backend"])
        self.net = net
        self._engine_kind = engine
        self._train_backend = train_backend
        if device is not None:
            self._device = torch.device(device)
            self.net.to(self._device)

    def define_bnn(self) -> None:  # bayesian.py:45-98
        if not self.hparams.pretrain_epochs == 0:
            self.net.apply(weights_init)
        prior = tyxe.priors.IIDPrior(tyxe.Normal(self.hparams.prior_loc, self.hparams.prior_scale))
        if self.hparams.fit_context == "lrt":
            self.fit_ctxt = tyxe.poutine.local_reparameterization
        elif self.hparams.fit_context == "flipout":
            self.fit_ctxt = tyxe.poutine.flipout
        else:
            self.fit_ctxt = contextlib.nullcontext
        likelihood = tyxe.likelihoods.HeteroskedasticGaussian(self.hparams.dataset_size, positive_scale=False)
        guide_kwargs = {"init_scale": self.hparams.q_scale}
        if self.hparams.guide == "normal":
            guide_base = tyxe.guides.AutoNormal
        elif self.hparams.guide == "radial":
            guide_base = AutoRadial
            self.fit_ctxt = contextlib.nullcontext
        else:
            raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
        if self.hparams.pretrain_epochs > 0:
            guide_kwargs["init_loc_fn"] = tyxe.guides.PretrainedInitializer.from_net(self.net)
        guide = partial(guide_base, **guide_kwargs)
        self.net.to(self.device)
        self.bnn = tyxe.VariationalBNN(self.net, prior, likelihood, guide, engine=self._engine_kind,
                                       train_backend=self._train_backend)

    def on_fit_start(self) -> None:  # bayesian.py:100-132
        self.define_bnn()
        param_store_to(self.device)
        self.configure_optimizers()
        self.loss = (pyro.TraceMeanField_ELBO(self.hparams.mc_samples_train) if self.hparams.guide != "radial"
                     else pyro.Trace_ELBO(self.hparams.mc_samples_train))
        scale = 1.0 / (self.hparams.dataset_size * self.net.win_length * self.net.n_features)
        self.svi = pyro.SVI(pyro.poutine.scale(self.bnn.model, scale=scale), pyro.poutine.scale(self.bnn.guide, scale=scale),
                            self.hparams.optimizer, self.loss)

    def _agg(self, out, n):
        # bnn.predict(aggregate = n > 1) (bayesian.py:149-153): precision-weighted aggregate when n > 1
        return self.bnn.engine.aggregate_predictions(out) if n > 1 else out[0]

    def _train_batch(self, x, y):
        """svi.step on one batch; the values training_step logs (bayesian.py:134-166)."""
        with self.fit_ctxt():
            elbo = self.svi.step(x, y.unsqueeze(-1))
            output = self._agg(self.svi.last["out"], self.hparams.mc_samples_train)
            loc, scale = output[:, 0], output[:, 1]
            kl = float(self.svi.last["scalars"][2].item())
        m = self.bnn.engine.step_metrics(loc, scale, y)  # mse, sharpness, rmsce (+ nll, mace) in one fused pass (N3)
        mse, sharp, rmsce = m[1].item(), m[2].float(), m[3].float()
        return {"mse/train": mse, "elbo/train": elbo, "kl/train": kl, "likelihood/train": elbo - kl, "rmsce/train": rmsce,
                "sharp/train": sharp}

    def training_step(self, batch, batch_idx):  # bayesian.py:134-166
        for k, v in self._train_batch(batch[0], batch[1]).items():
            self.log(k, v, on_step=False, on_epoch=True)

    def fit_epoch(self, x, y, batch_size: int, generator=None):
        """One training epoch over the DEVICE-resident split x [N,30,18], y [N]: what Lightning's fit does with training_step
        over the shuffled batches of a DataLoader, without a host round trip per batch.  The permutation is
        torch.randperm(N, generator=generator, device=x.device); its floor(N / batch_size) full batches run as ONE
        Engine.elbo_train_steps call, which continues the seed sequence of the BNN's steps and ClippedAdam's step count and
        advances both; the remainder batch goes through training_step.  Logs the epoch means of the keys training_step logs,
        each batch weighted by its size as Lightning's epoch mean weighs it, and returns dict(scalars [K,1,4], metrics [K,1,5],
        perm) of the K full batches (Engine.elbo_train_steps)."""
        N, bs = int(x.shape[0]), int(batch_size)
        if bs <= 0 or y.numel() != N:
            raise RuntimeError("bayesrul_b200: fit_epoch needs batch_size > 0 and one target per window")
        bnn, svi = self.bnn, self.svi
        opt, g = svi.optim, bnn.net_guide
        grad_factor = svi.model_scale / (1.0 / (bnn.likelihood.dataset_size * 30 * 18))  # what SVI.step multiplies the gradients by
        if svi.no_obs or grad_factor != 1.0 or not (hasattr(opt, "step_vi") and g.loc.is_contiguous() and g.log_scale.is_contiguous()):
            raise RuntimeError("bayesrul_b200: fit_epoch runs the ClippedAdam step of a mean-field guide at the ELBO's own scale")
        perm = torch.randperm(N, generator=generator, device=x.device)
        K = N // bs
        x, y = x.contiguous(), y.reshape(-1).contiguous()
        res = None
        sums, weight = {}, 0
        if K > 0:
            with self.fit_ctxt():
                ctx = tyxe.active_context()
            mode = ctx if (ctx and g.family == "normal") else "ws"
            be = bnn.train_backend
            if be == "auto":
                be = "fused" if getattr(self.net, "kind", "") == "inception" else "simt"
            eng = bnn.engine
            eng.set_gemm_backend(be)
            sts = [opt._slot(name, p) for name, p in (("loc", g.loc), ("log_scale", g.log_scale))]
            a = opt.args
            res = eng.elbo_train_steps(x, y, perm[: K * bs].view(K, bs), g.loc, g.log_scale, g.scale,
                                       (sts[0]["m"], sts[0]["v"], sts[1]["m"], sts[1]["v"]), step0=sts[0]["step"], lr=a["lr"],
                                       betas=tuple(a["betas"]), eps=a["eps"], clip_norm=a["clip_norm"], lrd=a["lrd"],
                                       weight_decay=a["weight_decay"], mode=mode, guide=g.family,
                                       particles=self.hparams.mc_samples_train, prior_loc=bnn.prior.loc, prior_scale=bnn.prior.scale,
                                       dataset_size=bnn.likelihood.dataset_size,
                                       seed=(bnn.seed + 0x9E3779B97F4A7C15 * bnn._step) & 0xFFFFFFFFFFFFFFFF)
            bnn._step += K
            for st in sts:
                st["step"] += K
            bnn._last_kl = res["scalars"][K - 1, 0, 2]
            sc, mt = res["scalars"][:, 0], res["metrics"][:, 0]
            elbo, kl = sc[:, 0].sum(), sc[:, 2].sum()
            sums = {"mse/train": mt[:, 1].sum(), "elbo/train": elbo, "kl/train": kl, "likelihood/train": elbo - kl,
                    "rmsce/train": mt[:, 3].float().double().sum(), "sharp/train": mt[:, 2].float().double().sum()}  # logged as float32
            sums = {k: v * bs for k, v in sums.items()}
            weight = K * bs
        if K * bs < N:
            rest = perm[K * bs:]
            vals = self._train_batch(x[rest], y[rest])
            for k, v in vals.items():
                sums[k] = sums.get(k, 0.0) + v * rest.numel()
            weight += rest.numel()
        means = torch.stack([torch.as_tensor(v, dtype=torch.float64, device=x.device) for v in sums.values()]).div(weight).tolist()
        for k, v in zip(sums, means):
            self.log(k, v, on_step=False, on_epoch=True)
        return dict(scalars=res["scalars"] if res else None, metrics=res["metrics"] if res else None, perm=perm)

    def _val_batch(self, x, y):
        """svi.evaluate_loss, the predictive and the metrics of one batch; the values validation_step logs (bayesian.py:168-197)"""
        elbo = self.svi.evaluate_loss(x, y.unsqueeze(-1))
        kl = float(self.svi.last["scalars"][2].item())
        output = self.bnn.predict(x, num_predictions=self.hparams.mc_samples_eval,
                                  aggregate=self.hparams.mc_samples_eval > 1)
        if output.dim() == 3:
            output = output[0]
        loc, scale = output[:, 0], output[:, 1]
        m = self.bnn.engine.step_metrics(loc, scale, y)
        return {"elbo/val": elbo, "mse/val": m[1].float(), "kl/val": kl, "likelihood/val": elbo - kl, "rmsce/val": m[3].float(),
                "sharp/val": m[2].float()}

    def validation_step(self, batch, batch_idx):  # bayesian.py:168-197 (no fit context: weight sampling)
        for k, v in self._val_batch(batch[0], batch[1]).items():
            self.log(k, v)

    def validate_epoch(self, x, y, batch_size: int):
        """One validation epoch over the DEVICE-resident split x [N,30,18], y [N]: what Lightning does with validation_step over
        the batches of an unshuffled DataLoader, without two host reads per batch.  The floor(N / batch_size) full batches of
        arange(N), in order, run as ONE Engine.elbo_val_steps call with the BNN's guide, mc_samples_train particles,
        mc_samples_eval predictive samples, engine and ELBO back-end; it continues the BNN's seed sequence (two keys per batch, as
        validation_step draws them) and advances it.  The remainder batch goes through validation_step's own path.  Logs the epoch
        means of the keys validation_step logs, each batch weighted by its size as Lightning's epoch mean weighs it, each with the
        type validation_step logs it with; returns dict(scalars [K,4], metrics [K,5]) of the K full batches."""
        N, bs = int(x.shape[0]), int(batch_size)
        if bs <= 0 or y.numel() != N:
            raise RuntimeError("bayesrul_b200: validate_epoch needs batch_size > 0 and one target per window")
        bnn, svi = self.bnn, self.svi
        loss_factor = svi.model_scale / (1.0 / (bnn.likelihood.dataset_size * 30 * 18))  # what evaluate_loss multiplies the loss by
        if svi.no_obs or loss_factor != 1.0:
            raise RuntimeError("bayesrul_b200: validate_epoch evaluates the ELBO at its own scale (a scaled or KL-only loss is not supported)")
        K = N // bs
        x, y = x.contiguous(), y.reshape(-1).contiguous()
        res = None
        sums, weight = {}, 0
        if K > 0:
            g, eng = bnn.net_guide, bnn.engine
            be = bnn.train_backend
            if be == "auto":
                be = "fused" if getattr(self.net, "kind", "") == "inception" else "simt"
            eng.set_gemm_backend(be)
            idx = torch.arange(K * bs, device=x.device).view(K, bs)
            res = eng.elbo_val_steps(x, y, idx, g.loc, g.scale, guide=g.family, particles=self.hparams.mc_samples_train,
                                     S=self.hparams.mc_samples_eval, prior_loc=bnn.prior.loc, prior_scale=bnn.prior.scale,
                                     dataset_size=bnn.likelihood.dataset_size,
                                     seed=(bnn.seed + 0x9E3779B97F4A7C15 * bnn._step) & 0xFFFFFFFFFFFFFFFF, engine=bnn.engine_kind)
            bnn._step += 2 * K
            bnn._last_kl = res["scalars"][K - 1, 2]
            sc, mt = res["scalars"], res["metrics"]
            elbo, kl = sc[:, 0].sum(), sc[:, 2].sum()
            f32 = lambda t: t.float().double().sum()  # logged as float32 by validation_step
            sums = {"elbo/val": elbo, "mse/val": f32(mt[:, 1]), "kl/val": kl, "likelihood/val": elbo - kl, "rmsce/val": f32(mt[:, 3]),
                    "sharp/val": f32(mt[:, 2])}
            sums = {k: v * bs for k, v in sums.items()}
            weight = K * bs
        if K * bs < N:
            vals = self._val_batch(x[K * bs:], y[K * bs:])
            for k, v in vals.items():
                sums[k] = sums.get(k, 0.0) + (v.double() if isinstance(v, torch.Tensor) else v) * (N - K * bs)
            weight += N - K * bs
        tensor_keys = ("mse/val", "rmsce/val", "sharp/val")
        means = torch.stack([torch.as_tensor(v, dtype=torch.float64, device=x.device) for v in sums.values()]).div(weight).tolist()
        for k, v in zip(sums, means):
            self.log(k, torch.tensor(v, dtype=torch.float32, device=x.device) if k in tensor_keys else v)
        return dict(scalars=res["scalars"] if res else None, metrics=res["metrics"] if res else None)

    def on_test_start(self) -> None:
        self.define_bnn()
        param_store_to(self.device)

    def test_step(self, batch, batch_idx):  # bayesian.py:203-225
        (x, y) = batch[0].to(self.device, non_blocking=True), batch[1].to(self.device, non_blocking=True)
        loc, scale, _, _ = self.bnn.predict_moments(x, self.hparams.mc_samples_eval)
        m = self.bnn.engine.step_metrics(loc, scale, y)  # nll, mse, sharpness, rmsce (+ mace) in one pass
        self.log("nll/test", m[0])
        self.log("mse/test", m[1])
        self.log("rmsce/test", m[3])
        self.log("sharp/test", m[2])
        return m[0]

    def on_predict_start(self) -> None:
        self.define_bnn()
        param_store_to(self.device)

    def predict_step(self, batch, batch_idx, dataloader_idx=0):  # bayesian.py:231-250
        pred = dict()
        if batch[0].device.type == "cpu" and batch[0].dtype == torch.float32 and int(os.environ.get("BRL_HOST_CHUNKS", "0")) != 1:
            # host batch (the DataLoader's): brl_predict_moments_host copies it in window chunks underneath the compute and
            # writes the four result vectors into one pinned host tensor.  (BRL_HOST_CHUNKS >= 2: the Python-level chunking,
            # measured slower: every extra call repeats the weight sampling / packing; = 1: plain .to(device) + device call.)
            loc, scale, ep_var, al_var = self.bnn.predict_moments_host(
                batch[0], self.hparams.mc_samples_eval, float(os.environ.get("BRL_HOST_FIRST", "0.25")),
                int(os.environ.get("BRL_HOST_CHUNKS", "0")))
        else:
            loc, scale, ep_var, al_var = self.bnn.predict_moments(batch[0].to(self.device), self.hparams.mc_samples_eval)
        packed = torch.stack([ep_var, al_var, loc, scale]).cpu()  # one D2H instead of four
        pred["labels"] = batch[1].cpu().numpy()
        pred["ep_vars"], pred["al_vars"], pred["preds"], pred["stds"] = (packed[i].numpy() for i in range(4))
        return pred

    def configure_optimizers(self):
        return None

    def on_save_checkpoint(self, checkpoint):  # bayesian.py:255-257
        checkpoint["param_store"] = pyro.get_param_store().get_state()

    def on_load_checkpoint(self, checkpoint):  # bayesian.py:259-264
        pyro.get_param_store().set_state(checkpoint["param_store"])
        if not hasattr(self, "bnn") and "state_dict" in checkpoint:
            checkpoint["state_dict"] = remove_dict_entry_startswith(checkpoint["state_dict"], "bnn")


def param_store_to(device):  # bayesian.py:267-271
    ps = pyro.get_param_store().get_state()
    moved = {k: v.to(device) for k, v in ps["params"].items()}
    if any(moved[k] is not ps["params"][k] for k in moved):
        pyro.get_param_store().set_state({"params": moved, "constraints": ps["constraints"]})


def remove_dict_entry_startswith(dictionary, string):
    return {k: v for k, v in dictionary.items() if not k.startswith(string)}
