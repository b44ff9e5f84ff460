"""Stand-ins for the TyXe@368bf62 names bayesrul touches (bayesrul/models/bayesian.py:50-98,146,149):
tyxe.priors.IIDPrior, tyxe.likelihoods.HeteroskedasticGaussian, tyxe.guides.AutoNormal /
PretrainedInitializer, tyxe.bnn.VariationalBNN, tyxe.poutine.local_reparameterization / flipout.
The objects only carry configuration; the arithmetic is the CUDA engine's."""
from __future__ import annotations

import contextlib
import copy
from typing import Optional

import torch

from ..engine import Engine, Noise
from . import pyro_shim

_CTX_STACK = []  # active fit context: "lrt" | "flipout"


@contextlib.contextmanager
def local_reparameterization():
    _CTX_STACK.append("lrt")
    try:
        yield
    finally:
        _CTX_STACK.pop()


@contextlib.contextmanager
def flipout():
    _CTX_STACK.append("flipout")
    try:
        yield
    finally:
        _CTX_STACK.pop()


def active_context() -> Optional[str]:
    return _CTX_STACK[-1] if _CTX_STACK else None


class Normal:
    """pyro.distributions.Normal(loc, scale) as used for the IID prior (bayesian.py:50-64)."""

    def __init__(self, loc, scale):
        self.loc, self.scale = float(loc), float(scale)


class IIDPrior:
    def __init__(self, distribution, **kwargs):
        if kwargs.get("hide_all") or kwargs.get("hide"):
            raise NotImplementedError("bayesrul exposes every parameter (expose_all=True, bayesian.py:49)")
        self.loc, self.scale = float(distribution.loc), float(distribution.scale)


class HeteroskedasticGaussian:
    def __init__(self, dataset_size: int, positive_scale: bool = False):
        if positive_scale:
            raise NotImplementedError("bayesrul uses positive_scale=False (bayesian.py:73-76)")
        self.dataset_size, self.positive_scale = int(dataset_size), positive_scale


class PretrainedInitializer:
    def __init__(self, theta: torch.Tensor):
        self.theta = theta

    @classmethod
    def from_net(cls, net):
        return cls(net.flat().detach().clone())


class AutoNormal:
    """Per-site Normal(loc, scale); trainable state = flat `loc` [P] and `log_scale` [P]."""

    family = "normal"

    def __init__(self, net, init_scale: float = 1e-1, init_loc_fn=None, prior: Optional[IIDPrior] = None):
        dev = net.flat().device
        self.net = net
        if isinstance(init_loc_fn, PretrainedInitializer):
            self.loc = init_loc_fn.theta.to(dev).clone()
        else:
            # init_to_median: median of 15 prior draws per element (SURVEY A.2)
            g = torch.Generator(device="cpu").manual_seed(torch.initial_seed() % (2**31))
            pl, ps = (prior.loc, prior.scale) if prior else (0.0, 1.0)
            draws = pl + ps * torch.randn(15, net.P, generator=g)
            self.loc = draws.median(0).values.to(dev)
        self.log_scale = torch.full((net.P,), float(init_scale), device=dev).log()
        self.scale = self.log_scale.exp()
        pending = pyro_shim.get_param_store().pending()
        pend = dict(pending)
        pyro_shim.get_param_store().bind(self)
        if pend:
            pyro_shim.get_param_store().set_state({"params": pend})
            self.refresh()

    def refresh(self):
        torch.exp(self.log_scale, out=self.scale)

    def named_site_views(self):
        for name, (off, shape) in zip(self.net.site_names, self.net._sites):
            n = 1
            for s in shape:
                n *= s
            yield ("net_guide.net." + name, self.loc[off: off + n].view(shape), self.log_scale[off: off + n].view(shape))


class guides:  # namespace mirror of tyxe.guides
    AutoNormal = AutoNormal
    PretrainedInitializer = PretrainedInitializer


class VariationalBNN:
    """tyxe.bnn.VariationalBNN(net, prior, likelihood, guide_builder)."""

    def __init__(self, net, prior: IIDPrior, likelihood: HeteroskedasticGaussian, net_guide_builder, engine="simt",
                 train_backend="auto"):
        self.net, self.prior, self.likelihood = net, prior, likelihood
        try:
            self.net_guide = net_guide_builder(net, prior=prior)
        except TypeError:
            self.net_guide = net_guide_builder(net)
        self.engine_kind = engine
        # kernels of the ELBO step: "auto" = the level-fused tcgen05 kernels where they exist (Inception: LRT, Flipout and the
        # weight-sampling ELBO; fp16 / bf16 operands, loss 5e-3, gradient cosine > 0.999), else the fp32 FFMA kernels; "simt" = always the fp32 parity
        # back-end (rtol 1e-3 against the oracle); "fused" / "tc" force a back-end ("fused" also covers the Linear and Conv-D3
        # nets, with the same bound)
        self.train_backend = train_backend
        self.seed = int(torch.initial_seed() % (2**62))
        self._step = 0
        self._last_kl = None

    @property
    def engine(self) -> Engine:
        return self.net.engine()

    # handles passed to SVI / poutine.scale (bayesian.py:111-129)
    class _Handle:
        def __init__(self, owner, is_model):
            self.__self__, self._is_model = owner, is_model

    @property
    def model(self):
        if not hasattr(self, "_model_h"):
            self._model_h = VariationalBNN._Handle(self, True)
        return self._model_h

    @property
    def guide(self):
        if not hasattr(self, "_guide_h"):
            self._guide_h = VariationalBNN._Handle(self, False)
        return self._guide_h

    def __call__(self, x):
        """One guided forward (a fresh weight draw, or LRT / flipout if the caller sits in the context)."""
        return self.predict(x, num_predictions=1, aggregate=False)[0]

    def _noise(self):
        self._step += 1
        return Noise(seed=(self.seed + 0x9E3779B97F4A7C15 * self._step) & 0xFFFFFFFFFFFFFFFF)

    def _elbo(self, x, y, particles: int, analytic_kl: bool, grads: bool):
        g = self.net_guide
        ctx = active_context()
        mode = ctx if (ctx and g.family == "normal") else "ws"
        N = self.likelihood.dataset_size
        be = self.train_backend
        if be == "auto":
            be = "fused" if getattr(self.net, "kind", "") == "inception" else "simt"  # lrt / flipout / weight sampling (radial)
        self.engine.set_gemm_backend(be)
        res = self.engine.elbo_step(x.contiguous(), y.reshape(-1).contiguous(), g.loc, g.scale, mode=mode, guide=g.family,
                                    particles=particles, prior_loc=self.prior.loc, prior_scale=self.prior.scale,
                                    dataset_size=N, noise=self._noise(), compute_grads=grads)
        res["c"] = 1.0 / (N * 30 * 18)
        self._last_kl = res["scalars"][2]
        self._last_out = res["out"]
        return res

    def predict(self, x, num_predictions: int = 1, aggregate: bool = True):
        """[S,B,2] (aggregate=False) or the precision-weighted [B,2] aggregate (A.5)."""
        g = self.net_guide
        ctx = active_context()
        nz = self._noise()
        if ctx == "lrt" and g.family == "normal":
            out = self.engine.forward(x.contiguous(), "lrt", theta=g.loc, sigma=g.scale, S=num_predictions, noise=nz)
        else:
            w = self.engine.sample_weights(g.loc, g.scale, g.family, num_predictions, nz)
            if ctx == "flipout" and g.family == "normal":
                out = self.engine.forward(x.contiguous(), "flipout", theta=g.loc, wsamp=w, S=num_predictions, noise=nz)
            else:
                out = self.engine.forward(x.contiguous(), "ws", wsamp=w, S=num_predictions, noise=nz, engine=self.engine_kind)
        return self.engine.aggregate_predictions(out) if aggregate else out

    def predict_moments(self, x, num_predictions: int):
        """Fused S-sample forward + moment reduction ([S,B,2] never materialised)."""
        g = self.net_guide
        return self.engine.predict_moments(x.contiguous(), g.loc, g.scale, S=num_predictions, guide=g.family,
                                           noise=self._noise(), engine=self.engine_kind)

    def predict_moments_host(self, x_host, num_predictions: int, first_fraction: float = 0.25, n_chunks: int = 2):
        """predict_moments for a HOST batch (pinned memory for a truly asynchronous copy): the windows travel in
        chunks on a copy stream while the previous chunk is being computed, so only the first (small) chunk's
        transfer is exposed.  The weight draws do not depend on the window index and per-window noise is keyed by
        the global window index (Noise.window0), so the result equals the un-chunked call."""
        g = self.net_guide
        dev = g.loc.device
        B = x_host.shape[0]
        if n_chunks == 0:  # the library's own host entry point (window chunks share the packed weight images)
            out = self.engine.predict_moments_host(x_host, g.loc, g.scale, S=num_predictions, guide=g.family,
                                                   noise=self._noise(), engine=self.engine_kind)
            return tuple(out[i] for i in range(4))
        if B < 2048 or n_chunks < 2:
            return self.predict_moments(x_host.to(dev, non_blocking=True), num_predictions)
        first = max(512, int(B * first_fraction))
        rest = (B - first + n_chunks - 2) // (n_chunks - 1)
        bounds = [0, first]
        while bounds[-1] < B:
            bounds.append(min(B, bounds[-1] + rest))
        if getattr(self, "_xstage", None) is None or self._xstage.shape[0] < B:
            self._xstage = torch.empty((B,) + tuple(x_host.shape[1:]), device=dev)
            self._copy_stream = torch.cuda.Stream(dev)
        stage, cs, main = self._xstage, self._copy_stream, torch.cuda.current_stream(dev)
        cs.wait_stream(main)  # the staging buffer may still be read by the previous call's kernels
        events = []
        with torch.cuda.stream(cs):
            for a, b in zip(bounds[:-1], bounds[1:]):
                stage[a:b].copy_(x_host[a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cs)
                events.append(ev)
        nz = self._noise()
        outs = [torch.empty(B, device=dev) for _ in range(4)]
        for (a, b), ev in zip(zip(bounds[:-1], bounds[1:]), events):
            main.wait_event(ev)
            part = self.engine.predict_moments(stage[a:b], g.loc, g.scale, S=num_predictions, guide=g.family,
                                               noise=Noise(seed=nz.seed, window0=nz.window0 + a), engine=self.engine_kind)
            for o, p in zip(outs, part):
                o[a:b] = p
        return tuple(outs)


class bnn:  # namespace mirror of tyxe.bnn
    VariationalBNN = VariationalBNN


class priors:
    IIDPrior = IIDPrior


class likelihoods:
    HeteroskedasticGaussian = HeteroskedasticGaussian


class poutine:
    local_reparameterization = staticmethod(local_reparameterization)
    flipout = staticmethod(flipout)
