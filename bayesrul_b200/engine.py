"""Thin PyTorch-side host of the C ABI: tensors in, tensors out, device memory and streams from torch.

`Engine(net)` owns a `brl_ctx` and a grow-on-demand workspace tensor.  Every method validates its
inputs (device, dtype, contiguity, shape) and raises RuntimeError on failure -- no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib
from ._lib import ENGINE_IDS, GUIDE_IDS, MODE_IDS, NET_IDS, BrlNoise

WIN_LENGTH, N_FEATURES = 30, 18


@dataclass
class Noise:
    """Noise specification: Philox (seed) unless a tensor is injected (SURVEY Appendix C layouts)."""

    seed: int = 0
    sample0: int = 0
    window0: int = 0
    weight_eps: Optional[torch.Tensor] = None  # [S,P]
    radial_r: Optional[torch.Tensor] = None  # [S,n_sites]
    lrt_eps: Dict[int, torch.Tensor] = field(default_factory=dict)  # layer -> [S,B,out_elems]
    flip_in: Dict[int, torch.Tensor] = field(default_factory=dict)  # layer -> [S,B,Cin]
    flip_out: Dict[int, torch.Tensor] = field(default_factory=dict)  # layer -> [S,B,Cout]
    drop_mask: Dict[int, torch.Tensor] = field(default_factory=dict)  # layer -> [S,B,out_elems]

    def to_struct(self, device) -> Tuple[BrlNoise, list]:
        keep = []

        def ptr(t):
            if t is None:
                return None
            t = _chk(t, device, "noise tensor")
            keep.append(t)
            return t.data_ptr()

        s = BrlNoise()
        s.seed = self.seed & 0xFFFFFFFFFFFFFFFF
        s.sample0, s.window0 = int(self.sample0), int(self.window0)
        s.weight_eps, s.radial_r = ptr(self.weight_eps), ptr(self.radial_r)
        for name in ("lrt_eps", "flip_in", "flip_out", "drop_mask"):
            arr = getattr(s, name)
            for layer, t in getattr(self, name).items():
                arr[int(layer)] = ptr(t)
        return s, keep


def _chk(t: torch.Tensor, device, what: str, dtype=torch.float32) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise RuntimeError(f"bayesrul_b200: {what} must be a torch.Tensor")
    if t.device != device:
        raise RuntimeError(f"bayesrul_b200: {what} is on {t.device}, expected {device}")
    if t.dtype != dtype:
        raise RuntimeError(f"bayesrul_b200: {what} has dtype {t.dtype}, expected {dtype}")
    if not t.is_contiguous():
        raise RuntimeError(f"bayesrul_b200: {what} must be contiguous")
    return t


def net_info(net: str):
    """Static description from the library: P, sites [(offset, shape)], layers [(cout, cin, out_elems, drop_factor)]."""
    lib = _lib.load()
    nid = NET_IDS[net]
    P = lib.brl_net_num_params(nid)
    sites = []
    for j in range(lib.brl_net_num_sites(nid)):
        off, nd, shp = C.c_int64(), C.c_int(), (C.c_int64 * 4)()
        _lib.check(lib.brl_net_site(nid, j, C.byref(off), C.byref(nd), C.byref(shp)))
        sites.append((off.value, tuple(shp[i] for i in range(nd.value))))
    layers = []
    for l in range(lib.brl_net_num_layers(nid)):
        co, ci, oe, df = C.c_int(), C.c_int(), C.c_int(), C.c_float()
        _lib.check(lib.brl_net_layer(nid, l, C.byref(co), C.byref(ci), C.byref(oe), C.byref(df)))
        layers.append((co.value, ci.value, oe.value, df.value))
    return dict(P=P, sites=sites, layers=layers, flops_fwd=lib.brl_net_flops_fwd(nid))


class Engine:
    def __init__(self, net: str = "inception", device=None):
        if net not in NET_IDS:
            raise RuntimeError(f"bayesrul_b200: unknown net {net!r}")
        if not torch.cuda.is_available():
            raise RuntimeError("bayesrul_b200: no CUDA device available (B200 / sm_100a required, no CPU fallback)")
        self.lib = _lib.load()
        self.net = net
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.info = net_info(net)
        self.P = self.info["P"]
        ctx = C.c_void_p()
        _lib.check(self.lib.brl_create(C.byref(ctx), NET_IDS[net], self.device.index))
        self.ctx = ctx
        self._ws: Optional[torch.Tensor] = None
        self.max_workspace_bytes = 8 << 30  # 180 GB of HBM per GPU: S = 100 x B = 10 000 on the fused engine is one 4.9 GB pass

    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.lib.brl_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    def has_tc(self) -> bool:
        """True when the tcgen05 (fp16 operand / fp32 accumulate) engine supports this net."""
        return bool(self.lib.brl_engine_available(self.ctx, ENGINE_IDS["tc"]))
    def set_gemm_backend(self, backend: str) -> None:
        """'simt' (fp32 FFMA, parity back-end) or 'tc' (tcgen05 TF32 dual GEMMs) for the per-layer kernels of
        forward(engine='simt') / elbo_step / hnn_step."""
        _lib.check(self.lib.brl_set_gemm_backend(self.ctx, {"simt": 0, "tc": 7, "fused": 8}.get(backend, backend)))

    def set_step_graph(self, enable: bool) -> None:
        """CUDA-graph replay of elbo_step with native noise (on by default; identical results, far less host time)."""
        _lib.check(self.lib.brl_set_step_graph(self.ctx, int(enable)))

    def gemm_status(self) -> int:
        """0 = ok; else the code of the first mbarrier time-out inside a TF32 per-layer kernel (synchronises)."""
        return int(self.lib.brl_gemm_status())

    def tc_timing(self, enable: bool) -> None:
        """Bracket every tc_conv_kernel launch with CUDA events on the launching stream (bench.py roofline)."""
        _lib.check(self.lib.brl_tc_timing(self.ctx, int(enable)))

    def tc_timing_read(self):
        """{kernel: (summed milliseconds, launches)} since the last enable / read; synchronises the recorded events."""
        ms, n = (C.c_double * 2)(), (C.c_int64 * 2)()
        _lib.check(self.lib.brl_tc_timing_read(self.ctx, ms, n))
        return {"tc_conv_kernel": (ms[0], n[0]), "tc_fc_kernel": (ms[1], n[1])}

    def tc_status(self) -> int:
        """0 = ok; >0 = an mbarrier wait inside a tcgen05 kernel timed out (synchronises)."""
        return int(self.lib.brl_tc_status(self.ctx))


    # -- helpers ------------------------------------------------------------------------------
    def _on_device(self):
        """Context manager for the entry points that take no brl_ctx (moments, mixture, metrics, optimiser): their kernels
        launch on a stream of THIS engine's device, which must then be the current one (the ctx entry points guard
        themselves inside the library)."""
        return torch.cuda.device(self.device)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def workspace(self, nbytes: int) -> torch.Tensor:
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        return self._ws

    def _ws_for(self, B: int, S: int, train: bool, engine: str) -> torch.Tensor:
        n = self.lib.brl_workspace_bytes(self.ctx, B, S, int(train), ENGINE_IDS[engine])
        if n < 0:
            raise RuntimeError("bayesrul_b200: bad workspace query")
        return self.workspace(n)

    def _x(self, x: torch.Tensor) -> torch.Tensor:
        x = _chk(x, self.device, "x")
        if x.dim() != 3 or x.shape[1] != WIN_LENGTH or x.shape[2] != N_FEATURES:
            raise RuntimeError(f"bayesrul_b200: x must be [B,{WIN_LENGTH},{N_FEATURES}], got {tuple(x.shape)}")
        if x.shape[0] == 0:
            raise RuntimeError("bayesrul_b200: empty batch")
        return x

    def _theta(self, t: torch.Tensor, what: str, lead=()) -> torch.Tensor:
        t = _chk(t, self.device, what)
        if tuple(t.shape) != tuple(lead) + (self.P,):
            raise RuntimeError(f"bayesrul_b200: {what} must have shape {tuple(lead) + (self.P,)}, got {tuple(t.shape)}")
        return t

    def _noise(self, noise: Optional[Noise]):
        noise = noise if noise is not None else Noise()
        s, keep = noise.to_struct(self.device)
        return C.byref(s), (s, keep)

    # -- A7 / A8: guide samplers -----------------------------------------------------------------
    def sample_weights(self, mu, sigma, guide: str = "normal", S: int = 1, noise: Optional[Noise] = None,
                       return_delta: bool = False):
        mu, sigma = self._theta(mu, "mu"), self._theta(sigma, "sigma")
        if guide not in GUIDE_IDS:
            raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
        w = torch.empty(S, self.P, device=self.device)
        delta = torch.empty(S, self.P, device=self.device) if return_delta else None
        ws = self.workspace(max(4096, S * 64 * 4 + 1024))
        nz, keep = self._noise(noise)
        _lib.check(self.lib.brl_sample_weights(self.ctx, mu.data_ptr(), sigma.data_ptr(), GUIDE_IDS[guide], S, nz,
                                               w.data_ptr(), delta.data_ptr() if delta is not None else None,
                                               ws.data_ptr(), ws.numel(), self._stream()))
        return (w, delta) if return_delta else w

    # -- A1-A6: forward ----------------------------------------------------------------------------
    def forward(self, x, mode: str = "det", theta=None, sigma=None, wsamp=None, S: int = 1, p_dropout: float = 0.0,
                noise: Optional[Noise] = None, engine: str = "simt") -> torch.Tensor:
        x = self._x(x)
        B = x.shape[0]
        if mode not in MODE_IDS:
            raise RuntimeError(f"bayesrul_b200: unknown mode {mode!r}")
        if theta is not None:
            theta = self._theta(theta, "theta")
        if sigma is not None:
            sigma = self._theta(sigma, "sigma")
        if wsamp is not None:
            wsamp = self._theta(wsamp, "wsamp", (S,))
        out = torch.empty(S, B, 2, device=self.device)
        ws = self._ws_for(B, S, 2 if mode == "flipout" else 0, engine)
        nz, keep = self._noise(noise)
        p = lambda t: t.data_ptr() if t is not None else None
        _lib.check(self.lib.brl_forward(self.ctx, x.data_ptr(), B, S, MODE_IDS[mode], p(theta), p(sigma), p(wsamp),
                                        float(p_dropout), nz, out.data_ptr(), ENGINE_IDS[engine], ws.data_ptr(),
                                        ws.numel(), self._stream()))
        return out

    # -- A11 / A12: predictive moments ---------------------------------------------------------------
    def predict_moments(self, x, mu, sigma=None, S: int = 20, guide: Optional[str] = "normal", p_dropout: float = 0.0,
                        noise: Optional[Noise] = None, engine: str = "simt", chunk: Optional[int] = None):
        """Returns (pred, std, ep_var, al_var), each [B].  guide=None: MC-dropout / deterministic weights `mu`."""
        x = self._x(x)
        B = x.shape[0]
        mu = self._theta(mu, "mu")
        if guide is not None:
            if guide not in GUIDE_IDS:
                raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
            sigma = self._theta(sigma, "sigma")
        eid = ENGINE_IDS[engine]
        sc = min(S, chunk or (128 if engine == "tc" else 16))
        while sc > 1 and self.lib.brl_workspace_bytes(self.ctx, B, sc, 0, eid) > self.max_workspace_bytes:
            sc -= 1
        ws = self.workspace(self.lib.brl_workspace_bytes(self.ctx, B, sc, 0, eid))
        nbytes = self.lib.brl_workspace_bytes(self.ctx, B, sc, 0, eid)
        outs = [torch.empty(B, device=self.device) for _ in range(4)]
        nz, keep = self._noise(noise)
        _lib.check(self.lib.brl_predict_moments(self.ctx, x.data_ptr(), B, S, GUIDE_IDS[guide] if guide else -1,
                                                mu.data_ptr(), sigma.data_ptr() if sigma is not None else None,
                                                float(p_dropout), nz, *[o.data_ptr() for o in outs], eid,
                                                ws.data_ptr(), nbytes, self._stream()))
        return tuple(outs)

    def predict_moments_ensemble(self, x, mu, sigma=None, S: int = 20, guide: Optional[str] = "normal", p_dropout: float = 0.0,
                                 noise: Optional[Noise] = None, engine: str = "simt", chunk: Optional[int] = None):
        """predict_moments of M models over one batch x [B,30,18] in one call: mu (and sigma with a guide) [M,P].  Member m is
        predict_moments(x, mu[m], sigma[m], S, guide, p_dropout, noise with sample0 + m * S); injected noise is member-major
        ([M * S, ...]).  Returns (pred, std, ep_var, al_var), each an [M,B] view of one [4,M,B] tensor (pred / std are the
        inputs of mixture_moments).  `chunk` caps the draws per pass of the flattened M * S sample axis."""
        x = self._x(x)
        B = x.shape[0]
        mu = _chk(mu, self.device, "mu")
        if mu.dim() != 2 or mu.shape[0] == 0 or mu.shape[1] != self.P:
            raise RuntimeError(f"bayesrul_b200: mu must have shape (M, {self.P}), got {tuple(mu.shape)}")
        M = mu.shape[0]
        if guide is not None:
            if guide not in GUIDE_IDS:
                raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
            if sigma is None:
                raise RuntimeError("bayesrul_b200: sigma is required with a guide")
            sigma = self._theta(sigma, "sigma", (M,))
        eid = ENGINE_IDS[engine]
        sc = min(M * S, chunk or (128 if engine == "tc" else 16))
        while sc > 1 and self.lib.brl_workspace_bytes(self.ctx, B, sc, 0, eid) > self.max_workspace_bytes:
            sc -= 1
        nbytes = self.lib.brl_workspace_bytes(self.ctx, B, sc, 0, eid) + (M * 4 * B * 4 + 255) // 256 * 256  # + Welford state
        ws = self.workspace(nbytes)
        out = torch.empty(4, M, B, device=self.device)
        nz, keep = self._noise(noise)
        _lib.check(self.lib.brl_predict_moments_ensemble(self.ctx, x.data_ptr(), M, B, S, GUIDE_IDS[guide] if guide else -1,
                                                         mu.data_ptr(), sigma.data_ptr() if guide is not None else None,
                                                         float(p_dropout), nz, out.data_ptr(), eid, ws.data_ptr(), nbytes,
                                                         self._stream()))
        return tuple(out.unbind(0))

    def predict_moments_host(self, x_host: torch.Tensor, mu, sigma=None, S: int = 20, guide: Optional[str] = "normal",
                             p_dropout: float = 0.0, noise: Optional[Noise] = None, engine: str = "simt") -> torch.Tensor:
        """predict_moments for a HOST batch [B,30,18] (pinned memory makes the copies asynchronous).  Returns a pinned
        host tensor [4,B] = (pred, std, ep_var, al_var); the call synchronises the current stream before returning.
        On the fused engine the batch travels in window chunks while the previous chunk is computed."""
        if not isinstance(x_host, torch.Tensor) or x_host.device.type != "cpu" or x_host.dtype != torch.float32:
            raise RuntimeError("bayesrul_b200: x_host must be a float32 CPU tensor")
        if x_host.dim() != 3 or x_host.shape[1] != WIN_LENGTH or x_host.shape[2] != N_FEATURES or x_host.shape[0] == 0:
            raise RuntimeError(f"bayesrul_b200: x_host must be [B,{WIN_LENGTH},{N_FEATURES}], got {tuple(x_host.shape)}")
        x_host = x_host.contiguous()
        B = x_host.shape[0]
        mu = self._theta(mu, "mu")
        if guide is not None:
            if guide not in GUIDE_IDS:
                raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
            sigma = self._theta(sigma, "sigma")
        eid = ENGINE_IDS[engine]
        nbytes = self.lib.brl_workspace_bytes_host(self.ctx, B, S, eid)
        if nbytes < 0:
            raise RuntimeError("bayesrul_b200: bad workspace query")
        ws = self.workspace(nbytes)
        out = torch.empty(4, B, dtype=torch.float32, pin_memory=True)
        nz, keep = self._noise(noise)
        _lib.check(self.lib.brl_predict_moments_host(self.ctx, x_host.data_ptr(), B, S, GUIDE_IDS[guide] if guide else -1,
                                                     mu.data_ptr(), sigma.data_ptr() if sigma is not None else None,
                                                     float(p_dropout), nz, out.data_ptr(), eid, ws.data_ptr(), ws.numel(),
                                                     self._stream()))
        torch.cuda.current_stream(self.device).synchronize()
        return out

    def moments(self, out: torch.Tensor):
        out = _chk(out, self.device, "out")
        if out.dim() != 3 or out.shape[2] != 2:
            raise RuntimeError("bayesrul_b200: out must be [S,B,2]")
        S, B = out.shape[0], out.shape[1]
        r = [torch.empty(B, device=self.device) for _ in range(4)]
        with self._on_device():
            _lib.check(self.lib.brl_moments(out.data_ptr(), S, B, *[t.data_ptr() for t in r], self._stream()))
        return tuple(r)

    def aggregate_predictions(self, out: torch.Tensor) -> torch.Tensor:
        out = _chk(out, self.device, "out")
        S, B = out.shape[0], out.shape[1]
        agg = torch.empty(B, 2, device=self.device)
        with self._on_device():
            _lib.check(self.lib.brl_aggregate_predictions(out.data_ptr(), S, B, agg.data_ptr(), self._stream()))
        return agg

    # -- A9 / A10: ELBO step ---------------------------------------------------------------------------
    def elbo_step(self, x, y, mu, sigma, *, mode: str = "lrt", guide: str = "normal", particles: int = 1,
                  prior_loc: float = 0.0, prior_scale: float = 1.0, dataset_size: int, noise: Optional[Noise] = None,
                  compute_grads: bool = True, out_flat: Optional[torch.Tensor] = None):
        """One `svi.step` worth of work.  Returns dict(scalars[4] (device, float64: loss, nll_sum, kl, mse),
        grad_mu, grad_sigma, grad_log_sigma, out [particles,B,2])."""
        x = self._x(x)
        B = x.shape[0]
        y = _chk(y, self.device, "y")
        if y.numel() != B:
            raise RuntimeError(f"bayesrul_b200: y must have {B} elements")
        mu, sigma = self._theta(mu, "mu"), self._theta(sigma, "sigma")
        if guide not in GUIDE_IDS:
            raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
        if mode is None:
            mode = "ws"
        scalars = torch.empty(4, dtype=torch.float64, device=self.device)
        out = torch.empty(particles, B, 2, device=self.device)
        # ONE flat fp32 buffer [grad_mu | grad_log_sigma | 4 scalars | grad_sigma]: data-parallel ranks all-reduce its first
        # 2 P + 4 floats in a single collective (dist.allreduce_elbo_grads) -- no concatenation, no slicing copies
        # (`out_flat`: a caller-owned buffer of >= 2 P + 4 floats for the reduced part, e.g. symmetric memory of
        # dist.FlatGradAllReduce; grad_sigma then lives in its own tensor)
        flat, g = None, [None] * 3
        if compute_grads and out_flat is not None:
            flat = _chk(out_flat, self.device, "out_flat")
            if flat.numel() < 2 * self.P + 4:
                raise RuntimeError("bayesrul_b200: out_flat needs at least 2 P + 4 floats")
            g = [flat[: self.P], torch.empty(self.P, device=self.device), flat[self.P: 2 * self.P]]
        elif compute_grads:
            flat = torch.empty(3 * self.P + 4, device=self.device)
            g = [flat[: self.P], flat[2 * self.P + 4:], flat[self.P: 2 * self.P]]
        ws = self._ws_for(B, 2 if particles > 1 else 1, True, "simt")  # S >= 2: room for two particles side by side
        nz, keep = self._noise(noise)
        p = lambda t: t.data_ptr() if t is not None else None
        _lib.check(self.lib.brl_elbo_step(self.ctx, x.data_ptr(), y.data_ptr(), B, mu.data_ptr(), sigma.data_ptr(),
                                          MODE_IDS[mode], GUIDE_IDS[guide], particles, float(prior_loc),
                                          float(prior_scale), int(dataset_size), nz, int(compute_grads),
                                          scalars.data_ptr(), p(g[0]), p(g[1]), p(g[2]), out.data_ptr(), ws.data_ptr(),
                                          ws.numel(), self._stream()))
        return dict(scalars=scalars, grad_mu=g[0], grad_sigma=g[1], grad_log_sigma=g[2], out=out, flat=flat)

    def elbo_step_ensemble(self, x, y, mu, sigma, *, mode: str = "lrt", guide: str = "normal", particles: int = 1,
                           prior_loc: float = 0.0, prior_scale: float = 1.0, dataset_size: int, noise: Optional[Noise] = None,
                           compute_grads: bool = True):
        """elbo_step of M independent variational posteriors (the seeds of an experiment) in one call: x [M,B,30,18], y [M,B],
        mu / sigma [M,P].  Member m is elbo_step(x[m], y[m], mu[m], sigma[m], noise with sample0 + m * particles); injected
        noise is member-major, particle-minor ([M * particles, ...]).  Returns dict(scalars [M,4] (device, float64: loss,
        nll_sum, kl, mse), grad_mu, grad_sigma, grad_log_sigma [M,P], out [M,particles,B,2]).  clipped_adam_vi over the
        [M,P] stacks is elementwise: M independent optimisers."""
        x = _chk(x, self.device, "x")
        if x.dim() != 4 or x.shape[2] != WIN_LENGTH or x.shape[3] != N_FEATURES:
            raise RuntimeError(f"bayesrul_b200: x must be [M,B,{WIN_LENGTH},{N_FEATURES}], got {tuple(x.shape)}")
        M, B = x.shape[0], x.shape[1]
        if M == 0 or B == 0:
            raise RuntimeError("bayesrul_b200: empty ensemble or batch")
        y = _chk(y, self.device, "y")
        if tuple(y.shape) != (M, B):
            raise RuntimeError(f"bayesrul_b200: y must have shape {(M, B)}, got {tuple(y.shape)}")
        mu, sigma = self._theta(mu, "mu", (M,)), self._theta(sigma, "sigma", (M,))
        if guide not in GUIDE_IDS:
            raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
        if mode is None:
            mode = "ws"
        scalars = torch.empty(M, 4, dtype=torch.float64, device=self.device)
        out = torch.empty(M, particles, B, 2, device=self.device)
        g = [torch.empty(M, self.P, device=self.device) for _ in range(3)] if compute_grads else [None] * 3
        ws = self._ws_for(B, M, 4, "simt")
        nz, keep = self._noise(noise)
        p = lambda t: t.data_ptr() if t is not None else None
        _lib.check(self.lib.brl_elbo_step_ensemble(self.ctx, x.data_ptr(), y.data_ptr(), M, B, mu.data_ptr(), sigma.data_ptr(),
                                                   MODE_IDS[mode], GUIDE_IDS[guide], particles, float(prior_loc),
                                                   float(prior_scale), int(dataset_size), nz, int(compute_grads),
                                                   scalars.data_ptr(), p(g[0]), p(g[1]), p(g[2]), out.data_ptr(), ws.data_ptr(),
                                                   ws.numel(), self._stream()))
        return dict(scalars=scalars, grad_mu=g[0], grad_sigma=g[1], grad_log_sigma=g[2], out=out)

    # -- A13: HNN step -----------------------------------------------------------------------------------
    def hnn_step(self, x, y, theta, p_dropout: float = 0.0, noise: Optional[Noise] = None, compute_grads: bool = True,
                 out_grad: Optional[torch.Tensor] = None):
        x = self._x(x)
        B = x.shape[0]
        y = _chk(y, self.device, "y")
        theta = self._theta(theta, "theta")
        scalars = torch.empty(2, dtype=torch.float64, device=self.device)
        out = torch.empty(B, 2, device=self.device)
        grad = None
        if compute_grads:  # out_grad: a caller-owned buffer of >= P floats (e.g. dist.FlatGradAllReduce(...).flat)
            grad = _chk(out_grad, self.device, "out_grad")[: self.P] if out_grad is not None else torch.empty(self.P, device=self.device)
        ws = self._ws_for(B, 1, True, "simt")
        nz, keep = self._noise(noise)
        _lib.check(self.lib.brl_hnn_step(self.ctx, x.data_ptr(), y.data_ptr(), B, theta.data_ptr(), float(p_dropout), nz,
                                         int(compute_grads), scalars.data_ptr(),
                                         grad.data_ptr() if grad is not None else None, out.data_ptr(), ws.data_ptr(),
                                         ws.numel(), self._stream()))
        return dict(scalars=scalars, grad=grad, out=out)

    def hnn_step_ensemble(self, x, y, theta, p_dropout: float = 0.0, noise: Optional[Noise] = None, compute_grads: bool = True,
                          out_grad: Optional[torch.Tensor] = None):
        """hnn_step of the M members of a deep ensemble (models/deepens.py) in one call: x [M,B,30,18], y [M,B], theta [M,P].
        Member m is hnn_step(x[m], y[m], theta[m], p_dropout, noise with sample0 + m); injected masks are [M,B,out_elems].
        Returns dict(scalars [M,2] (device, float64: loss, mse), grad [M,P], out [M,B,2]).  torch.optim.Adam or clipped_adam
        over the [M,P] parameter tensor are elementwise: M independent optimisers."""
        x = _chk(x, self.device, "x")
        if x.dim() != 4 or x.shape[2] != WIN_LENGTH or x.shape[3] != N_FEATURES:
            raise RuntimeError(f"bayesrul_b200: x must be [M,B,{WIN_LENGTH},{N_FEATURES}], got {tuple(x.shape)}")
        M, B = x.shape[0], x.shape[1]
        if M == 0 or B == 0:
            raise RuntimeError("bayesrul_b200: empty ensemble or batch")
        y = _chk(y, self.device, "y")
        if tuple(y.shape) != (M, B):
            raise RuntimeError(f"bayesrul_b200: y must have shape {(M, B)}, got {tuple(y.shape)}")
        theta = self._theta(theta, "theta", (M,))
        scalars = torch.empty(M, 2, dtype=torch.float64, device=self.device)
        out = torch.empty(M, B, 2, device=self.device)
        grad = None
        if compute_grads:  # out_grad: a caller-owned buffer of >= M P floats
            if out_grad is not None:
                grad = _chk(out_grad, self.device, "out_grad")
                if grad.numel() < M * self.P:
                    raise RuntimeError(f"bayesrul_b200: out_grad needs at least {M * self.P} floats")
                grad = grad.view(-1)[: M * self.P].view(M, self.P)
            else:
                grad = torch.empty(M, self.P, device=self.device)
        ws = self._ws_for(B, M, 3, "simt")
        nz, keep = self._noise(noise)
        _lib.check(self.lib.brl_hnn_step_ensemble(self.ctx, x.data_ptr(), y.data_ptr(), M, B, theta.data_ptr(), float(p_dropout),
                                                  nz, int(compute_grads), scalars.data_ptr(),
                                                  grad.data_ptr() if grad is not None else None, out.data_ptr(), ws.data_ptr(),
                                                  ws.numel(), self._stream()))
        return dict(scalars=scalars, grad=grad, out=out)

    # -- K training steps per call over a device-resident dataset ---------------------------------------
    def _train_inputs(self, X, Y, idx, params, shared_idx=False):
        """Checks the dataset, the index tensor and the [M,P] (or [P] for M = 1) parameter / optimiser-state tensors; returns
        (X, Y, idx [K,M,B], M).  shared_idx: idx must be [K,B], the windows of every member (returned as [K,1,B]).  The index range
        check is one device reduction and one host read: the only synchronisation of a K-step call."""
        X = _chk(X, self.device, "X")
        if X.dim() != 3 or X.shape[1] != WIN_LENGTH or X.shape[2] != N_FEATURES or X.shape[0] == 0:
            raise RuntimeError(f"bayesrul_b200: X must be [N,{WIN_LENGTH},{N_FEATURES}] with N > 0, got {tuple(X.shape)}")
        N = X.shape[0]
        if X.data_ptr() % 16:
            raise RuntimeError("bayesrul_b200: X must be 16-byte aligned")
        Y = _chk(Y, self.device, "Y")
        if Y.numel() != N:
            raise RuntimeError(f"bayesrul_b200: Y must have {N} elements, got {Y.numel()}")
        lead = tuple(params[0][0].shape[:-1]) if isinstance(params[0][0], torch.Tensor) else ()
        if len(lead) > 1:
            raise RuntimeError(f"bayesrul_b200: parameters must be [M,{self.P}] or [{self.P}]")
        M = lead[0] if lead else 1
        for t, what in params:
            self._theta(t, what, lead)
        idx = _chk(idx, self.device, "idx", dtype=torch.int64)
        if shared_idx and idx.dim() != 2:
            raise RuntimeError(f"bayesrul_b200: idx must be [K,B] (every member sees the same windows), got {tuple(idx.shape)}")
        if idx.dim() == 2 and (shared_idx or not lead):
            idx = idx.view(idx.shape[0], 1, idx.shape[1])
        if idx.dim() != 3 or idx.shape[1] != (1 if shared_idx else M) or idx.shape[0] == 0 or idx.shape[2] == 0:
            raise RuntimeError(f"bayesrul_b200: idx must be [K,{M},B] (or [K,B] for one member) with K, B > 0, got {tuple(idx.shape)}")
        lo, hi = torch.stack(torch.aminmax(idx)).tolist()
        if lo < 0 or hi >= N:
            raise RuntimeError(f"bayesrul_b200: idx holds windows outside [0, {N}): min {lo}, max {hi}")
        return X, Y, idx, M

    def elbo_train_steps(self, X, Y, idx, loc, log_scale, scale, opt_state, *, step0: int, lr: float, betas=(0.95, 0.999),
                         eps: float = 1e-8, clip_norm: float = 15.0, lrd: float = 1.0, weight_decay: float = 0.0, mode: str = "lrt",
                         guide: str = "normal", particles: int = 1, prior_loc: float = 0.0, prior_scale: float = 1.0,
                         dataset_size: int, seed: int, sample0: int = 0, window0: int = 0):
        """K ELBO training steps in one call over the device-resident split X [N,30,18], Y [N].  idx [K,M,B] (int64; [K,B] with
        [P] parameters) names the windows of member m's minibatch at step k.  Step k is elbo_step_ensemble (elbo_step at M = 1)
        on X[idx[k]], Y[idx[k]] with Noise(seed + 0x9E3779B97F4A7C15 (k + 1) mod 2**64, sample0, window0), then
        clipped_adam_vi at step step0 + k + 1, then step_metrics_ensemble of the logged predictions (particle 0, or the aggregate
        of several particles).  loc / log_scale / scale [M,P] and opt_state = (m_loc, v_loc, m_log_scale, v_log_scale) [M,P] are
        updated in place.  Returns dict(scalars [K,M,4] = (loss, nll_sum, kl, mse), metrics [K,M,5] = (nll, mse, sharpness,
        rmsce, mace)), float64 device tensors.  The index range check before the launches is the call's only synchronisation;
        from the third step of a configuration on, each step is one CUDA-graph launch."""
        if len(opt_state) != 4:
            raise RuntimeError("bayesrul_b200: opt_state must be (m_loc, v_loc, m_log_scale, v_log_scale)")
        ts = (loc, log_scale, scale) + tuple(opt_state)
        names = ("loc", "log_scale", "scale", "m_loc", "v_loc", "m_log_scale", "v_log_scale")
        X, Y, idx, M = self._train_inputs(X, Y, idx, list(zip(ts, names)))
        if guide not in GUIDE_IDS:
            raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
        if mode is None:
            mode = "ws"
        K, B = idx.shape[0], idx.shape[2]
        scalars = torch.empty(K, M, 4, dtype=torch.float64, device=self.device)
        metrics = torch.empty(K, M, 5, dtype=torch.float64, device=self.device)
        ws = self._ws_for(B, M, 5, "simt")
        _lib.check(self.lib.brl_elbo_train_steps(self.ctx, X.data_ptr(), Y.data_ptr(), X.shape[0], idx.data_ptr(), K, M, B,
                                                 *[t.data_ptr() for t in ts], int(step0), float(lr), float(betas[0]), float(betas[1]),
                                                 float(eps), float(clip_norm), float(lrd), float(weight_decay), MODE_IDS[mode],
                                                 GUIDE_IDS[guide], int(particles), float(prior_loc), float(prior_scale),
                                                 int(dataset_size), int(seed) & 0xFFFFFFFFFFFFFFFF, int(sample0), int(window0),
                                                 scalars.data_ptr(), metrics.data_ptr(), ws.data_ptr(), ws.numel(), self._stream()))
        return dict(scalars=scalars, metrics=metrics)

    def elbo_val_steps(self, X, Y, idx, loc, scale, *, guide: str = "normal", particles: int = 1, S: int = 1, prior_loc: float = 0.0,
                       prior_scale: float = 1.0, dataset_size: int, seed: int, sample0: int = 0, window0: int = 0,
                       engine: str = "simt"):
        """K validation batches of one variational BNN in one call over the device-resident split X [N,30,18], Y [N]; idx [K,B]
        (int64) names the windows of batch k.  Batch k is elbo_step(X[idx[k]], Y[idx[k]], loc, scale, mode="ws", compute_grads=False)
        with Noise(seed + 0x9E3779B97F4A7C15 (2k + 1) mod 2**64, sample0, window0) on the current gemm back-end, then
        sample_weights(S) with Noise(seed + 0x9E3779B97F4A7C15 (2k + 2) mod 2**64, sample0, window0), forward("ws", engine) and,
        for S > 1, aggregate_predictions, then step_metrics of that (loc, scale).  loc / scale [P] are not changed.  Returns
        dict(scalars [K,4] = (loss, nll_sum, kl, mse), metrics [K,5] = (nll, mse, sharpness, rmsce, mace)), float64 device tensors.
        The index range check is the call's only synchronisation; from the third batch of a configuration on, each batch is one
        CUDA-graph launch.

        loc / scale [M,P]: the M seeds of an experiment, validated together on the same batches idx [K,B].  Member m of batch k is
        the batch above with its elbo_step's particles at sample0 + m particles and its S weight draws at sample0 + m S
        (elbo_step_ensemble's and predict_moments_ensemble's conventions); the members share every launch they can.  Returns
        dict(scalars [K,M,4], metrics [K,M,5])."""
        ens = isinstance(loc, torch.Tensor) and loc.dim() == 2
        X, Y, idx, M = self._train_inputs(X, Y, idx, [(loc, "loc"), (scale, "scale")], shared_idx=ens)
        if M == 0:
            raise RuntimeError("bayesrul_b200: empty ensemble (loc / scale have M = 0 rows)")
        if guide not in GUIDE_IDS:
            raise RuntimeError("Guide unknown. Choose from 'normal', 'radial'.")
        if engine not in ENGINE_IDS:
            raise RuntimeError(f"bayesrul_b200: unknown engine {engine!r}")
        K, B = idx.shape[0], idx.shape[2]
        if ens:
            scalars = torch.empty(K, M, 4, dtype=torch.float64, device=self.device)
            metrics = torch.empty(K, M, 5, dtype=torch.float64, device=self.device)
            n = self.lib.brl_workspace_bytes_val(self.ctx, B, M, int(S), ENGINE_IDS[engine])
            if n < 0:
                raise RuntimeError(f"bayesrul_b200: bad workspace query (B = {B}, M = {M}, S = {S})")
            ws = self.workspace(n)
            _lib.check(self.lib.brl_elbo_val_steps_ensemble(
                self.ctx, X.data_ptr(), Y.data_ptr(), X.shape[0], idx.data_ptr(), K, M, B, loc.data_ptr(), scale.data_ptr(),
                GUIDE_IDS[guide], int(particles), int(S), ENGINE_IDS[engine], float(prior_loc), float(prior_scale), int(dataset_size),
                int(seed) & 0xFFFFFFFFFFFFFFFF, int(sample0), int(window0), scalars.data_ptr(), metrics.data_ptr(), ws.data_ptr(),
                ws.numel(), self._stream()))
            return dict(scalars=scalars, metrics=metrics)
        scalars = torch.empty(K, 4, dtype=torch.float64, device=self.device)
        metrics = torch.empty(K, 5, dtype=torch.float64, device=self.device)
        n = self.lib.brl_workspace_bytes(self.ctx, B, int(S), 7, ENGINE_IDS[engine])
        if n < 0:
            raise RuntimeError(f"bayesrul_b200: bad workspace query (B = {B}, S = {S})")
        ws = self.workspace(n)
        _lib.check(self.lib.brl_elbo_val_steps(self.ctx, X.data_ptr(), Y.data_ptr(), X.shape[0], idx.data_ptr(), K, B, loc.data_ptr(),
                                               scale.data_ptr(), GUIDE_IDS[guide], int(particles), int(S), ENGINE_IDS[engine],
                                               float(prior_loc), float(prior_scale), int(dataset_size), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                               int(sample0), int(window0), scalars.data_ptr(), metrics.data_ptr(), ws.data_ptr(),
                                               ws.numel(), self._stream()))
        return dict(scalars=scalars, metrics=metrics)

    def hnn_train_steps(self, X, Y, idx, theta, opt_state, *, step0: int, lr: float, betas=(0.9, 0.999), eps: float = 1e-8,
                        clip_norm: Optional[float] = None, lrd: Optional[float] = None, weight_decay: float = 0.0,
                        p_dropout: float = 0.0, seed: int, sample0: int = 0, window0: int = 0, optimizer: str = "clipped_adam"):
        """K heteroscedastic-NN training steps in one call (the members of a deep ensemble): step k is hnn_step_ensemble
        (hnn_step at M = 1) on X[idx[k]], Y[idx[k]] with Noise(seed + 0x9E3779B97F4A7C15 (k + 1) mod 2**64, sample0, window0),
        then the optimizer over theta [M,P] with opt_state = (exp_avg, exp_avg_sq) at step step0 + k + 1, then
        step_metrics_ensemble of the step's (loc, scale).  optimizer="clipped_adam" is clipped_adam (clip_norm defaults to 1e30,
        which disables the clip, and lrd to 1.0); optimizer="adam" is Engine.adam, torch.optim.Adam's update, and takes no
        clip_norm or lrd.  Returns dict(scalars [K,M,2] = (loss, mse), metrics [K,M,5]); synchronises only for the index range
        check, as elbo_train_steps."""
        if optimizer not in ("clipped_adam", "adam"):
            raise RuntimeError(f"bayesrul_b200: optimizer must be 'clipped_adam' or 'adam', got {optimizer!r}")
        if optimizer == "adam" and (clip_norm is not None or lrd is not None):
            raise RuntimeError("bayesrul_b200: optimizer='adam' (torch.optim.Adam) has no clip_norm or lrd")
        if len(opt_state) != 2:
            raise RuntimeError("bayesrul_b200: opt_state must be (exp_avg, exp_avg_sq)")
        ts = (theta,) + tuple(opt_state)
        X, Y, idx, M = self._train_inputs(X, Y, idx, list(zip(ts, ("theta", "exp_avg", "exp_avg_sq"))))
        K, B = idx.shape[0], idx.shape[2]
        scalars = torch.empty(K, M, 2, dtype=torch.float64, device=self.device)
        metrics = torch.empty(K, M, 5, dtype=torch.float64, device=self.device)
        ws = self._ws_for(B, M, 6, "simt")
        head = (self.ctx, X.data_ptr(), Y.data_ptr(), X.shape[0], idx.data_ptr(), K, M, B, *[t.data_ptr() for t in ts], int(step0))
        tail = (float(p_dropout), int(seed) & 0xFFFFFFFFFFFFFFFF, int(sample0), int(window0), scalars.data_ptr(), metrics.data_ptr(),
                ws.data_ptr(), ws.numel(), self._stream())
        if optimizer == "adam":
            _lib.check(self.lib.brl_hnn_train_steps_adam(*head, float(lr), float(betas[0]), float(betas[1]), float(eps),
                                                         float(weight_decay), *tail))
        else:
            _lib.check(self.lib.brl_hnn_train_steps(*head, float(lr), float(betas[0]), float(betas[1]), float(eps),
                                                    float(1e30 if clip_norm is None else clip_norm), float(1.0 if lrd is None else lrd),
                                                    float(weight_decay), *tail))
        return dict(scalars=scalars, metrics=metrics)

    # -- A14 / A15 / N1 ------------------------------------------------------------------------------------
    def mixture_moments(self, mu_m: torch.Tensor, sigma_m: torch.Tensor):
        mu_m, sigma_m = _chk(mu_m, self.device, "mu_m"), _chk(sigma_m, self.device, "sigma_m")
        if mu_m.shape != sigma_m.shape or mu_m.dim() != 2:
            raise RuntimeError("bayesrul_b200: mu_m / sigma_m must both be [M,n]")
        M, n = mu_m.shape
        mu, sd = torch.empty(n, device=self.device), torch.empty(n, device=self.device)
        with self._on_device():
            _lib.check(self.lib.brl_mixture_moments(mu_m.data_ptr(), sigma_m.data_ptr(), M, n, mu.data_ptr(), sd.data_ptr(),
                                                    self._stream()))
        return mu, sd

    def test_metrics(self, pred, std, y) -> torch.Tensor:
        """device float64[4]: gaussian_nll, mse, sharpness, rmsce (bayesian.py:217-224)."""
        pred, std, y = (_chk(t, self.device, n) for t, n in ((pred, "pred"), (std, "std"), (y, "y")))
        if not (pred.shape == std.shape == y.shape):
            raise RuntimeError("bayesrul_b200: pred / std / y shapes differ")
        scalars = torch.empty(4, dtype=torch.float64, device=self.device)
        ws = self.workspace(4096)
        with self._on_device():
            _lib.check(self.lib.brl_test_metrics(pred.data_ptr(), std.data_ptr(), y.data_ptr(), pred.numel(),
                                                 scalars.data_ptr(), ws.data_ptr(), ws.numel(), self._stream()))
        return scalars

    def step_metrics(self, pred, std, y) -> torch.Tensor:
        """device float64[5]: gaussian_nll, mse, sharpness, rmsce, mace -- every scalar a training / validation / test step
        logs (bayesian.py:158-166; results/metrics.py:210-297) from one fused pass."""
        pred, std, y = (_chk(t.reshape(-1).contiguous(), self.device, n) for t, n in ((pred, "pred"), (std, "std"), (y, "y")))
        if not (pred.shape == std.shape == y.shape):
            raise RuntimeError("bayesrul_b200: pred / std / y shapes differ")
        scalars = torch.empty(5, dtype=torch.float64, device=self.device)
        if getattr(self, "_metrics_ws", None) is None:
            self._metrics_ws = torch.empty(4096, dtype=torch.uint8, device=self.device)  # its own scratch: survives workspace growth
        with self._on_device():
            _lib.check(self.lib.brl_step_metrics(pred.data_ptr(), std.data_ptr(), y.data_ptr(), pred.numel(), scalars.data_ptr(),
                                                 self._metrics_ws.data_ptr(), self._metrics_ws.numel(), self._stream()))
        return scalars

    def step_metrics_ensemble(self, pred, std, y) -> torch.Tensor:
        """step_metrics of M rows in one pass: pred / std / y [M,n] -> device float64 [M,5], row m = step_metrics(pred[m],
        std[m], y[m])."""
        pred, std, y = (_chk(t, self.device, n) for t, n in ((pred, "pred"), (std, "std"), (y, "y")))
        if pred.dim() != 2 or not (pred.shape == std.shape == y.shape) or pred.numel() == 0:
            raise RuntimeError("bayesrul_b200: pred / std / y must all be [M,n] with M, n > 0")
        M, n = pred.shape
        scalars = torch.empty(M, 5, dtype=torch.float64, device=self.device)
        if getattr(self, "_metrics_ws", None) is None or self._metrics_ws.numel() < M * 1024:
            self._metrics_ws = torch.empty(max(4096, M * 1024), dtype=torch.uint8, device=self.device)
        with self._on_device():
            _lib.check(self.lib.brl_step_metrics_ensemble(pred.data_ptr(), std.data_ptr(), y.data_ptr(), M, n, scalars.data_ptr(),
                                                          self._metrics_ws.data_ptr(), self._metrics_ws.numel(), self._stream()))
        return scalars

    def clipped_adam(self, param, grad, exp_avg, exp_avg_sq, step: int, lr: float, betas=(0.95, 0.999), eps=1e-8,
                     clip_norm=15.0, lrd=1.0, weight_decay=0.0) -> None:
        for t, n in ((param, "param"), (grad, "grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
            _chk(t, self.device, n)
        with self._on_device():
            _lib.check(self.lib.brl_clipped_adam(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(),
                                                 exp_avg_sq.data_ptr(), param.numel(), int(step), lr, betas[0], betas[1],
                                                 eps, clip_norm, lrd, weight_decay, self._stream()))

    def adam(self, param, grad, exp_avg, exp_avg_sq, step: int, lr: float, betas=(0.9, 0.999), eps: float = 1e-8,
             weight_decay: float = 0.0) -> None:
        """One torch.optim.Adam step (amsgrad=False, maximize=False; L2 weight decay) over flat fp32 tensors, in place:
        step `step` >= 1 of the optimizer, with the hyper-parameters it holds.  The update is torch's single-tensor formula, one
        rounding per torch op (DESIGN §4.8.1)."""
        ts = (param, grad, exp_avg, exp_avg_sq)
        for t, n in zip(ts, ("param", "grad", "exp_avg", "exp_avg_sq")):
            _chk(t, self.device, n)
            if t.numel() != param.numel():
                raise RuntimeError("bayesrul_b200: adam tensors must have the same number of elements")
        with self._on_device():
            _lib.check(self.lib.brl_adam(*[t.data_ptr() for t in ts], param.numel(), int(step), float(lr), float(betas[0]),
                                         float(betas[1]), float(eps), float(weight_decay), self._stream()))

    def clipped_adam_vi(self, loc, log_scale, scale, grad_loc, grad_log_scale, m_loc, v_loc, m_ls, v_ls, step: int, lr: float,
                        betas=(0.95, 0.999), eps=1e-8, clip_norm=15.0, lrd=1.0, weight_decay=0.0, grad_scale: float = 1.0) -> None:
        """One launch: ClippedAdam on `loc` and on `log_scale`, then scale = exp(log_scale) (all in place).  grad_scale multiplies
        the gradients before the clamp (1 / world after a SUM all-reduce)."""
        ts = (loc, log_scale, scale, grad_loc, grad_log_scale, m_loc, v_loc, m_ls, v_ls)
        for t in ts:
            _chk(t, self.device, "clipped_adam_vi tensor")
            if t.numel() != loc.numel():
                raise RuntimeError("bayesrul_b200: clipped_adam_vi tensors must have the same number of elements")
        with self._on_device():
            if grad_scale != 1.0:
                _lib.check(self.lib.brl_clipped_adam_vi_scaled(*[t.data_ptr() for t in ts], loc.numel(), int(step), lr, betas[0], betas[1],
                                                               eps, clip_norm, lrd, weight_decay, float(grad_scale), self._stream()))
            else:
                _lib.check(self.lib.brl_clipped_adam_vi(*[t.data_ptr() for t in ts], loc.numel(), int(step), lr, betas[0], betas[1], eps,
                                                        clip_norm, lrd, weight_decay, self._stream()))
