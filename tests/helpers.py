"""Shared helpers of the GPU parity tests (oracle <-> engine noise conversion) and the golden-fixture loader."""
import ast
import functools
import hashlib
import math
import os

import numpy as np
import torch

from oracle import bnn_oracle as O

GOLDEN_NETS = ("inception", "conv", "linear")  # the order in which tests/golden/make_golden.py draws the nets


def golden_digest(t):
    """SHA-256 of a float32 tensor's values: how a fixture pins an array it does not store."""
    return hashlib.sha256(t.detach().numpy().astype("<f4").tobytes()).hexdigest()


def load_golden(golden_dir, net):
    """tests/golden/<net>.npz as tests/golden/make_golden.py computed it.  The parameter-sized inputs (theta, sigma,
    ws_eps) and the LRT noise are not stored but regenerated from make_golden.py's seeds, each checked bit for bit
    against the SHA-256 stored in its place."""
    return {k: v.copy() for k, v in _golden(golden_dir)[net].items()}


def _default_init(shapes):
    """torch's default init of the reference's Conv / Linear layers, (weight, bias) pairs in named_parameters() order:
    kaiming_uniform_(a=sqrt(5)) weights and uniform biases, both U(-1/sqrt(fan_in), 1/sqrt(fan_in))."""
    ps = [torch.empty(s) for s in shapes]
    for w, b in zip(ps[0::2], ps[1::2]):
        bound = 1.0 / math.sqrt(w[0].numel())
        w.uniform_(-bound, bound)
        b.uniform_(-bound, bound)
    return ps


@functools.lru_cache(maxsize=None)
def _golden(golden_dir):
    fixtures = {net: dict(np.load(os.path.join(golden_dir, f"{net}.npz"))) for net in GOLDEN_NETS}

    def regenerated(key, t, digest):
        assert golden_digest(t) == str(digest), f"golden {key}: regenerated values differ from the fixture's"
        return t.numpy()

    def same(fx, key, t):
        assert np.array_equal(fx[key], t.numpy()), f"golden {key}: random stream out of step with make_golden.py"

    # make_golden.py draws from two streams, each running through the three nets in turn: torch.manual_seed(12345)
    # initialises the reference net (default init + weights_init) and then builds its dropout variant (default init);
    # Generator(777) draws x, the weight-sampling eps [S,P], the LRT noise and the Flipout signs.
    g = torch.Generator().manual_seed(777)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(12345)
        for net in GOLDEN_NETS:
            fx = fixtures[net]
            shapes = [ast.literal_eval(s) for s in fx["shapes"]]
            ps = _default_init(shapes)
            for w in ps[0::2]:  # weights_init: xavier_normal_ for conv weights, kaiming_normal_ for linear weights
                torch.nn.init.xavier_normal_(w) if w.dim() > 2 else torch.nn.init.kaiming_normal_(w)
            theta = torch.cat([p.flatten() for p in ps])
            _default_init(shapes)
            fx["theta"] = regenerated("theta", theta, fx["theta_sha256"])
            fx["sigma"] = np.full(theta.numel(), fx["sigma_value"], dtype=np.float32)
            same(fx, "x", torch.randn(fx["x"].shape, generator=g))
            eps = torch.randn(fx["out_ws"].shape[0], theta.numel(), generator=g)
            fx["ws_eps"] = regenerated("ws_eps", eps, fx["ws_eps_sha256"])
            for i, (shape, digest) in enumerate(zip(fx["lrt_eps_shapes"], fx["lrt_eps_sha256"])):
                e = torch.randn(ast.literal_eval(shape), generator=g)
                fx[f"lrt_eps_call{i}"] = regenerated(f"lrt_eps_call{i}", e, digest)
            for i in range(sum(k.startswith("flip_in_call") for k in fx)):
                same(fx, f"flip_in_call{i}", (torch.rand(fx[f"flip_in_call{i}"].shape, generator=g) > 0.5).float() * 2 - 1)
                same(fx, f"flip_out_call{i}", (torch.rand(fx[f"flip_out_call{i}"].shape, generator=g) > 0.5).float() * 2 - 1)
    return fixtures


def injected_to_engine(net, noises, B, device):
    """list (one per MC sample) of oracle noise dicts -> bayesrul_b200.Noise with [S,...] tensors."""
    from bayesrul_b200 import Noise

    S = len(noises)
    nz = Noise()

    def stack(key):
        return torch.stack([n[key].float() for n in noises]).contiguous().to(device)

    keys = noises[0].keys()
    if "weight_eps" in keys:
        nz.weight_eps = stack("weight_eps")
    if "radial_r" in keys:
        nz.radial_r = stack("radial_r")
    for k in keys:
        if "." in k:
            name, layer = k.split(".")
            getattr(nz, name)[int(layer)] = stack(k).reshape(S, B, -1).contiguous()
    return nz


def assert_close(a, b, rtol=1e-3, atol_scale=1e-5, what=""):
    a = a.detach().double().cpu()
    b = b.detach().double().cpu()
    scale = b.abs().max().item() + 1e-30
    err = (a - b).abs()
    tol = rtol * b.abs() + atol_scale * scale
    bad = err > tol
    assert not bad.any(), f"{what}: {int(bad.sum())}/{bad.numel()} mismatches, max err {err.max().item():.3e}, scale {scale:.3e}"


def synth(net, B, seed=0, sigma=0.05, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 30, 18, generator=g, dtype=torch.float64).to(dtype)
    y = (torch.rand(B, generator=g, dtype=torch.float64) * 100).to(dtype)
    mu = O.init_params(net, seed + 1, dtype)
    sg = torch.full_like(mu, sigma)
    return x, y, mu, sg
