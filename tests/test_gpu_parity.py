"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle and the golden fixtures.
Tolerance: fp32 SIMT engine rtol 1e-3 (north_star injected-noise bound)."""
import os

import numpy as np
import pytest
import torch

from oracle import bnn_oracle as O
from tests.helpers import assert_close, injected_to_engine, synth, load_golden as _fx

pytestmark = pytest.mark.gpu
NETS = ["inception", "conv", "linear"]
DROP_ORDER = {"inception": [0, 1, 2, 3, 4, 6, 8, 9, 10], "conv": [0, 1, 2], "linear": [0, 1, 2, 3]}
DEV = "cuda:0"


@pytest.fixture(scope="module")
def engines():
    from bayesrul_b200 import Engine
    return {n: Engine(n, DEV) for n in NETS}


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).float().to(DEV)


# ----------------------------------------------------------------------------- golden fixtures
@pytest.mark.parametrize("net", NETS)
def test_golden_det(engines, golden_dir, net):
    fx = _fx(golden_dir, net)
    out = engines[net].forward(_t(fx["x"]), "det", theta=_t(fx["theta"]))
    assert_close(out[0], torch.from_numpy(fx["out_det"]), what="det")


@pytest.mark.parametrize("net", NETS)
def test_golden_dropout(engines, golden_dir, net):
    from bayesrul_b200 import Noise
    fx = _fx(golden_dir, net)
    B = fx["x"].shape[0]
    nz = Noise(drop_mask={i: _t(fx[f"drop_mask_call{j}"]).reshape(1, B, -1).contiguous() for j, i in enumerate(DROP_ORDER[net])})
    out = engines[net].forward(_t(fx["x"]), "det", theta=_t(fx["theta"]), p_dropout=float(fx["drop_p"]), noise=nz)
    assert_close(out[0], torch.from_numpy(fx["out_drop"]), what="dropout")


@pytest.mark.parametrize("net", NETS)
def test_golden_weight_sampling_and_moments(engines, golden_dir, net):
    from bayesrul_b200 import Noise
    fx = _fx(golden_dir, net)
    e = engines[net]
    S = fx["ws_eps"].shape[0]
    nz = Noise(weight_eps=_t(fx["ws_eps"]))
    w = e.sample_weights(_t(fx["theta"]), _t(fx["sigma"]), "normal", S, nz)
    out = e.forward(_t(fx["x"]), "ws", wsamp=w, S=S)
    assert_close(out, torch.from_numpy(fx["out_ws"]), what="ws")
    pred, std, ep, al = e.predict_moments(_t(fx["x"]), _t(fx["theta"]), _t(fx["sigma"]), S=S, guide="normal", noise=nz, chunk=2)
    for a, k in ((pred, "pred"), (std, "std"), (ep, "ep_var"), (al, "al_var")):
        assert_close(a, torch.from_numpy(fx[k]), rtol=2e-3, atol_scale=1e-4, what=k)
    m = e.moments(out)
    for a, b in zip(m, (pred, std, ep, al)):
        assert_close(a, b, rtol=1e-5, what="moments")


@pytest.mark.parametrize("net", NETS)
def test_golden_lrt(engines, golden_dir, net):
    from bayesrul_b200 import Noise
    fx = _fx(golden_dir, net)
    B = fx["x"].shape[0]
    n = len(O.net_layers(net))
    nz = Noise(lrt_eps={i: _t(fx[f"lrt_eps_call{i}"]).reshape(1, B, -1).contiguous() for i in range(n)})
    out = engines[net].forward(_t(fx["x"]), "lrt", theta=_t(fx["theta"]), sigma=_t(fx["sigma"]), noise=nz)
    assert_close(out[0], torch.from_numpy(fx["out_lrt"]), what="lrt")


@pytest.mark.parametrize("net", NETS)
def test_golden_flipout(engines, golden_dir, net):
    from bayesrul_b200 import Noise
    fx = _fx(golden_dir, net)
    B = fx["x"].shape[0]
    n = len(O.net_layers(net))
    nz = Noise(flip_in={i: _t(fx[f"flip_in_call{i}"]).reshape(1, B, -1).contiguous() for i in range(n)},
               flip_out={i: _t(fx[f"flip_out_call{i}"]).reshape(1, B, -1).contiguous() for i in range(n)})
    w = (_t(fx["theta"]) + _t(fx["sigma"]) * _t(fx["ws_eps"][0])).reshape(1, -1).contiguous()
    out = engines[net].forward(_t(fx["x"]), "flipout", theta=_t(fx["theta"]), wsamp=w, noise=nz)
    assert_close(out[0], torch.from_numpy(fx["out_flipout"]), what="flipout")


def test_golden_deep_ensemble(engines, golden_dir):
    z = np.load(os.path.join(golden_dir, "deep_ensemble.npz"))
    mu, sd = engines["inception"].mixture_moments(_t(z["mu_m"]), _t(z["sigma_m"]))
    assert_close(mu, torch.from_numpy(z["preds"]), rtol=1e-5, what="de mu")
    assert_close(sd, torch.from_numpy(z["stds"]), rtol=1e-3, atol_scale=1e-4, what="de sd")


# ----------------------------------------------------------------------------- native Philox noise
@pytest.mark.parametrize("net", NETS)
def test_native_sampler_matches_numpy_philox(engines, net):
    from bayesrul_b200 import Noise
    e = engines[net]
    _, _, mu, sg = synth(net, 1)
    for guide in ("normal", "radial"):
        w = e.sample_weights(mu.to(DEV), sg.to(DEV), guide, 3, Noise(seed=1234, sample0=5))
        for s in range(3):
            ref = O.sample_weights(net, mu.double(), sg.double(), guide, O.PhiloxNoise(net, 1234, sample=5 + s, dtype=torch.float64))
            assert_close(w[s], ref, rtol=1e-4, atol_scale=1e-5, what=f"{guide} sample {s}")


@pytest.mark.parametrize("net", NETS)
@pytest.mark.parametrize("mode", ["lrt", "flipout", "dropout"])
def test_native_noise_forward(engines, net, mode):
    from bayesrul_b200 import Noise
    e = engines[net]
    B = 9
    x, _, mu, sg = synth(net, B, seed=3)
    nz = Noise(seed=99, sample0=2, window0=1000)
    pn = O.PhiloxNoise(net, 99, sample=2, window0=1000)
    if mode == "lrt":
        out = e.forward(x.to(DEV), "lrt", theta=mu.to(DEV), sigma=sg.to(DEV), noise=nz)
        ref = O.forward_lrt(net, x, mu, sg, pn)
    elif mode == "flipout":
        w = e.sample_weights(mu.to(DEV), sg.to(DEV), "normal", 1, nz)
        out = e.forward(x.to(DEV), "flipout", theta=mu.to(DEV), wsamp=w, noise=nz)
        ref = O.forward_flipout(net, x, mu, O.sample_weights(net, mu, sg, "normal", pn), pn)
    else:
        out = e.forward(x.to(DEV), "det", theta=mu.to(DEV), p_dropout=0.3, noise=nz)
        ref = O.forward_det(net, x, mu, 0.3, pn)
    assert_close(out[0], ref, rtol=2e-3, atol_scale=1e-4, what=mode)


def test_native_noise_is_shard_invariant(engines):
    """Philox is keyed by the GLOBAL window / sample index: a shard reproduces its slice bit-exactly."""
    from bayesrul_b200 import Noise
    e = engines["inception"]
    x, _, mu, sg = synth("inception", 12, seed=5)
    x, mu, sg = x.to(DEV), mu.to(DEV), sg.to(DEV)
    full = e.forward(x, "lrt", theta=mu, sigma=sg, noise=Noise(seed=7))
    part = e.forward(x[5:].contiguous(), "lrt", theta=mu, sigma=sg, noise=Noise(seed=7, window0=5))
    assert torch.equal(full[0, 5:], part[0])
    a = e.predict_moments(x, mu, sg, S=6, noise=Noise(seed=3), chunk=6)
    b = e.predict_moments(x, mu, sg, S=6, noise=Noise(seed=3), chunk=1)
    for u, v in zip(a, b):
        assert torch.equal(u, v)


# ----------------------------------------------------------------------------- predictive path
@pytest.mark.parametrize("net", NETS)
@pytest.mark.parametrize("guide", ["normal", "radial"])
def test_predict_moments_vs_oracle(engines, net, guide):
    from bayesrul_b200 import Noise
    e = engines[net]
    B, S = 37, 7
    x, _, mu, sg = synth(net, B, seed=11)
    g = torch.Generator().manual_seed(1)
    nzs = [O.make_injected_noise(net, B, "radial" if guide == "radial" else "ws", g) for _ in range(S)]
    ref = O.predictive_moments(O.predict(net, x, mu, sg, guide, [O.InjectedNoise(n) for n in nzs]))
    got = e.predict_moments(x.to(DEV), mu.to(DEV), sg.to(DEV), S=S, guide=guide, noise=injected_to_engine(net, nzs, B, DEV), chunk=3)
    for a, b, k in zip(got, ref, ("pred", "std", "ep", "al")):
        assert_close(a, b, rtol=2e-3, atol_scale=1e-4, what=k)


def test_predict_mcd_vs_oracle(engines):
    from bayesrul_b200 import Noise
    e = engines["inception"]
    B, S, p = 21, 5, 0.241437
    x, _, mu, _ = synth("inception", B, seed=12)
    g = torch.Generator().manual_seed(2)
    nzs = [O.make_injected_noise("inception", B, "det", g, p_dropout=p) for _ in range(S)]
    ref = O.predictive_moments(O.predict_mcd("inception", x, mu, p, [O.InjectedNoise(n) for n in nzs]))
    got = e.predict_moments(x.to(DEV), mu.to(DEV), None, S=S, guide=None, p_dropout=p,
                            noise=injected_to_engine("inception", nzs, B, DEV), chunk=2)
    for a, b, k in zip(got, ref, ("pred", "std", "ep", "al")):
        assert_close(a, b, rtol=2e-3, atol_scale=1e-4, what=k)


def test_aggregate_and_single_sample_nan(engines):
    e = engines["inception"]
    g = torch.Generator().manual_seed(3)
    out = torch.rand(6, 40, 2, generator=g) * 3 + 0.5
    assert_close(e.aggregate_predictions(out.to(DEV)), O.aggregate_predictions(out.double()), rtol=1e-4, what="aggregate")
    m = e.moments(out[:1].contiguous().to(DEV))
    assert torch.isnan(m[2]).all()  # loc.var(0) of one sample is NaN in torch too (bayesian.py:148 comment)


# ----------------------------------------------------------------------------- ELBO step
@pytest.mark.parametrize("net", NETS)
@pytest.mark.parametrize("mode,guide,particles", [("lrt", "normal", 1), ("flipout", "normal", 2), ("ws", "normal", 1),
                                                   ("ws", "radial", 1)])
@pytest.mark.parametrize("sigma", [0.05, 1.351e-3])
def test_elbo_step_vs_oracle(engines, net, mode, guide, particles, sigma):
    e = engines[net]
    B = 33
    x, y, mu, sg = synth(net, B, seed=21, sigma=sigma)
    g = torch.Generator().manual_seed(4)
    md = "radial" if guide == "radial" else mode
    nzs = [O.make_injected_noise(net, B, md, g) for _ in range(particles)]
    kw = dict(mode=mode, guide=guide, prior_loc=0.0, prior_scale=0.138793, dataset_size=238150)
    ref = O.elbo_loss_and_grads(net, x.double(), y.double(), mu.double(), sg.double(),
                                noises=[O.InjectedNoise({k: v.double() for k, v in n.items()}) for n in nzs], **kw)
    got = e.elbo_step(x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV), particles=particles,
                      noise=injected_to_engine(net, nzs, B, DEV), **kw)
    sc = got["scalars"].cpu()
    assert abs(sc[0].item() / ref["loss"].item() - 1) < 1e-4
    assert abs(sc[1].item() / ref["nll_sum"].item() - 1) < 1e-4
    assert abs(sc[2].item() / ref["kl"].item() - 1) < 1e-4
    assert_close(got["out"], ref["out"], what="out")
    assert_close(got["grad_mu"], ref["grad_mu"], rtol=1e-3, atol_scale=2e-5, what="grad_mu")
    assert_close(got["grad_sigma"], ref["grad_sigma"], rtol=1e-3, atol_scale=2e-5, what="grad_sigma")
    assert_close(got["grad_log_sigma"], ref["grad_log_sigma"], rtol=1e-3, atol_scale=2e-5, what="grad_log_sigma")
    ev = e.elbo_step(x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV), particles=particles,
                     noise=injected_to_engine(net, nzs, B, DEV), compute_grads=False, **kw)
    assert abs(ev["scalars"][0].item() - sc[0].item()) < 1e-6 * abs(sc[0].item())  # split-K atomics: summation order varies


@pytest.mark.parametrize("net", NETS)
@pytest.mark.parametrize("p", [0.0, 0.241437])
def test_hnn_step_vs_oracle(engines, net, p):
    e = engines[net]
    B = 29
    x, y, mu, _ = synth(net, B, seed=31)
    g = torch.Generator().manual_seed(5)
    nz = O.make_injected_noise(net, B, "det", g, p_dropout=p)
    th = mu.double().requires_grad_(True)
    loss, out = O.hnn_loss(net, x.double(), y.double(), th, p, O.InjectedNoise({k: v.double() for k, v in nz.items()}))
    (gref,) = torch.autograd.grad(loss, th)
    got = e.hnn_step(x.to(DEV), y.to(DEV), mu.to(DEV), p, injected_to_engine(net, [nz], B, DEV) if p > 0 else None)
    assert abs(got["scalars"][0].item() / loss.item() - 1) < 1e-4
    assert_close(got["out"], out, what="out")
    assert_close(got["grad"], gref, rtol=1e-3, atol_scale=2e-5, what="grad")


# ----------------------------------------------------------------------------- small reductions / optimiser
@pytest.mark.parametrize("n", [100, 256, 10000])
def test_step_metrics_vs_reference_formulas(engines, n):
    """N3: brl_step_metrics = {gaussian_nll, mse, sharpness, rmsce, mace} of results/metrics.py:210-297 (restated in torch by
    compat.metrics / the oracle) at the batch sizes of a train step (100 / 256) and of a test batch (10 000)."""
    from bayesrul_b200.compat import metrics as M
    e = engines["inception"]
    g = torch.Generator().manual_seed(60 + n)
    y = torch.rand(n, generator=g) * 100
    std = torch.rand(n, generator=g) * 20 + 0.5
    pred = y + torch.randn(n, generator=g) * std * 1.3  # mildly over-confident predictions: a non-trivial calibration curve
    sc = e.step_metrics(pred.to(DEV), std.to(DEV), y.to(DEV)).cpu()
    want = [torch.nn.functional.gaussian_nll_loss(pred, y, std**2).item(), torch.nn.functional.mse_loss(pred, y).item(),
            M.sharpness(std).item(), O.rms_calibration_error(pred.double(), std.double(), y.double()).item(),
            M.mean_absolute_calibration_error(pred.double(), std.double(), y.double()).item()]
    for k, (a, b) in enumerate(zip(sc.tolist(), want)):
        assert abs(a - b) <= 2e-3 * abs(b) + 2.0 / n, (k, sc, want)  # one residual on a bin edge moves a proportion by 1 / n


def test_test_metrics_and_adam(engines):
    e = engines["inception"]
    g = torch.Generator().manual_seed(6)
    n = 5000
    pred, y = torch.rand(n, generator=g) * 100, torch.rand(n, generator=g) * 100
    std = torch.rand(n, generator=g) * 30 + 1
    sc = e.test_metrics(pred.to(DEV), std.to(DEV), y.to(DEV)).cpu()
    want = [torch.nn.functional.gaussian_nll_loss(pred, y, std**2).item(), torch.nn.functional.mse_loss(pred, y).item(),
            O.sharpness(std).item(), O.rms_calibration_error(pred.double(), std.double(), y.double()).item()]
    for a, b in zip(sc.tolist(), want):
        assert abs(a - b) <= 2e-3 * abs(b) + 1e-4, (sc, want)
    p = torch.randn(1000, generator=g)
    q, m, v = p.clone().to(DEV), torch.zeros(1000, device=DEV), torch.zeros(1000, device=DEV)
    pr, mr, vr = p.double(), torch.zeros(1000, dtype=torch.float64), torch.zeros(1000, dtype=torch.float64)
    for step in range(1, 5):
        gr = torch.randn(1000, generator=g) * 20
        e.clipped_adam(q, gr.to(DEV), m, v, step, 1e-3)
        pr, mr, vr = O.clipped_adam_step(pr, gr.double(), mr, vr, step, 1e-3)
    assert_close(q, pr, rtol=1e-5, what="adam")
    # the fused step of a mean-field guide: both buffers in one launch + scale = exp(log scale)
    loc0, ls0 = torch.randn(1000, generator=g), torch.randn(1000, generator=g) * 0.1 - 6.0
    loc, ls, sc = loc0.clone().to(DEV), ls0.clone().to(DEV), torch.empty(1000, device=DEV)
    st = [torch.zeros(1000, device=DEV) for _ in range(4)]
    ref = [[loc0.double(), torch.zeros(1000, dtype=torch.float64), torch.zeros(1000, dtype=torch.float64)],
           [ls0.double(), torch.zeros(1000, dtype=torch.float64), torch.zeros(1000, dtype=torch.float64)]]
    for step in range(1, 5):
        g1, g2 = torch.randn(1000, generator=g) * 20, torch.randn(1000, generator=g) * 20
        e.clipped_adam_vi(loc, ls, sc, g1.to(DEV), g2.to(DEV), st[0], st[1], st[2], st[3], step, 1e-3)
        ref[0] = list(O.clipped_adam_step(ref[0][0], g1.double(), ref[0][1], ref[0][2], step, 1e-3))
        ref[1] = list(O.clipped_adam_step(ref[1][0], g2.double(), ref[1][1], ref[1][2], step, 1e-3))
    assert_close(loc, ref[0][0], rtol=1e-5, what="adam_vi loc")
    assert_close(ls, ref[1][0], rtol=1e-5, what="adam_vi log scale")
    assert_close(sc, ref[1][0].exp(), rtol=1e-5, what="adam_vi scale")


# ----------------------------------------------------------------------------- edge cases / errors
@pytest.mark.parametrize("B", [1, 5, 127, 129, 257])
def test_ragged_batches(engines, B):
    e = engines["inception"]
    x, _, mu, _ = synth("inception", B, seed=B)
    out = e.forward(x.to(DEV), "det", theta=mu.to(DEV))
    assert_close(out[0], O.forward_det("inception", x, mu), what=f"B={B}")


def test_error_behaviour(engines):
    e = engines["inception"]
    x, y, mu, sg = synth("inception", 4)
    with pytest.raises(RuntimeError):
        e.forward(torch.zeros(4, 30, 17, device=DEV), "det", theta=mu.to(DEV))
    with pytest.raises(RuntimeError):
        e.forward(x, "det", theta=mu.to(DEV))  # CPU tensor
    with pytest.raises(RuntimeError):
        e.forward(torch.zeros(0, 30, 18, device=DEV), "det", theta=mu.to(DEV))
    with pytest.raises(RuntimeError, match="Guide unknown"):
        e.sample_weights(mu.to(DEV), sg.to(DEV), "laplace")
    with pytest.raises(RuntimeError):
        e.forward(x.to(DEV), "det", theta=mu[:-1].contiguous().to(DEV))


def test_full_size_properties(engines):
    """BASELINE config size (B=10 000 windows): chunk invariance + linearity of the mixture moments."""
    from bayesrul_b200 import Noise
    e = engines["inception"]
    B, S = 10000, 6
    x, _, mu, sg = synth("inception", B, seed=77, sigma=0.02)
    x, mu, sg = x.to(DEV), mu.to(DEV), sg.to(DEV)
    a = e.predict_moments(x, mu, sg, S=S, noise=Noise(seed=11), chunk=3)
    b = e.predict_moments(x, mu, sg, S=S, noise=Noise(seed=11), chunk=2)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert torch.isfinite(a[1]).all() and (a[2] >= 0).all() and (a[3] > 0).all()
    assert_close(a[1] ** 2, a[2] + a[3], rtol=1e-5, what="std^2 = ep + al")
    # the first 64 windows against the oracle with the same Philox stream
    ref = O.predictive_moments(O.predict("inception", x[:64].cpu(), mu.cpu(), sg.cpu(), "normal",
                                         [O.PhiloxNoise("inception", 11, sample=s) for s in range(S)]))
    for u, v, k in zip(a, ref, ("pred", "std", "ep", "al")):
        assert_close(u[:64], v, rtol=5e-3, atol_scale=1e-3, what=k)


# ----------------------------------------------------------------------------- native-RNG mode: statistical parity
@pytest.mark.parametrize("engine", ["simt", "tc"])
def test_native_rng_statistical_parity(engines, engine):
    """north_star, native-RNG mode: predictive mean / variance / NLL / RMSE of the in-kernel Philox stream must agree
    statistically with the oracle fed by an INDEPENDENT generator (torch.randn), on the same inputs.  A weight draw is
    shared by every window (bayesian.py:235-239), so window averages do NOT average the Monte-Carlo error away: bounds
    are k standard errors of an S-sample estimate with fully correlated windows."""
    from bayesrul_b200 import Noise
    net, B, S = "inception", 256, 1024
    e = engines[net]
    if engine == "tc" and not e.has_tc():
        pytest.skip("tensor-core engine unavailable")
    x, y, mu, _ = synth(net, B, seed=41)
    sg = torch.full_like(mu, 0.02)
    g = torch.Generator().manual_seed(99)
    ref = O.predictive_moments(O.predict(net, x, mu, sg, "normal",
                                         [O.InjectedNoise({"weight_eps": torch.randn(mu.numel(), generator=g)}) for _ in range(S)]))
    got = e.predict_moments(x.to(DEV), mu.to(DEV), sg.to(DEV), S=S, guide="normal", noise=Noise(seed=2025), engine=engine)
    pred, std, ep, al = [t.cpu().double() for t in got]
    rpred, rstd, rep, ral = [t.double() for t in ref]
    yd = y.double()
    k = 4.5
    se_mean = (2.0 * rep.mean().item() / S) ** 0.5          # difference of two S-sample means, windows fully correlated
    rel_var = k * (2.0 * 2.0 / (S - 1)) ** 0.5               # relative s.e. of a variance estimate sqrt(2/(S-1)), two of them

    def nll(p, s):
        return (0.5 * (torch.log(s * s) + (p - yd) ** 2 / (s * s))).mean().item()

    assert abs(pred.mean().item() - rpred.mean().item()) <= k * se_mean, (engine, "mean pred", pred.mean().item(), rpred.mean().item())
    rm, rrm = ((pred - yd) ** 2).mean().sqrt().item(), ((rpred - yd) ** 2).mean().sqrt().item()
    assert abs(rm - rrm) <= k * se_mean, (engine, "rmse", rm, rrm)
    assert abs(ep.mean().item() / rep.mean().item() - 1) <= rel_var, (engine, "epistemic var", ep.mean().item(), rep.mean().item())
    # the aleatoric variance is a mean over samples of scale^2: its Monte-Carlo error is far below the epistemic one
    assert abs(al.mean().item() / ral.mean().item() - 1) <= 0.05, (engine, "aleatoric var", al.mean().item(), ral.mean().item())
    assert abs(std.mean().item() / rstd.mean().item() - 1) <= 0.05, (engine, "std", std.mean().item(), rstd.mean().item())
    assert abs(nll(pred, std) - nll(rpred, rstd)) <= 0.05 * abs(nll(rpred, rstd)) + k * se_mean, (engine, "nll")
    # per window: the two predictive means differ by less than k standard errors of their own estimate
    z = (pred - rpred).abs() / ((2.0 * rep / S).sqrt() + 1e-9)
    assert (z > k).double().mean().item() < 0.02, (engine, z.max().item())


def test_flipout_forward_multi_sample_workspace(engines):
    """brl_forward in Flipout mode with native signs needs [S,B,Cin] + [S,B,Cout] per layer on top of the activations
    (brl_workspace_bytes(train=2)); S = 3 samples x 256 windows used to overflow the default query."""
    from bayesrul_b200 import Noise
    e = engines["inception"]
    B, S = 256, 3
    x, _, mu, sg = synth("inception", B, seed=5, sigma=0.05)
    x, mu, sg = x.to(DEV), mu.to(DEV), sg.to(DEV)
    w = e.sample_weights(mu, sg, "normal", S, Noise(seed=5))
    out = e.forward(x, "flipout", theta=mu, wsamp=w, S=S, noise=Noise(seed=11))
    one = e.forward(x, "flipout", theta=mu, wsamp=w[1:2].contiguous(), S=1, noise=Noise(seed=11, sample0=1))
    assert out.shape == (S, B, 2) and torch.isfinite(out).all()
    assert_close(out[1], one[0], rtol=1e-6, what="sample 1 of a 3-sample call == single-sample call at sample0=1")
