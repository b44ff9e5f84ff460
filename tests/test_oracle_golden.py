"""Pin the CPU oracle against fixtures produced by the reference's own code
(tests/golden/make_golden.py) and against independent formulas (SURVEY section 4, items 1-7)."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bnn_oracle as O
from tests.helpers import load_golden as _load

NETS = ["inception", "conv", "linear"]
DROP_ORDER = {"inception": [0, 1, 2, 3, 4, 6, 8, 9, 10], "conv": [0, 1, 2], "linear": [0, 1, 2, 3]}


@pytest.mark.parametrize("net", NETS)
def test_site_table_matches_reference(golden_dir, net):
    fx = _load(golden_dir, net)
    sites = O.site_table(net)
    assert [s[0] for s in sites] == list(fx["names"])
    assert [str(tuple(s[1])) for s in sites] == list(fx["shapes"])
    assert O.num_params(net) == fx["theta"].size
    assert [s[0] for s in O.site_table(net, dropout=True)] == list(fx["names_dropout_variant"])
    assert O.num_params(net) == {"inception": 187142, "conv": 15810, "linear": 192098}[net]


@pytest.mark.parametrize("net", NETS)
def test_det_forward(golden_dir, net):
    fx = _load(golden_dir, net)
    out = O.forward_det(net, torch.from_numpy(fx["x"]), torch.from_numpy(fx["theta"]))
    np.testing.assert_allclose(out.numpy(), fx["out_det"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("net", NETS)
def test_dropout_forward(golden_dir, net):
    fx = _load(golden_dir, net)
    t = {f"drop_mask.{i}": torch.from_numpy(fx[f"drop_mask_call{j}"]) for j, i in enumerate(DROP_ORDER[net])}
    out = O.forward_det(net, torch.from_numpy(fx["x"]), torch.from_numpy(fx["theta"]),
                        float(fx["drop_p"]), O.InjectedNoise(t))
    np.testing.assert_allclose(out.numpy(), fx["out_drop"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("net", NETS)
def test_weight_sample_predict_and_moments(golden_dir, net):
    fx = _load(golden_dir, net)
    x, mu, sg = (torch.from_numpy(fx[k]) for k in ("x", "theta", "sigma"))
    noises = [O.InjectedNoise({"weight_eps": torch.from_numpy(e)}) for e in fx["ws_eps"]]
    out = O.predict(net, x, mu, sg, "normal", noises)
    np.testing.assert_allclose(out.numpy(), fx["out_ws"], rtol=1e-5, atol=1e-6)
    pred, std, ep, al = O.predictive_moments(out)
    for a, k in ((pred, "pred"), (std, "std"), (ep, "ep_var"), (al, "al_var")):
        np.testing.assert_allclose(a.numpy(), fx[k], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("net", NETS)
def test_lrt_composition(golden_dir, net):
    fx = _load(golden_dir, net)
    x, mu, sg = (torch.from_numpy(fx[k]) for k in ("x", "theta", "sigma"))
    n = len(O.net_layers(net))
    t = {f"lrt_eps.{i}": torch.from_numpy(fx[f"lrt_eps_call{i}"]) for i in range(n)}
    out = O.forward_lrt(net, x, mu, sg, O.InjectedNoise(t))
    np.testing.assert_allclose(out.numpy(), fx["out_lrt"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("net", NETS)
def test_flipout_composition(golden_dir, net):
    fx = _load(golden_dir, net)
    x, mu, sg = (torch.from_numpy(fx[k]) for k in ("x", "theta", "sigma"))
    n = len(O.net_layers(net))
    t = {f"flip_in.{i}": torch.from_numpy(fx[f"flip_in_call{i}"]) for i in range(n)}
    t.update({f"flip_out.{i}": torch.from_numpy(fx[f"flip_out_call{i}"]) for i in range(n)})
    w = mu + sg * torch.from_numpy(fx["ws_eps"][0])
    out = O.forward_flipout(net, x, mu, w, O.InjectedNoise(t))
    np.testing.assert_allclose(out.numpy(), fx["out_flipout"], rtol=1e-5, atol=1e-6)


def test_deep_ensemble(golden_dir):
    z = np.load(os.path.join(golden_dir, "deep_ensemble.npz"))
    mu, sd = O.deep_ensemble_moments(torch.from_numpy(z["mu_m"]), torch.from_numpy(z["sigma_m"]))
    np.testing.assert_allclose(mu.numpy(), z["preds"], rtol=1e-5)
    np.testing.assert_allclose(sd.numpy(), z["stds"], rtol=1e-3, atol=1e-4)


@pytest.mark.parametrize("net", NETS)
def test_init_params_std(golden_dir, net):
    ref = np.load(os.path.join(golden_dir, "weights_init_std.npz"))[net]
    th = O.init_params(net, 3)
    for (name, shape, off), r in zip(O.site_table(net), ref):
        n = int(np.prod(shape))
        if n >= 512:
            assert abs(th[off:off + n].std().item() / r - 1) < 0.15, name


# ------------------------------------------------------------------ independent formulas


def test_philox_known_answers():
    # Random123 kat_vectors: philox4x32-10
    kats = [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for c, k, want in kats:
        got = O.philox4x32_10(*[np.array([v]) for v in c], k[0], k[1])
        assert tuple(int(g[0]) for g in got) == want
    # Random123 kat_vectors: philox4x32-7 (the dropout-mask generator)
    kats7 = [
        ((0, 0, 0, 0), (0, 0), (0x5F6FB709, 0x0D893F64, 0x4F121F81, 0x4F730A48)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x5207DDC2, 0x45165E59, 0x4D8EE751, 0x8C52F662)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0x4DFCCABA, 0x190A87F0, 0xC47362BA, 0xB6B5242A)),
    ]
    for c, k, want in kats7:
        got = O.philox4x32_10(*[np.array([v]) for v in c], k[0], k[1], rounds=7)
        assert tuple(int(g[0]) for g in got) == want


def test_philox_normal_moments():
    z = O.philox_normal(42, O.KIND_WEIGHT_EPS, 0, 3, 0, np.arange(400_000))
    assert abs(z.mean()) < 5e-3 and abs(z.std() - 1) < 5e-3
    assert abs(np.mean(z**4) - 3) < 0.05
    s = O.PhiloxNoise("inception", 7).flip_in(2, 4000, 18).numpy()
    assert abs(s.mean()) < 0.02 and set(np.unique(s)) == {-1.0, 1.0}
    m = O.PhiloxNoise("inception", 7).drop_mask(4, (3000, 16, 30), 0.8).numpy()
    assert abs(m.mean() - 0.8) < 5e-3


def test_lrt_moments_match_weight_sampling_linear():
    # SURVEY section 4 item 1: for a linear layer LRT is distributionally exact
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 32, generator=g, dtype=torch.float64)
    mu_w, mu_b = torch.randn(8, 32, generator=g, dtype=torch.float64), torch.randn(8, generator=g, dtype=torch.float64)
    sw, sb = torch.rand(8, 32, generator=g, dtype=torch.float64) * 0.3, torch.rand(8, generator=g, dtype=torch.float64) * 0.3
    S = 200_000
    W = mu_w + sw * torch.randn(S, 8, 32, generator=g, dtype=torch.float64)
    b = mu_b + sb * torch.randn(S, 8, generator=g, dtype=torch.float64)
    o = torch.einsum("sok,k->so", W, x[0]) + b
    m = F.linear(x, mu_w, mu_b)[0]
    v = F.linear(x * x, sw**2, sb**2)[0]
    assert torch.allclose(o.mean(0), m, atol=0.02)
    assert torch.allclose(o.var(0), v, rtol=0.02)


def test_kl_matches_torch_distributions():
    g = torch.Generator().manual_seed(1)
    mu, sg = torch.randn(1000, generator=g, dtype=torch.float64), torch.rand(1000, generator=g, dtype=torch.float64) + 0.01
    want = torch.distributions.kl_divergence(torch.distributions.Normal(mu, sg),
                                             torch.distributions.Normal(0.3, 0.7)).sum()
    assert torch.allclose(O.kl_normal(mu, sg, 0.3, 0.7), want)
    w = mu + sg * torch.randn(1000, generator=g, dtype=torch.float64)
    want = (torch.distributions.Normal(mu, sg).log_prob(w) - torch.distributions.Normal(0.3, 0.7).log_prob(w)).sum()
    assert torch.allclose(O.logq_minus_logp(w, mu, sg, 0.3, 0.7), want)


def test_nll_matches_normal_log_prob():
    g = torch.Generator().manual_seed(2)
    out = torch.rand(50, 2, generator=g, dtype=torch.float64) * 5 + 0.1
    y = torch.rand(50, generator=g, dtype=torch.float64) * 10
    want = -torch.distributions.Normal(out[:, 0], F.softplus(out[:, 1])).log_prob(y).sum()
    assert torch.allclose(O.heteroskedastic_nll_sum(out, y), want)


def test_radial_norm_property():
    net = "conv"
    P = O.num_params(net)
    g = torch.Generator().manual_seed(3)
    mu, sg = torch.zeros(P, dtype=torch.float64), torch.full((P,), 0.1, dtype=torch.float64)
    nz = O.InjectedNoise(O.make_injected_noise(net, 1, "radial", g, dtype=torch.float64))
    w = O.sample_weights(net, mu, sg, "radial", nz)
    for j, (_, shape, off) in enumerate(O.site_table(net)):
        n = int(np.prod(shape))
        assert math.isclose(torch.linalg.vector_norm((w[off:off + n] - mu[off:off + n]) / 0.1).item(),
                            abs(nz.t["radial_r"][j].item()), rel_tol=1e-9)


def test_elbo_scaling_anchor():
    # SURVEY A.10: KL/(N*540) for the Flipout hyper-parameters ~ 0.0092
    P = O.num_params("inception")
    mu = torch.zeros(P, dtype=torch.float64)
    sg = torch.full((P,), 2.14e-4, dtype=torch.float64)
    kl = O.kl_normal(mu, sg, 0.0, 0.198768) / (238150 * 540)
    assert 0.0088 < kl.item() < 0.0096


@pytest.mark.parametrize("mode,guide", [("lrt", "normal"), ("flipout", "normal"), ("ws", "normal"), ("ws", "radial")])
def test_elbo_grads_finite_difference(mode, guide):
    net = "conv"
    g = torch.Generator().manual_seed(4)
    P = O.num_params(net)
    mu = O.init_params(net, 1, torch.float64)
    sg = torch.full((P,), 0.05, dtype=torch.float64)
    x = torch.randn(4, 30, 18, generator=g, dtype=torch.float64)
    y = torch.rand(4, generator=g, dtype=torch.float64) * 50
    md = "radial" if guide == "radial" else mode
    nz = [O.InjectedNoise(O.make_injected_noise(net, 4, md, g, dtype=torch.float64)) for _ in range(2)]
    kw = dict(mode=mode, guide=guide, prior_loc=0.0, prior_scale=0.2, dataset_size=1000, noises=nz)
    aux = O.elbo_loss_and_grads(net, x, y, mu, sg, **kw)
    idx = torch.randint(0, P, (6,), generator=g)
    for i in idx.tolist():
        for which, grad in (("mu", aux["grad_mu"]), ("sigma", aux["grad_sigma"])):
            h = 1e-6
            a, b = (mu.clone(), sg.clone()), (mu.clone(), sg.clone())
            k = 0 if which == "mu" else 1
            a[k][i] += h
            b[k][i] -= h
            fd = (O.elbo_loss(net, x, y, *a, **kw)[0] - O.elbo_loss(net, x, y, *b, **kw)[0]) / (2 * h)
            assert math.isclose(fd.item(), grad[i].item(), rel_tol=2e-4, abs_tol=1e-10), (which, i)


def test_clipped_adam_matches_torch_adam_when_unclipped():
    g = torch.Generator().manual_seed(5)
    p = torch.randn(100, generator=g, dtype=torch.float64)
    q = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([q], lr=1e-3, betas=(0.95, 0.999), eps=1e-8)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for step in range(1, 6):
        gr = torch.randn(100, generator=g, dtype=torch.float64)
        q.grad = gr.clone()
        opt.step()
        p, m, v = O.clipped_adam_step(p, gr, m, v, step, 1e-3)
    # pyro's ClippedAdam adds eps to sqrt(v) before bias correction (old-style Adam): eps-level difference
    assert torch.allclose(p, q.detach(), rtol=1e-6, atol=1e-8)


def test_aggregate_and_gaussian_nll():
    g = torch.Generator().manual_seed(6)
    out = torch.rand(7, 11, 2, generator=g, dtype=torch.float64) + 0.5
    agg = O.aggregate_predictions(out)
    assert torch.allclose(F.softplus(agg[:, 1]), ((out[:, :, 1] ** 2).mean(0) + out[:, :, 0].var(0)).sqrt())
    pred, std, ep, al = O.predictive_moments(out)
    assert torch.allclose(ep, out[:, :, 0].var(0, unbiased=True))
