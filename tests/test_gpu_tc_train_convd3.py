"""Level-fused tcgen05 training kernels of the Conv-D3 net (brl_set_gemm_backend 'fused': csrc/brl_tc_train_convd3.cuh).

The same checks as tests/test_gpu_tc_train_linear.py for the Linear net: one svi.step (LRT, Flipout, weight sampling) and one
HNN.step against the float64 oracle with the oracle's own noise injected, native Philox noise against the fp32 FFMA back-end
(same keys, same draws), graph replay against the eager step, ragged batches, and the public surfaces.  Stated bound of the
back-end (fp16 / bf16 operands, fp32 accumulation): outputs 1e-2, loss 5e-3, KL 1e-4, and for the likelihood part of the
gradient (the analytic KL gradient, identical on both sides, is subtracted) cosine > 0.999 and relative L2 error < 3e-2 per
layer group at B = 256 (cosine > 0.99 and relative L2 < 0.15 at small ragged batches)."""
import pytest
import torch

from oracle import bnn_oracle as O
from tests.helpers import injected_to_engine, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NET = "conv"
KW = dict(guide="normal", prior_loc=0.0, dataset_size=238150)
C = 1.0 / (238150 * 540.0)


@pytest.fixture(scope="module")
def eng():
    from bayesrul_b200 import Engine
    e = Engine(NET, DEV)
    yield e
    e.set_gemm_backend("simt")


def _kl_grads(mu, sg, prior_scale):
    return C * (mu / prior_scale**2), C * (-1.0 / sg + sg / prior_scale**2)


def _cos(a, b):
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-300))


def _groups(e):
    """(name, slice) of the whole net and of each layer (weight + bias)."""
    sites = [s[0] for s in e.info["sites"]] + [e.info["P"]]
    return [("all", slice(None))] + [(f"layer{ly}", slice(sites[2 * ly], sites[2 * ly + 2])) for ly in range(4)]


def _check_grads(e, got, ref, mu, sg, prior_scale, tag, cos_min=0.999, rel_max=3e-2):
    kmu, ksg = _kl_grads(mu.double(), sg.double(), prior_scale)
    for name, g, r, k in (("grad_mu", got["grad_mu"], ref["grad_mu"], kmu), ("grad_sigma", got["grad_sigma"], ref["grad_sigma"], ksg)):
        a = g.double().cpu() - k
        b = r.double().cpu() - k
        for part, sl in _groups(e):
            cs, rel = _cos(a[sl], b[sl]), float((a[sl] - b[sl]).norm() / (b[sl].norm() + 1e-300))
            print(f"[{tag}] {name}[{part}]: cosine {cs:.6f}, rel L2 err {rel:.2e}")
            assert cs > cos_min and rel < rel_max, (tag, name, part, cs, rel)


@pytest.mark.parametrize("mode,particles,sigma,prior_scale", [
    ("lrt", 1, 0.05, 0.138793), ("lrt", 1, 1.351e-3, 0.138793),
    ("flipout", 2, 0.05, 0.198768), ("flipout", 2, 2.14e-4, 0.198768)])
@pytest.mark.parametrize("B", [256, 37])
def test_fused_conv_elbo_step_vs_oracle(eng, mode, particles, sigma, prior_scale, B):
    x, y, mu, sg = synth(NET, B, seed=21 + B, sigma=sigma)
    g = torch.Generator().manual_seed(4)
    nzs = [O.make_injected_noise(NET, B, mode, g) for _ in range(particles)]
    kw = dict(mode=mode, prior_scale=prior_scale, **KW)
    ref = O.elbo_loss_and_grads(NET, x.double(), y.double(), mu.double(), sg.double(),
                                noises=[O.InjectedNoise({k: v.double() for k, v in n.items()}) for n in nzs], **kw)
    eng.set_gemm_backend("fused")
    got = eng.elbo_step(x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV), particles=particles,
                        noise=injected_to_engine(NET, nzs, B, DEV), **kw)
    eng.set_gemm_backend("simt")
    assert eng.tc_status() == 0
    tag = f"{mode} sigma={sigma} B={B}"
    sc = got["scalars"].cpu()
    out_err = ((got["out"].cpu().double() - ref["out"]).abs() / ref["out"].abs().clamp_min(1e-3)).max().item()
    print(f"\n[{tag}] loss {sc[0].item():.6e} vs {ref['loss'].item():.6e}, nll {sc[1].item():.5e} vs {ref['nll_sum'].item():.5e}, "
          f"max rel out err {out_err:.2e}")
    assert abs(sc[0].item() / ref["loss"].item() - 1) < 5e-3
    assert abs(sc[1].item() / ref["nll_sum"].item() - 1) < 5e-3
    assert abs(sc[2].item() / ref["kl"].item() - 1) < 1e-4
    assert out_err < 1e-2
    if B >= 256:
        _check_grads(eng, got, ref, mu, sg, prior_scale, tag)
    else:
        _check_grads(eng, got, ref, mu, sg, prior_scale, tag, cos_min=0.99, rel_max=1.5e-1)


@pytest.mark.parametrize("mode,particles", [("lrt", 1), ("flipout", 2)])
def test_fused_conv_native_noise_matches_fp32_backend(eng, mode, particles):
    """Native Philox noise: the fused back-end draws the same eps / signs as the fp32 back-end; a graph-replayed step equals
    the eager one; a new seed is a new draw."""
    from bayesrul_b200 import Noise
    B = 256
    x, y, mu, sg = synth(NET, B, seed=5, sigma=0.02)
    x, y, mu, sg = x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV)
    kw = dict(mode=mode, prior_scale=0.138793, particles=particles, **KW)
    eng.set_gemm_backend("simt")
    ref = eng.elbo_step(x, y, mu, sg, noise=Noise(seed=11), **kw)
    eng.set_gemm_backend("fused")
    runs = [eng.elbo_step(x, y, mu, sg, noise=Noise(seed=11), **kw) for _ in range(3)]  # eager, captured, replayed
    other = eng.elbo_step(x, y, mu, sg, noise=Noise(seed=12), **kw)
    eng.set_gemm_backend("simt")
    assert eng.tc_status() == 0
    got = runs[0]
    assert not torch.equal(got["out"], ref["out"])  # the fused kernels ran (the fp32 fall-back would match bit for bit)
    assert abs(got["scalars"][0].item() / ref["scalars"][0].item() - 1) < 5e-3
    for k in ("grad_mu", "grad_sigma"):
        cs = _cos(got[k].double(), ref[k].double())
        print(f"[{mode}] fused vs fp32 {k}: cosine {cs:.6f}")
        assert cs > 0.999, (k, cs)
    for r in runs[1:]:
        assert torch.allclose(r["scalars"], got["scalars"], rtol=1e-5)
        for k in ("grad_mu", "grad_sigma"):
            d = (r[k] - got[k]).abs().max().item() / got[k].abs().max().item()
            assert d < 1e-4, (k, d)
    assert abs(other["scalars"][1].item() - got["scalars"][1].item()) > 0


@pytest.mark.parametrize("B", [1, 5, 129, 1000])
def test_fused_conv_batch_sizes_match_fp32_backend(eng, B):
    """Ragged last M-tile (B * positions not a multiple of 128) and many M-tiles per weight-gradient CTA (B = 1000: conv1 has
    2032 M-tiles over 148 CTAs)."""
    from bayesrul_b200 import Noise
    x, y, mu, sg = synth(NET, B, seed=100 + B, sigma=0.01)
    x, y, mu, sg = x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV)
    for mode, particles in (("lrt", 1), ("flipout", 2)):
        kw = dict(mode=mode, prior_scale=0.138793, particles=particles, **KW)
        eng.set_gemm_backend("simt")
        ref = eng.elbo_step(x, y, mu, sg, noise=Noise(seed=3), **kw)
        eng.set_gemm_backend("fused")
        got = eng.elbo_step(x, y, mu, sg, noise=Noise(seed=3), **kw)
        eng.set_gemm_backend("simt")
        assert eng.tc_status() == 0
        assert abs(got["scalars"][0].item() / ref["scalars"][0].item() - 1) < 5e-3, (mode, B)
        assert torch.allclose(got["out"], ref["out"], rtol=1e-2, atol=1e-3), (mode, B)
        kmu, ksg = _kl_grads(mu.double().cpu(), sg.double().cpu(), 0.138793)
        for k, kk in (("grad_mu", kmu), ("grad_sigma", ksg)):
            cs = _cos(got[k].double().cpu() - kk, ref[k].double().cpu() - kk)
            assert cs > (0.999 if B >= 129 else 0.98), (mode, B, k, cs)


@pytest.mark.parametrize("guide", ["normal", "radial"])
@pytest.mark.parametrize("B", [256, 33])
def test_fused_conv_weight_sampling_elbo_vs_oracle(eng, guide, B):
    """Weight-sampling ELBO (no fit context / the radial guide's Trace_ELBO): one contraction with the particle's draw."""
    x, y, mu, sg = synth(NET, B, seed=70 + B, sigma=0.03)
    g = torch.Generator().manual_seed(8)
    nzs = [O.make_injected_noise(NET, B, "radial" if guide == "radial" else "ws", g)]
    kw = dict(mode="ws", guide=guide, prior_loc=0.0, prior_scale=0.138793, dataset_size=238150)
    ref = O.elbo_loss_and_grads(NET, x.double(), y.double(), mu.double(), sg.double(),
                                noises=[O.InjectedNoise({k: v.double() for k, v in n.items()}) for n in nzs], **kw)
    eng.set_gemm_backend("fused")
    got = eng.elbo_step(x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV), particles=1, noise=injected_to_engine(NET, nzs, B, DEV), **kw)
    eng.set_gemm_backend("simt")
    assert eng.tc_status() == 0
    sc = got["scalars"].cpu()
    assert abs(sc[0].item() / ref["loss"].item() - 1) < 5e-3
    assert abs(sc[1].item() / ref["nll_sum"].item() - 1) < 5e-3
    out_err = ((got["out"].cpu().double() - ref["out"]).abs() / ref["out"].abs().clamp_min(1e-3)).max().item()
    assert out_err < 1e-2, out_err
    cs = _cos(got["grad_mu"].double().cpu(), ref["grad_mu"])
    print(f"\n[ws {guide} B={B}] loss {sc[0].item():.6e} vs {ref['loss'].item():.6e}, out err {out_err:.2e}, grad_mu cosine {cs:.6f}")
    assert cs > (0.999 if B >= 256 else 0.99), cs


@pytest.mark.parametrize("p", [0.0, 0.3])
@pytest.mark.parametrize("B", [256, 29])
def test_fused_conv_hnn_step_vs_oracle(eng, p, B):
    """HNN.step (forward with the dropout sites, F.gaussian_nll_loss, backward) with the oracle's keep masks injected; native
    masks against the fp32 back-end; graph replay == eager."""
    from bayesrul_b200 import Noise
    x, y, mu, _ = synth(NET, B, seed=31 + B)
    g = torch.Generator().manual_seed(5)
    nz = O.make_injected_noise(NET, B, "det", g, p_dropout=p)
    th = mu.double().requires_grad_(True)
    loss, out = O.hnn_loss(NET, x.double(), y.double(), th, p, O.InjectedNoise({k: v.double() for k, v in nz.items()}))
    (gref,) = torch.autograd.grad(loss, th)
    eng.set_gemm_backend("fused")
    got = eng.hnn_step(x.to(DEV), y.to(DEV), mu.to(DEV), p, injected_to_engine(NET, [nz], B, DEV) if p > 0 else None)
    xd, yd, mud = x.to(DEV), y.to(DEV), mu.to(DEV)
    runs = [eng.hnn_step(xd, yd, mud, p, Noise(seed=9)) for _ in range(3)]
    eng.set_gemm_backend("simt")
    simt = eng.hnn_step(xd, yd, mud, p, Noise(seed=9))
    assert eng.tc_status() == 0
    assert abs(got["scalars"][0].item() / loss.item() - 1) < 5e-3
    out_err = ((got["out"].cpu().double() - out.detach()).abs() / out.detach().abs().clamp_min(1e-3)).max().item()
    cs = _cos(got["grad"].double().cpu(), gref)
    print(f"\n[hnn p={p} B={B}] loss {got['scalars'][0].item():.6e} vs {loss.item():.6e}, out err {out_err:.2e}, grad cosine {cs:.6f}")
    assert out_err < 1e-2
    assert cs > (0.99 if B < 256 else 0.999)
    assert abs(runs[0]["scalars"][0].item() / simt["scalars"][0].item() - 1) < 5e-3
    assert _cos(runs[0]["grad"].double(), simt["grad"].double()) > 0.999
    for r in runs[1:]:
        assert torch.allclose(r["scalars"], runs[0]["scalars"], rtol=1e-5)


def test_fused_conv_elbo_loss_op_is_differentiable():
    from bayesrul_b200.ops import elbo_loss
    B = 64
    x, y, mu, sg = synth(NET, B, seed=9, sigma=0.02)
    x, y = x.to(DEV), y.to(DEV)
    mu = mu.to(DEV).requires_grad_(True)
    ls = sg.log().to(DEV).requires_grad_(True)
    kw = dict(net=NET, mode="lrt", guide="normal", particles=1, prior_loc=0.0, prior_scale=0.138793, dataset_size=238150, seed=3)
    loss = elbo_loss(mu, ls, x, y, backend="fused", **kw)
    (2.0 * loss).backward()
    ref = O.elbo_loss_and_grads(NET, x.cpu().double(), y.cpu().double(), mu.detach().cpu().double(), ls.detach().exp().cpu().double(),
                                mode="lrt", guide="normal", prior_loc=0.0, prior_scale=0.138793, dataset_size=238150,
                                noises=[O.PhiloxNoise(NET, 3)])
    assert abs(loss.item() / ref["loss"].item() - 1) < 5e-3
    for g, r in ((mu.grad, ref["grad_mu"]), (ls.grad, ref["grad_log_sigma"])):
        cs = float((g.cpu().double() * 2.0 * r).sum() / (g.cpu().double().norm() * (2.0 * r).norm()))
        assert cs > 0.999 and abs(float(g.cpu().double().norm() / (2.0 * r).norm()) - 1) < 2e-2, cs


def _batch(B, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, 30, 18, generator=g).to(DEV), (torch.rand(B, generator=g) * 100).to(DEV)


def test_fused_conv_compat_bnn_and_hnn_training_step():
    import numpy as np
    from functools import partial
    from bayesrul_b200.compat import BNN, HNN, Conv, pyro_shim
    torch.manual_seed(12345)
    net = Conv(30, 18)
    opt = pyro_shim.ClippedAdam({"lr": 0.000857, "betas": [0.95, 0.999], "clip_norm": 15})
    m = BNN(net, opt, pretrain_epochs=5, mc_samples_train=1, mc_samples_eval=8, dataset_size=238150, fit_context="lrt",
            prior_loc=0.0, prior_scale=0.138793, guide="normal", q_scale=1.351e-3, device=DEV, train_backend="fused")
    m.on_fit_start()
    x, y = _batch(100)
    m.training_step((x, y), 0)
    assert all(np.isfinite(m.logged[k]) for k in ("elbo/train", "kl/train", "likelihood/train", "mse/train"))
    h = HNN(Conv(30, 18, dropout=0.3), partial(torch.optim.Adam, lr=1e-3), mc_samples=10, p_dropout=0.3, device=DEV,
            train_backend="fused")
    h.net.train()
    loss = h.training_step((x, y), 0)
    loss.backward()
    assert np.isfinite(float(loss)) and all(p.grad is not None and torch.isfinite(p.grad).all() for p in h.net.parameters())
    assert h.net.engine().tc_status() == 0
    h.net.engine().set_gemm_backend("simt")
    m.bnn.engine.set_gemm_backend("simt")


def test_fused_conv_small_workspace_falls_back_to_per_layer_kernels(eng):
    """A workspace sized without room for the Conv-D3 net's images: the 'fused' step runs the per-layer fp32 kernels (the same
    numbers as the 'simt' back-end)."""
    from bayesrul_b200 import Noise
    B = 256
    x, y, mu, sg = synth(NET, B, seed=6, sigma=0.02)
    x, y, mu, sg = x.to(DEV), y.to(DEV), mu.to(DEV), sg.to(DEV)
    kw = dict(mode="lrt", prior_scale=0.138793, particles=1, **KW)
    eng.set_gemm_backend("simt")
    ref = eng.elbo_step(x, y, mu, sg, noise=Noise(seed=2), **kw)
    full = eng.lib.brl_workspace_bytes(eng.ctx, B, 1, 1, 0)
    small = torch.empty(full - (1 << 20), dtype=torch.uint8, device=DEV)  # the images of one lane take > 90 MB
    ws_for = eng._ws_for
    eng._ws_for = lambda *a, **k: small
    try:
        eng.set_gemm_backend("fused")
        got = eng.elbo_step(x, y, mu, sg, noise=Noise(seed=2), **kw)
    finally:
        eng._ws_for = ws_for
        eng.set_gemm_backend("simt")
    assert torch.allclose(got["scalars"], ref["scalars"], rtol=1e-6)
    for k in ("grad_mu", "grad_sigma"):  # the fp32 weight-gradient kernels sum with atomics: equal up to summation order
        d = (got[k] - ref[k]).abs().max().item() / ref[k].abs().max().item()
        assert d < 1e-5, (k, d)
