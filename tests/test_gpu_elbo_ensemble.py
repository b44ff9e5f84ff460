"""Member-batched ELBO step over the seeds of a BNN experiment (brl_elbo_step_ensemble / Engine.elbo_step_ensemble).

Member m of an M-member step is elbo_step(x[m], y[m], mu[m], sigma[m], noise with sample0 + m * particles); injected noise is
member-major, particle-minor.  On the fused back-end with the Inception net the members share every launch (member = blockIdx.z
of the fused kernels, blockIdx.y of the sampler / sign / finalisation kernels); everywhere else they run one after another on
the single-member step.  Either way a member's result equals the single-member step's up to summation order: scalars and
outputs rtol 1e-5, gradient max |diff| / max |grad| < 3e-4 at B >= 256 (the bounds of tests/test_gpu_hnn_ensemble.py) and
< 1e-3 below.  The fc layer's split-K sums are fp32 atomics whose order depends on which CTAs run together; a last-bit change
flips the rounding of one bf16 gradient-image element, and the fewer windows a batch has, the more one element weighs in a
weight gradient.  Measured on a B200: eight single-member calls on the same inputs were up to 1.6e-4 apart (LRT grad_sigma,
B = 256); a member of a 3-member LRT step was 4.7e-4 from its single-member step at B = 37, i.e. 1.6e-4 scaled by 256 / 37
is the expected size.  Against the float64 oracle the fused
back-end's bounds hold (tests/test_gpu_tc_train.py): loss and nll 5e-3, kl 1e-4, outputs 1e-2, likelihood-gradient cosine
> 0.999 (> 0.99 for a ragged 37-window batch)."""
import pytest
import torch

from oracle import bnn_oracle as O
from tests.helpers import injected_to_engine, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NET = "inception"
KW = dict(prior_loc=0.0, prior_scale=0.138793, dataset_size=238150)
# (mode, guide, particles): LRT, Flipout, weight sampling with the normal guide, the radial guide (weight sampling)
CONFIGS = [("lrt", "normal", 1), ("flipout", "normal", 2), ("ws", "normal", 1), ("lrt", "radial", 1)]


@pytest.fixture(scope="module")
def eng():
    from bayesrul_b200 import Engine
    e = Engine(NET, DEV)
    e.set_gemm_backend("fused")
    yield e
    e.set_gemm_backend("simt")
    e.set_step_graph(True)


def _members(net, M, B, seed, sigma=0.02):
    """distinct windows, targets, locs and scales per member"""
    xs, ys, mus, sgs = zip(*[synth(net, B, seed=seed + 7 * m, sigma=sigma * (1 + 0.25 * m)) for m in range(M)])
    return tuple(torch.stack(t).to(DEV) for t in (xs, ys, mus, sgs))


def _singles(e, x, y, mu, sg, seed, s0, mode, guide, particles, compute_grads=True):
    from bayesrul_b200 import Noise
    return [e.elbo_step(x[m], y[m], mu[m], sg[m], mode=mode, guide=guide, particles=particles,
                        noise=Noise(seed=seed, sample0=s0 + m * particles), compute_grads=compute_grads, **KW)
            for m in range(x.shape[0])]


def _assert_member(got, ref, m, what, grads=True):
    assert torch.allclose(got["scalars"][m], ref["scalars"], rtol=1e-5, atol=0), (what, m, got["scalars"][m], ref["scalars"])
    assert torch.allclose(got["out"][m], ref["out"], rtol=1e-5, atol=1e-6), (what, m, (got["out"][m] - ref["out"]).abs().max())
    if grads:
        bound = 3e-4 if ref["out"].shape[-2] >= 256 else 1e-3
        for k in ("grad_mu", "grad_sigma", "grad_log_sigma"):
            rel = ((got[k][m] - ref[k]).abs().max() / ref[k].abs().max()).item()
            assert rel < bound, (what, m, k, rel)


def _cos(a, b):
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-300))


def _launches(e, fn):
    torch.cuda.synchronize()
    n0 = e.lib.brl_launch_count()
    fn()
    torch.cuda.synchronize()
    return e.lib.brl_launch_count() - n0


@pytest.mark.parametrize("mode,guide,particles", CONFIGS)
@pytest.mark.parametrize("B", [256, 37])
@pytest.mark.parametrize("M", [1, 3, 5])
def test_members_match_single_steps(eng, M, B, mode, guide, particles):
    from bayesrul_b200 import Noise
    x, y, mu, sg = _members(NET, M, B, seed=100 + M + B)
    got = eng.elbo_step_ensemble(x, y, mu, sg, mode=mode, guide=guide, particles=particles, noise=Noise(seed=11, sample0=3), **KW)
    refs = _singles(eng, x, y, mu, sg, 11, 3, mode, guide, particles)
    assert eng.tc_status() == 0
    assert got["scalars"].shape == (M, 4) and got["scalars"].dtype == torch.float64
    assert got["out"].shape == (M, particles, B, 2) and got["grad_mu"].shape == (M, eng.P)
    for m in range(M):
        _assert_member(got, refs[m], m, f"{mode}/{guide} M={M} B={B}")


@pytest.mark.parametrize("mode,particles", [("lrt", 1), ("flipout", 2)])
@pytest.mark.parametrize("B", [256, 37])
def test_injected_noise_vs_oracle(eng, B, mode, particles):
    M = 3
    x, y, mu, sg = _members(NET, M, B, seed=300 + B)
    g = torch.Generator().manual_seed(5)
    nzs = [[O.make_injected_noise(NET, B, mode, g) for _ in range(particles)] for _ in range(M)]
    flat = [n for per in nzs for n in per]  # member-major, particle-minor
    got = eng.elbo_step_ensemble(x, y, mu, sg, mode=mode, particles=particles, noise=injected_to_engine(NET, flat, B, DEV), **KW)
    assert eng.tc_status() == 0
    c = 1.0 / (KW["dataset_size"] * 540.0)
    for m in range(M):
        mu_m, sg_m = mu[m].cpu().double(), sg[m].cpu().double()
        ref = O.elbo_loss_and_grads(NET, x[m].cpu().double(), y[m].cpu().double(), mu_m, sg_m, mode=mode, guide="normal",
                                    noises=[O.InjectedNoise({k: v.double() for k, v in n.items()}) for n in nzs[m]], **KW)
        sc = got["scalars"][m].cpu()
        out_err = ((got["out"][m].cpu().double() - ref["out"]).abs() / ref["out"].abs().clamp_min(1e-3)).max().item()
        # the likelihood part of the gradient (the analytic KL gradient is the same on both sides)
        kl_mu = c * mu_m / KW["prior_scale"] ** 2
        cs = _cos(got["grad_mu"][m].cpu().double() - kl_mu, ref["grad_mu"] - kl_mu)
        print(f"\n[ensemble oracle {mode} B={B} member {m}] loss {sc[0].item():.6e} vs {ref['loss'].item():.6e}, "
              f"out err {out_err:.2e}, likelihood grad_mu cosine {cs:.6f}")
        assert abs(sc[0].item() / ref["loss"].item() - 1) < 5e-3
        assert abs(sc[1].item() / ref["nll_sum"].item() - 1) < 5e-3
        assert abs(sc[2].item() / ref["kl"].item() - 1) < 1e-4
        assert out_err < 1e-2
        assert cs > (0.999 if B >= 256 else 0.99), (m, cs)


def test_members_share_launches(eng):
    from bayesrul_b200 import Noise
    eng.set_step_graph(False)
    try:
        for mode, particles in (("lrt", 1), ("flipout", 2)):
            kw = dict(mode=mode, particles=particles, noise=Noise(seed=2), **KW)
            counts = {}
            for M in (1, 5):
                x, y, mu, sg = _members(NET, M, 256, seed=400)
                eng.elbo_step_ensemble(x, y, mu, sg, **kw)  # warm-up: workspace growth, kernel attributes
                counts[M] = _launches(eng, lambda: eng.elbo_step_ensemble(x, y, mu, sg, **kw))
            single = _launches(eng, lambda: eng.elbo_step(x[0], y[0], mu[0], sg[0], **kw))
            print(f"\n[ensemble launches {mode}] M=1: {counts[1]}, M=5: {counts[5]}, elbo_step: {single}")
            assert counts[1] == counts[5] == single > 0, (mode, counts, single)
    finally:
        eng.set_step_graph(True)
    assert eng.tc_status() == 0


@pytest.mark.parametrize("mode,particles", [("lrt", 1), ("flipout", 2)])
def test_graph_replay_equals_eager(eng, mode, particles):
    from bayesrul_b200 import Noise
    M, B = 4, 128
    _, _, mu, sg = _members(NET, M, B, seed=500)  # one parameter stack for the whole sequence: part of the graph key
    steps = [(_members(NET, M, B, seed=510 + 3 * i)[:2], Noise(seed=20 + i, sample0=5 * i)) for i in range(4)]
    kw = dict(mode=mode, particles=particles, **KW)
    replayed = []
    for (x, y), nz in steps + steps:  # first pass: eager, capture, then replays; the second pass replays every step
        r = eng.elbo_step_ensemble(x, y, mu, sg, noise=nz, **kw)
        replayed.append({k: v.clone() for k, v in r.items()})
    eng.set_step_graph(False)
    try:
        eager = [eng.elbo_step_ensemble(x, y, mu, sg, noise=nz, **kw) for (x, y), nz in steps]
    finally:
        eng.set_step_graph(True)
    assert eng.tc_status() == 0
    for i, ref in enumerate(eager):
        for got in (replayed[i], replayed[len(steps) + i]):
            for m in range(M):
                _assert_member(got, {k: v[m] for k, v in ref.items()}, m, f"{mode} graph step {i}")
    # a new seed draws new noise (same inputs, same sample0)
    (x, y), nz = steps[0]
    other = eng.elbo_step_ensemble(x, y, mu, sg, noise=Noise(seed=nz.seed + 1000, sample0=nz.sample0), **kw)
    for m in range(M):
        assert not torch.allclose(other["out"][m], eager[0]["out"][m], rtol=1e-3), m


@pytest.mark.parametrize("B", [1, 5, 129, 1000])
def test_ragged_batches(eng, B):
    from bayesrul_b200 import Noise
    M = 3
    x, y, mu, sg = _members(NET, M, B, seed=600 + B)
    for mode, particles in (("lrt", 1), ("flipout", 2)):
        got = eng.elbo_step_ensemble(x, y, mu, sg, mode=mode, particles=particles, noise=Noise(seed=4, sample0=1), **KW)
        refs = _singles(eng, x, y, mu, sg, 4, 1, mode, "normal", particles)
        assert eng.tc_status() == 0
        for m in range(M):
            _assert_member(got, refs[m], m, f"{mode} B={B}")


@pytest.mark.parametrize("net,backend", [("inception", "simt"), ("linear", "fused"), ("conv", "fused")])
def test_member_loop_fallback(net, backend):
    from bayesrul_b200 import Engine, Noise
    e = Engine(net, DEV)
    e.set_gemm_backend(backend)
    M, B = 3, 64
    x, y, mu, sg = _members(net, M, B, seed=700)
    got = e.elbo_step_ensemble(x, y, mu, sg, mode="lrt", noise=Noise(seed=6, sample0=2), **KW)
    refs = _singles(e, x, y, mu, sg, 6, 2, "lrt", "normal", 1)
    e.set_step_graph(False)
    one = _launches(e, lambda: e.elbo_step(x[0], y[0], mu[0], sg[0], mode="lrt", noise=Noise(seed=6), **KW))
    loop = _launches(e, lambda: e.elbo_step_ensemble(x, y, mu, sg, mode="lrt", noise=Noise(seed=6), **KW))
    assert e.tc_status() == 0
    assert loop == M * one, (loop, one)
    for m in range(M):
        _assert_member(got, refs[m], m, f"{net}/{backend}")


def test_one_member_workspace_and_too_small(eng):
    from bayesrul_b200 import Noise
    M, B = 3, 256
    x, y, mu, sg = _members(NET, M, B, seed=800)
    refs = _singles(eng, x, y, mu, sg, 8, 0, "lrt", "normal", 1)

    def call(nbytes):
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=DEV)
        sc = torch.empty(M, 4, dtype=torch.float64, device=DEV)
        out = torch.empty(M, 1, B, 2, device=DEV)
        g = [torch.empty(M, eng.P, device=DEV) for _ in range(3)]
        nz, keep = eng._noise(Noise(seed=8))
        rc = eng.lib.brl_elbo_step_ensemble(eng.ctx, x.data_ptr(), y.data_ptr(), M, B, mu.data_ptr(), sg.data_ptr(), 2, 0, 1,
                                            KW["prior_loc"], KW["prior_scale"], KW["dataset_size"], nz, 1, sc.data_ptr(),
                                            g[0].data_ptr(), g[1].data_ptr(), g[2].data_ptr(), out.data_ptr(), ws.data_ptr(),
                                            ws.numel(), eng._stream())
        torch.cuda.synchronize()
        return rc, dict(scalars=sc, out=out, grad_mu=g[0], grad_sigma=g[1], grad_log_sigma=g[2])

    one_member = eng.lib.brl_workspace_bytes(eng.ctx, B, 1, 1, 0)
    assert one_member < eng.lib.brl_workspace_bytes(eng.ctx, B, M, 4, 0)
    eng.set_step_graph(False)
    try:
        single = _launches(eng, lambda: eng.elbo_step(x[0], y[0], mu[0], sg[0], mode="lrt", noise=Noise(seed=8), **KW))
        n0 = eng.lib.brl_launch_count()
        rc, got = call(one_member)
        loop = eng.lib.brl_launch_count() - n0
        rc_small, _ = call(1 << 16)
    finally:
        eng.set_step_graph(True)
    assert rc == 0 and eng.tc_status() == 0
    assert loop == M * single, (loop, single)  # one member after another
    for m in range(M):
        _assert_member(got, refs[m], m, "one-member workspace")
    assert rc_small != 0 and "workspace too small" in eng.lib.brl_last_error().decode()


def test_validation(eng):
    x, y, mu, sg = _members(NET, 3, 64, seed=850)
    for args in ((x[:, :, :, :17].contiguous(), y, mu, sg), (x, y[:2], mu, sg), (x, y, mu[:2], sg), (x, y, mu, sg[:, :-1]),
                 (x[:0], y[:0], mu[:0], sg[:0])):
        with pytest.raises(RuntimeError):
            eng.elbo_step_ensemble(*args, **KW)


def test_compute_grads_false(eng):
    from bayesrul_b200 import Noise
    x, y, mu, sg = _members(NET, 5, 256, seed=900)
    for mode, particles in (("lrt", 1), ("flipout", 2)):
        kw = dict(mode=mode, particles=particles, noise=Noise(seed=3), **KW)
        a = eng.elbo_step_ensemble(x, y, mu, sg, **kw)
        b = eng.elbo_step_ensemble(x, y, mu, sg, compute_grads=False, **kw)
        assert b["grad_mu"] is None and b["grad_sigma"] is None and b["grad_log_sigma"] is None
        assert eng.tc_status() == 0
        assert torch.allclose(a["scalars"], b["scalars"], rtol=1e-5, atol=0), mode
        assert torch.allclose(a["out"], b["out"], rtol=1e-5, atol=1e-6), mode


def test_training_matches_independent_seeds(eng):
    """Ten steps of elbo_step_ensemble + ONE clipped_adam_vi over [5, P] loc / log-scale stacks follow five independent
    elbo_step + clipped_adam_vi runs; a trained member's (loc, scale) then predicts what the member trained alone predicts."""
    from bayesrul_b200 import Noise
    M, B, steps, lr = 5, 256, 10, 1e-3
    x, y, mu0, sg0 = _members(NET, M, B, seed=1000)

    def state(mu, sg):
        return dict(loc=mu.clone(), ls=sg.log(), scale=sg.clone(), m_loc=torch.zeros_like(mu), v_loc=torch.zeros_like(mu),
                    m_ls=torch.zeros_like(mu), v_ls=torch.zeros_like(mu))

    def adam(s, r, k):
        eng.clipped_adam_vi(s["loc"], s["ls"], s["scale"], r["grad_mu"], r["grad_log_sigma"], s["m_loc"], s["v_loc"], s["m_ls"],
                            s["v_ls"], step=k + 1, lr=lr)

    ens = state(mu0, sg0)
    ind = [state(mu0[m], sg0[m]) for m in range(M)]
    for k in range(steps):
        r = eng.elbo_step_ensemble(x, y, ens["loc"], ens["scale"], mode="lrt", noise=Noise(seed=40 + k), **KW)
        adam(ens, r, k)
        for m in range(M):
            s = eng.elbo_step(x[m], y[m], ind[m]["loc"], ind[m]["scale"], mode="lrt", noise=Noise(seed=40 + k, sample0=m), **KW)
            adam(ind[m], s, k)
            rel = abs(r["scalars"][m, 0].item() / s["scalars"][0].item() - 1)
            assert rel < 1e-3, (k, m, rel)
    assert eng.tc_status() == 0
    for m in (0, M - 1):
        a = eng.predict_moments(x[m], ens["loc"][m].contiguous(), ens["scale"][m].contiguous(), S=8, noise=Noise(seed=9))
        b = eng.predict_moments(x[m], ind[m]["loc"], ind[m]["scale"], S=8, noise=Noise(seed=9))
        for u, v in zip(a, b):
            err = ((u - v).abs() / v.abs().clamp_min(1e-3)).max().item()
            assert err < 1e-2, (m, err)
