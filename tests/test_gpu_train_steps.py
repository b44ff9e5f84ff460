"""K training steps per call over a device-resident dataset (brl_elbo_train_steps / brl_hnn_train_steps, Engine.*_train_steps,
compat BNN.fit_epoch).

Step k of a K-step call is, by contract, the per-step sequence a training loop issues: elbo_step_ensemble (elbo_step at M = 1)
on X[idx[k]] with the Philox seed seed + 0x9E3779B97F4A7C15 (k + 1), clipped_adam_vi at step step0 + k + 1 and
step_metrics_ensemble of the logged predictions (hnn_step{,_ensemble} and clipped_adam for the HNN).  Each comparison runs
that reference loop several times from the same state: fp32 atomics in the backward make repeated steps differ in the last bits,
and the K-step call must lie within twice the largest distance between the reference runs (bit for bit where they all agree).
Three runs, not two: on the nondeterministic paths the distance of a single pair is a noisy estimate of the run-to-run spread,
and a measured K-step result fell 2.2-3.8x one pair's distance while differing from the loop only in the last bits.  The bound
also allows 1e-5 of the quantity's largest magnitude: the order of fp32 atomics depends on what else is in flight, so reruns of
the same launch sequence agree more closely with each other than with a different sequence.  Measured on a B200: the K-step
call's first Adam moment of loc on the simt back-end at B = 37 was 1.6e-6 of its magnitude from the loop, whose three runs were
2e-8 apart; an epoch-mean rmsce of fit_epoch 3e-10 from three loops that agreed exactly (one window in a neighbouring bin).
The final parameters and optimizer moments are compared in L2 norm, with 1e-3 of the norm allowed: Adam's normalised update
m / sqrt(v) turns a last-bit difference in a near-zero gradient into a parameter difference of up to lr per step (measured: one
loc element 2.1e-4 apart in the fused M = 5 LRT case, whose loop runs were 9e-6 apart at most; m of log_scale 7e-8 apart in L2
after Flipout steps whose loop runs agreed to 4e-10).  A wrong seed, step size or minibatch moves every quantity by O(1)."""
import math

import pytest
import torch

from oracle import bnn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W = 0x9E3779B97F4A7C15
KW = dict(prior_loc=0.0, prior_scale=0.138793, dataset_size=238150)
OPT = dict(lr=1e-3, betas=(0.95, 0.999), eps=1e-8, clip_norm=15.0, lrd=0.99995, weight_decay=0.0)
HOPT = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, clip_norm=1e30, lrd=1.0, weight_decay=0.0)
P_MCD = 0.241437


_ENGINES = {}


def _eng(net, backend, tag):
    """one engine per (net, back-end, role): the K-step call and each reference run keep their own workspace and graphs"""
    from bayesrul_b200 import Engine
    key = (net, backend, tag)
    if key not in _ENGINES:
        e = Engine(net, DEV)
        e.set_gemm_backend(backend)
        _ENGINES[key] = e
    return _ENGINES[key]


@pytest.fixture(scope="module", autouse=True)
def _cleanup():
    yield
    _ENGINES.clear()


def _data(N, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, 30, 18, generator=g).to(DEV), (torch.rand(N, generator=g) * 100).to(DEV)


def _idx(K, M, B, N, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.stack([torch.randperm(N, generator=g)[:B] for _ in range(M)]) for _ in range(K)]).to(DEV)


def _vi_state(net, M, seed):
    loc = torch.stack([O.init_params(net, seed + m) for m in range(M)]).to(DEV)
    log_scale = torch.full_like(loc, math.log(0.02)) + 0.1 * torch.rand(loc.shape, generator=torch.Generator().manual_seed(seed)).to(DEV)
    z = torch.zeros_like(loc)
    return dict(loc=loc, log_scale=log_scale, scale=log_scale.exp(), m_loc=z.clone(), v_loc=z.clone(), m_ls=z.clone(), v_ls=z.clone())


def _hnn_state(net, M, seed):
    theta = torch.stack([O.init_params(net, seed + m) for m in range(M)]).to(DEV)
    return dict(theta=theta, m=torch.zeros_like(theta), v=torch.zeros_like(theta))


def _clone(st):
    return {k: v.clone() for k, v in st.items()}


def _logged(e, out, yb, particles):
    """step_metrics_ensemble of particle 0's (loc, scale), or of each member's aggregate of several particles (BNN._agg)"""
    M = yb.shape[0]
    lo = torch.stack([out[m, 0] if particles == 1 else e.aggregate_predictions(out[m]) for m in range(M)])
    return e.step_metrics_ensemble(lo[..., 0].contiguous(), lo[..., 1].contiguous(), yb)


def _ref_elbo(e, X, Y, idx, st, cfg, seed, step0, sample0=0, window0=0):
    """the per-step loop of the contract, on `st` in place; returns scalars [K,M,4], metrics [K,M,5]"""
    from bayesrul_b200 import Noise
    mode, guide, particles = cfg
    K, M, B = idx.shape
    sc, mt = [], []
    for k in range(K):
        xb, yb = X[idx[k]], Y[idx[k]]
        nz = Noise(seed=(seed + W * (k + 1)) & 0xFFFFFFFFFFFFFFFF, sample0=sample0, window0=window0)
        if M == 1:
            r = e.elbo_step(xb[0], yb[0], st["loc"][0], st["scale"][0], mode=mode, guide=guide, particles=particles, noise=nz, **KW)
            r = {k2: (v.unsqueeze(0) if v is not None and k2 != "flat" else v) for k2, v in r.items()}
        else:
            r = e.elbo_step_ensemble(xb, yb, st["loc"], st["scale"], mode=mode, guide=guide, particles=particles, noise=nz, **KW)
        e.clipped_adam_vi(st["loc"], st["log_scale"], st["scale"], r["grad_mu"].contiguous(), r["grad_log_sigma"].contiguous(),
                          st["m_loc"], st["v_loc"], st["m_ls"], st["v_ls"], step0 + k + 1, **OPT)
        sc.append(r["scalars"].clone())
        mt.append(_logged(e, r["out"], yb, particles))
    return torch.stack(sc), torch.stack(mt)


def _ref_hnn(e, X, Y, idx, st, p, seed, step0):
    from bayesrul_b200 import Noise
    K, M, B = idx.shape
    sc, mt = [], []
    for k in range(K):
        xb, yb = X[idx[k]], Y[idx[k]]
        nz = Noise(seed=(seed + W * (k + 1)) & 0xFFFFFFFFFFFFFFFF)
        if M == 1:
            r = e.hnn_step(xb[0], yb[0], st["theta"][0], p, nz)
            r = dict(scalars=r["scalars"].unsqueeze(0), grad=r["grad"], out=r["out"].unsqueeze(0))
        else:
            r = e.hnn_step_ensemble(xb, yb, st["theta"], p, nz)
        e.clipped_adam(st["theta"], r["grad"], st["m"], st["v"], step0 + k + 1, **HOPT)
        sc.append(r["scalars"].clone())
        mt.append(_logged(e, r["out"].unsqueeze(1), yb, 1))
    return torch.stack(sc), torch.stack(mt)


NREF = 3  # runs of the reference loop


def _within(got, refs, what, state=False):
    """|got - refs[0]| <= 2 max_ij |refs[i] - refs[j]| + rtol |refs[0]|: per column of a [K,M,c] result in max norm with
    rtol 1e-5; a final parameter or optimizer moment (state=True) in L2 norm with rtol 1e-3"""
    if got.dim() == 3:
        for c in range(got.shape[-1]):
            _within(got[..., c], [r[..., c] for r in refs], f"{what}[{c}]")
        return
    assert torch.isfinite(got).all(), what
    size = (lambda t: t.double().norm().item()) if state else (lambda t: t.abs().max().item())
    err = size(got - refs[0])
    spread = max(size(a - b) for i, a in enumerate(refs) for b in refs[i + 1:])
    assert err <= 2 * spread + (1e-3 if state else 1e-5) * size(refs[0]), (what, err, spread)


def _elbo_call(e, X, Y, idx, st, cfg, seed, step0, **kw):
    mode, guide, particles = cfg
    return e.elbo_train_steps(X, Y, idx, st["loc"], st["log_scale"], st["scale"], (st["m_loc"], st["v_loc"], st["m_ls"], st["v_ls"]),
                              step0=step0, mode=mode, guide=guide, particles=particles, seed=seed, **OPT, **KW, **kw)


def _hnn_call(e, X, Y, idx, st, p, seed, step0):
    return e.hnn_train_steps(X, Y, idx, st["theta"], (st["m"], st["v"]), step0=step0, p_dropout=p, seed=seed, **HOPT)


ELBO_CASES = [  # net, back-end, (mode, guide, particles), M, B
    ("inception", "fused", ("lrt", "normal", 1), 1, 100),
    ("inception", "fused", ("lrt", "normal", 1), 5, 100),
    ("inception", "fused", ("ws", "radial", 1), 1, 100),
    ("inception", "fused", ("ws", "radial", 1), 5, 100),
    ("inception", "fused", ("flipout", "normal", 2), 1, 100),
    ("inception", "simt", ("lrt", "normal", 1), 1, 37),
    ("linear", "fused", ("lrt", "normal", 1), 2, 100),
    ("conv", "fused", ("ws", "normal", 1), 1, 100),
]


@pytest.mark.parametrize("net,backend,cfg,M,B", ELBO_CASES)
def test_elbo_train_steps_match_the_step_loop(net, backend, cfg, M, B):
    K, N = 7, 1500
    X, Y = _data(N, 1)
    idx = _idx(K, M, B, N, 2)
    st0 = _vi_state(net, M, 3)
    seed, step0 = 0x1234_5678_9ABC_DEF0 + 3 * M + B, 11
    refs = []
    for i in range(NREF):
        st = _clone(st0)
        refs.append((st,) + _ref_elbo(_eng(net, backend, f"ref{i}"), X, Y, idx, st, cfg, seed, step0))
    st = _clone(st0)
    got = _elbo_call(_eng(net, backend, "ksteps"), X, Y, idx, st, cfg, seed, step0)
    assert got["scalars"].shape == (K, M, 4) and got["metrics"].shape == (K, M, 5)
    _within(got["scalars"], [r[1] for r in refs], "scalars")
    _within(got["metrics"], [r[2] for r in refs], "metrics")
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)


@pytest.mark.parametrize("M,p", [(5, P_MCD), (1, 0.0)])
def test_hnn_train_steps_match_the_step_loop(M, p):
    K, N, B, net = 7, 1500, 100, "inception"
    X, Y = _data(N, 4)
    idx = _idx(K, M, B, N, 5)
    st0 = _hnn_state(net, M, 6)
    seed, step0 = 987654321 + M, 3
    refs = []
    for i in range(NREF):
        st = _clone(st0)
        refs.append((st,) + _ref_hnn(_eng(net, "fused", f"ref{i}"), X, Y, idx, st, p, seed, step0))
    st = _clone(st0)
    got = _hnn_call(_eng(net, "fused", "ksteps"), X, Y, idx, st, p, seed, step0)
    assert got["scalars"].shape == (K, M, 2) and got["metrics"].shape == (K, M, 5)
    _within(got["scalars"], [r[1] for r in refs], "scalars")
    _within(got["metrics"], [r[2] for r in refs], "metrics")
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)


def _launches(e, fn):
    torch.cuda.synchronize()
    n0 = e.lib.brl_launch_count()
    r = fn()
    torch.cuda.synchronize()
    return e.lib.brl_launch_count() - n0, r


def test_second_call_replays_with_new_indices_and_seed():
    """a second call with new X / idx tensors, a new seed and step0 continues the loop exactly, from the captured graph:
    both calls issue one setup launch plus the same launches per step"""
    net, cfg, M, B, K, N = "inception", ("lrt", "normal", 1), 5, 100, 7, 1500
    X, Y = _data(N, 7)
    idx1, idx2 = _idx(K, M, B, N, 8), _idx(K, M, B, N, 9)
    st0 = _vi_state(net, M, 10)
    refs = []
    for i in range(NREF):
        st = _clone(st0)
        a = _ref_elbo(_eng(net, "fused", f"ref{i}"), X, Y, idx1, st, cfg, 5, 0)
        b = _ref_elbo(_eng(net, "fused", f"ref{i}"), X, Y, idx2, st, cfg, 77, K)
        refs.append((st,) + a + b)
    e = _eng(net, "fused", "second_call")
    st = _clone(st0)
    n1, got1 = _launches(e, lambda: _elbo_call(e, X, Y, idx1, st, cfg, 5, 0))
    n2, got2 = _launches(e, lambda: _elbo_call(e, X.clone(), Y.clone(), idx2, st, cfg, 77, K))
    assert n1 == n2 and (n2 - 1) % K == 0, (n1, n2)
    n3, _ = _launches(e, lambda: _elbo_call(e, X, Y, idx2[:3], _clone(st), cfg, 1, 0))
    assert n2 - n3 == (K - 3) * (n3 - 1) // 3, (n2, n3)
    for i, (got, name) in enumerate(((got1, "call 1"), (got2, "call 2"))):
        _within(got["scalars"], [r[1 + 2 * i] for r in refs], name + " scalars")
        _within(got["metrics"], [r[2 + 2 * i] for r in refs], name + " metrics")
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)


@pytest.mark.parametrize("kind", ["elbo", "hnn"])
def test_graphs_off_gives_the_same_results(kind):
    net, M, B, K, N = "inception", 5, 100, 7, 1500
    X, Y = _data(N, 11)
    idx = _idx(K, M, B, N, 12)
    cfg = ("lrt", "normal", 1)
    st0 = _vi_state(net, M, 13) if kind == "elbo" else _hnn_state(net, M, 13)
    runs = []
    for tag, graphs in (("nograph", False), ("g1", True), ("g2", True), ("g3", True)):
        e = _eng(net, "fused", tag)
        e.set_step_graph(graphs)
        st = _clone(st0)
        r = _elbo_call(e, X, Y, idx, st, cfg, 21, 0) if kind == "elbo" else _hnn_call(e, X, Y, idx, st, P_MCD, 21, 0)
        e.set_step_graph(True)
        runs.append((st, r))
    (s0, r0), refs = runs[0], runs[1:]
    for k in ("scalars", "metrics"):
        _within(r0[k], [r[k] for _, r in refs], k)
    for k in s0:
        _within(s0[k], [s[k] for s, _ in refs], k, state=True)


def test_call_returns_before_the_gpu_is_done():
    """K = 500 steps at B = 256: the call enqueues them and returns; nothing in it waits for the stream"""
    net, M, B, K, N = "inception", 1, 256, 500, 20000
    X, Y = _data(N, 14)
    idx = torch.randperm(N, device=DEV)[: 256 * 78].view(78, 1, 256).repeat(7, 1, 1)[:K].contiguous()
    e = _eng(net, "fused", "busy")
    st = _vi_state(net, M, 15)
    torch.cuda.synchronize()
    r = _elbo_call(e, X, Y, idx, st, ("lrt", "normal", 1), 3, 0)
    busy = not torch.cuda.current_stream().query()
    torch.cuda.synchronize()
    assert busy
    assert torch.isfinite(r["scalars"]).all() and torch.isfinite(st["loc"]).all()


def test_bnn_fit_epoch_matches_training_step_loop():
    """compat: one epoch over a 1 037-window split with batch size 100 (ten full batches in one K-step call, the remainder of
    37 through training_step) against Lightning's loop of training_step over the same permutation"""
    from bayesrul_b200.compat import BNN, Inception, pyro_shim
    N, bs = 1037, 100
    X, Y = _data(N, 16)
    keys = ("mse/train", "elbo/train", "kl/train", "likelihood/train", "rmsce/train", "sharp/train")

    def model():
        torch.manual_seed(12345)
        net = Inception(30, 18)
        with torch.no_grad():
            net.last.bias.fill_(3.0)
        opt = pyro_shim.ClippedAdam({"lr": 0.000857, "betas": [0.95, 0.999], "clip_norm": 15})
        m = BNN(net, opt, pretrain_epochs=5, mc_samples_train=1, mc_samples_eval=8, dataset_size=238150, fit_context="lrt",
                prior_loc=0.0, prior_scale=0.138793, guide="normal", q_scale=1.351e-3, device=DEV)
        m.on_fit_start()
        return m

    def loop():
        m = model()
        perm = torch.randperm(N, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV)
        sums = dict.fromkeys(keys, 0.0)
        for i, a in enumerate(range(0, N, bs)):
            b = perm[a: a + bs]
            m.training_step((X[b], Y[b]), i)
            for k in keys:
                sums[k] += float(m.logged[k]) * b.numel()
        return m, {k: v / N for k, v in sums.items()}

    refs = [loop() for _ in range(NREF)]
    m = model()
    res = m.fit_epoch(X, Y, bs, generator=torch.Generator(device=DEV).manual_seed(5))
    assert res["scalars"].shape == (10, 1, 4) and res["metrics"].shape == (10, 1, 5)
    for k in keys:
        vals = [r[1][k] for r in refs]
        spread = max(vals) - min(vals)
        assert abs(m.logged[k] - vals[0]) <= 2 * spread + 1e-5 * abs(vals[0]), (k, m.logged[k], vals)
    for k in ("loc", "log_scale", "scale"):
        _within(getattr(m.bnn.net_guide, k), [getattr(r[0].bnn.net_guide, k) for r in refs], k, state=True)
    assert m.bnn._step == refs[0][0].bnn._step == 11
    for name in ("loc", "log_scale"):
        st = m.svi.optim.state[name]
        assert st["step"] == refs[0][0].svi.optim.state[name]["step"] == 11
        for k in ("m", "v"):
            _within(st[k], [r[0].svi.optim.state[name][k] for r in refs], f"{name}.{k}", state=True)


# brl_workspace_bytes(ctx, B, S, train, engine) of the Inception net at the parent commit: the new train codes leave 0-4 as they were
PARENT_WORKSPACE_BYTES = {
    "37,1,0,0": 2727680,
    "37,1,0,1": 1897216,
    "37,1,1,0": 36606464,
    "37,1,1,1": 35776000,
    "37,1,2,0": 3245056,
    "37,1,2,1": 2414592,
    "37,1,3,0": 35856128,
    "37,1,3,1": 35856128,
    "37,1,4,0": 35856128,
    "37,1,4,1": 35856128,
    "37,2,0,0": 5368576,
    "37,2,0,1": 3660032,
    "37,2,1,0": 75099392,
    "37,2,1,1": 73390848,
    "37,2,2,0": 6399744,
    "37,2,2,1": 4691200,
    "37,2,3,0": 49772800,
    "37,2,3,1": 49772800,
    "37,2,4,0": 59811584,
    "37,2,4,1": 59811584,
    "37,5,0,0": 13292032,
    "37,5,0,1": 8948736,
    "37,5,1,0": 83022848,
    "37,5,1,1": 78679552,
    "37,5,2,0": 15869440,
    "37,5,2,1": 11526144,
    "37,5,3,0": 88947200,
    "37,5,3,1": 88947200,
    "37,5,4,0": 114041088,
    "37,5,4,1": 114041088,
    "100,1,0,0": 6086912,
    "100,1,0,1": 2101504,
    "100,1,1,0": 62744320,
    "100,1,1,1": 58758912,
    "100,1,2,0": 7480320,
    "100,1,2,1": 3494912,
    "100,1,3,0": 61992448,
    "100,1,3,1": 61992448,
    "100,1,4,0": 61992448,
    "100,1,4,1": 61992448,
    "100,2,0,0": 11950336,
    "100,2,0,1": 3864832,
    "100,2,1,0": 130596096,
    "100,2,1,1": 122510592,
    "100,2,2,0": 14734848,
    "100,2,2,1": 6649344,
    "100,2,3,0": 87605760,
    "100,2,3,1": 87605760,
    "100,2,4,0": 99437056,
    "100,2,4,1": 99437056,
    "100,5,0,0": 29541888,
    "100,5,0,1": 9155072,
    "100,5,1,0": 148187648,
    "100,5,1,1": 127800832,
    "100,5,2,0": 36498688,
    "100,5,2,1": 16111872,
    "100,5,3,0": 161314560,
    "100,5,3,1": 161314560,
    "100,5,4,0": 190885888,
    "100,5,4,1": 190885888,
    "256,1,0,0": 14405120,
    "256,1,0,1": 3200768,
    "256,1,1,0": 131943936,
    "256,1,1,1": 120739584,
    "256,1,2,0": 17966592,
    "256,1,2,1": 6762240,
    "256,1,3,0": 131188736,
    "256,1,3,1": 131188736,
    "256,1,4,0": 131188736,
    "256,1,4,1": 131188736,
    "256,2,0,0": 28248576,
    "256,2,0,1": 5579776,
    "256,2,1,0": 276972032,
    "256,2,1,1": 254303232,
    "256,2,2,0": 35371520,
    "256,2,2,1": 12702720,
    "256,2,3,0": 190238464,
    "256,2,3,1": 190238464,
    "256,2,4,0": 206505728,
    "256,2,4,1": 206505728,
    "256,5,0,0": 69779200,
    "256,5,0,1": 12717056,
    "256,5,1,0": 318502656,
    "256,5,1,1": 261440512,
    "256,5,2,0": 87586560,
    "256,5,2,1": 30524416,
    "256,5,3,0": 362882560,
    "256,5,3,1": 362882560,
    "256,5,4,0": 403547904,
    "256,5,4,1": 403547904,
}


def test_errors_and_workspace_codes():
    e = _eng("inception", "fused", "errors")
    X, Y = _data(300, 17)
    st = _vi_state("inception", 1, 18)
    cfg = ("lrt", "normal", 1)
    good = _idx(3, 1, 50, 300, 19)
    with pytest.raises(RuntimeError, match="outside"):
        _elbo_call(e, X, Y, torch.where(good == good[1, 0, 7], 300, good), st, cfg, 1, 0)
    with pytest.raises(RuntimeError, match="outside"):
        _elbo_call(e, X, Y, good - good.max(), st, cfg, 1, 0)
    with pytest.raises(RuntimeError, match="idx"):
        _elbo_call(e, X, Y, good.view(3, 50, 1), st, cfg, 1, 0)
    with pytest.raises(RuntimeError, match="idx"):
        _elbo_call(e, X, Y, good.view(-1), st, cfg, 1, 0)
    with pytest.raises(RuntimeError, match="int64"):
        _elbo_call(e, X, Y, good.int(), st, cfg, 1, 0)
    with pytest.raises(RuntimeError, match="idx"):
        _elbo_call(e, X, Y, good[:0], st, cfg, 1, 0)
    hs = _hnn_state("inception", 1, 18)
    with pytest.raises(RuntimeError, match="idx"):
        _hnn_call(e, X, Y, good.view(3, 50, 1), hs, 0.0, 1, 0)
    # the library's own checks: K = 0 and a workspace below brl_workspace_bytes(B, M, 5 / 6)
    lib = e.lib
    sc = torch.empty(3, 1, 5, dtype=torch.float64, device=DEV)
    for code, fn, params, opt in ((5, lib.brl_elbo_train_steps, [st[k] for k in ("loc", "log_scale", "scale", "m_loc", "v_loc", "m_ls", "v_ls")],
                                   [2, 0, 1, 0.0, 1.0, 238150, 1, 0, 0]),
                                  (6, lib.brl_hnn_train_steps, [hs["theta"], hs["m"], hs["v"]], [0.0, 1, 0, 0])):
        need = lib.brl_workspace_bytes(e.ctx, 50, 1, code, 0)
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        for K, nbytes in ((0, need), (3, need - 256)):
            rc = fn(e.ctx, X.data_ptr(), Y.data_ptr(), 300, good.data_ptr(), K, 1, 50, *[t.data_ptr() for t in params], 0, 1e-3,
                    0.9, 0.999, 1e-8, 15.0, 1.0, 0.0, *opt, sc.data_ptr(), sc.data_ptr(), ws.data_ptr(), nbytes,
                    torch.cuda.current_stream().cuda_stream)
            assert rc != 0, (code, K, nbytes)
            with pytest.raises(RuntimeError):
                from bayesrul_b200 import _lib
                _lib.check(rc)
    got = {f"{B},{S},{t},{en}": lib.brl_workspace_bytes(e.ctx, B, S, t, en)
           for B in (37, 100, 256) for S in (1, 2, 5) for t in range(5) for en in (0, 1)}
    assert got == PARENT_WORKSPACE_BYTES
