"""Member-batched predictive moments and step metrics (brl_predict_moments_ensemble / Engine.predict_moments_ensemble,
brl_step_metrics_ensemble / Engine.step_metrics_ensemble).

Member m of an M-member call is predict_moments(x, mu[m], sigma[m], S, noise with sample0 + m S): every weight draw and
dropout mask is keyed by its MC-sample index, every tile row of the engines is computed on its own and the Welford update
is sequential per window, so a member's moments are BIT-identical to its single call on the same engine, whichever chunk
of the flattened M S sample axis its samples fall in.  Step metrics: the coverage histogram is exact (rmsce, mace equal);
nll, mse and sharpness are sums of fp64 atomics (1e-12 relative)."""
import ctypes as C

import pytest
import torch

from tests.helpers import synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
P_DROP = 0.241437
BRL_ERR_WORKSPACE = -3


def _eq(a, b, what):
    torch.testing.assert_close(a, b, rtol=0, atol=0, equal_nan=True, msg=lambda m: f"{what}: {m}")


@pytest.fixture(scope="module")
def engines():
    from bayesrul_b200 import Engine
    return {}, Engine


def _eng(engines, net):
    cache, Engine = engines
    if net not in cache:
        cache[net] = Engine(net, DEV)
    return cache[net]


def _stack(net, M, B, seed):
    """one batch of windows, M distinct parameter vectors (and scales)"""
    x = synth(net, B, seed=seed)[0].to(DEV)
    mus, sgs = zip(*[synth(net, 1, seed=seed + 11 * (m + 1), sigma=0.02 + 0.01 * m)[2:] for m in range(M)])
    return x, torch.stack(mus).to(DEV), torch.stack(sgs).to(DEV)


# (guide, p_dropout): weight sampling of M posteriors, MC-dropout and deterministic members (guide None)
CASES = {"normal": ("normal", 0.0), "radial": ("radial", 0.0), "mcd": (None, P_DROP), "det": (None, 0.0)}


def _run(e, case, x, mu, sg, S, noise_kw, engine, chunk=None):
    from bayesrul_b200 import Noise
    guide, p = CASES[case]
    return e.predict_moments_ensemble(x, mu, sg if guide else None, S=S, guide=guide, p_dropout=p, noise=Noise(**noise_kw),
                                      engine=engine, chunk=chunk)


def _singles(e, case, x, mu, sg, S, noise_kw, engine):
    from bayesrul_b200 import Noise
    guide, p = CASES[case]
    refs = []
    for m in range(mu.shape[0]):
        kw = dict(noise_kw, sample0=noise_kw.get("sample0", 0) + m * S)
        refs.append(e.predict_moments(x, mu[m], sg[m] if guide else None, S=S, guide=guide, p_dropout=p, noise=Noise(**kw),
                                      engine=engine))
    return refs


def _assert_members(got, refs, what):
    M = len(refs)
    for k, name in enumerate(("pred", "std", "ep_var", "al_var")):
        assert got[k].shape == (M, refs[0][k].shape[0]), (what, name, got[k].shape)
        for m in range(M):
            _eq(got[k][m], refs[m][k], f"{what} member {m} {name}")


@pytest.mark.parametrize("case", ["normal", "radial", "mcd"])
@pytest.mark.parametrize("S", [7, 20])
@pytest.mark.parametrize("B", [1, 37, 300, 1000])
@pytest.mark.parametrize("M", [1, 3, 5])
def test_inception_tc_members_equal_singles(engines, M, B, S, case):
    e = _eng(engines, "inception")
    x, mu, sg = _stack("inception", M, B, seed=10 * M + B + S)
    nkw = dict(seed=7, sample0=3, window0=1234)
    got = _run(e, case, x, mu, sg, S, nkw, "tc")
    refs = _singles(e, case, x, mu, sg, S, nkw, "tc")
    assert e.tc_status() == 0
    _assert_members(got, refs, f"inception tc {case} M={M} B={B} S={S}")


@pytest.mark.parametrize("B", [1, 37, 300, 1000])
@pytest.mark.parametrize("M", [1, 3, 5])
def test_inception_tc_deterministic_members(engines, M, B):
    e = _eng(engines, "inception")
    x, mu, sg = _stack("inception", M, B, seed=500 + M + B)
    nkw = dict(seed=1, window0=77)
    got = _run(e, "det", x, mu, sg, 1, nkw, "tc")
    refs = _singles(e, "det", x, mu, sg, 1, nkw, "tc")
    assert e.tc_status() == 0
    _assert_members(got, refs, f"inception tc det M={M} B={B}")
    assert torch.isnan(got[2]).all()  # one sample: the unbiased epistemic variance is 0 / 0, as in the single call


@pytest.mark.parametrize("case", ["normal", "det"])
@pytest.mark.parametrize("net", ["linear", "conv"])
def test_linear_convd3_tc_members_equal_singles(engines, net, case):
    e = _eng(engines, net)
    M, B, S = 3, 300, 1 if case == "det" else 20
    x, mu, sg = _stack(net, M, B, seed=600)
    nkw = dict(seed=4, sample0=2, window0=9)
    got = _run(e, case, x, mu, sg, S, nkw, "tc")
    refs = _singles(e, case, x, mu, sg, S, nkw, "tc")
    assert e.tc_status() == 0
    _assert_members(got, refs, f"{net} tc {case}")


@pytest.mark.parametrize("net", ["linear", "conv"])
def test_linear_convd3_tc_mc_dropout_raises(engines, net):
    e = _eng(engines, net)
    x, mu, sg = _stack(net, 3, 64, seed=700)
    with pytest.raises(RuntimeError, match="dropout"):
        e.predict_moments(x, mu[0], None, S=5, guide=None, p_dropout=P_DROP, engine="tc")
    with pytest.raises(RuntimeError, match="dropout"):
        _run(e, "mcd", x, mu, sg, 5, dict(seed=1), "tc")


def _launches(e, fn):
    torch.cuda.synchronize()
    n0 = e.lib.brl_launch_count()
    fn()
    torch.cuda.synchronize()
    return e.lib.brl_launch_count() - n0


@pytest.mark.parametrize("case", ["normal", "mcd"])
def test_simt_loop_equals_singles(engines, case):
    e = _eng(engines, "inception")
    M, B, S = 3, 37, 5
    x, mu, sg = _stack("inception", M, B, seed=800)
    nkw = dict(seed=5, sample0=1, window0=3)
    got = _run(e, case, x, mu, sg, S, nkw, "simt")
    refs = _singles(e, case, x, mu, sg, S, nkw, "simt")
    _assert_members(got, refs, f"simt {case}")
    loop = _launches(e, lambda: _run(e, case, x, mu, sg, S, nkw, "simt"))
    single = _launches(e, lambda: _singles(e, case, x, mu[:1], sg[:1], S, nkw, "simt"))
    assert loop == M * single > 0, (loop, single)


@pytest.mark.parametrize("case", ["normal", "radial", "mcd"])
def test_members_share_launches(engines, case):
    """M S <= one chunk: the M = 5 call issues as many launches as the M = 1 call and as one predict_moments call"""
    e = _eng(engines, "inception")
    B, S = 256, 20
    x, mu, sg = _stack("inception", 5, B, seed=900)
    nkw = dict(seed=8)
    _run(e, case, x, mu, sg, S, nkw, "tc")  # warm-up: workspace growth
    counts = {M: _launches(e, lambda: _run(e, case, x, mu[:M], sg[:M], S, nkw, "tc")) for M in (1, 5)}
    single = _launches(e, lambda: _singles(e, case, x, mu[:1], sg[:1], S, nkw, "tc"))
    assert e.tc_status() == 0
    print(f"\n[predict ensemble launches, {case}] M=1: {counts[1]}, M=5: {counts[5]}, predict_moments: {single}")
    assert counts[1] == counts[5] == single > 0


@pytest.mark.parametrize("case", ["normal", "radial", "mcd"])
def test_injected_noise_rows(engines, case):
    """injected noise [M S, ...]: member m equals its single call given rows [m S, (m + 1) S)"""
    from bayesrul_b200 import Noise
    e = _eng(engines, "inception")
    M, B, S = 3, 37, 7
    x, mu, sg = _stack("inception", M, B, seed=1000)
    guide, p = CASES[case]
    g = torch.Generator().manual_seed(3)
    layers = e.info["layers"]
    full = {}
    if guide:
        full["weight_eps"] = torch.randn(M * S, e.P, generator=g)
    if guide == "radial":
        full["radial_r"] = torch.randn(M * S, 2 * len(layers), generator=g)
    masks = {}
    if p > 0:
        masks = {l: (torch.rand(M * S, B, oe, generator=g) > p * df).float() for l, (_, _, oe, df) in enumerate(layers) if df > 0}
    dev = lambda t: t.to(DEV).contiguous()
    nz = Noise(seed=2, window0=5, drop_mask={l: dev(t) for l, t in masks.items()}, **{k: dev(t) for k, t in full.items()})
    got = e.predict_moments_ensemble(x, mu, sg if guide else None, S=S, guide=guide, p_dropout=p, noise=nz, engine="tc")
    refs = []
    for m in range(M):
        rows = slice(m * S, (m + 1) * S)
        nm = Noise(seed=2, window0=5, drop_mask={l: dev(t[rows]) for l, t in masks.items()},
                   **{k: dev(t[rows]) for k, t in full.items()})
        refs.append(e.predict_moments(x, mu[m], sg[m] if guide else None, S=S, guide=guide, p_dropout=p, noise=nm, engine="tc"))
    assert e.tc_status() == 0
    _assert_members(got, refs, f"injected {case}")


def test_chunking_and_workspace(engines):
    """the minimum workspace (one draw per chunk) and chunks that straddle members give the same bits; one byte less is refused"""
    from bayesrul_b200 import Noise
    e = _eng(engines, "inception")
    M, B, S = 3, 300, 7
    x, mu, sg = _stack("inception", M, B, seed=1100)
    nkw = dict(seed=6, sample0=4)
    refs = _singles(e, "normal", x, mu, sg, S, nkw, "tc")
    _assert_members(_run(e, "normal", x, mu, sg, S, nkw, "tc", chunk=5), refs, "chunk 5")
    eid = 1
    need = e.lib.brl_workspace_bytes(e.ctx, B, 1, 0, eid) + (M * 4 * B * 4 + 255) // 256 * 256
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    out = torch.empty(4, M, B, device=DEV)
    nz = Noise(**nkw).to_struct(torch.device(DEV))[0]

    def call(nbytes):
        return e.lib.brl_predict_moments_ensemble(e.ctx, x.data_ptr(), M, B, S, 0, mu.data_ptr(), sg.data_ptr(), 0.0, C.byref(nz),
                                                  out.data_ptr(), eid, ws.data_ptr(), nbytes,
                                                  torch.cuda.current_stream().cuda_stream)

    launches = _launches(e, lambda: call(need))
    assert e.tc_status() == 0
    _assert_members(tuple(out), refs, "minimum workspace")
    assert launches >= M * S  # one draw per chunk
    assert call(need - 1) == BRL_ERR_WORKSPACE
    assert "workspace too small" in e.lib.brl_last_error().decode()


def test_bad_arguments(engines):
    e = _eng(engines, "inception")
    x, mu, sg = _stack("inception", 2, 16, seed=1200)
    with pytest.raises(RuntimeError):
        e.predict_moments_ensemble(x, mu[0], sg[0], S=3, engine="tc")  # mu not [M,P]
    with pytest.raises(RuntimeError):
        e.predict_moments_ensemble(x, torch.cat([mu, mu[:, :1]], 1), sg, S=3, engine="tc")
    with pytest.raises(RuntimeError):
        e.predict_moments_ensemble(x, mu, None, S=3, guide="normal", engine="tc")  # sigma missing with a guide
    with pytest.raises(RuntimeError):
        e.predict_moments_ensemble(x, mu, sg[:1], S=3, guide="normal", engine="tc")
    with pytest.raises(RuntimeError):
        e.predict_moments_ensemble(x, mu[:0], sg[:0], S=3, engine="tc")  # M = 0
    with pytest.raises(RuntimeError):
        e.predict_moments_ensemble(x, mu, None, S=3, guide=None, p_dropout=1.0, engine="tc")
    with pytest.raises(RuntimeError, match="Guide unknown"):
        e.predict_moments_ensemble(x, mu, sg, S=3, guide="laplace", engine="tc")


@pytest.mark.parametrize("n", [1, 97, 10000])
@pytest.mark.parametrize("M", [1, 5])
def test_step_metrics_rows(engines, M, n):
    e = _eng(engines, "inception")
    g = torch.Generator().manual_seed(M * n)
    y = (torch.rand(M, n, generator=g) * 100).to(DEV)
    pred = (y.cpu() + torch.randn(M, n, generator=g) * 12).to(DEV)
    std = (torch.rand(M, n, generator=g) * 20 + 0.5).to(DEV)
    got = e.step_metrics_ensemble(pred, std, y)
    assert got.shape == (M, 5) and got.dtype == torch.float64
    for m in range(M):
        ref = e.step_metrics(pred[m], std[m], y[m])
        _eq(got[m, 3:], ref[3:], f"M={M} n={n} member {m} rmsce / mace")
        torch.testing.assert_close(got[m, :3], ref[:3], rtol=1e-12, atol=0)
    rc = e.lib.brl_step_metrics_ensemble(pred.data_ptr(), std.data_ptr(), y.data_ptr(), M, n, got.data_ptr(),
                                         e._metrics_ws.data_ptr(), M * 1024 - 1, torch.cuda.current_stream().cuda_stream)
    assert rc == BRL_ERR_WORKSPACE
    with pytest.raises(RuntimeError):
        e.step_metrics_ensemble(pred.reshape(-1), std.reshape(-1), y.reshape(-1))


def test_full_size(engines):
    e = _eng(engines, "inception")
    M, B, S = 5, 10000, 100
    x, mu, sg = _stack("inception", M, B, seed=1300)
    nkw = dict(seed=12)
    got = _run(e, "normal", x, mu, sg, S, nkw, "tc")
    refs = _singles(e, "normal", x, mu, sg, S, nkw, "tc")
    assert e.tc_status() == 0
    for t in got:
        assert torch.isfinite(t).all()
    assert (got[1] > 0).all() and (got[2] >= 0).all()
    _assert_members(got, refs, "full size")


def test_end_to_end_deep_ensemble(engines):
    """five members trained with hnn_step_ensemble + Adam, then predict_moments_ensemble (MC-dropout) -> step_metrics_ensemble ->
    mixture_moments equals the per-member singles followed by the same mixture"""
    from bayesrul_b200 import Noise
    e = _eng(engines, "inception")
    M, B, S = 5, 256, 20
    xs, ys, ths = zip(*[synth("inception", B, seed=1400 + 7 * m)[:3] for m in range(M)])
    x, y, th = torch.stack(xs).to(DEV), torch.stack(ys).to(DEV), torch.stack(ths).to(DEV)
    ens = torch.nn.Parameter(th.clone())
    opt = torch.optim.Adam([ens], lr=1e-3)
    e.set_gemm_backend("fused")
    try:
        for k in range(3):
            ens.grad = e.hnn_step_ensemble(x, y, ens.data, P_DROP, Noise(seed=50 + k))["grad"]
            opt.step()
    finally:
        e.set_gemm_backend("simt")
    xt, yt = synth("inception", 300, seed=1500)[:2]
    xt, yt = xt.to(DEV), yt.to(DEV)
    theta = ens.data.contiguous()
    pred, std, ep, al = e.predict_moments_ensemble(xt, theta, S=S, guide=None, p_dropout=P_DROP, noise=Noise(seed=60), engine="tc")
    scal = e.step_metrics_ensemble(pred, std, yt.expand(M, -1).contiguous())
    mix = e.mixture_moments(pred, std)
    refs = [e.predict_moments(xt, theta[m], S=S, guide=None, p_dropout=P_DROP, noise=Noise(seed=60, sample0=m * S), engine="tc")
            for m in range(M)]
    assert e.tc_status() == 0
    _assert_members((pred, std, ep, al), refs, "end to end")
    for m in range(M):
        ref = e.step_metrics(refs[m][0], refs[m][1], yt)
        _eq(scal[m, 3:], ref[3:], f"metrics member {m}")
        torch.testing.assert_close(scal[m, :3], ref[:3], rtol=1e-12, atol=0)
    ref_mix = e.mixture_moments(torch.stack([r[0] for r in refs]), torch.stack([r[1] for r in refs]))
    _eq(mix[0], ref_mix[0], "mixture mean")
    _eq(mix[1], ref_mix[1], "mixture std")
