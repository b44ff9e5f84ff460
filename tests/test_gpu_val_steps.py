"""K validation batches of one variational BNN per call over a device-resident split (brl_elbo_val_steps, Engine.elbo_val_steps,
compat BNN.validate_epoch).

Batch k of a call is, by contract, the sequence of Engine calls that validation_step issues: elbo_step(mode="ws",
compute_grads=False) with the Philox seed seed + 0x9E3779B97F4A7C15 (2k + 1), then sample_weights(S), forward("ws", engine) and
(S > 1) aggregate_predictions with seed + 0x9E3779B97F4A7C15 (2k + 2), then step_metrics.  Each comparison runs that loop three
times (the scheme of tests/test_gpu_train_steps.py): fp64 / fp32 atomics in the ELBO's reductions make repeated runs differ in the
last bits, and the call must lie within twice the largest distance between the loop's runs plus 1e-6 of the quantity's largest
magnitude, per column of scalars and metrics.  A wrong key moves the ELBO or the predictive by a weight draw, far outside that
bound; the negative controls below check that the bound sees it."""
import pytest
import torch

from tests.test_gpu_hnn_fit_epoch import PARENT_TRAIN_STEPS_BYTES
from tests.test_gpu_train_steps import (KW, NREF, PARENT_WORKSPACE_BYTES, W, _ENGINES, _clone, _data, _elbo_call, _eng, _idx,
                                        _launches, _vi_state, _within)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MASK = 0xFFFFFFFFFFFFFFFF


@pytest.fixture(scope="module", autouse=True)
def _cleanup():
    yield
    _ENGINES.clear()


def _params(net, seed):
    st = _vi_state(net, 1, seed)
    return st["loc"][0].contiguous(), st["log_scale"][0].contiguous(), st["scale"][0].contiguous()


def _ref_val(e, X, Y, idx, loc, scale, cfg, seed, swap=False):
    """the loop of the contract; swap=True draws the ELBO with the predictive's key and the other way round"""
    from bayesrul_b200 import Noise
    guide, particles, S, engine = cfg
    sc, mt = [], []
    for k in range(idx.shape[0]):
        xb, yb = X[idx[k]], Y[idx[k]]
        k1, k2 = (seed + W * (2 * k + 1)) & MASK, (seed + W * (2 * k + 2)) & MASK
        if swap:
            k1, k2 = k2, k1
        r = e.elbo_step(xb, yb, loc, scale, mode="ws", guide=guide, particles=particles, noise=Noise(seed=k1), compute_grads=False, **KW)
        sc.append(r["scalars"].clone())
        w = e.sample_weights(loc, scale, guide, S, Noise(seed=k2))
        out = e.forward(xb, "ws", wsamp=w, S=S, noise=Noise(seed=k2), engine=engine)
        o = e.aggregate_predictions(out) if S > 1 else out[0]
        mt.append(e.step_metrics(o[:, 0], o[:, 1], yb))
    return torch.stack(sc), torch.stack(mt)


def _call(e, X, Y, idx, loc, scale, cfg, seed):
    guide, particles, S, engine = cfg
    return e.elbo_val_steps(X, Y, idx, loc, scale, guide=guide, particles=particles, S=S, seed=seed, engine=engine, **KW)


def _excess(got, refs):
    """largest ratio, over the columns, of the distance to refs[0] to the bound that _within allows (> 1: outside it)"""
    worst = 0.0
    for c in range(got.shape[-1]):
        g, rs = got[..., c], [r[..., c] for r in refs]
        err = (g - rs[0]).abs().max().item()
        spread = max((a - b).abs().max().item() for i, a in enumerate(rs) for b in rs[i + 1:])
        worst = max(worst, err / (2 * spread + 1e-6 * rs[0].abs().max().item() + 1e-300))
    return worst


def _close(got, refs, what, rtol=1e-6):
    """|got - refs[0]| <= 2 max_ij |refs[i] - refs[j]| + rtol |refs[0]| per column of a [K,c] (or [K,1,c]) result, in max norm"""
    got, refs = got.reshape(got.shape[0], -1), [r.reshape(r.shape[0], -1) for r in refs]
    assert torch.isfinite(got).all(), what
    for c in range(got.shape[1]):
        g, rs = got[:, c], [r[:, c] for r in refs]
        err = (g - rs[0]).abs().max().item()
        spread = max((a - b).abs().max().item() for i, a in enumerate(rs) for b in rs[i + 1:])
        assert err <= 2 * spread + rtol * rs[0].abs().max().item(), (f"{what}[{c}]", err, spread)


def _check(got, refs, what):
    for key, i in (("scalars", 0), ("metrics", 1)):
        _close(got[key], [r[i] for r in refs], f"{what} {key}")


CASES = [  # net, back-end, (guide, particles, S, engine), B
    ("inception", "fused", ("normal", 1, 8, "tc"), 100),
    ("inception", "fused", ("normal", 1, 1, "tc"), 100),
    ("inception", "fused", ("radial", 1, 8, "tc"), 100),
    ("inception", "fused", ("normal", 2, 8, "tc"), 100),
    ("inception", "simt", ("normal", 1, 8, "simt"), 37),
    ("linear", "fused", ("normal", 1, 8, "tc"), 100),
    ("conv", "fused", ("normal", 1, 8, "simt"), 100),
]


@pytest.mark.parametrize("net,backend,cfg,B", CASES)
def test_val_steps_match_the_loop(net, backend, cfg, B):
    K, N = 7, 1500
    X, Y = _data(N, 101)
    idx = _idx(K, 1, B, N, 102)[:, 0]
    loc, log_scale, scale = _params(net, 103)
    before = [t.clone() for t in (loc, log_scale, scale)]
    seed = 0x0123_4567_89AB_CDEF + B
    refs = [_ref_val(_eng(net, backend, f"vref{i}"), X, Y, idx, loc, scale, cfg, seed) for i in range(NREF)]
    e = _eng(net, backend, "val")
    got = _call(e, X, Y, idx, loc, scale, cfg, seed)
    assert got["scalars"].shape == (K, 4) and got["metrics"].shape == (K, 5)
    _check(got, refs, "call")
    for a, b in zip((loc, log_scale, scale), before):
        assert torch.equal(a, b)
    if net == "inception" and cfg == ("normal", 1, 8, "tc"):
        # negative controls: a call one key further along the sequence, and the loop with the two keys of each batch swapped
        bad = _call(e, X, Y, idx, loc, scale, cfg, (seed + W) & MASK)
        assert _excess(bad["scalars"], [r[0] for r in refs]) > 1 and _excess(bad["metrics"], [r[1] for r in refs]) > 1
        sw = _ref_val(_eng(net, backend, "vref0"), X, Y, idx, loc, scale, cfg, seed, swap=True)
        assert _excess(sw[0], [r[0] for r in refs]) > 1 and _excess(sw[1], [r[1] for r in refs]) > 1


def test_second_call_replays_with_new_indices_and_seed():
    """a second call with new X / idx tensors and a new seed comes from the first call's graph: both calls issue one setup launch
    plus the same launches per batch"""
    net, cfg, B, K, N = "inception", ("normal", 1, 8, "tc"), 100, 7, 1500
    X, Y = _data(N, 104)
    idx1, idx2 = _idx(K, 1, B, N, 105)[:, 0], _idx(K, 1, B, N, 106)[:, 0]
    loc, _, scale = _params(net, 107)
    refs1 = [_ref_val(_eng(net, "fused", f"vref{i}"), X, Y, idx1, loc, scale, cfg, 5) for i in range(NREF)]
    refs2 = [_ref_val(_eng(net, "fused", f"vref{i}"), X, Y, idx2, loc, scale, cfg, 77) for i in range(NREF)]
    e = _eng(net, "fused", "val_second")
    n1, got1 = _launches(e, lambda: _call(e, X, Y, idx1, loc, scale, cfg, 5))
    n2, got2 = _launches(e, lambda: _call(e, X.clone(), Y.clone(), idx2, loc, scale, cfg, 77))
    assert n1 == n2 and (n2 - 1) % K == 0, (n1, n2)
    n3, _ = _launches(e, lambda: _call(e, X, Y, idx2[:3], loc, scale, cfg, 1))
    assert n2 - n3 == (K - 3) * (n3 - 1) // 3, (n2, n3)
    _check(got1, refs1, "call 1")
    _check(got2, refs2, "call 2")


@pytest.mark.parametrize("cfg", [("normal", 1, 8, "tc"), ("radial", 2, 4, "simt")])
def test_graphs_off_gives_the_same_results(cfg):
    net, B, K, N = "inception", 100, 7, 1500
    X, Y = _data(N, 108)
    idx = _idx(K, 1, B, N, 109)[:, 0]
    loc, _, scale = _params(net, 110)
    runs = []
    for tag, graphs in (("vnograph", False), ("vg1", True), ("vg2", True), ("vg3", True)):
        e = _eng(net, "fused", tag)
        e.set_step_graph(graphs)
        runs.append(_call(e, X, Y, idx, loc, scale, cfg, 21))
        e.set_step_graph(True)
    _check(runs[0], [(r["scalars"], r["metrics"]) for r in runs[1:]], "graphs off")


def test_tc_timing_runs_eagerly_with_the_same_results():
    """with the tensor-core engine's timing hooks on, every batch runs eagerly (the hooks record events at enqueue time) and
    gives the loop's results; the hooks see every batch's tc_conv_kernel"""
    net, cfg, B, K, N = "inception", ("normal", 1, 8, "tc"), 100, 7, 1500
    X, Y = _data(N, 111)
    idx = _idx(K, 1, B, N, 112)[:, 0]
    loc, _, scale = _params(net, 113)
    refs = [_ref_val(_eng(net, "fused", f"vref{i}"), X, Y, idx, loc, scale, cfg, 9) for i in range(NREF)]
    e = _eng(net, "fused", "val_timing")
    _call(e, X, Y, idx, loc, scale, cfg, 9)  # a graph of this configuration exists ...
    e.tc_timing(True)
    try:
        got = _call(e, X, Y, idx, loc, scale, cfg, 9)  # ... and is not replayed while the hooks are on
        timed = e.tc_timing_read()
    finally:
        e.tc_timing(False)
    assert timed["tc_conv_kernel"][1] == K and timed["tc_fc_kernel"][1] == K, timed
    _check(got, refs, "timed call")


def test_train_val_train_on_the_same_pointers():
    """elbo_train_steps, elbo_val_steps, elbo_train_steps on one engine (one workspace, graphs on) against the same sequence with
    graphs off"""
    net, cfg, B, K, N = "inception", ("normal", 1, 8, "tc"), 100, 7, 1500
    X, Y = _data(N, 114)
    idx1, idx2, idx3 = (_idx(K, 1, B, N, s) for s in (115, 116, 117))
    st0 = _vi_state(net, 1, 118)

    def seq(e):
        st = _clone(st0)
        a = _elbo_call(e, X, Y, idx1, st, ("lrt", "normal", 1), 31, 0)
        b = _call(e, X, Y, idx2[:, 0], st["loc"][0], st["scale"][0], cfg, 32)
        c = _elbo_call(e, X, Y, idx3, st, ("lrt", "normal", 1), 33, K)
        return st, a, b, c

    refs = []
    for i in range(NREF):
        e = _eng(net, "fused", f"vseq_eager{i}")
        e.set_step_graph(False)
        refs.append(seq(e))
    e = _eng(net, "fused", "vseq_graph")
    seq(e)  # first sight of each configuration: eager, then captured
    st, a, b, c = seq(e)  # every step / batch after the first of each call replays
    for i, (got, name) in enumerate(((a, "train 1"), (b, "val"), (c, "train 2"))):
        for key in ("scalars", "metrics"):
            _close(got[key], [r[1 + i][key] for r in refs], f"{name} {key}", rtol=1e-6 if name == "val" else 1e-5)
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)


def test_out_of_range_index_gives_a_nan_row():
    e = _eng("inception", "fused", "vnan")
    X, Y = _data(300, 119)
    loc, _, scale = _params("inception", 120)
    idx = _idx(3, 1, 50, 300, 121)[:, 0].contiguous()
    idx[1, 7] = 300
    lib = e.lib
    need = lib.brl_workspace_bytes(e.ctx, 50, 4, 7, 1)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    sc = torch.empty(3, 4, dtype=torch.float64, device=DEV)
    mt = torch.empty(3, 5, dtype=torch.float64, device=DEV)
    rc = lib.brl_elbo_val_steps(e.ctx, X.data_ptr(), Y.data_ptr(), 300, idx.data_ptr(), 3, 50, loc.data_ptr(), scale.data_ptr(), 0, 1,
                                4, 1, 0.0, 0.138793, 238150, 5, 0, 0, sc.data_ptr(), mt.data_ptr(), ws.data_ptr(), need,
                                torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.isnan(sc[1]).all() and torch.isnan(mt[1]).all()
    assert torch.isfinite(sc[0]).all() and torch.isfinite(sc[2]).all() and torch.isfinite(mt[0]).all() and torch.isfinite(mt[2]).all()


def test_errors_and_workspace_codes():
    from bayesrul_b200 import _lib
    e = _eng("inception", "fused", "verrors")
    X, Y = _data(300, 122)
    loc, _, scale = _params("inception", 123)
    good = _idx(3, 1, 50, 300, 124)[:, 0].contiguous()
    cfg = ("normal", 1, 4, "tc")
    with pytest.raises(RuntimeError, match="outside"):
        _call(e, X, Y, torch.where(good == good[1, 7], 300, good), loc, scale, cfg, 1)
    with pytest.raises(RuntimeError, match="idx"):
        _call(e, X, Y, good.view(-1), loc, scale, cfg, 1)
    with pytest.raises(RuntimeError, match="int64"):
        _call(e, X, Y, good.int(), loc, scale, cfg, 1)
    with pytest.raises(RuntimeError, match="loc"):
        _call(e, X, Y, good, loc[:-1], scale, cfg, 1)
    with pytest.raises(RuntimeError, match="Guide unknown"):
        _call(e, X, Y, good, loc, scale, ("laplace", 1, 4, "tc"), 1)
    with pytest.raises(RuntimeError, match="engine"):
        _call(e, X, Y, good, loc, scale, ("normal", 1, 4, "fp8"), 1)
    with pytest.raises(RuntimeError, match="particles"):
        _call(e, X, Y, good, loc, scale, ("normal", 9, 4, "tc"), 1)
    with pytest.raises(RuntimeError, match="S"):
        _call(e, X, Y, good, loc, scale, ("normal", 1, 0, "tc"), 1)
    # the library's own checks: K = 0, S = 0, and a workspace one byte below brl_workspace_bytes(B, S, 7, engine)
    lib = e.lib
    sc = torch.empty(3, 5, dtype=torch.float64, device=DEV)
    for eng_id in (0, 1):
        need = lib.brl_workspace_bytes(e.ctx, 50, 4, 7, eng_id)
        assert need > 0
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        for K, S, nbytes, code in ((0, 4, need, -1), (3, 0, need, -1), (3, 4, need - 1, -3)):
            rc = lib.brl_elbo_val_steps(e.ctx, X.data_ptr(), Y.data_ptr(), 300, good.data_ptr(), K, 50, loc.data_ptr(), scale.data_ptr(),
                                        0, 1, S, eng_id, 0.0, 0.138793, 238150, 1, 0, 0, sc.data_ptr(), sc.data_ptr(), ws.data_ptr(),
                                        nbytes, torch.cuda.current_stream().cuda_stream)
            assert rc == code, (eng_id, K, S, nbytes, rc)
            with pytest.raises(RuntimeError, match="workspace too small" if code == -3 else "bad"):
                _lib.check(rc)
    # the codes of the other calls are as they were
    got = {f"{B},{S},{t},{en}": lib.brl_workspace_bytes(e.ctx, B, S, t, en)
           for B in (37, 100, 256) for S in (1, 2, 5) for t in range(5) for en in (0, 1)}
    assert got == PARENT_WORKSPACE_BYTES
    got = {f"{B},{S},{t}": lib.brl_workspace_bytes(e.ctx, B, S, t, 0) for B in (37, 100, 256) for S in (1, 2, 5) for t in (5, 6)}
    assert got == PARENT_TRAIN_STEPS_BYTES


def _bnn(engine="tc", mc_train=1, mc_eval=8):
    from bayesrul_b200.compat import BNN, Inception, pyro_shim
    torch.manual_seed(12345)
    net = Inception(30, 18)
    with torch.no_grad():
        net.last.bias.fill_(3.0)
    opt = pyro_shim.ClippedAdam({"lr": 0.000857, "betas": [0.95, 0.999], "clip_norm": 15})
    m = BNN(net, opt, pretrain_epochs=5, mc_samples_train=mc_train, mc_samples_eval=mc_eval, dataset_size=238150, fit_context="lrt",
            prior_loc=0.0, prior_scale=0.138793, guide="normal", q_scale=1.351e-3, device=DEV, engine=engine)
    m.on_fit_start()
    m.bnn._step = 5  # as after some training batches
    return m


VKEYS = ("elbo/val", "mse/val", "kl/val", "likelihood/val", "rmsce/val", "sharp/val")


@pytest.mark.parametrize("N", [1000, 1037])
def test_bnn_validate_epoch_matches_validation_step_loop(N):
    """compat: one validation epoch at batch size 100 (ten full batches in one call, and at N = 1037 a remainder of 37 through
    validation_step) against Lightning's loop of validation_step over the same in-order batches; then one training_step on each
    model continues from the same seed sequence"""
    bs = 100
    X, Y = _data(N, 125)

    def loop():
        m = _bnn()
        sums = dict.fromkeys(VKEYS, 0.0)
        for i, a in enumerate(range(0, N, bs)):
            b = slice(a, min(a + bs, N))
            m.validation_step((X[b], Y[b]), i)
            for k in VKEYS:
                sums[k] += float(m.logged[k]) * (b.stop - b.start)
        return m, {k: v / N for k, v in sums.items()}

    refs = [loop() for _ in range(NREF)]
    m = _bnn()
    g = m.bnn.net_guide
    before = [t.clone() for t in (g.loc, g.log_scale, g.scale)]
    res = m.validate_epoch(X, Y, bs)
    assert res["scalars"].shape == (10, 4) and res["metrics"].shape == (10, 5)
    for a, b in zip((g.loc, g.log_scale, g.scale), before):
        assert torch.equal(a, b)
    for k in VKEYS:
        vals = [r[1][k] for r in refs]
        spread = max(vals) - min(vals)
        got = m.logged[k]
        assert type(got) is type(refs[0][0].logged[k]), (k, type(got))
        if isinstance(got, torch.Tensor):
            assert got.dtype == refs[0][0].logged[k].dtype
        assert abs(float(got) - vals[0]) <= 2 * spread + 1e-6 * abs(vals[0]), (k, float(got), vals)
    assert m.bnn._step == refs[0][0].bnn._step == 5 + 2 * (-(-N // bs))
    assert float(m.bnn._last_kl) == pytest.approx(float(refs[0][0].bnn._last_kl), rel=1e-6)
    # one training batch on each: the same seed, hence the same step
    xb, yb = X[:bs].clone(), Y[:bs].clone()
    m.training_step((xb, yb), 0)
    for r in refs:
        r[0].training_step((xb, yb), 0)
    for k in ("elbo/train", "kl/train", "mse/train"):
        vals = [float(r[0].logged[k]) for r in refs]
        assert abs(float(m.logged[k]) - vals[0]) <= 2 * (max(vals) - min(vals)) + 1e-5 * abs(vals[0]), (k, m.logged[k], vals)


def test_bnn_validate_epoch_refuses_a_scaled_loss():
    from bayesrul_b200.compat import pyro_shim
    m = _bnn()
    X, Y = _data(300, 126)
    m.svi = pyro_shim.SVI(pyro_shim.poutine.scale(m.bnn.model, scale=1.0), pyro_shim.poutine.scale(m.bnn.guide, scale=1.0),
                          m.hparams.optimizer, m.loss)
    with pytest.raises(RuntimeError, match="validate_epoch"):
        m.validate_epoch(X, Y, 100)
    assert m.bnn._step == 5
