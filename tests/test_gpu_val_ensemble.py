"""K validation batches of the M seeds of a BNN experiment per call (brl_elbo_val_steps_ensemble, Engine.elbo_val_steps with [M,P]
parameters).

Member m of batch k is, by contract, the sequence of Engine calls that validates seed m on its own: elbo_step(mode="ws",
compute_grads=False) with the Philox seed seed + 0x9E3779B97F4A7C15 (2k + 1) at sample0 + m particles, then sample_weights(S),
forward("ws", engine) and (S > 1) aggregate_predictions with seed + 0x9E3779B97F4A7C15 (2k + 2) at sample0 + m S, then
step_metrics; every member sees the same windows idx[k].  The comparison scheme is that of tests/test_gpu_val_steps.py: three
runs of the loop, and the call within twice their largest distance plus 1e-6 of the quantity's largest magnitude, per member and
column (fp64 / fp32 atomics in the ELBO's reductions make repeated runs differ in the last bits).  A member drawn at another MC-sample
index, or with the wrong key, moves by a weight draw: the negative controls check that the bound sees it."""
import pytest
import torch

from tests.test_gpu_hnn_fit_epoch import PARENT_TRAIN_STEPS_BYTES
from tests.test_gpu_train_steps import (KW, NREF, PARENT_WORKSPACE_BYTES, W, _ENGINES, _clone, _data, _elbo_call, _eng, _idx,
                                        _launches, _vi_state, _within)
from tests.test_gpu_val_steps import _call, _check, _close, _excess

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MASK = 0xFFFFFFFFFFFFFFFF


@pytest.fixture(scope="module", autouse=True)
def _cleanup():
    yield
    _ENGINES.clear()


def _params(net, M, seed):
    st = _vi_state(net, M, seed)
    return st["loc"], st["log_scale"], st["scale"]


def _ref_members(e, X, Y, idx, loc, scale, cfg, seed, same_sample0=False, swap=False):
    """the per-member loop of the contract, [K,M,4] and [K,M,5]; same_sample0=True draws every member at sample0 = 0, swap=True
    draws the ELBO with the predictive's key and the other way round"""
    from bayesrul_b200 import Noise
    guide, particles, S, engine = cfg
    sc, mt = [], []
    for k in range(idx.shape[0]):
        xb, yb = X[idx[k]], Y[idx[k]]
        k1, k2 = (seed + W * (2 * k + 1)) & MASK, (seed + W * (2 * k + 2)) & MASK
        if swap:
            k1, k2 = k2, k1
        scs, mts = [], []
        for m in range(loc.shape[0]):
            s1, s2 = (0, 0) if same_sample0 else (m * particles, m * S)
            r = e.elbo_step(xb, yb, loc[m], scale[m], mode="ws", guide=guide, particles=particles, noise=Noise(seed=k1, sample0=s1),
                            compute_grads=False, **KW)
            scs.append(r["scalars"].clone())
            w = e.sample_weights(loc[m], scale[m], guide, S, Noise(seed=k2, sample0=s2))
            out = e.forward(xb, "ws", wsamp=w, S=S, noise=Noise(seed=k2, sample0=s2), engine=engine)
            o = e.aggregate_predictions(out) if S > 1 else out[0]
            mts.append(e.step_metrics(o[:, 0], o[:, 1], yb))
        sc.append(torch.stack(scs))
        mt.append(torch.stack(mts))
    return torch.stack(sc), torch.stack(mt)


CASES = [  # net, back-end, (guide, particles, S, engine), M, B
    ("inception", "fused", ("normal", 1, 8, "tc"), 5, 100),
    ("inception", "fused", ("normal", 1, 1, "tc"), 5, 100),
    ("inception", "fused", ("radial", 1, 8, "tc"), 5, 100),
    ("inception", "fused", ("normal", 2, 8, "tc"), 5, 100),
    ("inception", "simt", ("normal", 1, 8, "simt"), 3, 37),
    ("linear", "fused", ("normal", 1, 8, "tc"), 3, 100),
    ("conv", "fused", ("normal", 1, 8, "simt"), 3, 100),
]


@pytest.mark.parametrize("net,backend,cfg,M,B", CASES)
def test_val_ensemble_matches_the_member_loop(net, backend, cfg, M, B):
    K, N = 7, 1500
    X, Y = _data(N, 201)
    idx = _idx(K, 1, B, N, 202)[:, 0]
    loc, log_scale, scale = _params(net, M, 203)
    before = [t.clone() for t in (loc, log_scale, scale)]
    seed = 0x0FED_CBA9_8765_4321 + B
    refs = [_ref_members(_eng(net, backend, f"evref{i}"), X, Y, idx, loc, scale, cfg, seed) for i in range(NREF)]
    e = _eng(net, backend, "eval")
    got = _call(e, X, Y, idx, loc, scale, cfg, seed)
    assert got["scalars"].shape == (K, M, 4) and got["metrics"].shape == (K, M, 5)
    _check(got, refs, "call")
    for a, b in zip((loc, log_scale, scale), before):
        assert torch.equal(a, b)
    if net == "inception" and cfg == ("normal", 1, 8, "tc"):
        # negative controls: the loop with every member at sample0 = 0, a call one key further along the sequence, and the loop
        # with the two keys of each batch swapped
        ref0 = _eng(net, backend, "evref0")
        z = _ref_members(ref0, X, Y, idx, loc, scale, cfg, seed, same_sample0=True)
        assert _excess(z[0], [r[0] for r in refs]) > 1 and _excess(z[1], [r[1] for r in refs]) > 1
        bad = _call(e, X, Y, idx, loc, scale, cfg, (seed + W) & MASK)
        assert _excess(bad["scalars"], [r[0] for r in refs]) > 1 and _excess(bad["metrics"], [r[1] for r in refs]) > 1
        sw = _ref_members(ref0, X, Y, idx, loc, scale, cfg, seed, swap=True)
        assert _excess(sw[0], [r[0] for r in refs]) > 1 and _excess(sw[1], [r[1] for r in refs]) > 1


@pytest.mark.parametrize("cfg", [("normal", 1, 8, "tc"), ("radial", 2, 4, "simt")])
def test_one_member_is_elbo_val_steps(cfg):
    """M = 1: the ensemble call gives what elbo_val_steps gives, with the same launches per batch"""
    net, B, K, N = "inception", 100, 7, 1500
    X, Y = _data(N, 204)
    idx = _idx(K, 1, B, N, 205)[:, 0]
    loc, _, scale = _params(net, 1, 206)
    refs = []
    for i in range(NREF):
        e = _eng(net, "fused", f"e1single{i}")
        n_single, r = _launches(e, lambda: _call(e, X, Y, idx, loc[0], scale[0], cfg, 41))
        refs.append((r["scalars"], r["metrics"]))
    e = _eng(net, "fused", "e1ens")
    n_ens, got = _launches(e, lambda: _call(e, X, Y, idx, loc, scale, cfg, 41))
    assert got["scalars"].shape == (K, 1, 4) and got["metrics"].shape == (K, 1, 5)
    assert n_ens == n_single, (n_ens, n_single)
    _check(got, refs, "M = 1")


def test_second_call_replays_with_new_indices_and_seed():
    """a second call with new X / idx tensors and a new seed comes from the first call's graph: both calls issue one setup launch
    plus the same launches per batch"""
    net, cfg, M, B, K, N = "inception", ("normal", 1, 8, "tc"), 5, 100, 7, 1500
    X, Y = _data(N, 207)
    idx1, idx2 = _idx(K, 1, B, N, 208)[:, 0], _idx(K, 1, B, N, 209)[:, 0]
    loc, _, scale = _params(net, M, 210)
    refs1 = [_ref_members(_eng(net, "fused", f"evref{i}"), X, Y, idx1, loc, scale, cfg, 5) for i in range(NREF)]
    refs2 = [_ref_members(_eng(net, "fused", f"evref{i}"), X, Y, idx2, loc, scale, cfg, 77) for i in range(NREF)]
    e = _eng(net, "fused", "eval_second")
    n1, got1 = _launches(e, lambda: _call(e, X, Y, idx1, loc, scale, cfg, 5))
    n2, got2 = _launches(e, lambda: _call(e, X.clone(), Y.clone(), idx2, loc, scale, cfg, 77))
    assert n1 == n2 and (n2 - 1) % K == 0, (n1, n2)
    n3, _ = _launches(e, lambda: _call(e, X, Y, idx2[:3], loc, scale, cfg, 1))
    assert n2 - n3 == (K - 3) * (n3 - 1) // 3, (n2, n3)
    _check(got1, refs1, "call 1")
    _check(got2, refs2, "call 2")


@pytest.mark.parametrize("cfg", [("normal", 1, 8, "tc"), ("radial", 2, 4, "simt")])
def test_graphs_off_gives_the_same_results(cfg):
    net, M, B, K, N = "inception", 5, 100, 7, 1500
    X, Y = _data(N, 211)
    idx = _idx(K, 1, B, N, 212)[:, 0]
    loc, _, scale = _params(net, M, 213)
    runs = []
    for tag, graphs in (("evnograph", False), ("evg1", True), ("evg2", True), ("evg3", True)):
        e = _eng(net, "fused", tag)
        e.set_step_graph(graphs)
        runs.append(_call(e, X, Y, idx, loc, scale, cfg, 21))
        e.set_step_graph(True)
    _check(runs[0], [(r["scalars"], r["metrics"]) for r in runs[1:]], "graphs off")


def test_tc_timing_runs_eagerly_with_the_same_results():
    """with the tensor-core engine's timing hooks on, every batch runs eagerly and gives the loop's results; the M S draws of a
    batch are one forward: the hooks see one tc_conv_kernel and one tc_fc_kernel per batch"""
    net, cfg, M, B, K, N = "inception", ("normal", 1, 8, "tc"), 5, 100, 7, 1500
    X, Y = _data(N, 214)
    idx = _idx(K, 1, B, N, 215)[:, 0]
    loc, _, scale = _params(net, M, 216)
    refs = [_ref_members(_eng(net, "fused", f"evref{i}"), X, Y, idx, loc, scale, cfg, 9) for i in range(NREF)]
    e = _eng(net, "fused", "eval_timing")
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
    """elbo_train_steps (M = 5), the val ensemble call, elbo_train_steps on one engine (one workspace, graphs on): no call replays
    another's graph.  The training calls are compared with the same sequence with graphs off.  The val call is compared with the
    per-member loop on the parameters it validated: the five members' fused training step sums in fp32 atomics whose order differs
    between the eager and the replayed step, and Adam's normalised update turns those last bits into parameter differences
    (tests/test_gpu_train_steps.py) that move the val ELBO by more than the 1e-6 of the val bound (measured on a B200: one member's
    val loss 7.6e-6 of its magnitude from the graphs-off sequence, whose three runs agreed to 1e-8)."""
    net, cfg, M, B, K, N = "inception", ("normal", 1, 8, "tc"), 5, 100, 7, 1500
    X, Y = _data(N, 217)
    idx1, idx2, idx3 = (_idx(K, M, B, N, s) for s in (218, 219, 220))
    vidx = idx2[:, 0].contiguous()
    st0 = _vi_state(net, M, 221)

    def seq(e):
        st = _clone(st0)
        a = _elbo_call(e, X, Y, idx1, st, ("lrt", "normal", 1), 31, 0)
        seen = (st["loc"].clone(), st["scale"].clone())
        b = _call(e, X, Y, vidx, st["loc"], st["scale"], cfg, 32)
        c = _elbo_call(e, X, Y, idx3, st, ("lrt", "normal", 1), 33, K)
        return st, a, b, c, seen

    refs = []
    for i in range(NREF):
        e = _eng(net, "fused", f"evseq_eager{i}")
        e.set_step_graph(False)
        refs.append(seq(e))
    e = _eng(net, "fused", "evseq_graph")
    seq(e)  # first sight of each configuration: eager, then captured
    st, a, b, c, (loc, scale) = seq(e)  # every step / batch after the first of each call replays
    for i, (got, name) in ((0, (a, "train 1")), (2, (c, "train 2"))):
        for key in ("scalars", "metrics"):
            _close(got[key], [r[1 + i][key] for r in refs], f"{name} {key}", rtol=1e-5)
    vrefs = [_ref_members(_eng(net, "fused", f"evref{i}"), X, Y, vidx, loc, scale, cfg, 32) for i in range(NREF)]
    _check(b, vrefs, "val")
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)


def _raw(e, X, Y, N, idx, K, M, B, loc, scale, S, eng_id, sc, mt, ws, nbytes, guide=0, particles=1):
    return e.lib.brl_elbo_val_steps_ensemble(e.ctx, X, Y, N, idx, K, M, B, loc, scale, guide, particles, S, eng_id, 0.0, 0.138793,
                                             238150, 5, 0, 0, sc, mt, ws, nbytes, torch.cuda.current_stream().cuda_stream)


def test_out_of_range_index_gives_nan_rows_for_every_member():
    e = _eng("inception", "fused", "evnan")
    M, B, K, N = 3, 50, 3, 300
    X, Y = _data(N, 222)
    loc, _, scale = _params("inception", M, 223)
    idx = _idx(K, 1, B, N, 224)[:, 0].contiguous()
    idx[1, 7] = N
    need = e.lib.brl_workspace_bytes_val(e.ctx, B, M, 4, 1)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    sc = torch.empty(K, M, 4, dtype=torch.float64, device=DEV)
    mt = torch.empty(K, M, 5, dtype=torch.float64, device=DEV)
    rc = _raw(e, X.data_ptr(), Y.data_ptr(), N, idx.data_ptr(), K, M, B, loc.data_ptr(), scale.data_ptr(), 4, 1, sc.data_ptr(),
              mt.data_ptr(), ws.data_ptr(), need)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.isnan(sc[1]).all() and torch.isnan(mt[1]).all()
    for k in (0, 2):
        assert torch.isfinite(sc[k]).all() and torch.isfinite(mt[k]).all()


def test_errors_and_workspace_codes():
    from bayesrul_b200 import _lib
    e = _eng("inception", "fused", "everrors")
    M, B, K, N = 3, 50, 3, 300
    X, Y = _data(N, 225)
    loc, _, scale = _params("inception", M, 226)
    good = _idx(K, 1, B, N, 227)[:, 0].contiguous()
    cfg = ("normal", 1, 4, "tc")
    with pytest.raises(RuntimeError, match="outside"):
        _call(e, X, Y, torch.where(good == good[1, 7], N, good), loc, scale, cfg, 1)
    with pytest.raises(RuntimeError, match="idx"):
        _call(e, X, Y, good.view(K, 1, B).expand(K, M, B).contiguous(), loc, scale, cfg, 1)  # [K,M,B]: the members share idx [K,B]
    with pytest.raises(RuntimeError, match="scale"):
        _call(e, X, Y, good, loc, scale[:2], cfg, 1)
    with pytest.raises(RuntimeError, match="scale"):
        _call(e, X, Y, good, loc, scale[0], cfg, 1)
    with pytest.raises(RuntimeError, match="loc"):
        _call(e, X, Y, good, loc[:, :-1].contiguous(), scale, cfg, 1)
    with pytest.raises(RuntimeError, match="empty ensemble"):
        _call(e, X, Y, good, loc[:0], scale[:0], cfg, 1)
    with pytest.raises(RuntimeError, match="engine"):
        _call(e, X, Y, good, loc, scale, ("normal", 1, 4, "fp8"), 1)
    with pytest.raises(RuntimeError, match="particles"):
        _call(e, X, Y, good, loc, scale, ("normal", 9, 4, "tc"), 1)
    with pytest.raises(RuntimeError, match="S"):
        _call(e, X, Y, good, loc, scale, ("normal", 1, 0, "tc"), 1)
    with pytest.raises(RuntimeError, match="S"):
        _call(e, X, Y, good, loc, scale, ("normal", 1, 1 << 15, "tc"), 1)  # M S >= 65536
    # the library's own checks
    lib = e.lib
    sc = torch.empty(K, M, 5, dtype=torch.float64, device=DEV)
    for eng_id in (0, 1):
        need = lib.brl_workspace_bytes_val(e.ctx, B, M, 4, eng_id)
        assert need > 0
        ws = torch.empty(need, dtype=torch.uint8, device=DEV)
        p = dict(X=X.data_ptr(), Y=Y.data_ptr(), N=N, idx=good.data_ptr(), K=K, M=M, B=B, loc=loc.data_ptr(), scale=scale.data_ptr(),
                 S=4, eng_id=eng_id, sc=sc.data_ptr(), mt=sc.data_ptr(), ws=ws.data_ptr(), nbytes=need)
        for bad, code in ((dict(loc=None), -1), (dict(scale=None), -1), (dict(X=None), -1), (dict(idx=None), -1), (dict(sc=None), -1),
                          (dict(ws=None), -1), (dict(K=0), -1), (dict(M=0), -1), (dict(M=1 << 16), -1), (dict(B=0), -1),
                          (dict(N=0), -1), (dict(S=0), -1), (dict(S=1 << 15), -1), (dict(eng_id=2), -1), (dict(guide=2), -1),
                          (dict(particles=0), -1), (dict(particles=9), -1), (dict(nbytes=need - 1), -3)):
            rc = _raw(e, **{**p, **bad})
            assert rc == code, (eng_id, bad, rc)
            with pytest.raises(RuntimeError):
                _lib.check(rc)
        # one member's workspace is brl_elbo_val_steps'
        for b in (37, 100, 256):
            for s in (1, 4, 8):
                assert lib.brl_workspace_bytes_val(e.ctx, b, 1, s, eng_id) == lib.brl_workspace_bytes(e.ctx, b, s, 7, eng_id), (b, s)
    for args in ((0, 1, 4, 1), (B, 0, 4, 1), (B, 1, 0, 1), (B, 4, 1 << 14, 1), (B, 1, 4, 2)):
        assert lib.brl_workspace_bytes_val(e.ctx, *args) < 0, args
    # the codes of the other calls are as they were
    got = {f"{b},{s},{t},{en}": lib.brl_workspace_bytes(e.ctx, b, s, t, en)
           for b in (37, 100, 256) for s in (1, 2, 5) for t in range(5) for en in (0, 1)}
    assert got == PARENT_WORKSPACE_BYTES
    got = {f"{b},{s},{t}": lib.brl_workspace_bytes(e.ctx, b, s, t, 0) for b in (37, 100, 256) for s in (1, 2, 5) for t in (5, 6)}
    assert got == PARENT_TRAIN_STEPS_BYTES
