"""torch.optim.Adam on the device (brl_adam / Engine.adam), inside the K-step HNN training call (brl_hnn_train_steps_adam /
Engine.hnn_train_steps(optimizer="adam")) and under compat HNN.fit_epoch.

Engine.adam computes torch.optim.Adam's single-tensor update, so it is compared with torch itself: after 100 steps its parameters
and moments must lie no further from torch's single-tensor path than torch's own foreach path lies from it, plus four fp32 ulps of
the quantity's largest magnitude.  Measured on a B200: both moments bit-identical to torch's without weight decay; parameters
bit-identical in 97.6 % of the elements and at most 5.3e-8 of the largest magnitude apart, as far as foreach lies from single-tensor.

The K-step call and fit_epoch are compared with the per-step loop of their contract by the three-run spread scheme of
tests/test_gpu_train_steps.py (its helpers are reused): fp32 atomics in the backward make repeated steps differ in the last bits,
and the K-step result must lie within twice the largest distance between three reference runs, plus 1e-5 of the magnitude for a
step's scalars and metrics and 1e-3 in L2 norm for the final parameters and moments, which Adam's normalised update amplifies.
The reference loop runs torch.optim.Adam as users configure it (the default foreach path)."""
from functools import partial

import pytest
import torch

from tests.test_gpu_train_steps import (NREF, P_MCD, W, _ENGINES, _clone, _data, _eng, _hnn_state, _idx, _launches, _logged,
                                        _within)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
AOPT = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
ULP = 2.0 ** -23


@pytest.fixture(scope="module", autouse=True)
def _cleanup():
    yield
    _ENGINES.clear()


def _rel(a, b):
    return (a.double() - b.double()).abs().max().item() / max(b.double().abs().max().item(), 1e-30)


def _torch_adam_run(p0, grads, foreach, **kw):
    p = p0.clone()
    opt = torch.optim.Adam([p], foreach=foreach, **kw)
    for g in grads:
        p.grad = g
        opt.step()
    st = opt.state[p]
    return p, st["exp_avg"], st["exp_avg_sq"]


@pytest.mark.parametrize("weight_decay", [0.0, 0.01])
def test_adam_matches_torch_optim_adam(weight_decay):
    """100 steps over 200 003 elements with seeded gradients that include zeros, near-zero (1e-30 to 1e-12) and large (1e4)
    elements, on the same flat tensor as torch.optim.Adam"""
    from bayesrul_b200 import Engine
    e = Engine("inception", DEV)
    n, steps = 200_003, 100
    g = torch.Generator().manual_seed(7)
    p0 = torch.randn(n, generator=g).to(DEV)
    grads = []
    for _ in range(steps):
        gr = torch.randn(n, generator=g) * 1e-2
        gr[::97] = 0.0
        gr[1::97] = 1e-30
        gr[2::97] = -1e-12
        gr[3::101] *= 1e6
        grads.append(gr.to(DEV))
    kw = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=weight_decay)
    single = _torch_adam_run(p0, grads, False, **kw)
    foreach = _torch_adam_run(p0, grads, True, **kw)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for t, gr in enumerate(grads, 1):
        e.adam(p, gr, m, v, t, **kw)
    torch.cuda.synchronize()
    for name, got, ref, other in zip(("param", "exp_avg", "exp_avg_sq"), (p, m, v), single, foreach):
        spread, err = _rel(other, ref), _rel(got, ref)
        same, same_f = (got == ref).double().mean().item(), (got == other).double().mean().item()
        print(f"adam wd={weight_decay} {name}: |ours - single| {err:.3e}, |foreach - single| {spread:.3e}, |ours - foreach| "
              f"{_rel(got, other):.3e}; bit-identical to single {same:.6f}, to foreach {same_f:.6f}")
        assert err <= spread + 4 * ULP, (name, err, spread)


def _torch_adam_ref(e, X, Y, idx, st, p, seed, step0, opt_kw):
    """the loop of the contract: hnn_step{,_ensemble} on X[idx[k]], torch.optim.Adam on the flat theta, step_metrics"""
    from bayesrul_b200 import Noise
    K, M, B = idx.shape
    th = st["theta"]
    opt = torch.optim.Adam([th], **opt_kw)
    if step0:
        opt.state[th] = {"step": torch.tensor(float(step0)), "exp_avg": st["m"], "exp_avg_sq": st["v"]}
    sc, mt = [], []
    for k in range(K):
        xb, yb = X[idx[k]], Y[idx[k]]
        nz = Noise(seed=(seed + W * (k + 1)) & 0xFFFFFFFFFFFFFFFF)
        if M == 1:
            r = e.hnn_step(xb[0], yb[0], th[0], p, nz)
            r = dict(scalars=r["scalars"].unsqueeze(0), grad=r["grad"], out=r["out"].unsqueeze(0))
        else:
            r = e.hnn_step_ensemble(xb, yb, th, p, nz)
        th.grad = r["grad"].view_as(th)
        opt.step()
        sc.append(r["scalars"].clone())
        mt.append(_logged(e, r["out"].unsqueeze(1), yb, 1))
    s = opt.state[th]
    st["m"], st["v"] = s["exp_avg"], s["exp_avg_sq"]
    return torch.stack(sc), torch.stack(mt)


def _adam_state(net, M, seed, step0):
    """theta, and at step0 > 0 moments as Adam leaves them (m of either sign, v > 0)"""
    st = _hnn_state(net, M, seed)
    if step0:
        g = torch.Generator().manual_seed(seed + 1)
        st["m"] = (torch.randn(st["theta"].shape, generator=g) * 1e-3).to(DEV)
        st["v"] = (torch.rand(st["theta"].shape, generator=g) * 1e-6).to(DEV)
    return st


def _adam_call(e, X, Y, idx, st, p, seed, step0, **kw):
    return e.hnn_train_steps(X, Y, idx, st["theta"], (st["m"], st["v"]), step0=step0, p_dropout=p, seed=seed, optimizer="adam",
                             **{**AOPT, **kw})


CASES = [  # net, back-end, M, B, p
    ("inception", "fused", 1, 100, P_MCD),
    ("inception", "fused", 1, 100, 0.0),
    ("inception", "fused", 5, 100, P_MCD),
    ("linear", "fused", 1, 100, P_MCD),
    ("conv", "fused", 1, 100, P_MCD),
    ("inception", "simt", 1, 37, P_MCD),
]


@pytest.mark.parametrize("net,backend,M,B,p", CASES)
def test_hnn_train_steps_adam_match_the_step_loop(net, backend, M, B, p):
    K, N, step0 = 7, 1500, 3
    X, Y = _data(N, 21)
    idx = _idx(K, M, B, N, 22)
    st0 = _adam_state(net, M, 23, step0)
    seed = 0x2468ACE + 7 * M + B
    refs = []
    for i in range(NREF):
        st = _clone(st0)
        refs.append((st,) + _torch_adam_ref(_eng(net, backend, f"aref{i}"), X, Y, idx, st, p, seed, step0, AOPT))
    st = _clone(st0)
    got = _adam_call(_eng(net, backend, "aksteps"), X, Y, idx, st, p, seed, step0)
    assert got["scalars"].shape == (K, M, 2) and got["metrics"].shape == (K, M, 5)
    _within(got["scalars"], [r[1] for r in refs], "scalars")
    _within(got["metrics"], [r[2] for r in refs], "metrics")
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)


def test_adam_second_call_replays_and_matches_clipped_launches():
    """a second call with new X / idx tensors, seed and step0 continues the loop from the captured graph with the same launches
    (one setup launch plus the same launches per step), and a step costs as many launches as in the ClippedAdam call"""
    net, M, B, K, N = "inception", 5, 100, 7, 1500
    X, Y = _data(N, 24)
    idx1, idx2 = _idx(K, M, B, N, 25), _idx(K, M, B, N, 26)
    st0 = _adam_state(net, M, 27, 0)
    refs = []
    for i in range(NREF):
        st = _clone(st0)
        a = _torch_adam_ref(_eng(net, "fused", f"aref{i}"), X, Y, idx1, st, P_MCD, 5, 0, AOPT)
        b = _torch_adam_ref(_eng(net, "fused", f"aref{i}"), X, Y, idx2, st, P_MCD, 77, K, AOPT)
        refs.append((st,) + a + b)
    e = _eng(net, "fused", "asecond")
    st = _clone(st0)
    n1, got1 = _launches(e, lambda: _adam_call(e, X, Y, idx1, st, P_MCD, 5, 0))
    n2, got2 = _launches(e, lambda: _adam_call(e, X.clone(), Y.clone(), idx2, st, P_MCD, 77, K))
    assert n1 == n2 and (n2 - 1) % K == 0, (n1, n2)
    for i, (got, name) in enumerate(((got1, "call 1"), (got2, "call 2"))):
        _within(got["scalars"], [r[1 + 2 * i] for r in refs], name + " scalars")
        _within(got["metrics"], [r[2 + 2 * i] for r in refs], name + " metrics")
    for k in st:
        _within(st[k], [r[0][k] for r in refs], k, state=True)
    ec = _eng(net, "fused", "aclipped")
    sc = _clone(st0)
    kw = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
    c1, _ = _launches(ec, lambda: ec.hnn_train_steps(X, Y, idx1, sc["theta"], (sc["m"], sc["v"]), step0=0, p_dropout=P_MCD, seed=5, **kw))
    c2, _ = _launches(ec, lambda: ec.hnn_train_steps(X, Y, idx2, sc["theta"], (sc["m"], sc["v"]), step0=K, p_dropout=P_MCD, seed=77, **kw))
    assert (c1, c2) == (n1, n2), (c1, c2, n1, n2)


def test_adam_graphs_off_gives_the_same_results():
    net, M, B, K, N = "inception", 5, 100, 7, 1500
    X, Y = _data(N, 28)
    idx = _idx(K, M, B, N, 29)
    st0 = _adam_state(net, M, 30, 2)
    runs = []
    for tag, graphs in (("anograph", False), ("ag1", True), ("ag2", True), ("ag3", True)):
        e = _eng(net, "fused", tag)
        e.set_step_graph(graphs)
        st = _clone(st0)
        r = _adam_call(e, X, Y, idx, st, P_MCD, 31, 2)
        e.set_step_graph(True)
        runs.append((st, r))
    (s0, r0), refs = runs[0], runs[1:]
    for k in ("scalars", "metrics"):
        _within(r0[k], [r[k] for _, r in refs], k)
    for k in s0:
        _within(s0[k], [s[k] for s, _ in refs], k, state=True)


def test_clipped_then_adam_on_the_same_pointers_share_no_graph():
    """ClippedAdam (a clamp of 1e-4 and eps 1e-3, far from Adam's update) then Adam on the same tensors and workspace, graphs
    on: each must match an eager run of its own optimizer"""
    net, M, B, K, N = "inception", 1, 100, 5, 1500
    X, Y = _data(N, 32)
    idx = _idx(K, M, B, N, 33)
    st0 = _adam_state(net, M, 34, 0)
    ckw = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-3, clip_norm=1e-4, lrd=1.0, weight_decay=0.0)
    akw = dict(eps=1e-3)

    def clipped(e, st):
        return e.hnn_train_steps(X, Y, idx, st["theta"], (st["m"], st["v"]), step0=0, p_dropout=P_MCD, seed=35, **ckw)

    eager = {}
    for kind in ("clipped", "adam"):
        outs = []
        for i in range(NREF):
            e = _eng(net, "fused", f"aeager{i}")
            e.set_step_graph(False)
            st = _clone(st0)
            r = clipped(e, st) if kind == "clipped" else _adam_call(e, X, Y, idx, st, P_MCD, 35, 0, **akw)
            e.set_step_graph(True)
            outs.append((st, r))
        eager[kind] = outs
    e = _eng(net, "fused", "amixed")
    st = _clone(st0)
    for kind in ("clipped", "adam"):
        for k in st:
            st[k].copy_(st0[k])  # the same pointers for both calls
        r = clipped(e, st) if kind == "clipped" else _adam_call(e, X, Y, idx, st, P_MCD, 35, 0, **akw)
        refs = eager[kind]
        _within(r["scalars"], [o[1]["scalars"] for o in refs], kind + " scalars")
        for k in st:
            _within(st[k], [o[0][k] for o in refs], f"{kind} {k}", state=True)
    # the two optimizers must be told apart by the comparison above
    a, c = eager["adam"][0][0]["theta"], eager["clipped"][0][0]["theta"]
    assert (a - c).norm() > 0.1 * (a - st0["theta"]).norm()


def _hnn_model(net_kind, p):
    from bayesrul_b200.compat import HNN, Conv, Inception, Linear
    torch.manual_seed(12345)
    net = {"inception": Inception, "linear": Linear, "conv": Conv}[net_kind](30, 18, dropout=p)
    m = HNN(net, partial(torch.optim.Adam, lr=1e-3), mc_samples=10, p_dropout=p, device=DEV)
    return m, m.configure_optimizers()


def _lightning_batch(m, opt, x, y, i):
    """Lightning's automatic optimisation of one batch: training_step, zero_grad, backward, step"""
    loss = m.training_step((x, y), i)
    opt.zero_grad()
    loss.backward()
    opt.step()


KEYS = ("nll/train", "mse/train", "rmsce/train", "sharp/train")


@pytest.mark.parametrize("N", [1000, 1037])
def test_hnn_fit_epoch_matches_lightning_loop(N):
    """compat: one epoch at batch size 100 (ten full batches in one K-step call, and at N = 1037 a remainder of 37 through
    training_step) against Lightning's loop over the same permutation; then one more batch on each continues the trajectory"""
    bs = 100
    X, Y = _data(N, 36)
    xn, yn = X[:bs].clone(), Y[:bs].clone()

    def loop():
        m, opt = _hnn_model("inception", P_MCD)
        perm = torch.randperm(N, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV)
        sums = dict.fromkeys(KEYS, 0.0)
        for i, a in enumerate(range(0, N, bs)):
            b = perm[a: a + bs]
            _lightning_batch(m, opt, X[b], Y[b], i)
            for k in KEYS:
                sums[k] += float(torch.as_tensor(m.logged[k]).detach()) * b.numel()
        return m, opt, {k: v / N for k, v in sums.items()}

    refs = [loop() for _ in range(NREF)]
    m, opt = _hnn_model("inception", P_MCD)
    res = m.fit_epoch(X, Y, bs, opt, generator=torch.Generator(device=DEV).manual_seed(5))
    assert res["scalars"].shape == (10, 1, 2) and res["metrics"].shape == (10, 1, 5)
    assert torch.equal(res["perm"], torch.randperm(N, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV))
    for k in KEYS:
        vals = [r[2][k] for r in refs]
        spread = max(vals) - min(vals)
        assert abs(m.logged[k] - vals[0]) <= 2 * spread + 1e-5 * abs(vals[0]), (k, m.logged[k], vals)
    _within(m.net.theta, [r[0].net.theta for r in refs], "theta", state=True)
    nsteps = -(-N // bs)
    assert m._it == refs[0][0]._it == nsteps
    for i, p in enumerate(m.net._params):
        st = opt.state[p]
        rsts = [r[1].state[r[0].net._params[i]] for r in refs]
        assert float(st["step"]) == float(rsts[0]["step"]) == nsteps
        assert st["step"].dtype == rsts[0]["step"].dtype and st["step"].device == rsts[0]["step"].device
        for k in ("exp_avg", "exp_avg_sq"):
            assert st[k].shape == p.shape
    for k in ("exp_avg", "exp_avg_sq"):
        flat = lambda mm, o: torch.cat([o.state[q][k].reshape(-1) for q in mm.net._params])
        _within(flat(m, opt), [flat(r[0], r[1]) for r in refs], k, state=True)
    # one more batch: the torch optimizer continues from the state fit_epoch left
    _lightning_batch(m, opt, xn, yn, 0)
    got = float(m.logged["nll/train"].detach())
    for r in refs:
        _lightning_batch(r[0], r[1], xn, yn, 0)
    vals = [float(r[0].logged["nll/train"].detach()) for r in refs]
    assert abs(got - vals[0]) <= 2 * (max(vals) - min(vals)) + 1e-5 * abs(vals[0]), (got, vals)
    _within(m.net.theta, [r[0].net.theta for r in refs], "theta after one more batch", state=True)


def test_hnn_fit_epoch_errors():
    X, Y = _data(300, 37)
    m, _ = _hnn_model("inception", P_MCD)
    ps = list(m.parameters())
    bad = [torch.optim.Adam(ps, lr=1e-3, amsgrad=True), torch.optim.Adam(ps, lr=1e-3, maximize=True),
           torch.optim.Adam([{"params": ps[:4]}, {"params": ps[4:]}], lr=1e-3), torch.optim.SGD(ps, lr=1e-3),
           torch.optim.AdamW(ps, lr=1e-3), torch.optim.Adam(ps[1:], lr=1e-3)]
    for opt in bad:
        with pytest.raises(RuntimeError, match="fit_epoch"):
            m.fit_epoch(X, Y, 100, opt)
    assert m._it == 0 and torch.isfinite(m.net.theta).all()
    e = m.net.engine()
    st = _hnn_state("inception", 1, 38)
    idx = _idx(2, 1, 50, 300, 39)
    for kw in (dict(clip_norm=15.0), dict(lrd=0.999), dict(clip_norm=1e30, lrd=1.0)):
        with pytest.raises(RuntimeError, match="clip_norm or lrd"):
            e.hnn_train_steps(X, Y, idx, st["theta"], (st["m"], st["v"]), step0=0, lr=1e-3, seed=1, optimizer="adam", **kw)
    with pytest.raises(RuntimeError, match="optimizer"):
        e.hnn_train_steps(X, Y, idx, st["theta"], (st["m"], st["v"]), step0=0, lr=1e-3, seed=1, optimizer="sgd")


def test_adam_call_marks_out_of_range_windows_nan():
    """the C ABI reads no memory for an index outside [0, N): that step's rows are NaN, the others are finite"""
    e = _eng("inception", "fused", "anan")
    X, Y = _data(300, 40)
    st = _hnn_state("inception", 1, 41)
    idx = _idx(3, 1, 50, 300, 42)
    idx[1, 0, 7] = 300
    lib = e.lib
    need = lib.brl_workspace_bytes(e.ctx, 50, 1, 6, 0)
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    sc = torch.empty(3, 1, 2, dtype=torch.float64, device=DEV)
    mt = torch.empty(3, 1, 5, dtype=torch.float64, device=DEV)
    rc = lib.brl_hnn_train_steps_adam(e.ctx, X.data_ptr(), Y.data_ptr(), 300, idx.data_ptr(), 3, 1, 50, st["theta"].data_ptr(),
                                      st["m"].data_ptr(), st["v"].data_ptr(), 0, 1e-3, 0.9, 0.999, 1e-8, 0.0, P_MCD, 1, 0, 0,
                                      sc.data_ptr(), mt.data_ptr(), ws.data_ptr(), need, torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.isnan(sc[1]).all() and torch.isnan(mt[1]).all()
    assert torch.isfinite(sc[0]).all() and torch.isfinite(mt[0]).all()
    # the library's own checks: K = 0 and a workspace below brl_workspace_bytes(B, M, 6)
    for K, nbytes in ((0, need), (3, need - 256)):
        rc = lib.brl_hnn_train_steps_adam(e.ctx, X.data_ptr(), Y.data_ptr(), 300, idx.data_ptr(), K, 1, 50, st["theta"].data_ptr(),
                                          st["m"].data_ptr(), st["v"].data_ptr(), 0, 1e-3, 0.9, 0.999, 1e-8, 0.0, P_MCD, 1, 0, 0,
                                          sc.data_ptr(), mt.data_ptr(), ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
        assert rc != 0, (K, nbytes)


# brl_workspace_bytes(ctx, B, S, 5 / 6, 0) of the Inception net at the parent commit (codes 0-4 are pinned by
# tests/test_gpu_train_steps.py): torch's Adam shares code 6 and leaves both as they were
PARENT_TRAIN_STEPS_BYTES = {
    "37,1,5": 77435136, "37,1,6": 37442048, "37,2,5": 64477184, "37,2,6": 51438848, "37,5,5": 125694976, "37,5,6": 93103104,
    "100,1,5": 133072896, "100,1,6": 63717120, "100,2,5": 104385280, "100,2,6": 89546496, "100,5,5": 203246592, "100,5,6": 166157312,
    "256,1,5": 279798272, "256,1,6": 133256192, "256,2,5": 212153088, "256,2,6": 192858368, "256,5,5": 417658624, "256,5,6": 369425408,
}


def test_train_steps_workspace_codes_unchanged():
    e = _eng("inception", "fused", "aws")
    got = {f"{B},{S},{t}": e.lib.brl_workspace_bytes(e.ctx, B, S, t, 0) for B in (37, 100, 256) for S in (1, 2, 5) for t in (5, 6)}
    assert got == PARENT_TRAIN_STEPS_BYTES
