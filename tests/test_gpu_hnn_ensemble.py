"""Member-batched HNN step of a deep ensemble (brl_hnn_step_ensemble / Engine.hnn_step_ensemble).

Member m of an M-member step is hnn_step(x[m], y[m], theta[m], p, noise with sample0 + m).  On the fused back-end with the
Inception net the members share every launch of the level-fused kernels (member = blockIdx.z); everywhere else they run one
after another on the single-member step.  Either way a member's result equals the single-member step's up to summation order
(atomics, and the backward CTA grouping that counts all members): scalars and outputs rtol 1e-5, gradient
max |diff| / max |grad| < 3e-4.  That is the spread of the fused back-end itself: a last-bit change of an fp32 atomic sum
that flips the rounding of one bf16 gradient-image element moves the largest gradient entries by up to about 1e-4, and two
calls of the single-member step on the same inputs have been measured 1.1e-4 apart.
Against the float64 oracle the fused back-end's bounds hold: loss 5e-3, outputs 1e-2, gradient cosine > 0.999 (> 0.99 for a
ragged 37-window batch)."""
import pytest
import torch

from oracle import bnn_oracle as O
from tests.helpers import injected_to_engine, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NET = "inception"
P_DROP = 0.241437


@pytest.fixture(scope="module")
def eng():
    from bayesrul_b200 import Engine
    e = Engine(NET, DEV)
    e.set_gemm_backend("fused")
    yield e
    e.set_gemm_backend("simt")
    e.set_step_graph(True)


def _members(net, M, B, seed):
    """distinct windows, targets and parameters per member"""
    xs, ys, ths = zip(*[synth(net, B, seed=seed + 7 * m)[:3] for m in range(M)])
    return torch.stack(xs).to(DEV), torch.stack(ys).to(DEV), torch.stack(ths).to(DEV)


def _singles(e, x, y, th, p, seed, s0, compute_grads=True):
    from bayesrul_b200 import Noise
    return [e.hnn_step(x[m], y[m], th[m], p, Noise(seed=seed, sample0=s0 + m), compute_grads=compute_grads) for m in range(x.shape[0])]


def _assert_member(got, ref, m, what, grads=True):
    assert torch.allclose(got["scalars"][m], ref["scalars"], rtol=1e-5, atol=0), (what, m, got["scalars"][m], ref["scalars"])
    assert torch.allclose(got["out"][m], ref["out"], rtol=1e-5, atol=1e-6), (what, m, (got["out"][m] - ref["out"]).abs().max())
    if grads:
        rel = ((got["grad"][m] - ref["grad"]).abs().max() / ref["grad"].abs().max()).item()
        assert rel < 3e-4, (what, m, rel)


def _cos(a, b):
    return float((a * b).sum() / (a.norm() * b.norm() + 1e-300))


@pytest.mark.parametrize("p", [0.0, P_DROP])
@pytest.mark.parametrize("B", [256, 37])
@pytest.mark.parametrize("M", [1, 3, 5])
def test_members_match_single_steps(eng, M, B, p):
    from bayesrul_b200 import Noise
    x, y, th = _members(NET, M, B, seed=100 + M + B)
    got = eng.hnn_step_ensemble(x, y, th, p, Noise(seed=11, sample0=3))
    refs = _singles(eng, x, y, th, p, 11, 3)
    assert eng.tc_status() == 0
    assert got["scalars"].shape == (M, 2) and got["scalars"].dtype == torch.float64
    assert got["out"].shape == (M, B, 2) and got["grad"].shape == (M, eng.P)
    for m in range(M):
        _assert_member(got, refs[m], m, f"M={M} B={B} p={p}")


@pytest.mark.parametrize("B", [256, 37])
def test_injected_masks_vs_oracle(eng, B):
    M = 3
    x, y, th = _members(NET, M, B, seed=300 + B)
    g = torch.Generator().manual_seed(5)
    nzs = [O.make_injected_noise(NET, B, "det", g, p_dropout=P_DROP) for _ in range(M)]
    got = eng.hnn_step_ensemble(x, y, th, P_DROP, injected_to_engine(NET, nzs, B, DEV))
    assert eng.tc_status() == 0
    for m in range(M):
        t = th[m].cpu().double().requires_grad_(True)
        loss, out = O.hnn_loss(NET, x[m].cpu().double(), y[m].cpu().double(), t, P_DROP,
                               O.InjectedNoise({k: v.double() for k, v in nzs[m].items()}))
        (gref,) = torch.autograd.grad(loss, t)
        out = out.detach()
        out_err = ((got["out"][m].cpu().double() - out).abs() / out.abs().clamp_min(1e-3)).max().item()
        cs = _cos(got["grad"][m].cpu().double(), gref)
        print(f"\n[ensemble oracle B={B} member {m}] loss {got['scalars'][m, 0].item():.6e} vs {loss.item():.6e}, "
              f"out err {out_err:.2e}, grad cosine {cs:.6f}")
        assert abs(got["scalars"][m, 0].item() / loss.item() - 1) < 5e-3
        assert out_err < 1e-2
        assert cs > (0.999 if B >= 256 else 0.99)


def _launches(e, fn):
    torch.cuda.synchronize()
    n0 = e.lib.brl_launch_count()
    fn()
    torch.cuda.synchronize()
    return e.lib.brl_launch_count() - n0


def test_members_share_launches(eng):
    from bayesrul_b200 import Noise
    eng.set_step_graph(False)
    try:
        counts = {}
        for M in (1, 5):
            x, y, th = _members(NET, M, 256, seed=400)
            eng.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=2))  # warm-up: workspace growth, kernel attributes
            counts[M] = _launches(eng, lambda: eng.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=2)))
        single = _launches(eng, lambda: eng.hnn_step(x[0], y[0], th[0], P_DROP, Noise(seed=2)))
    finally:
        eng.set_step_graph(True)
    assert eng.tc_status() == 0
    print(f"\n[ensemble launches] M=1: {counts[1]}, M=5: {counts[5]}, hnn_step: {single}")
    assert counts[1] == counts[5] == single > 0


def test_graph_replay_equals_eager(eng):
    from bayesrul_b200 import Noise
    M, B = 4, 128
    th = _members(NET, M, B, seed=500)[2]  # one parameter tensor for the whole sequence: part of the graph key
    steps = [(_members(NET, M, B, seed=510 + 3 * i)[:2], Noise(seed=20 + i, sample0=5 * i)) for i in range(4)]
    replayed = []
    for (x, y), nz in steps + steps:  # first pass: eager, capture, then replays; the second pass replays every step
        r = eng.hnn_step_ensemble(x, y, th, P_DROP, nz)
        replayed.append({k: v.clone() for k, v in r.items()})
    eng.set_step_graph(False)
    try:
        eager = [eng.hnn_step_ensemble(x, y, th, P_DROP, nz) for (x, y), nz in steps]
    finally:
        eng.set_step_graph(True)
    assert eng.tc_status() == 0
    for i, ref in enumerate(eager):
        for got in (replayed[i], replayed[len(steps) + i]):
            for m in range(M):
                _assert_member(got, {k: v[m] for k, v in ref.items()}, m, f"graph step {i}")
    # a new seed draws new masks (same inputs, same sample0)
    (x, y), nz = steps[0]
    other = eng.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=nz.seed + 1000, sample0=nz.sample0))
    for m in range(M):
        assert not torch.allclose(other["out"][m], eager[0]["out"][m], rtol=1e-3), m


@pytest.mark.parametrize("B", [1, 5, 129, 1000])
def test_ragged_batches(eng, B):
    from bayesrul_b200 import Noise
    M = 3
    x, y, th = _members(NET, M, B, seed=600 + B)
    got = eng.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=4, sample0=1))
    refs = _singles(eng, x, y, th, P_DROP, 4, 1)
    assert eng.tc_status() == 0
    for m in range(M):
        _assert_member(got, refs[m], m, f"B={B}")


@pytest.mark.parametrize("net,backend", [("inception", "simt"), ("linear", "fused"), ("conv", "fused")])
def test_member_loop_fallback(net, backend):
    from bayesrul_b200 import Engine, Noise
    e = Engine(net, DEV)
    e.set_gemm_backend(backend)
    M, B = 3, 64
    x, y, th = _members(net, M, B, seed=700)
    got = e.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=6, sample0=2))
    refs = _singles(e, x, y, th, P_DROP, 6, 2)
    e.set_step_graph(False)
    one = _launches(e, lambda: e.hnn_step(x[0], y[0], th[0], P_DROP, Noise(seed=6)))
    loop = _launches(e, lambda: e.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=6)))
    assert e.tc_status() == 0
    assert loop == M * one, (loop, one)
    for m in range(M):
        _assert_member(got, refs[m], m, f"{net}/{backend}")


def test_one_lane_workspace_and_too_small(eng):
    from bayesrul_b200 import Noise
    M, B = 3, 256
    x, y, th = _members(NET, M, B, seed=800)
    refs = _singles(eng, x, y, th, P_DROP, 8, 0)

    def call(nbytes):
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=DEV)
        sc = torch.empty(M, 2, dtype=torch.float64, device=DEV)
        out, grad = torch.empty(M, B, 2, device=DEV), torch.empty(M, eng.P, device=DEV)
        nz, keep = eng._noise(Noise(seed=8))
        rc = eng.lib.brl_hnn_step_ensemble(eng.ctx, x.data_ptr(), y.data_ptr(), M, B, th.data_ptr(), P_DROP, nz, 1, sc.data_ptr(),
                                           grad.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), eng._stream())
        torch.cuda.synchronize()
        return rc, dict(scalars=sc, out=out, grad=grad)

    one_lane = eng.lib.brl_workspace_bytes(eng.ctx, B, 1, 1, 0)
    assert one_lane < eng.lib.brl_workspace_bytes(eng.ctx, B, M, 3, 0)
    eng.set_step_graph(False)
    try:
        single = _launches(eng, lambda: eng.hnn_step(x[0], y[0], th[0], P_DROP, Noise(seed=8)))
        n0 = eng.lib.brl_launch_count()
        rc, got = call(one_lane)
        loop = eng.lib.brl_launch_count() - n0
        rc_small, _ = call(1 << 16)
    finally:
        eng.set_step_graph(True)
    assert rc == 0 and eng.tc_status() == 0
    assert loop == M * single, (loop, single)  # one member after another
    for m in range(M):
        _assert_member(got, refs[m], m, "one-lane workspace")
    assert rc_small != 0 and "workspace too small" in eng.lib.brl_last_error().decode()
    with pytest.raises(RuntimeError):
        eng.hnn_step_ensemble(x[:, :, :, :17].contiguous(), y, th)
    with pytest.raises(RuntimeError):
        eng.hnn_step_ensemble(x, y[:2], th)
    with pytest.raises(RuntimeError):
        eng.hnn_step_ensemble(x, y, th[:2])


def test_compute_grads_false(eng):
    from bayesrul_b200 import Noise
    x, y, th = _members(NET, 5, 256, seed=900)
    a = eng.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=3))
    b = eng.hnn_step_ensemble(x, y, th, P_DROP, Noise(seed=3), compute_grads=False)
    assert b["grad"] is None and eng.tc_status() == 0
    assert torch.allclose(a["scalars"], b["scalars"], rtol=1e-5, atol=0)
    assert torch.allclose(a["out"], b["out"], rtol=1e-5, atol=1e-6)


def test_adam_training_matches_independent_members(eng):
    """Ten Adam steps over one [5, P] parameter follow five independent hnn_step + Adam runs; a trained member then loads into
    compat.nets.Inception."""
    from bayesrul_b200 import Noise
    from bayesrul_b200.compat.nets import Inception
    M, B, steps = 5, 256, 10
    x, y, th0 = _members(NET, M, B, seed=1000)
    ens = torch.nn.Parameter(th0.clone())
    opt = torch.optim.Adam([ens], lr=1e-3)
    ind = [torch.nn.Parameter(th0[m].clone()) for m in range(M)]
    opts = [torch.optim.Adam([t], lr=1e-3) for t in ind]
    for k in range(steps):
        r = eng.hnn_step_ensemble(x, y, ens.data, P_DROP, Noise(seed=40 + k))
        ens.grad = r["grad"]
        opt.step()
        for m in range(M):
            s = eng.hnn_step(x[m], y[m], ind[m].data, P_DROP, Noise(seed=40 + k, sample0=m))
            ind[m].grad = s["grad"]
            opts[m].step()
            rel = abs(r["scalars"][m, 0].item() / s["scalars"][0].item() - 1)
            assert rel < 1e-3, (k, m, rel)
    assert eng.tc_status() == 0
    final = eng.hnn_step_ensemble(x, y, ens.data, 0.0, compute_grads=False)
    net = Inception(30, 18).to(DEV).eval()
    for m in (0, M - 1):
        with torch.no_grad():
            net.theta.copy_(ens.data[m])
            out = net(x[m])
        err = ((out - final["out"][m]).abs() / final["out"][m].abs().clamp_min(1e-3)).max().item()
        assert err < 1e-2, (m, err)
