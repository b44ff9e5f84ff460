"""HNN training with torch.optim.Adam: the compat per-batch loop against HNN.fit_epoch / one K-step call.

    python tools/probe_hnn_fit_epoch.py [K]

On a synthetic 238 150-window split on the device, each case runs K = 2000 steps (or the given K) two ways, CUDA events around
each, and reports ms per step:
  (a) the compat per-batch loop, as Lightning's automatic optimisation runs it: HNN.training_step (the fused step and the logged
      metrics), zero_grad, backward and torch.optim.Adam.step (default foreach path) per batch.  Batches are gathered from the
      device-resident split, so no host copy is timed;
  (b) HNN.fit_epoch over the first K * B windows (one Engine.hnn_train_steps(optimizer="adam") call), or, where K * B exceeds
      the split, over the whole split (floor(N / B) steps; K then shrinks to that).
Cases: the Inception net at p = 0.241437 (B = 100 and 250) and p = 0 (B = 250); the Linear and Conv-D3 nets on the fused
back-end (p = 0.241437, B = 100); and five deep-ensemble members (Inception, p = 0.241437, B = 100), five compat loops against
one Engine.hnn_train_steps(optimizer="adam") call over [5, P].  The device name, power limit and max SM clock are read in the
same run."""
import os
import subprocess
import sys
from functools import partial

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200.compat import HNN, Conv, Inception, Linear

dev = torch.device("cuda", 0)
K0 = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
except OSError:
    q = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(dev)} | {q}", flush=True)
N = 238150
P_MCD = 0.241437
g = torch.Generator().manual_seed(0)
X = torch.randn(N, 30, 18, generator=g).to(dev)
Y = (torch.rand(N, generator=g) * 100).to(dev)
NETS = {"inception": Inception, "linear": Linear, "conv": Conv}
CASES = [  # name, net, p, B, members, train back-end
    ("Inception p=0.241437", "inception", P_MCD, 100, 1, "auto"),
    ("Inception p=0.241437", "inception", P_MCD, 250, 1, "auto"),
    ("Inception p=0", "inception", 0.0, 250, 1, "auto"),
    ("Linear p=0.241437 fused", "linear", P_MCD, 100, 1, "fused"),
    ("Conv-D3 p=0.241437 fused", "conv", P_MCD, 100, 1, "fused"),
    ("Inception p=0.241437, M=5", "inception", P_MCD, 100, 5, "auto"),
]


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def model(net, p, backend, seed):
    torch.manual_seed(seed)
    m = HNN(NETS[net](30, 18, dropout=p), partial(torch.optim.Adam, lr=1e-3), mc_samples=10, p_dropout=p, device=dev,
            train_backend=backend)
    return m, m.configure_optimizers()


def lightning_loop(pairs, batches):
    for i, b in enumerate(batches):
        xb, yb = X[b], Y[b]
        for m, opt in pairs:
            loss = m.training_step((xb, yb), i)
            opt.zero_grad()
            loss.backward()
            opt.step()


for name, net, p, B, M, backend in CASES:
    K = min(K0, N // B)
    perm = torch.randperm(N, device=dev)
    batches = [perm[k * B: (k + 1) * B] for k in range(K)]
    loops = [model(net, p, backend, 12345 + m) for m in range(M)]
    lightning_loop(loops, batches[:20])  # warm-up: module loads, step graphs
    ms_a = timed(lambda: lightning_loop(loops, batches)) / K
    if M == 1:
        m, opt = model(net, p, backend, 12345)
        m.fit_epoch(X[: 20 * B], Y[: 20 * B], B, opt)  # warm-up: the K-step graph is captured here and replayed below
        xs, ys = X[: K * B], Y[: K * B]
        ms_b = timed(lambda: m.fit_epoch(xs, ys, B, opt)) / K
        ok = bool(torch.isfinite(m.net.theta).all())
    else:
        from bayesrul_b200 import Engine
        e = Engine(net, dev)
        e.set_gemm_backend("fused")
        theta = torch.stack([model(net, p, backend, 12345 + i)[0].net.flat().detach().clone() for i in range(M)])
        mv = (torch.zeros_like(theta), torch.zeros_like(theta))
        idx = torch.stack([torch.randperm(N, device=dev)[: M * B].view(M, B) for _ in range(K)])
        call = lambda n, s0: e.hnn_train_steps(X, Y, idx[:n], theta, mv, step0=s0, lr=1e-3, p_dropout=p, seed=7, optimizer="adam")
        call(20, 0)
        ms_b = timed(lambda: call(K, 20)) / K
        ok = bool(torch.isfinite(theta).all())
    print(f"{name:28s} B={B:4d} K={K:5d}: (a) compat loop {ms_a:.4f} ms/step | (b) one call {ms_b:.4f} ms/step | "
          f"(a)/(b) {ms_a / ms_b:.2f}x | finite {ok}", flush=True)
    del loops
