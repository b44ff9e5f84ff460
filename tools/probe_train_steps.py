"""K training steps per call over a device-resident split, against the per-step loops a training run issues today.

    python tools/probe_train_steps.py [K] [B ...]

On a synthetic 238 150-window split (514 MB on the device), K = 2000 steps (or the given K) of each configuration: LRT,
Flipout with 2 particles, the radial guide, the M = 5 seeds of LRT (all Inception, fused back-end) and the HNN deep ensemble
with M = 5 and p = 0.241437; at B = 100 and 256 (or the given sizes).  Three versions of the same steps, CUDA events around
each:
  (a) the compat per-batch loop: BNN.training_step (svi.step + the logged metrics, with their .item() reads) per batch and
      per seed; for the HNN, the Engine per-step loop (hnn_step_ensemble + clipped_adam + step_metrics_ensemble) with one
      .item() per step.  The batches are gathered from the device-resident split (X[idx[k]]), so no host copy is timed;
  (b) the Engine per-step loop without any synchronisation: elbo_step{,_ensemble} / hnn_step_ensemble + the optimizer + the
      step metrics per step;
  (c) ONE Engine.elbo_train_steps / hnn_train_steps call over the K steps (after a short warm-up call that captures its graph).
Also the host time of call (c) per step (index check included), and the device name, power limit and max SM clock, read in
the same run."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200 import Engine, Noise
from bayesrul_b200.compat import BNN, Inception, pyro_shim
from bayesrul_b200.compat.nets import init_flat_params

dev = torch.device("cuda", 0)
K = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
sizes = [int(a) for a in sys.argv[2:]] or [100, 256]
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
except OSError:
    q = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(dev)} | {q}", flush=True)
N = 238150
W = 0x9E3779B97F4A7C15
KW = dict(prior_loc=0.0, prior_scale=0.138793, dataset_size=N)
OPT = dict(lr=0.000857, betas=(0.95, 0.999), eps=1e-8, clip_norm=15.0, lrd=1.0, weight_decay=0.0)
HOPT = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, clip_norm=1e30, lrd=1.0, weight_decay=0.0)
P_MCD = 0.241437
g = torch.Generator().manual_seed(0)
X = torch.randn(N, 30, 18, generator=g).to(dev)
Y = (torch.rand(N, generator=g) * 100).to(dev)
CASES = [  # name, kind, fit context, guide, particles, M
    ("LRT", "elbo", "lrt", "normal", 1, 1),
    ("Flipout x2", "elbo", "flipout", "normal", 2, 1),
    ("radial", "elbo", None, "radial", 1, 1),
    ("LRT, M=5 seeds", "elbo", "lrt", "normal", 1, 5),
    ("HNN p=0.241437, M=5", "hnn", None, None, 1, 5),
]


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def vi_state(M):
    loc = torch.stack([init_flat_params("inception", 12345 + m) for m in range(M)]).to(dev)
    ls = torch.full_like(loc, -6.6)
    return [loc, ls, ls.exp()] + [torch.zeros_like(loc) for _ in range(4)]


def bnn_model(ctx, guide, particles, seed):
    torch.manual_seed(seed)
    net = Inception(30, 18)
    with torch.no_grad():
        net.last.bias.fill_(3.0)
    m = BNN(net, pyro_shim.ClippedAdam(dict(OPT)), pretrain_epochs=5, mc_samples_train=particles, mc_samples_eval=8,
            dataset_size=N, fit_context=ctx, prior_loc=0.0, prior_scale=0.138793, guide=guide, q_scale=1.351e-3, device=dev)
    m.on_fit_start()
    return m


def logged(e, out, yb, particles):
    M = yb.shape[0]
    lo = torch.stack([out[m, 0] if particles == 1 else e.aggregate_predictions(out[m]) for m in range(M)])
    return e.step_metrics_ensemble(lo[..., 0].contiguous(), lo[..., 1].contiguous(), yb)


for B in sizes:
    for name, kind, ctx, guide, particles, M in CASES:
        idx = torch.stack([torch.randperm(N, device=dev)[: M * B].view(M, B) for _ in range(K)])
        mode = "ws" if (ctx is None or guide == "radial") else ctx
        eb, ec = Engine("inception", dev), Engine("inception", dev)
        for e in (eb, ec):
            e.set_gemm_backend("fused")
        res = {}
        if kind == "elbo":
            models = [bnn_model(ctx, guide, particles, 12345 + m) for m in range(M)]
            sb, sc = vi_state(M), vi_state(M)

            def run_a(n=K):
                for k in range(n):
                    xb, yb = X[idx[k]], Y[idx[k]]
                    for m, mdl in enumerate(models):
                        mdl.training_step((xb[m], yb[m]), k)

            def run_b(n=K):
                for k in range(n):
                    xb, yb = X[idx[k]], Y[idx[k]]
                    nz = Noise(seed=(7 + W * (k + 1)) & 0xFFFFFFFFFFFFFFFF)
                    if M == 1:
                        r = eb.elbo_step(xb[0], yb[0], sb[0][0], sb[2][0], mode=mode, guide=guide, particles=particles, noise=nz, **KW)
                        out = r["out"].unsqueeze(0)
                    else:
                        r = eb.elbo_step_ensemble(xb, yb, sb[0], sb[2], mode=mode, guide=guide, particles=particles, noise=nz, **KW)
                        out = r["out"]
                    eb.clipped_adam_vi(sb[0], sb[1], sb[2], r["grad_mu"], r["grad_log_sigma"], *sb[3:], step=k + 1, **OPT)
                    logged(eb, out, yb, particles)

            def run_c(n=K):
                return ec.elbo_train_steps(X, Y, idx[:n], sc[0], sc[1], sc[2], sc[3:], step0=0, mode=mode, guide=guide,
                                           particles=particles, seed=7, **OPT, **KW)
        else:
            th = lambda: torch.stack([init_flat_params("inception", 99 + m) for m in range(M)]).to(dev)
            sa, sb, sc = [[th(), None, None] for _ in range(3)]
            for s in (sa, sb, sc):
                s[1], s[2] = torch.zeros_like(s[0]), torch.zeros_like(s[0])

            def hnn_loop(e, s, n, sync):
                for k in range(n):
                    xb, yb = X[idx[k]], Y[idx[k]]
                    r = e.hnn_step_ensemble(xb, yb, s[0], P_MCD, Noise(seed=(7 + W * (k + 1)) & 0xFFFFFFFFFFFFFFFF))
                    e.clipped_adam(s[0], r["grad"], s[1], s[2], k + 1, **HOPT)
                    logged(e, r["out"].unsqueeze(1), yb, 1)
                    if sync:
                        r["scalars"][0, 0].item()

            ea = Engine("inception", dev)
            ea.set_gemm_backend("fused")
            run_a = lambda n=K: hnn_loop(ea, sa, n, True)
            run_b = lambda n=K: hnn_loop(eb, sb, n, False)
            run_c = lambda n=K: ec.hnn_train_steps(X, Y, idx[:n], sc[0], (sc[1], sc[2]), step0=0, p_dropout=P_MCD, seed=7, **HOPT)
        for f in (run_a, run_b, run_c):  # warm-up: module loads, graph captures
            f(20)
        torch.cuda.synchronize()
        ms = {"a": timed(run_a) / K, "b": timed(run_b) / K}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = run_c()
        host = (time.perf_counter() - t0) * 1e3 / K
        b.record()
        torch.cuda.synchronize()
        ms["c"] = a.elapsed_time(b) / K
        ms_b2 = timed(run_b) / K  # (b) again after (c): the run-to-run spread of the per-step loop
        ok = bool(torch.isfinite(r["scalars"]).all())
        print(f"B={B:4d} {name:22s}: (a) compat loop {ms['a']:.4f} ms/step | (b) Engine loop {ms['b']:.4f} / {ms_b2:.4f} ms/step | "
              f"(c) one call {ms['c']:.4f} ms/step, host {host:.4f} ms/step | (a)/(c) {ms['a'] / ms['c']:.2f}x, "
              f"(b)/(c) {min(ms['b'], ms_b2) / ms['c']:.2f}x | finite {ok}", flush=True)
        del eb, ec
