"""Test-time evaluation of M models over one batch: one predict_moments_ensemble + one step_metrics_ensemble call against M
sequential predict_moments + step_metrics calls, on the tensor-core engine.

    python tools/probe_predict_ensemble.py [B ...]

M in {1, 2, 5, 8}, B in {100, 1000, 10000} (or the given sizes), S in {20, 100}; cases: Inception with the normal guide, the
radial guide and MC-dropout (p = 0.241437), Linear and Conv-D3 with the normal guide.  CUDA events around a window of about
0.2 s per variant after warm-up, median of 3 alternated repeats and their spread; the device name, power limit and max SM clock
read in the same run.  "launches" counts the library's kernel launches of one evaluation of each variant."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200 import Engine, Noise
from bayesrul_b200.compat.nets import init_flat_params

dev = torch.device("cuda", 0)
sizes = [int(a) for a in sys.argv[1:]] or [100, 1000, 10000]
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
except OSError:
    q = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(dev)} | {q}", flush=True)
P_DROP = 0.241437
CASES = [("inception", "normal", 0.0), ("inception", "radial", 0.0), ("inception", None, P_DROP), ("linear", "normal", 0.0),
         ("conv", "normal", 0.0)]
engines = {}


def timed(f, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        f()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


for net, guide, p in CASES:
    eng = engines.setdefault(net, Engine(net, dev))
    for B in sizes:
        for S in (20, 100):
            for M in (1, 2, 5, 8):
                g = torch.Generator().manual_seed(1)
                x = torch.randn(B, 30, 18, generator=g).to(dev)
                y = (torch.rand(M, B, generator=g) * 100).to(dev)
                mu = torch.stack([init_flat_params(net, 12345 + m) for m in range(M)]).to(dev)
                sg = torch.full_like(mu, 0.02) if guide else None

                def ens():
                    r = eng.predict_moments_ensemble(x, mu, sg, S=S, guide=guide, p_dropout=p, noise=Noise(seed=5), engine="tc")
                    return r, eng.step_metrics_ensemble(r[0], r[1], y)

                def loop():
                    for m in range(M):
                        r = eng.predict_moments(x, mu[m], sg[m] if guide else None, S=S, guide=guide, p_dropout=p,
                                                noise=Noise(seed=5, sample0=m * S), engine="tc")
                        eng.step_metrics(r[0], r[1], y[m])
                    return r

                variants = {"ens": ens, "loop": loop}
                n = {}
                for k, f in variants.items():
                    for _ in range(3):
                        f()
                    torch.cuda.synchronize()
                    n[k] = max(3, min(500, int(200.0 / max(timed(f, 3), 1e-3))))
                times = {k: [] for k in variants}
                for _ in range(3):  # alternated repeats
                    for k, f in variants.items():
                        times[k].append(timed(f, n[k]))
                med = {k: sorted(v)[1] for k, v in times.items()}
                spread = {k: (max(v) - min(v)) / sorted(v)[1] for k, v in times.items()}
                nl = {}
                for k, f in variants.items():
                    torch.cuda.synchronize()
                    n0 = eng.lib.brl_launch_count()
                    f()
                    torch.cuda.synchronize()
                    nl[k] = eng.lib.brl_launch_count() - n0
                print(f"{net:9s} {guide or 'mc-dropout':10s} B={B:5d} S={S:3d} M={M}: ensemble {med['ens']:.4f} ms, "
                      f"{M} x single {med['loop']:.4f} ms, speed-up {med['loop'] / med['ens']:.2f}x | "
                      f"spread {spread['ens']:.1%} / {spread['loop']:.1%} | launches {nl['ens']} / {nl['loop']} | "
                      f"status {eng.tc_status()}", flush=True)
