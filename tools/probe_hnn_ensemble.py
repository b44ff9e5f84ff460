"""Replayed deep-ensemble HNN training step: M members in one hnn_step_ensemble + one clipped_adam over M x P, against M
sequential hnn_step + clipped_adam calls, on the fused back-end (Inception).

    python tools/probe_hnn_ensemble.py [B ...]

M in {1, 2, 5, 8}, B in {64, 256, 1024} (or the given sizes), p in {0, 0.241437}; CUDA events around 200 steps after warm-up,
median of 3 alternated repeats; the device name, power limit and max SM clock read in the same run.  "launches" counts the
library's kernel launches of one step of each (graph replays included): the ensemble step issues those of ONE member."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200 import Engine, Noise
from bayesrul_b200.compat.nets import init_flat_params

dev = torch.device("cuda", 0)
sizes = [int(a) for a in sys.argv[1:]] or [64, 256, 1024]
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
except OSError:
    q = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(dev)} | {q}")
eng = Engine("inception", dev)
eng.set_gemm_backend("fused")
P = eng.P
for B in sizes:
    for p in (0.0, 0.241437):
        for M in (1, 2, 5, 8):
            g = torch.Generator().manual_seed(1)
            x = torch.randn(M, B, 30, 18, generator=g).to(dev)
            y = (torch.rand(M, B, generator=g) * 100).to(dev)
            th0 = torch.stack([init_flat_params("inception", 12345 + m) for m in range(M)]).to(dev)
            th_e, th_s = th0.clone(), th0.clone()
            opt_e = [torch.zeros_like(th0) for _ in range(2)]
            opt_s = [torch.zeros_like(th0) for _ in range(2)]
            it = {"ens": 0, "seq": 0}

            def ens():
                it["ens"] += 1
                r = eng.hnn_step_ensemble(x, y, th_e, p, Noise(seed=5000 + it["ens"]))
                eng.clipped_adam(th_e, r["grad"], opt_e[0], opt_e[1], it["ens"], 1e-3, (0.95, 0.999), 1e-8, 15.0)
                return r

            def seq():
                it["seq"] += 1
                for m in range(M):
                    r = eng.hnn_step(x[m], y[m], th_s[m], p, Noise(seed=5000 + it["seq"], sample0=m))
                    eng.clipped_adam(th_s[m], r["grad"], opt_s[0][m], opt_s[1][m], it["seq"], 1e-3, (0.95, 0.999), 1e-8, 15.0)
                return r

            steps = {"ens": ens, "seq": seq}
            for f in steps.values():
                for _ in range(10):
                    f()
            torch.cuda.synchronize()
            times = {k: [] for k in steps}
            for _ in range(3):  # alternated repeats
                for k, f in steps.items():
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    n = 200
                    a.record()
                    for _ in range(n):
                        f()
                    b.record()
                    torch.cuda.synchronize()
                    times[k].append(a.elapsed_time(b) / n)
            med = {k: sorted(v)[1] for k, v in times.items()}
            nl = {}
            for k, f in steps.items():
                n0 = eng.lib.brl_launch_count()
                f()
                nl[k] = eng.lib.brl_launch_count() - n0
            spread = {k: (max(v) - min(v)) / sorted(v)[1] for k, v in times.items()}
            dl = (th_e - th_s).abs().max().item()
            print(f"B={B:5d} p={p:.3f} M={M}: ensemble {med['ens']:.4f} ms/step, {M} x hnn_step {med['seq']:.4f} ms/step, "
                  f"speed-up {med['seq'] / med['ens']:.2f}x | spread {spread['ens']:.1%} / {spread['seq']:.1%} | "
                  f"launches {nl['ens']} / {nl['seq']} | max |theta diff| after {it['ens']} steps {dl:.2e} | status {eng.tc_status()}")
eng.set_gemm_backend("simt")
