"""Replayed BNN training step over the seeds of an experiment: M variational posteriors in one elbo_step_ensemble + one
clipped_adam_vi over M x P, against M sequential elbo_step + clipped_adam_vi calls, on the fused back-end (Inception).

    python tools/probe_elbo_ensemble.py [B ...]

M in {1, 2, 5, 8}, B in {100, 256, 1024} (or the given sizes), three configurations: LRT with 1 particle, Flipout with 2, the
radial guide with 1; CUDA events around 200 steps after warm-up, median of 3 alternated repeats; the device name, power limit
and max SM clock read in the same run.  "launches" counts the library's kernel launches of one step of each (graph replays
included): the ensemble step issues those of ONE member."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200 import Engine, Noise
from bayesrul_b200.compat.nets import init_flat_params

dev = torch.device("cuda", 0)
sizes = [int(a) for a in sys.argv[1:]] or [100, 256, 1024]
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
except OSError:
    q = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(dev)} | {q}")
eng = Engine("inception", dev)
eng.set_gemm_backend("fused")
P = eng.P
KW = dict(prior_loc=0.0, prior_scale=0.138793, dataset_size=238150)
CONFIGS = [("lrt", "normal", 1), ("flipout", "normal", 2), ("lrt", "radial", 1)]


def state(M):
    loc = torch.stack([init_flat_params("inception", 12345 + m) for m in range(M)]).to(dev)
    ls = torch.full_like(loc, -4.0)
    return [loc, ls, ls.exp()] + [torch.zeros_like(loc) for _ in range(4)]  # loc, log_scale, scale, m_loc, v_loc, m_ls, v_ls


for B in sizes:
    for mode, guide, particles in CONFIGS:
        for M in (1, 2, 5, 8):
            g = torch.Generator().manual_seed(1)
            x = torch.randn(M, B, 30, 18, generator=g).to(dev)
            y = (torch.rand(M, B, generator=g) * 100).to(dev)
            se, ss = state(M), state(M)
            it = {"ens": 0, "seq": 0}
            kw = dict(mode=mode, guide=guide, particles=particles, **KW)

            def ens():
                it["ens"] += 1
                r = eng.elbo_step_ensemble(x, y, se[0], se[2], noise=Noise(seed=5000 + it["ens"]), **kw)
                eng.clipped_adam_vi(se[0], se[1], se[2], r["grad_mu"], r["grad_log_sigma"], *se[3:], step=it["ens"], lr=1e-3)
                return r

            def seq():
                it["seq"] += 1
                for m in range(M):
                    r = eng.elbo_step(x[m], y[m], ss[0][m], ss[2][m], noise=Noise(seed=5000 + it["seq"], sample0=m * particles), **kw)
                    eng.clipped_adam_vi(ss[0][m], ss[1][m], ss[2][m], r["grad_mu"], r["grad_log_sigma"], *[t[m] for t in ss[3:]],
                                        step=it["seq"], lr=1e-3)
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
            dl = (se[0] - ss[0]).abs().max().item()
            print(f"B={B:5d} {mode}/{guide} particles={particles} M={M}: ensemble {med['ens']:.4f} ms/step, "
                  f"{M} x elbo_step {med['seq']:.4f} ms/step, speed-up {med['seq'] / med['ens']:.2f}x | "
                  f"spread {spread['ens']:.1%} / {spread['seq']:.1%} | launches {nl['ens']} / {nl['seq']} | "
                  f"max |loc diff| after {it['ens']} steps {dl:.2e} | status {eng.tc_status()}", flush=True)
eng.set_gemm_backend("simt")
