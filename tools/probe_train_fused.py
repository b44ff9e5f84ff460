"""Replayed training-step time (graph replay + the optimizer step) of the fp32 FFMA back-end vs the level-fused tcgen05 back-end.

    python tools/probe_train_fused.py [B] [net]

net = inception (default): ELBO step (LRT 1 particle, Flipout 2 particles) at B (default 256) on simt / fused.
net = linear / conv: at B = 64 / 256 / 1024 (or the given B) the ELBO step (LRT 1 particle, Flipout 2 particles, weight sampling
with the radial guide) + clipped_adam_vi and hnn_step at p = 0.3 + clipped_adam, on simt / tc / fused; CUDA events around
200 steps after warm-up, median of 3 alternated repeats; the device name and power limit; at each size the fused-vs-fp32 loss
ratio and gradient cosine of the first step."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200 import Engine, Noise
from bayesrul_b200.compat.nets import init_flat_params

dev = torch.device("cuda", 0)
B_arg = int(sys.argv[1]) if len(sys.argv) > 1 and int(sys.argv[1]) > 0 else None
net = sys.argv[2] if len(sys.argv) > 2 else "inception"


def inception():
    eng = Engine("inception", dev)
    B = B_arg or 256
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 30, 18, generator=g).to(dev)
    y = (torch.rand(B, generator=g) * 100).to(dev)
    mu0 = init_flat_params("inception", 12345).to(dev)
    for mode, particles, q, ps in (("lrt", 1, 1.351e-3, 0.138793), ("flipout", 2, 2.14e-4, 0.198768)):
        for backend in ("simt", "fused"):
            eng.set_gemm_backend(backend)
            mu = mu0.clone(); ls = torch.full_like(mu, float(torch.log(torch.tensor(q)))); sg = torch.full_like(mu, q)
            opt = [torch.zeros_like(mu) for _ in range(4)]
            it = [0]
            def step():
                it[0] += 1
                r = eng.elbo_step(x, y, mu, sg, mode=mode, guide="normal", particles=particles, prior_loc=0.0, prior_scale=ps,
                                  dataset_size=238150, noise=Noise(seed=5000 + it[0]))
                eng.clipped_adam_vi(mu, ls, sg, r["grad_mu"], r["grad_log_sigma"], *opt, it[0], 1e-3, (0.95, 0.999), 1e-8, 15.0)
                return r
            for _ in range(10): r = step()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 200
            a.record()
            for _ in range(n): r = step()
            b.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(b) / n
            print(f"{mode:8s} {backend:6s} B={B}: {ms:.4f} ms/step  {B / ms:.0f} k windows/s  loss {r['scalars'][0].item():.5f}  status {eng.tc_status()}")
    eng.set_gemm_backend("simt")


def small_net(name):
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    except OSError:
        q = "nvidia-smi unavailable"
    print(f"device: {torch.cuda.get_device_name(dev)} | {q}")
    eng = Engine(name, dev)
    mu0 = init_flat_params(name, 12345).to(dev)
    cases = (("lrt", 1, "normal", 1.351e-3, 0.138793), ("flipout", 2, "normal", 2.14e-4, 0.198768), ("ws", 1, "radial", 1.351e-3, 0.138793),
             ("hnn", 1, None, 0.0, 0.0))
    for B in ([B_arg] if B_arg else [64, 256, 1024]):
        g = torch.Generator().manual_seed(1)
        x = torch.randn(B, 30, 18, generator=g).to(dev)
        y = (torch.rand(B, generator=g) * 100).to(dev)
        for mode, particles, guide, q, ps in cases:
            steps, first = {}, {}
            for backend in ("simt", "tc", "fused"):
                mu = mu0.clone(); opt = [torch.zeros_like(mu) for _ in range(4)]
                ls = torch.full_like(mu, float(torch.log(torch.tensor(max(q, 1e-30))))); sg = torch.full_like(mu, q)
                it = [0]
                def step(backend=backend, mu=mu, ls=ls, sg=sg, opt=opt, it=it):
                    eng.set_gemm_backend(backend)
                    it[0] += 1
                    if mode == "hnn":
                        r = eng.hnn_step(x, y, mu, 0.3, Noise(seed=5000 + it[0]))
                        eng.clipped_adam(mu, r["grad"], opt[0], opt[1], it[0], 1e-3, (0.95, 0.999), 1e-8, 15.0)
                    else:
                        r = eng.elbo_step(x, y, mu, sg, mode=mode, guide=guide, particles=particles, prior_loc=0.0, prior_scale=ps,
                                          dataset_size=238150, noise=Noise(seed=5000 + it[0]))
                        eng.clipped_adam_vi(mu, ls, sg, r["grad_mu"], r["grad_log_sigma"], *opt, it[0], 1e-3, (0.95, 0.999), 1e-8, 15.0)
                    return r
                r = step()
                first[backend] = (r["scalars"][0].item(), (r["grad"] if mode == "hnn" else r["grad_mu"]).double().clone())
                for _ in range(10): step()
                steps[backend] = step
            torch.cuda.synchronize()
            times = {b: [] for b in steps}
            for _ in range(3):  # alternated repeats
                for backend, step in steps.items():
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    n = 200
                    a.record()
                    for _ in range(n): step()
                    b.record(); torch.cuda.synchronize()
                    times[backend].append(a.elapsed_time(b) / n)
            med = {k: sorted(v)[1] for k, v in times.items()}
            l0, g0 = first["simt"]
            lf, gf = first["fused"]
            cs = float((gf * g0).sum() / (gf.norm() * g0.norm()))
            name = f"{mode}{'' if mode == 'hnn' else f' P={particles}'}{' radial' if guide == 'radial' else ''}"
            print(f"B={B:5d} {name:14s} ms/step simt {med['simt']:.4f} tc {med['tc']:.4f} fused {med['fused']:.4f} | "
                  f"fused/simt loss {lf / l0:.6f} grad cosine {cs:.6f} | status {eng.tc_status()}")
    eng.set_gemm_backend("simt")


small_net(net) if net in ("linear", "conv") else inception()
