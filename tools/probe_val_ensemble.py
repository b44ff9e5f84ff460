"""Validation of the M seeds of a BNN experiment: M Engine.elbo_val_steps calls against one ensemble call.

    python tools/probe_val_ensemble.py [N]

On a synthetic N-window split on the device (default 60 000: 600 batches of 100, 240 of 250), each case validates M = 5 Inception
BNNs (normal guide, one ELBO particle, S = 8 predictive draws, ELBO on the fused back-end) over the same in-order full batches two
ways, CUDA events around each, and reports ms per batch (all five members):
  (a) M sequential Engine.elbo_val_steps calls, one per member with its [P] loc / scale;
  (b) one Engine.elbo_val_steps call with the [M,P] loc / scale (brl_elbo_val_steps_ensemble).
Cases: B = 100 and 250, with the tensor-core and the fp32 SIMT predictive engine.  Each path has its own Engine (its own workspace
and graphs) and is warmed up first (module loads, captured batches); each time is the median of three epochs.  Member 0 draws at
the same MC-sample indices in both paths, so its rows must agree to the run-to-run spread of the ELBO's atomics; the largest
relative difference is printed as a check.  The device name, power limit and max SM clock are read in the same run."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200 import Engine
from oracle import bnn_oracle as O

dev = torch.device("cuda", 0)
N = int(sys.argv[1]) if len(sys.argv) > 1 else 60000
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
except OSError:
    q = "nvidia-smi unavailable"
print(f"device: {torch.cuda.get_device_name(dev)} | {q}", flush=True)
g = torch.Generator().manual_seed(0)
X = torch.randn(N, 30, 18, generator=g).to(dev)
Y = (torch.rand(N, generator=g) * 100).to(dev)
M, S = 5, 8
CASES = [(100, "tc"), (250, "tc"), (100, "simt"), (250, "simt")]  # B, predictive engine
loc = torch.stack([O.init_params("inception", 1 + m) for m in range(M)]).to(dev)
scale = torch.full_like(loc, 0.02) * (1 + 0.1 * torch.rand(loc.shape, generator=g).to(dev))
KW = dict(guide="normal", particles=1, S=S, prior_loc=0.0, prior_scale=0.138793, dataset_size=238150, seed=7)


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), r


def engine():
    e = Engine("inception", dev)
    e.set_gemm_backend("fused")
    return e


for B, eng in CASES:
    K = N // B
    xs, ys = X[: K * B], Y[: K * B]
    idx = torch.arange(K * B, device=dev).view(K, B)
    ea, eb = engine(), engine()
    seq = lambda ix: [ea.elbo_val_steps(xs, ys, ix, loc[m], scale[m], engine=eng, **KW) for m in range(M)]
    one = lambda ix: eb.elbo_val_steps(xs, ys, ix, loc, scale, engine=eng, **KW)
    seq(idx[:20])  # warm-up: every member's batch graph is captured here and replayed below
    one(idx[:20])
    runs_a = [timed(lambda: seq(idx)) for _ in range(3)]
    runs_b = [timed(lambda: one(idx)) for _ in range(3)]
    ms_a = sorted(t for t, _ in runs_a)[1] / K
    ms_b = sorted(t for t, _ in runs_b)[1] / K
    ra, rb = runs_a[0][1][0], runs_b[0][1]
    diff = max(((rb[key][:, 0] - ra[key]).abs().max() / ra[key].abs().max()).item() for key in ("scalars", "metrics"))
    ok = bool(torch.isfinite(rb["scalars"]).all() and torch.isfinite(rb["metrics"]).all())
    print(f"Inception M={M} B={B:4d} S={S} engine={eng:4s} K={K:4d}: (a) {M} calls {ms_a:.4f} ms/batch | (b) one call {ms_b:.4f} "
          f"ms/batch | (a)/(b) {ms_a / ms_b:.2f}x | member 0 max rel diff {diff:.2e} | finite {ok}", flush=True)
    del ea, eb
    torch.cuda.empty_cache()
