"""BNN validation epoch: the compat loop of validation_step against BNN.validate_epoch (one Engine.elbo_val_steps call).

    python tools/probe_val_epoch.py [N]

On a synthetic N-window split on the device (default 60 000: 600 batches of 100, 240 of 250), each case runs one validation
epoch over the in-order full batches two ways, CUDA events around each, and reports ms per batch:
  (a) the compat loop, as Lightning's validation loop runs it: BNN.validation_step per batch (svi.evaluate_loss with its .item()
      read, the kl read, bnn.predict with mc_samples_eval draws and the aggregate, step_metrics).  Batches are sliced from the
      device-resident split, so no host copy is timed;
  (b) BNN.validate_epoch over the same batches: one Engine.elbo_val_steps call.
Cases: the Inception BNN (LRT fit context, normal guide, mc_samples_train = 1, mc_samples_eval = 8, ELBO on the fused back-end) at
B = 100 and 250, with the tensor-core and the fp32 SIMT predictive engine.  Both paths are warmed up first (module loads, the
ELBO step graph of the loop, the call's captured batch).  Then the host enqueue time of one Engine.elbo_val_steps call over
the same batches, with step graphs on and off (the call returns before the GPU is done; the index check is its one
synchronisation, before the launches).  The device name, power limit and max SM clock are read in the same run."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bayesrul_b200.compat import BNN, Inception, pyro_shim

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
CASES = [(100, "tc"), (250, "tc"), (100, "simt"), (250, "simt")]  # B, predictive engine
S_EVAL = 8


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def model(engine):
    torch.manual_seed(12345)
    net = Inception(30, 18)
    opt = pyro_shim.ClippedAdam({"lr": 0.000857, "betas": [0.95, 0.999], "clip_norm": 15})
    m = BNN(net, opt, pretrain_epochs=5, mc_samples_train=1, mc_samples_eval=S_EVAL, dataset_size=238150, fit_context="lrt",
            prior_loc=0.0, prior_scale=0.138793, guide="normal", q_scale=1.351e-3, device=dev, engine=engine)
    m.on_fit_start()
    return m


def loop(m, B, K):
    for k in range(K):
        m.validation_step((X[k * B: (k + 1) * B], Y[k * B: (k + 1) * B]), k)


for B, engine in CASES:
    K = N // B
    xs, ys = X[: K * B], Y[: K * B]
    m = model(engine)
    loop(m, B, 20)  # warm-up
    ms_a = timed(lambda: loop(m, B, K)) / K
    m.validate_epoch(X[: 20 * B], Y[: 20 * B], B)  # warm-up: the call's batch graph is captured here and replayed below
    ms_b = timed(lambda: m.validate_epoch(xs, ys, B)) / K
    ok = all(torch.isfinite(torch.as_tensor(float(v))) for v in m.logged.values())
    e, gd, idx = m.bnn.engine, m.bnn.net_guide, torch.arange(K * B, device=dev).view(K, B)
    enq = []
    for graphs in (True, False):
        e.set_step_graph(graphs)
        call = lambda: e.elbo_val_steps(xs, ys, idx, gd.loc, gd.scale, guide="normal", particles=1, S=S_EVAL, prior_loc=0.0,
                                        prior_scale=0.138793, dataset_size=238150, seed=7, engine=engine)
        call()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        call()
        enq.append((time.perf_counter() - t0) * 1e3 / K)
        torch.cuda.synchronize()
    e.set_step_graph(True)
    print(f"Inception B={B:4d} S={S_EVAL} engine={engine:4s} K={K:4d}: (a) compat loop {ms_a:.4f} ms/batch | (b) one call "
          f"{ms_b:.4f} ms/batch | (a)/(b) {ms_a / ms_b:.2f}x | call enqueue {enq[0]:.4f} ms/batch with graphs, {enq[1]:.4f} "
          f"without | finite {ok}", flush=True)
    del m
