#!/usr/bin/env python
"""Benchmark of the MC variational-BNN hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--engine tc|simt] [--dump-outputs DIR]

Headline workload (config.workload): the LRT experiment's Inception BNN (experiment=ncmapss_lrt,
q_scale 1.351e-3, prior 0.138793) predicting B=10 000 synthetic N-CMAPSS windows [30x18] with S=100
Monte-Carlo weight samples per step (reference semantics: bnn.predict draws one full weight sample
per MC sample, bayesian.py:235-249) + the predictive-moment reduction.
A "step" = one such batch; `value` = window x samples / s with inputs resident in HBM; `e2e` = the
same through BNN.predict_step -> brl_predict_moments_host with pinned HOST inputs and host results.
Riding along: "train" (one whole svi.step of the LRT / Flipout experiments at B=256 per GPU: ELBO
forward + backward + ClippedAdam, + the NCCL all-reduce at N > 1; level-fused tcgen05 kernels, with
the fp32 and TF32 per-layer back-ends and the CPU port beside them), "mcd_predict" (configs[1]),
"flipout_predict" (configs[2]: q_scale 2.14e-4, S=20), "radial_sweep" (configs[3], MC samples sharded
over the ranks + moment merge), "deep_ensemble" (five members as one launch) and "deep_ensemble_full"
(configs[4] at its stated scale: 1M windows, 5 members + LRT BNN at S=1000, members / samples sharded
over the ranks, NCCL moment merges inside the timed region).  One process per GPU; windows are sharded across ranks, no data-path collective in the
headline (weak scaling).  Only the JSON line is written to stdout.
--dump-outputs DIR: after the timed headline steps, the (pred, std, ep_var, al_var) vectors of the last one are
written as DIR/<name>.npy (float32, 4 x 40 KB per rank; `_rank<r>` suffix when several ranks run).  Inputs, weights
and noise are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NET = "inception"
B_PRED, S_PRED = 10000, 100
B_TRAIN = 256
N_DATASET = 238150
CFG = dict(q_scale=1.351e-3, prior_scale=0.138793, prior_loc=0.0)
F_FWD = 2_289_376  # GEMM FLOPs / window / weight sample (SURVEY 8(d))
F_FC = 2 * (2400 * 64 + 64 * 2)  # of which the fc + head layers (tc_fc_kernel); the rest is the conv stack (tc_conv_kernel)
F_CONV = F_FWD - F_FC
F_TRAIN_LRT = 13_036_416
METRIC = "mc_predictive_window_samples_per_s"
UNIT = "window*samples/s"


def synth(n, seed=12345):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 30, 18, generator=g)
    y = torch.rand(n, generator=g) * 100.0
    return x, y


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            pass

    def stop(self):
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons, power = [], 0.0, set(), 0.0
        for r in rows:
            try:
                sm.append(float(r[1]))
                smax = max(smax, float(r[2]))
                power = max(power, float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        busy = [c for c in sm if c > 0.5 * smax] or sm
        return dict(sm_mhz=statistics.median(busy) if busy else None, sm_max_mhz=smax or None, reasons=sorted(reasons),
                    power_w_max=power, samples=len(sm))


def flush_l2(buf):
    buf.add_(1.0)  # 256 MiB read+write > 126 MB L2


def timed_steps(fn, steps, warmup, flush_buf, dist):
    """W warm-ups, then K steps each bracketed by its own CUDA events (L2 flushed in between, outside the
    timed regions); barrier + synchronize on both sides; returns per-rank total seconds."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    evs = []
    for i in range(steps):
        flush_l2(flush_buf)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(i)
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / 1e3


def dump_outputs(out_dir, arrays, rank, world):
    """Each [B] result tensor as out_dir/<name>.npy in float32 (<name>_rank<r>.npy when several ranks run)."""
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a.detach().float().cpu().numpy())


def max_over_ranks(t, dist, device):
    if dist is None:
        return t
    v = torch.tensor([t], dtype=torch.float64, device=device)
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    return v.item()


def cpu_predict_rate(n_windows, n_samples, threads):
    """Oracle port of the same workload on the host cores (bounded sample)."""
    from oracle import bnn_oracle as O

    torch.set_num_threads(threads)
    x, _ = synth(n_windows)
    mu = O.init_params(NET, 12345)
    sg = torch.full_like(mu, CFG["q_scale"])
    g = torch.Generator().manual_seed(1)

    def run():
        nz = [O.InjectedNoise({"weight_eps": torch.randn(mu.numel(), generator=g)}) for _ in range(n_samples)]
        return O.predictive_moments(O.predict(NET, x, mu, sg, "normal", nz))

    run_small = n_samples
    t0 = time.perf_counter()
    run()
    dt = time.perf_counter() - t0
    return n_windows * run_small / dt, dt


def cpu_train_rate(mode, particles, q, prior_scale, threads, steps=10, warmup=3):
    """Oracle port of one ELBO step (forward + autograd backward) on the host cores, B = 256: `warmup` untimed steps, then
    the MEDIAN of `steps` timed ones (BASELINE.md section 2)."""
    from oracle import bnn_oracle as O

    torch.set_num_threads(threads)
    x, y = synth(B_TRAIN, seed=777)
    mu = O.init_params(NET, 12345)
    sg = torch.full_like(mu, q)
    g = torch.Generator().manual_seed(3)
    kw = dict(mode=mode, guide="normal", prior_loc=0.0, prior_scale=prior_scale, dataset_size=N_DATASET)

    def step():
        nz = [O.InjectedNoise(O.make_injected_noise(NET, B_TRAIN, mode, g)) for _ in range(particles)]
        return O.elbo_loss_and_grads(NET, x, y, mu, sg, noises=nz, **kw)

    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    dt = statistics.median(ts)
    return B_TRAIN / dt, dt


def workload_config(engine, world):
    """`config` of both arms: the headline workload (BASELINE.json configs[0], predictive half)."""
    return {"workload": f"ncmapss_lrt Inception BNN predict (configs[0]), B={B_PRED} windows x S={S_PRED} weight samples "
                        "+ predictive moments per step per GPU", "net": NET, "engine": engine,
            "windows_per_step_per_gpu": B_PRED, "mc_samples": S_PRED, "q_scale": CFG["q_scale"],
            "l2": "256 MiB flush between timed steps + 8 rotating input batches", "parallelism": f"windows sharded x{world}"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the plain-PyTorch restatement
    (oracle port; pyro/tyxe are not installable, DESIGN.md) on all host threads; bounded sample per step."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    nb, ns = B_PRED, 10
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_predict_rate(nb // 4, 2, threads)
    t = 0.0
    units = 0
    for _ in range(args.steps):
        r, dt = cpu_predict_rate(nb, ns, threads)
        t += dt
        units += nb * ns
    v = units / t
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config("cpu-port (plain PyTorch restatement)", 1), l2="n/a (CPU)", parallelism="rank 0 only, all host threads",
                       sample=f"each step = {nb} windows x {ns} of the {S_PRED} MC samples"),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"each step = {nb} windows x {ns} of the {S_PRED} MC samples (plain-PyTorch restatement, "
                                   f"torch {torch.__version__} CPU, {threads} threads)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--engine", default=os.environ.get("BRL_ENGINE", "auto"))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-full", action="store_true", help="skip the 1M-window configs[4] pass (about 5 s at one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed headline step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's results; the reference arm computes a bounded sample")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    # stdout carries ONE JSON line: whatever libraries print to fd 1 (NCCL's version banner, NCCL_DEBUG=INFO logs) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist_mod.init_process_group("nccl", device_id=device)
        dist = dist_mod

    from bayesrul_b200 import Engine, Noise, _lib
    from bayesrul_b200.compat import BNN, Inception

    lib = _lib.load()
    eng = Engine(NET, device)
    engine = args.engine
    if engine == "auto":
        engine = "tc" if eng.has_tc() else "simt"

    # ---- synthetic workload: each rank owns its own shard of windows (global window index offset)
    n_rot = 8  # rotate 8 distinct batches (8 x 21.6 MB of windows > L2 together with the flush)
    xs = [synth(B_PRED, seed=12345 + 17 * rank + i)[0].to(device) for i in range(n_rot)]
    from bayesrul_b200.compat.nets import init_flat_params
    mu = init_flat_params(NET, 12345).to(device)  # weights_init under manual_seed(12345), SURVEY 8(d)
    sigma = torch.full_like(mu, CFG["q_scale"])
    flush_buf = torch.zeros(64 * 1024 * 1024, device=device)
    outs = {}

    def pred_step(i=0):
        outs["m"] = eng.predict_moments(xs[i % n_rot], mu, sigma, S=S_PRED, guide="normal",
                                        noise=Noise(seed=2024, window0=rank * B_PRED), engine=engine)

    sampler = ClockSampler(local)
    l0 = lib.brl_launch_count()
    for _ in range(args.warmup):
        pred_step()
    if engine == "tc":
        eng.tc_timing(True)  # CUDA events around every tc_conv_kernel launch, on the launching stream
    t_local = timed_steps(pred_step, args.steps, 0, flush_buf, dist)
    conv_ms, conv_launches, fc_ms, fc_launches = 0.0, 0, 0.0, 0
    if engine == "tc":
        kt = eng.tc_timing_read()
        (conv_ms, conv_launches), (fc_ms, fc_launches) = kt["tc_conv_kernel"], kt["tc_fc_kernel"]
        eng.tc_timing(False)
    launches = lib.brl_launch_count() - l0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("pred", "std", "ep_var", "al_var"), outs["m"])), rank, world)
    launches_timed = launches * args.steps // (args.steps + args.warmup)  # warm-up steps launch the same kernels
    t = max_over_ranks(t_local, dist, device)
    units_per_step = B_PRED * S_PRED
    value = world * units_per_step * args.steps / t
    pk = peaks()
    flops_step = units_per_step * F_FWD
    step_tf = flops_step * args.steps / t_local / 1e12
    traffic = None
    kernels = []
    tpath = os.path.join(ROOT, "profiles", "conv_traffic.json")
    if engine == "tc" and conv_launches > 0:
        # dominant kernel: algorithmic conv-stack FLOPs of the timed steps / summed tc_conv_kernel time (CUDA events)
        achieved_tf = units_per_step * args.steps * F_CONV / (conv_ms * 1e-3) / 1e12
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            # ncu dram bytes of one 16-sample launch, scaled to the average launch of this run
            traffic = tj["dram_bytes_per_window_sample"] * units_per_step * args.steps / conv_launches
        roof_note = (f"tc_conv_kernel: {F_CONV} algorithmic GEMM FLOPs per window-sample x "
                     f"{units_per_step * args.steps // conv_launches} window-samples per launch (average of {conv_launches} launches) / "
                     f"{conv_ms / conv_launches:.3f} ms per launch (CUDA events on the launch stream inside the timed region); "
                     f"kernel share of the step {conv_ms / (t_local * 1e3):.2f}; whole step incl. fc/pack/sampler/moments = {step_tf:.1f} TFLOP/s; "
                     f"peak = BURST bf16 cuBLAS of {pk['src']} MEASURED_PEAKS.json (the kernel is event-timed per launch); traffic = ncu dram read+write per launch "
                     f"(profiles/conv_traffic.json)")
        # second kernel: [128 windows x 2400] x [2400 x 64] + head; bound by the read of the fp16 feature tensor
        fc_bytes = units_per_step * args.steps * 4800.0
        kernels.append({"kernel": "tc_fc_kernel", "bound": "hbm", "achieved": fc_bytes / (fc_ms * 1e-3) / 1e9, "peak": pk["hbm"],
                        "unit": "GB/s", "frac": fc_bytes / (fc_ms * 1e-3) / 1e9 / pk["hbm"], "ms_per_launch": fc_ms / max(fc_launches, 1),
                        "share_of_step": fc_ms / (t_local * 1e3), "algorithmic": "4800 B of fp16 features read per window-sample"})
    else:
        achieved_tf = step_tf
        roof_note = (f"fp32 SIMT engine: algorithmic GEMM FLOPs of the whole step ({F_FWD} per window-sample) / step time; "
                     f"peak = burst bf16 cuBLAS of {pk['src']} MEASURED_PEAKS.json")

    # ---- e2e: BNN.predict_step through the reference-facing class, pinned host inputs, host results
    net = Inception(30, 18)
    model = BNN(net, optimizer=None, pretrain_epochs=0, mc_samples_train=1, mc_samples_eval=S_PRED, dataset_size=N_DATASET,
                fit_context="lrt", prior_loc=CFG["prior_loc"], prior_scale=CFG["prior_scale"], guide="normal",
                q_scale=CFG["q_scale"], device=device, engine=engine)
    model.on_predict_start()
    hx = [synth(B_PRED, seed=999 + i) for i in range(2)]
    hx = [(x.pin_memory(), y.pin_memory()) for x, y in hx]
    res = {}

    def e2e_step(i=0):
        x, y = hx[i % 2]
        res["p"] = model.predict_step((x, y), i)  # H2D of the batch + D2H of 5 result vectors inside

    t_e2e_local = timed_steps(e2e_step, args.steps, args.warmup, flush_buf, dist)
    t_e2e = max_over_ranks(t_e2e_local, dist, device)
    e2e_value = world * units_per_step * args.steps / t_e2e
    h2d = B_PRED * (30 * 18 + 1) * 4
    d2h = B_PRED * 4 * 4

    # ---- ELBO-train throughput (second half of the BASELINE metric), B=256
    train = {}
    if not args.no_train:
        xt, yt = synth(B_TRAIN, seed=777 + rank)
        xt, yt = xt.to(device), yt.to(device)
        from bayesrul_b200.dist import FlatGradAllReduce
        reducer = FlatGradAllReduce(mu.numel(), device) if dist is not None else None  # NVLS multimem all-reduce when available
        NT = 40
        pk_t = peaks()
        for mode, particles, q, ps, lr in (("lrt", 1, 1.351e-3, 0.138793, 1.0e-3), ("flipout", 2, 2.14e-4, 0.198768, 1.0e-3)):
            # one svi.step of the reference (bayesian.py:147): ELBO forward + backward, then pyro's ClippedAdam on (loc, log scale)
            # (conf/model/bnn.yaml:6-10); data-parallel ranks average the step's flat result buffer with ONE NCCL all-reduce first
            P = mu.numel()
            par = {"mu": mu.clone(), "ls": torch.full_like(mu, float(torch.log(torch.tensor(q)))), "sg": torch.full_like(mu, q)}
            opt = {k: torch.zeros(P, device=device) for k in ("m_mu", "v_mu", "m_ls", "v_ls")}
            st = {"i": 0}

            def train_step(i=0):
                st["i"] += 1
                r = eng.elbo_step(xt, yt, par["mu"], par["sg"], mode=mode, guide="normal", particles=particles, prior_loc=0.0,
                                  prior_scale=ps, dataset_size=N_DATASET, noise=Noise(seed=5000 + st["i"], window0=rank * B_TRAIN),
                                  out_flat=reducer.flat if reducer is not None else None)
                gs = 1.0
                if reducer is not None:
                    r = reducer.reduce(r)
                    gs = reducer.grad_scale
                eng.clipped_adam_vi(par["mu"], par["ls"], par["sg"], r["grad_mu"], r["grad_log_sigma"],
                                    opt["m_mu"], opt["v_mu"], opt["m_ls"], opt["v_ls"], st["i"], lr, (0.95, 0.999), 1e-8, 15.0, grad_scale=gs)

            res = {}
            # level-fused tcgen05 kernels (fp16 / bf16 operands: the default of compat.BNN) / fp32 FFMA parity kernels /
            # per-layer tcgen05 TF32 dual GEMMs (brl_set_gemm_backend: 8 / 0 / 7)
            l0t = lib.brl_launch_count()
            for backend in ("fused", "simt", "tc"):
                eng.set_gemm_backend(backend)
                res[backend] = max_over_ranks(timed_steps(train_step, NT, 6, flush_buf, dist), dist, device)
            eng.set_gemm_backend("fused")
            eng.set_step_graph(False)  # the same step without the CUDA-graph replay (eager launches), for the record
            t_eager = max_over_ranks(timed_steps(train_step, NT, 3, flush_buf, dist), dist, device)
            eng.set_step_graph(True)
            eng.set_gemm_backend("simt")
            tt = res["fused"]
            flops = F_TRAIN_LRT * particles * B_TRAIN  # 13 036 416 per window per particle (SURVEY 8(d))
            ach = flops / (tt / NT) / 1e12
            train[mode] = {"windows_per_s": world * B_TRAIN * NT / tt, "ms_per_step": 1e3 * tt / NT, "batch_per_gpu": B_TRAIN,
                           "particles": particles, "gemm_backend": "level-fused tcgen05 (fp16 / bf16 operands, fp32 accumulate)",
                           "ms_per_step_by_backend": {"fused_tcgen05": 1e3 * res["fused"] / NT, "simt_fp32": 1e3 * res["simt"] / NT,
                                                      "per_layer_tcgen05_tf32": 1e3 * res["tc"] / NT},
                           "ms_per_step_eager_fused": 1e3 * t_eager / NT,
                           "roofline": {"bound": "tensor", "achieved": ach, "peak": pk_t["tf_burst"], "unit": "TFLOP/s",
                                        "frac": ach / pk_t["tf_burst"], "traffic": None, "kernel": "svi.step (whole step)",
                                        "note": f"{F_TRAIN_LRT} algorithmic GEMM FLOPs per window-particle x {particles} x {B_TRAIN} windows / "
                                                "step time; a 256-window minibatch is 3.3 GFLOP -- the step is a chain of 16 latency-bound "
                                                "launches, not tensor-pipe throughput (profiles/r02_ncu_train_fused.txt); peak = burst bf16 "
                                                f"cuBLAS of {pk_t['src']} MEASURED_PEAKS.json"},
                           "includes": "ELBO forward + backward + KL + gradient finalisation (CUDA-graph replay) + ClippedAdam on (loc, log scale)"
                                       + (f" + ONE all-reduce of the step's flat result buffer over {world} ranks ({reducer.mode})" if dist is not None else "")}
            if world == 1 and not args.no_cpu:
                v, dt = cpu_train_rate(mode, particles, q, ps, os.cpu_count() or 1)
                train[mode]["cpu_windows_per_s"] = v
                train[mode]["cpu_ms_per_step"] = 1e3 * dt
                train[mode]["cpu_sample"] = "oracle port, 3 warm-up + 10 timed steps, median"
                train[mode]["speedup_vs_cpu_port"] = train[mode]["windows_per_s"] / v

        # the frequentist twin (configs[1] / [4] train their HNNs with it): HNN.step (frequentist.py:39-48: forward with dropout,
        # gaussian_nll_loss, backward) + Adam on the flat parameter buffer (brl_clipped_adam with the clip disabled)
        th = mu.clone()
        hm, hv = torch.zeros_like(th), torch.zeros_like(th)
        hs = {"i": 0}

        hred = FlatGradAllReduce(0, device, numel=mu.numel()) if dist is not None else None

        def hnn_train_step(i=0):
            hs["i"] += 1
            r = eng.hnn_step(xt, yt, th, p_dropout=0.241437, noise=Noise(seed=7000 + hs["i"], window0=rank * B_TRAIN),
                             out_grad=hred.flat if hred is not None else None)
            g = r["grad"]
            if hred is not None and hred.reduce_flat() != 1.0:
                g = g * hred.grad_scale  # SUM (multimem) -> mean; NCCL's AVG needs nothing
            eng.clipped_adam(th, g, hm, hv, hs["i"], 1e-3, (0.9, 0.999), 1e-8, 1e30)

        eng.set_gemm_backend("simt")
        th_s = max_over_ranks(timed_steps(hnn_train_step, NT, 6, flush_buf, dist), dist, device)
        eng.set_gemm_backend("fused")
        th_t = max_over_ranks(timed_steps(hnn_train_step, NT, 6, flush_buf, dist), dist, device)
        eng.set_step_graph(False)
        th_e = max_over_ranks(timed_steps(hnn_train_step, NT, 3, flush_buf, dist), dist, device)
        eng.set_step_graph(True)
        eng.set_gemm_backend("simt")
        train["hnn_mcd"] = {"windows_per_s": world * B_TRAIN * NT / th_t, "ms_per_step": 1e3 * th_t / NT, "batch_per_gpu": B_TRAIN,
                            "p_dropout": 0.241437, "ms_per_step_eager": 1e3 * th_e / NT,
                            "gemm_backend": "level-fused tcgen05 (fp16 / bf16 operands, fp32 accumulate)",
                            "ms_per_step_by_backend": {"fused_tcgen05": 1e3 * th_t / NT, "simt_fp32": 1e3 * th_s / NT},
                            "includes": "HNN.step forward (fused dropout masks) + gaussian_nll_loss + backward (CUDA-graph replay) + Adam"
                                        + (f" + NCCL all-reduce over {world} ranks" if dist is not None else "")}

    # ---- MC-dropout predictive (configs[1]: ncmapss_mcd, p = 0.241437, 100 masks), same engine
    mcd = {}
    if not args.no_train:
        def mcd_step(i=0):
            eng.predict_moments(xs[i % n_rot], mu, None, S=S_PRED, guide=None, p_dropout=0.241437,
                                noise=Noise(seed=4048, window0=rank * B_PRED), engine=engine)

        tm = max_over_ranks(timed_steps(mcd_step, 3, 2, flush_buf, dist), dist, device)
        mcd = {"window_samples_per_s": world * units_per_step * 3 / tm, "ms_per_step": 1e3 * tm / 3, "p_dropout": 0.241437,
               "masks": S_PRED, "noise": "in-kernel Philox masks (fused)"}

    # ---- configs[2], prediction half: the Flipout experiment's BNN (ncmapss_fo.yaml:17-25: q_scale 2.14e-4, S = 20 weight samples;
    #      outside fit_ctxt the predictive path is plain weight sampling, SURVEY F6)
    fo_pred = {}
    if not args.no_train:
        sg_fo = torch.full_like(mu, 2.14e-4)

        def fo_step(i=0):
            eng.predict_moments(xs[i % n_rot], mu, sg_fo, S=20, guide="normal", noise=Noise(seed=6060, window0=rank * B_PRED), engine=engine)

        tf = max_over_ranks(timed_steps(fo_step, 5, 3, flush_buf, dist), dist, device)
        fo_pred = {"window_samples_per_s": world * B_PRED * 20 * 5 / tf, "ms_per_step": 1e3 * tf / 5, "mc_samples": 20, "q_scale": 2.14e-4,
                   "windows_per_step_per_gpu": B_PRED}

    # ---- configs[3]: Radial BNN (ncmapss_rad: q_scale 1.241e-3), MC-sample sweep over a FIXED batch of windows, sharded 2-D:
    #      the ranks form a (window shards) x (sample shards) grid; MC samples are split only while every rank keeps >= 16 of them
    #      (a fused launch wants tens of samples: S = 10 over 8 ranks would leave 1 - 2 per launch), the remaining factor of the
    #      world splits the windows.  Ranks that share a window shard merge their per-window (n, mean, M2, sum sigma^2) with one
    #      all-gather + Chan's formula inside the timed region.
    radial = {}
    if not args.no_train:
        from bayesrul_b200.dist import merge_moments, shard_range
        sg_rad = torch.full_like(mu, 1.241e-3)
        x_rad = synth(B_PRED, seed=4242)[0].to(device)  # the same windows on every rank
        for S_tot in (10, 100, 1000):
            ss = 1
            while ss * 2 <= world and world % (ss * 2) == 0 and S_tot // (ss * 2) >= 16:
                ss *= 2
            wsh = world // ss
            wi, si = rank // ss, rank % ss
            w_lo, w_hi = shard_range(B_PRED, wi, wsh)
            s_lo, s_hi = shard_range(S_tot, si, ss)
            xr = x_rad[w_lo:w_hi].contiguous()

            def rad_step(i=0):
                m = eng.predict_moments(xr, mu, sg_rad, S=s_hi - s_lo, guide="radial", noise=Noise(seed=777, sample0=s_lo, window0=w_lo),
                                        engine=engine)
                if ss > 1:  # one all-gather over the world ([4, windows of a shard], padded to the largest shard); merge my row of the grid
                    nmax = -(-B_PRED // wsh)
                    packed = torch.zeros(4, nmax, device=device)
                    packed[0, : w_hi - w_lo] = float(s_hi - s_lo)
                    packed[1, : w_hi - w_lo], packed[2, : w_hi - w_lo], packed[3, : w_hi - w_lo] = m[0], m[2].nan_to_num(0.0), m[3]
                    allp = torch.empty(world * 4, nmax, device=device)
                    dist.all_gather_into_tensor(allp, packed)
                    allp = allp.view(world, 4, nmax)[wi * ss:(wi + 1) * ss, :, : w_hi - w_lo]
                    m = merge_moments([(allp[r, 0], allp[r, 1], allp[r, 2], allp[r, 3]) for r in range(ss)])
                outs["rad"] = m

            nrep = 3
            tr = max_over_ranks(timed_steps(rad_step, nrep, 2, flush_buf, dist), dist, device)
            radial[f"S={S_tot}"] = {"window_samples_per_s": B_PRED * S_tot * nrep / tr, "ms_per_step": 1e3 * tr / nrep,
                                    "samples_per_rank": s_hi - s_lo, "windows_per_rank": w_hi - w_lo, "grid": f"{wsh} window x {ss} sample shards"}
        radial["note"] = (f"{B_PRED} windows in total (strong scaling), AutoRadial guide (eps/||eps||*r sampler, two-phase norm), "
                          f"{world} rank(s) as a window x sample grid"
                          + ("; NCCL all-gather of the per-window moments + Chan merge inside the timed region where samples are split" if dist is not None else ""))

    # ---- configs[4]: deep ensemble of 5 HNN members (deterministic heteroscedastic nets) + mixture moments (deepens.py:21-24);
    #      windows sharded across the ranks like the headline workload
    deepens = {}
    if not args.no_train:
        members = torch.stack([init_flat_params(NET, 100 + k) for k in range(5)]).to(device)  # [5,P]: five trained-net stand-ins

        def de_step(i=0):
            # the members are five weight sets: ONE forward in weight-sample mode (wsamp = [M,P]) instead of five launches
            o = eng.forward(xs[i % n_rot], "ws", wsamp=members, S=5, engine=engine)  # [5,B,2]
            outs["de"] = eng.mixture_moments(o[:, :, 0].contiguous(), o[:, :, 1].contiguous())

        td = max_over_ranks(timed_steps(de_step, 5, 2, flush_buf, dist), dist, device)
        deepens = {"window_members_per_s": world * B_PRED * 5 * 5 / td, "ms_per_step": 1e3 * td / 5, "members": 5,
                   "windows_per_step_per_gpu": B_PRED}

    # ---- the two nets no shipped config selects (nets/conv.py:47-61 Conv-D3, nets/linear.py:44-55 Linear): weight-sampling predict on the
    #      per-layer engines (fp32 FFMA and tcgen05 TF32 GEMMs) and, for the Linear net, on its fused tcgen05 engine (DESIGN.md 4.6 / 8(i))
    other_nets = {}
    if not args.no_train and world == 1:
        from bayesrul_b200 import Engine as _Engine
        for net_name in ("conv", "linear"):
            en = _Engine(net_name, device)
            mu_n = init_flat_params(net_name, 12345).to(device)
            sg_n = torch.full_like(mu_n, CFG["q_scale"])
            rec = {}
            for be in ("simt", "tc"):
                en.set_gemm_backend(be)

                def on_step(i=0):
                    outs["on"] = en.predict_moments(xs[i % n_rot], mu_n, sg_n, S=20, guide="normal", noise=Noise(seed=9000 + i), engine="simt")

                t_on = timed_steps(on_step, 3, 2, flush_buf, None)
                rec[{"simt": "fp32_ffma", "tc": "per_layer_tcgen05_tf32"}[be]] = B_PRED * 20 * 3 / t_on
            en.set_gemm_backend("simt")
            if en.has_tc():  # Linear: the fused fp16 tcgen05 engine (csrc/brl_tc_linear.cuh), at the headline's S as well

                def on_tc(i=0, S=20):
                    outs["on"] = en.predict_moments(xs[i % n_rot], mu_n, sg_n, S=S, guide="normal", noise=Noise(seed=9100 + i), engine="tc")

                rec["fused_tcgen05_fp16"] = B_PRED * 20 * 3 / timed_steps(on_tc, 3, 2, flush_buf, None)
                rec[f"fused_tcgen05_fp16_S{S_PRED}"] = B_PRED * S_PRED * 3 / timed_steps(lambda i=0: on_tc(i, S_PRED), 3, 2, flush_buf, None)
            other_nets[net_name] = {"window_samples_per_s": rec, "mc_samples": 20, "windows_per_step": B_PRED, "params": int(mu_n.numel())}
            del en

    # ---- configs[4] at its stated scale: 1 000 000 windows, deep ensemble of 5 HNN members + the LRT-trained BNN at S = 1000.
    #      Members and MC samples are SHARDED over the ranks (every rank sees all windows); per window chunk the ranks merge
    #      their per-window moments with one NCCL all-gather (BNN: Chan merge) and one all-reduce (ensemble mixture) inside
    #      the timed region.  One timed pass (+ one warm-up chunk): 1.005e9 window-(samples + members) per pass.
    de_full = {}
    if not args.no_train and not args.no_full:
        from bayesrul_b200.dist import all_gather_moments, mixture_across_ranks, shard_range
        n_full, S_full, chunk = 1_000_000, 1000, 100_000
        gdev = torch.Generator(device=device).manual_seed(31337)
        s_lo, s_hi = shard_range(S_full, rank, world)
        m_lo, m_hi = shard_range(5, rank, world)
        res_full = {}

        def full_chunk(xc, c):
            m = eng.predict_moments(xc, mu, sigma, S=s_hi - s_lo, guide="normal", noise=Noise(seed=99, sample0=s_lo), engine=engine)
            if m_hi > m_lo:
                o = eng.forward(xc, "ws", wsamp=members[m_lo:m_hi].contiguous(), S=m_hi - m_lo, engine=engine)
                mu_m, sd_m = o[:, :, 0].contiguous(), o[:, :, 1].contiguous()
            else:
                mu_m = sd_m = torch.zeros(0, xc.shape[0], device=device)
            if dist is not None:
                m = all_gather_moments(s_hi - s_lo, m[0], m[2], m[3])
                de = mixture_across_ranks(mu_m, sd_m)
            else:
                de = eng.mixture_moments(mu_m, sd_m)
            res_full[c] = (m[0], m[1], de[0], de[1])

        xw = torch.randn(chunk, 30, 18, device=device, generator=gdev)
        full_chunk(xw[:10_000].contiguous(), -1)  # warm-up (workspace growth, graph-free path)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_full = 0.0
        for c in range(n_full // chunk):
            xw = torch.randn(chunk, 30, 18, device=device, generator=gdev)  # the chunk's windows, resident before the clock starts
            ev0.record()
            full_chunk(xw, c)
            ev1.record()
            torch.cuda.synchronize()
            t_full += ev0.elapsed_time(ev1) / 1e3
        t_full = max_over_ranks(t_full, dist, device)
        units = n_full * (S_full + 5)
        de_full = {"window_units_per_s": units / t_full, "seconds_per_pass": t_full, "windows": n_full, "bnn_mc_samples": S_full,
                   "members": 5, "window_chunk": chunk,
                   "sharding": f"MC samples {S_full} and members 5 over {world} rank(s); per chunk one all-gather of [4, {chunk}] moments + "
                               "one all-reduce of the mixture sums" if dist is not None else "single rank: no collective",
                   "unit": "window x (BNN samples + ensemble members) / s"}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands / f32 accumulate" if engine == "tc" else "f32", "data": "synthetic",
        "config": workload_config(engine, world),
        "clocks": clocks, "gpu_launches": int(launches_timed),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "bayesrul_b200.compat.BNN.predict_step -> brl_predict_moments_host (pinned host batch -> host results)"},
        "roofline": {"bound": "tensor", "achieved": achieved_tf, "peak": pk["tf_burst"], "unit": "TFLOP/s",
                     "frac": achieved_tf / pk["tf_burst"], "traffic": traffic, "kernel": "tc_conv_kernel" if engine == "tc" else "step",
                     "ms_per_launch": conv_ms / max(conv_launches, 1), "share_of_step": conv_ms / (t_local * 1e3) if conv_launches else None,
                     "note": roof_note, "other_kernels": kernels},
        "train": train, "mcd_predict": mcd, "flipout_predict": fo_pred, "radial_sweep": radial, "deep_ensemble": deepens,
        "other_nets_predict": other_nets,
        "deep_ensemble_full": de_full,
    }
    if world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        cpu_predict_rate(1000, 2, threads)  # warm-up
        v, dt = cpu_predict_rate(B_PRED, S_PRED, threads)  # one whole step of the workload: ~11 s on the 16-core GPU box
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{B_PRED} windows x all {S_PRED} MC samples = one step ({dt:.1f} s), plain-PyTorch "
                                          f"restatement on torch {torch.__version__} CPU"}
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
