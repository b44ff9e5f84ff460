"""Every engine and back-end on exactly representable nets: outputs bit for bit per window, gradients per element.

The other parity tests hold the fp16 / bf16 / TF32 paths to aggregate bounds (1e-2 on outputs, cosine and relative L2 per
layer group on gradients), because under operand rounding a ReLU gate within one rounding of zero flips and moves a whole
row (DESIGN §4.3).  A defect confined to one tile, one K-chunk, one tap or one member slot passes those bounds.  Here the
inputs are chosen so that nothing rounds in the forward pass:

  x      integers in -3..3, and feature 0 a time ramp +-(t - 15) + c with its own sign and offset c in -6..6 per window
  theta  every hidden output row 2-4 non-zeros of value +-1, biases integers; the head rows 8-16 non-zeros of +-1/16,
         biases multiples of 1/4.  Non-zeros sit on input channels that vary across the batch's windows.  Layer 0
         (Inception conv1) rows read the ramp only, and branch4's 1x1 conv reads only those channels, so that every
         max-pool window it routes a gradient through has a strictly ordered maximum
  sigma  half the layer's grid (1/2 hidden, 1/32 head)
  eps    injected weight noise, integers on theta's support only, chosen so that W = mu + sigma eps = +-mu or 2 mu:
         W stays sparse and on the layer's grid (eps = 0 on biases)
  signs  Flipout signs +-1
  drop   dropout at p = 0.5 where every site keeps 1/2 (Linear, Conv-D3): T = 8192 of 2^14 and 1 / keep = 2, both exact;
         the kernels draw their own Philox masks, replayed here by PhiloxNoise.drop_mask

Rows are drawn in topological order against the batch itself and redrawn until every pre-activation of every scenario
(sample, particle, mask) stays within LIMIT grid units and the head's pre-activations within |o| <= O_LIMIT, so every
activation is an integer below 2^8 (pooled values: halves and quarters), exact in fp16, bf16 and TF32, every product is
exact and every fp32 sum is exact.  test_construction_is_exact checks that on every case the GPU tests use, and fails
when one is not; it also requires the outputs to tell the windows apart (DISTINCT_MIN, TILE_DISTINCT_MIN), since a
window written into another window's slot shows only where their outputs differ.  Building the cases takes one to three
minutes of CPU, depending on the host (once per session: the GPU tests share them); the whole GPU run of this file,
case building included, took 65 s on a B200 host.  The forward pass of every engine must then reproduce the float64
oracle up to the head's softplus: at most OUT_ULPS float32 ulps per output (softplus is the only rounding left; measured on a B200: see DESIGN §4.3).

The Inception net's MC dropout is not in this construction: its branch sites keep 1 - p/4, whose reciprocal is not a
power of two for any p > 0, so the kernels' fp32 1 / keep factor rounds (not a defect; DESIGN §4.3).

Gradients: with the forward exact and every gate and route identical, a gradient entry differs from float64 autograd
only by the rounding of the gradient operands (bf16 on 'fused', TF32 on 'tc', none on 'simt') and by fp32 accumulation.
A magnitude pass runs the same backward with |W|, the recorded gates and routes, |activations| and |dL/do| taken from the
kernel's own outputs, and yields A = sum |terms| for every entry; the test asserts |g - g_ref| <= kappa A with kappa
derived in `kappa` below, and prints per layer the number of live entries (A > 0) and max and median err / (kappa A).
A layer no output reads in a case (A = 0 everywhere) is printed as empty and left out of the summary."""
import functools
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bnn_oracle as O
from tests.helpers import injected_to_engine

DEV = "cuda:0"
NETS = ["inception", "linear", "conv"]
KW = dict(prior_loc=0.0, prior_scale=0.5, dataset_size=1000)
LIMIT = 64  # grid units: |pre-activation| of every hidden layer (after dropout's x2 the next layer still reads < 2^8)
O_LIMIT = 12.0  # |head pre-activation|: softplus(-12) = 6e-6, far above the 1e-9 floor, below the o > 20 pass-through
# the head's fp32 softplus / threshold is the forward's only rounding: a few ulps of the output (and an ulp near 0)
OUT_ULPS = 4
# a per-window check sees a window written into another window's slot only where their outputs differ: every case keeps
# this share of distinct output rows in the batch and in its last (ragged) 128-window tile
DISTINCT_MIN, TILE_DISTINCT_MIN = 0.45, 0.8  # measured minima 0.49 (Linear, p = 0.5, B = 1000) and 0.82
U32, U_TF32, U_BF16 = 2.0**-24, 2.0**-10, 2.0**-8  # TF32 operands may be truncated: 2^-10 relative; bf16 round to nearest


def _grid(net, i):
    return 1.0 / 16 if i == len(O.net_layers(net)) - 1 else 1.0


def _sigma_of(net, i):
    return _grid(net, i) / 2


def _fan(L):
    return int(np.prod(L.wshape[1:]))


# ---------------------------------------------------------------------------------------------------------- construction
def _passes(net, mode, mu, sigma, eps, flip, rec):
    """lay(i, inp) of `mode` ('det': W = mu, 'ws': W = mu + sigma eps, 'flipout') for O.run_net; records each pre-activation"""
    layers = O.net_layers(net)
    m_ = O.unflatten(mu, net)
    w_ = m_ if mode == "det" else O.unflatten(mu + sigma * eps, net)

    def lay(i, inp):
        L = layers[i]
        if mode == "flipout":
            s_in = O._bcast(flip[f"flip_in.{i}"].to(inp.dtype), inp.dim())
            mean = O._op(L, inp, m_[i][0], None)
            pert = O._op(L, inp * s_in, w_[i][0] - m_[i][0], None)
            s_out = O._bcast(flip[f"flip_out.{i}"].to(inp.dtype), mean.dim())
            v = mean + pert * s_out + O._bcast(w_[i][1][None, :], mean.dim())
        else:
            v = O._op(L, inp, w_[i][0], w_[i][1])
        rec[i] = v
        return v

    return lay


def _drop(net, p, masks):
    return O.make_dropout(net, p, O.InjectedNoise(masks)) if p > 0 else None


def _cat_scen(scen, key_fn):
    return {k: torch.cat([key_fn(s)[k] for s in scen]) for k in key_fn(scen[0])}


def _build_theta(net, x, scen, mode, p, g):
    """mu, eps [n_scen, P] drawn row by row in topological order against all scenarios (each one a [B] batch)"""
    layers = O.net_layers(net)
    P = O.num_params(net)
    mu = torch.zeros(P, dtype=torch.float64)
    eps = torch.zeros(len(scen), P, dtype=torch.float64)
    sites = O.site_table(net)
    sigma = torch.zeros(P, dtype=torch.float64)
    for i in range(len(layers)):
        (_, _, wo), (_, _, bo) = sites[2 * i], sites[2 * i + 1]
        sigma[wo: bo + layers[i].cout] = _sigma_of(net, i)
    S, B = len(scen), x.shape[0]
    xs = x.repeat(S, 1, 1)
    flip = _cat_scen(scen, lambda s: s["flip"]) if mode == "flipout" else None
    masks = _cat_scen(scen, lambda s: s["masks"]) if p > 0 else {}
    n_last = len(layers) - 1

    def rows(i, idx, varies):
        """(weight rows, bias, eps rows [S]) for output channels idx of layer i; the non-zeros sit on input channels that
        vary across the batch's windows (all of them at B = 1), so that no row settles on window-constant (dead) inputs"""
        L, gr = layers[i], _grid(net, i)
        fan = _fan(L)
        ok = varies if varies.any() else torch.ones_like(varies)
        if net == "inception" and i == 0:
            ok = torch.arange(18) == 0  # conv1 (k = 1): the ramp feature only
        if net == "inception" and i == 9:
            ok = ok & (torch.arange(108) < 27)  # branch4 reads the max-pooled conv1 channels only
        allowed = np.flatnonzero(np.repeat(ok.numpy(), fan // L.wshape[1]))
        W = torch.zeros(len(idx), fan, dtype=torch.float64)
        E = torch.zeros(S, len(idx), fan, dtype=torch.float64)
        for r in range(len(idx)):
            # 2-4 non-zeros; the head 8-16, so that its two outputs tell the windows apart
            k = min(int(g.integers(8, 17) if i == n_last else g.integers(2, 5)), len(allowed))
            pos = g.choice(allowed, size=k, replace=False)
            s = g.choice([-1.0, 1.0], size=k)
            W[r, pos] = torch.from_numpy(s * gr)
            # W = mu + sigma eps in {mu, 2 mu, -mu}: sigma = grid / 2, eps in {0, 2 s, -4 s} (conv1: Flipout's mu +- (W - mu)
            # never 0, so the ramp rows stay strictly monotone)
            choices = [0.0, -4.0] if (net == "inception" and i == 0) else [0.0, 2.0, -4.0]
            for sc in range(S):
                E[sc, r, pos] = torch.from_numpy(g.choice(choices, size=k) * s) * (gr / 2 / _sigma_of(net, i))
        if i == n_last:
            b = torch.from_numpy(g.integers(-8, 9, size=len(idx)).astype(np.float64)) / 4
        elif net == "inception" and i == 0:
            b = torch.from_numpy(g.integers(-12, 13, size=len(idx)).astype(np.float64))
        else:
            b = torch.from_numpy(g.integers(-1, 3, size=len(idx)).astype(np.float64)) * gr
        return W, b, E

    def lay(i, inp):
        L = layers[i]
        (_, _, wo), (_, _, bo) = sites[2 * i], sites[2 * i + 1]
        fan, co = _fan(L), L.cout
        lim = O_LIMIT if i == n_last else LIMIT * _grid(net, i)
        varies = (inp != inp[:1]).reshape(inp.shape[0], inp.shape[1], -1).any(2).any(0)  # per input channel
        todo = torch.arange(co)
        for attempt in range(60):
            W, b, E = rows(i, todo, varies)
            if attempt >= 50:  # last resort: the bias alone (never reached by the seeds in use; the check below would say)
                W.zero_(), E.zero_(), b.zero_()
            wv = mu[wo: wo + co * fan].view(co, fan)
            wv[todo] = W
            mu[bo + todo] = b
            for sc in range(S):
                eps[sc, wo: wo + co * fan].view(co, fan)[todo] = E[sc]
            pre = _scen_pre(net, mode, i, inp, mu, sigma, eps, flip, S, B)
            bad = pre.abs().transpose(0, 1).reshape(co, -1).amax(1) > lim
            todo = todo[bad[todo]]
            if len(todo) == 0:
                break
        return pre

    O.run_net(net, xs, lay, _drop(net, p, masks))
    return mu, sigma, eps


def _scen_pre(net, mode, i, inp, mu, sigma, eps, flip, S, B):
    L = O.net_layers(net)[i]
    outs = []
    for sc in range(S):
        sl = slice(sc * B, (sc + 1) * B)
        fl = {k: v[sl] for k, v in flip.items()} if flip is not None else None
        rec = {}
        outs.append(_passes(net, mode, mu, sigma, eps[sc], fl, rec)(i, inp[sl]))
    return torch.cat(outs)


@functools.lru_cache(maxsize=None)
def exact_case(net, B, seed, mode="det", S=1, p=0.0, member=0):
    """x [B,30,18], y [B], mu / sigma [P], eps [S,P], flip (list of S dicts), masks (list of S dicts) -- float64 -- and the
    oracle's per-sample outputs out [S,B,2], head pre-activations o [S,B,2] and recorded pre-activations (see the module
    docstring for the construction).  x and y depend on (seed, B) only: the members of an ensemble share them."""
    gx = np.random.default_rng([seed, B])
    x = torch.from_numpy(gx.integers(-3, 4, size=(B, 30, 18)).astype(np.float64))
    # feature 0: a time ramp, strictly monotone in every window, with its own sign and offset per window
    sgn = torch.from_numpy(gx.choice([-1.0, 1.0], size=(B, 1)))
    off = torch.from_numpy(gx.integers(-6, 7, size=(B, 1)).astype(np.float64))
    x[:, :, 0] = sgn * (torch.arange(30, dtype=torch.float64) - 15) + off
    y = torch.from_numpy(gx.integers(0, 8, size=B).astype(np.float64))
    g = np.random.default_rng([seed, B, S, NETS.index(net), int(p * 8), ["det", "ws", "flipout"].index(mode), member])
    tg = torch.Generator().manual_seed(int(g.integers(1 << 30)))
    drop_seed = int(g.integers(1 << 62))
    scen = []
    for sc in range(S):
        s = {}
        if mode == "flipout":
            s["flip"] = {k: v.double() for k, v in O.make_injected_noise(net, B, "flipout", tg).items() if k.startswith("flip")}
        if p > 0:  # the kernels' own Philox masks (Noise(seed=drop_seed)), replayed
            pn = O.PhiloxNoise(net, drop_seed, sample=sc, dtype=torch.float64)
            s["masks"] = {f"drop_mask.{i}": pn.drop_mask(i, (B,) + O.layer_out_shape(net, i), 1.0 - p * f)
                          for i, f in O.DROPOUT_SITES[net].items()}
        scen.append(s)
    mu, sigma, eps = _build_theta(net, x, scen, mode, p, g)
    case = dict(net=net, B=B, mode=mode, S=S, p=p, x=x, y=y, mu=mu, sigma=sigma, eps=eps, scen=scen, drop_seed=drop_seed)
    case.update(oracle(case))
    return case


def oracle(case, mu=None, x=None):
    """float64 forward of every scenario: out [S,B,2], o [S,B,2], pre (list of {layer: pre-activation}), acts"""
    net, mode, p = case["net"], case["mode"], case["p"]
    mu = case["mu"] if mu is None else mu
    x = case["x"] if x is None else x
    outs, os_, pres = [], [], []
    for sc, s in enumerate(case["scen"]):
        rec = {}
        lay = _passes(net, mode, mu, case["sigma"], case["eps"][sc], s.get("flip"), rec)
        outs.append(O.run_net(net, x, lay, _drop(net, p, s.get("masks", {}))))
        os_.append(rec[len(O.net_layers(net)) - 1])
        pres.append(rec)
    return dict(out=torch.stack(outs), o=torch.stack(os_), pre=pres)


def _all_intermediates(case, sc=0):
    """every tensor a kernel stores between layers: pre-activations, activations, module concatenations, pooled values,
    fc features (re-run with hooks around relu / cat / pools)"""
    net, p, s = case["net"], case["p"], case["scen"][sc]
    seen = []
    rec = {}
    lay = _passes(net, case["mode"], case["mu"], case["sigma"], case["eps"][sc], s.get("flip"), rec)
    orig = (torch.relu, torch.cat, F.max_pool1d, F.avg_pool2d)

    def hook(fn, tag):
        def f(*a, **k):
            v = fn(*a, **k)
            seen.append((tag, v))
            return v
        return f

    torch.relu, torch.cat = hook(orig[0], "relu"), hook(orig[1], "cat")
    F.max_pool1d, F.avg_pool2d = hook(orig[2], "maxpool"), hook(orig[3], "avgpool")
    try:
        O.run_net(net, case["x"], lay, _drop(net, p, s.get("masks", {})))
    finally:
        torch.relu, torch.cat, F.max_pool1d, F.avg_pool2d = orig
    seen += [(f"pre {i}", v) for i, v in rec.items()]
    return seen


def diversity(out):
    """(share of distinct output rows in the batch, share of distinct rows in the last 128-window tile) of out [B,2]"""
    B = out.shape[0]
    last = out[128 * ((B - 1) // 128):]
    return len(torch.unique(out, dim=0)) / B, len(torch.unique(last, dim=0)) / last.shape[0]


def check_exact(case):
    """raises AssertionError unless every intermediate of every scenario equals its fp16 and bf16 rounding (the head's
    pre-activation: its fp32 rounding), no max-pool
    window that routes a gradient has a tie among positive maxima, the head pre-activations sit in |o| <= O_LIMIT, and
    the outputs tell the windows apart (DISTINCT_MIN of the batch, TILE_DISTINCT_MIN of its last 128-window tile)"""
    net = case["net"]
    for sc in range(case["S"]):
        if case["B"] > 1:
            d, dt = diversity(case["out"][sc])
            assert d >= DISTINCT_MIN and dt >= TILE_DISTINCT_MIN, (net, case["B"], case["mode"], sc, "windows too alike", d, dt)
        head = f"pre {len(O.net_layers(net)) - 1}"
        for tag, v in _all_intermediates(case, sc):
            v = v.detach()
            # the head's pre-activation is only ever an fp32 accumulator (the softplus input): exact in fp32 suffices
            for dt in ((torch.float32,) if tag == head else (torch.float16, torch.bfloat16)):
                bad = v.to(dt).double() != v
                assert not bad.any(), (f"{net} B={case['B']} {case['mode']} sample {sc}: {tag} not exact in {dt}: "
                                       f"{int(bad.sum())} values, e.g. {v[bad][0].item()!r}")
        o = case["o"][sc]
        assert o.abs().max() <= O_LIMIT, (net, "head pre-activation outside the softplus range", o.abs().max().item())
        if net == "inception":  # branch4's max pool over conv1's ramp channels (0..26 of module 1)
            a = torch.relu(case["pre"][sc][0])
            w = F.pad(a, (1, 1), value=-1.0).unfold(2, 3, 1)  # [B, 27, 30, 3]
            top = w.amax(-1, keepdim=True)
            ties = ((w == top).sum(-1) > 1) & (top[..., 0] > 0)
            assert not ties.any(), (net, "tie among positive max-pool maxima", int(ties.sum()))


# ---------------------------------------------------------------------------------------------------------- simt paths
# conv ops of the per-layer engine (csrc/brl_nets.cpp): (layer, Cin, Hin, Win, Cout, kh, kw, Hout, Wout, input gradient)
OPS = {
    "inception": [(0, 18, 30, 1, 27, 1, 1, 30, 1, False), (1, 18, 30, 1, 27, 3, 1, 30, 1, False),
                  (2, 18, 30, 1, 27, 5, 1, 30, 1, False), (3, 18, 30, 1, 27, 3, 1, 30, 1, False),
                  (4, 108, 30, 1, 16, 1, 1, 30, 1, True), (5, 108, 30, 1, 64, 1, 1, 30, 1, True),
                  (6, 64, 30, 1, 16, 3, 1, 30, 1, True), (7, 108, 30, 1, 64, 1, 1, 30, 1, True),
                  (8, 64, 30, 1, 16, 5, 1, 30, 1, True), (9, 108, 30, 1, 32, 1, 1, 30, 1, True),
                  (10, 2400, 1, 1, 64, 1, 1, 1, 1, True), (11, 64, 1, 1, 2, 1, 1, 1, 1, True)],
    "conv": [(0, 1, 30, 18, 16, 5, 9, 26, 10, False), (1, 16, 26, 10, 32, 2, 10, 25, 1, True),
             (2, 32, 12, 1, 64, 2, 1, 11, 1, True), (3, 320, 1, 1, 2, 1, 1, 1, 1, True)],
    "linear": [(0, 540, 1, 1, 256, 1, 1, 1, 1, False)] + [(i, ci, 1, 1, co, 1, 1, 1, 1, True) for i, (ci, co) in
                                                          enumerate([(256, 128), (128, 128), (128, 32), (32, 2)], 1)],
}


def _gemm_path(B, P, N, K, S):
    """(small_tiles, ksplit) of brl_gemm.cu's launch_conv_gemm / conv_gemm_ksplit (BN = 32, BK = 16; 148 SMs)"""
    ctas = -(-B * P // 128) * -(-N // 32)
    ks = 1 if (S != 1 or ctas >= 74 or K < 8 * 16) else max(1, min(K // 64, 296 // ctas))
    small = ctas * (ks if ks > 1 else S) < 4 * 148
    return small, ks


def _dw_split(B, P, N, K):
    """row splits of brl_gemm.cu's launch_conv_dw (DW_K = 128, DW_CO = 32, DW_M = 16, 148 CTAs)"""
    M = B * P
    gxy = -(-(K + 1) // 128) * -(-N // 32)
    split = max(1, min(-(-M // 32), -(-148 // gxy)))
    rows = -(-(-(-M // split)) // 16) * 16
    return -(-M // rows)


def simt_paths(net, B, S=1):
    """per conv op: dict(fwd=(small, ksplit), dx=(small, ksplit) or None, dw=splits)"""
    out = {}
    for (l, ci, hi, wi, co, kh, kw, ho, wo, dx) in OPS[net]:
        out[l] = dict(fwd=_gemm_path(B, ho * wo, co, ci * kh * kw, S),
                      dx=_gemm_path(B, hi * wi, ci, co * kh * kw, 1) if dx else None,
                      dw=_dw_split(B, ho * wo, co, ci * kh * kw))
    return out


def _fmt_paths(paths):
    f = lambda t: "-" if t is None else f"{'32' if t[0] else '128'}{'/k' + str(t[1]) if t[1] > 1 else ''}"
    return " ".join(f"L{l}[{f(d['fwd'])},{f(d['dx'])},dw{d['dw']}]" for l, d in paths.items())


# ---------------------------------------------------------------------------------------------------------- cases
BATCHES_TC = [1, 4, 127, 128, 129, 255, 257, 1000, 4097]
FWD_TC = [(n, m, B) for n in NETS for m, Bs in (("det", BATCHES_TC), ("ws", [5, 129, 1000])) for B in Bs]
BATCHES_SIMT = [1, 3, 129, 257, 1000]
FWD_SIMT = ([(n, m, p, B) for n in NETS for m in ("det", "ws", "flipout") for B in BATCHES_SIMT for p in (0.0,)]
            + [(n, "det", 0.5, B) for n in ("linear", "conv") for B in (5, 129, 1000)]
            + [("inception", "det", 0.0, 4097), ("linear", "det", 0.0, 4097)])
# (net, kind, p, backend, B): kind 'hnn' (p = 0 / 0.5) or the ELBO's 'ws' / 'flipout'
STEPS = ([(n, "hnn", 0.0, be, B) for n in NETS for be in ("simt", "tc", "fused") for B in (1, 4, 5, 129, 257)]
         + [(n, "hnn", 0.5, be, B) for n in ("linear", "conv") for be in ("simt", "tc", "fused") for B in (3, 129)]
         + [(n, k, 0.0, be, B) for n in NETS for k in ("ws", "flipout") for be in ("simt", "tc", "fused") for B in (4, 129)]
         + [("inception", "hnn", 0.0, be, 1000) for be in ("simt", "fused")]
         + [("inception", "ws", 0.0, "fused", 1000)])
MOMENTS = [(n, e, S) for n, e in (("inception", "simt"), ("inception", "tc"), ("linear", "tc"), ("conv", "simt"))
           for S in (1, 15, 16, 17)] + [("inception", "tc", 128), ("inception", "tc", 129)]
B_MOM = 37
ENSEMBLE = [(kind, M, B) for kind in ("hnn", "ws", "flipout") for M in (3, 5) for B in (5, 129)]
SEED = 11


def _case_for_step(net, kind, p, B, member=0):
    return exact_case(net, B, SEED, "det" if kind == "hnn" else kind, 1, p, member)


def all_cases():
    """every case the GPU tests run, built once"""
    for n, m, B in FWD_TC:
        yield exact_case(n, B, SEED, m, 2 if m == "ws" else 1)
    for n, m, p, B in FWD_SIMT:
        yield exact_case(n, B, SEED, m, 1, p)
    for n, k, p, be, B in STEPS:
        yield _case_for_step(n, k, p, B)
    for n, e, S in MOMENTS:
        yield exact_case(n, B_MOM, SEED, "ws", S)
    for kind, M, B in ENSEMBLE:
        for m in range(M):
            yield _case_for_step("inception", kind, 0.0, B, member=m)
    for M in (3, 5):
        for m in range(M):
            yield exact_case("inception", 129, SEED, "ws", 2, 0.0, m)


# ---------------------------------------------------------------------------------------------------------- CPU checks
def test_keep_half_is_exact():
    """p = 0.5 at a site of factor 1: T = 8192 of the 14-bit keep decisions and 1 / keep = 2, both exact in fp32"""
    assert O.keep_threshold(0.5) == 8192
    keep = np.float32(1.0) - np.float32(0.5) * np.float32(1.0)
    assert np.float32(1.0) / keep == np.float32(2.0)
    # the Inception net's branch sites keep 1 - p / 4: never a power of two, so its MC dropout stays out (module docstring)
    assert np.float64(np.float32(1.0) / np.float32(0.875)) != 8.0 / 7.0


def test_construction_is_exact():
    n = 0
    for case in all_cases():
        check_exact(case)
        n += 1
    print(f"[construction] {n} cases exact in fp16 and bf16")


def test_construction_check_fails_on_a_non_representable_intermediate():
    """one weight moved off the grid (1 -> 1 + 2^-9: exact in fp16, not in bf16) must make check_exact fail"""
    case = dict(exact_case("linear", 5, SEED, "det"))
    mu = case["mu"].clone()
    j = int(torch.nonzero(mu[:540 * 256]).flatten()[0])
    mu[j] += 2.0**-9 * torch.sign(mu[j])
    case["mu"] = mu
    case.update(oracle(case))
    with pytest.raises(AssertionError, match="not exact"):
        check_exact(case)


def test_simt_paths_cover_every_threshold():
    """the simt cases of this file reach both sides of small_tiles, conv_gemm_ksplit and the dw row split, for the forward,
    input-gradient and weight-gradient launches (the backward launches counted from the simt step cases only)"""
    seen = {k: set() for k in ("fwd small", "fwd ksplit", "dx small", "dx ksplit", "dw split")}
    steps = {(n, B, 1) for n, k, p, be, B in STEPS if be == "simt"}
    shapes = {(n, B, 1) for n, m, p, B in FWD_SIMT} | {(n, B_MOM, min(S, 16)) for n, e, S in MOMENTS if e == "simt"} | steps
    for net, B, S in sorted(shapes):
        paths = simt_paths(net, B, S)
        bwd = (net, B, S) in steps
        print(f"[simt paths] {net} B={B} S={S}{' (step)' if bwd else ''}: {_fmt_paths(paths)}")
        for d in paths.values():
            seen["fwd small"].add(d["fwd"][0])
            seen["fwd ksplit"].add(d["fwd"][1] > 1)
            if not bwd:
                continue
            seen["dw split"].add(d["dw"] > 1)
            if d["dx"] is not None:
                seen["dx small"].add(d["dx"][0])
                seen["dx ksplit"].add(d["dx"][1] > 1)
    print(f"[simt paths] reached: {seen}")
    for k, v in seen.items():
        assert v == {True, False}, (k, v)


# ---------------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def engines():
    from bayesrul_b200 import Engine
    es = {n: Engine(n, DEV) for n in NETS}
    yield es
    for e in es.values():
        e.set_gemm_backend("simt")
    # the module's summary, once every GPU test of it has run: worst forward ulps per engine, worst and median
    # err / (kappa A) per back-end and layer (layers with live entries only)
    for k, v in sorted(WORST.items()):
        print(f"[summary] forward {k}: worst {v:.1f} ulp")
    for (be, net, name, i), (mx, mds) in sorted(STATS.items()):
        print(f"[summary] {be} {net} {name} layer {i}: max err/(kA) {mx:.2e}, median of medians {float(np.median(mds)):.2e} "
              f"({len(mds)} checks)")


def _f32(t):
    return t.float().contiguous().to(DEV)


def _ulps(got, ref):
    """|got - ref| in float32 ulps of ref (ref float64)"""
    got, ref = got.detach().double().cpu(), ref.double()
    ulp = torch.from_numpy(np.spacing(np.abs(ref.float().numpy())).astype(np.float64))
    return (got - ref).abs() / ulp


WORST = {}


def check_out(got, ref, tag):
    """per window and channel: at most OUT_ULPS float32 ulps; returns the windows that fail (for the negative controls)"""
    u = _ulps(got, ref)
    worst = u.max().item()
    key = tag.split(" B=")[0]
    bad = (u > OUT_ULPS).reshape(-1, u.shape[-2], u.shape[-1]).any(-1).any(0)
    if not tag.startswith("control"):
        WORST[key] = max(WORST.get(key, 0.0), worst)
    return worst, torch.nonzero(bad).flatten().tolist()


def assert_out(got, ref, tag):
    worst, bad = check_out(got, ref, tag)
    print(f"[{tag}] worst {worst:.1f} ulp")
    assert not bad, (tag, f"{len(bad)} windows beyond {OUT_ULPS} ulps, first {bad[:8]}", worst)


def _noise(case):
    """the case's noise for bayesrul_b200: injected weight_eps [S,P] and flip signs; dropout as native Philox masks"""
    if case["p"] > 0:
        from bayesrul_b200 import Noise
        assert case["mode"] == "det"
        return Noise(seed=case["drop_seed"])
    dicts = []
    for sc, s in enumerate(case["scen"]):
        d = {}
        if case["mode"] in ("ws", "flipout"):
            d["weight_eps"] = case["eps"][sc]
        d.update(s.get("flip", {}))
        dicts.append(d)
    return injected_to_engine(case["net"], dicts, case["B"], DEV) if dicts[0] else None


def _wsamp(case):
    return _f32(case["mu"][None] + case["sigma"][None] * case["eps"])


# ---------------------------------------------------------------------------------------------------------- 2. forward
@pytest.mark.gpu
@pytest.mark.parametrize("net,mode,B", FWD_TC)
def test_tc_engine_forward_exact(engines, net, mode, B):
    e = engines[net]
    case = exact_case(net, B, SEED, mode, 2 if mode == "ws" else 1)
    x = _f32(case["x"])
    if mode == "det":
        out = e.forward(x, "det", theta=_f32(case["mu"]), engine="tc")
    else:
        out = e.forward(x, "ws", wsamp=_wsamp(case), S=case["S"], engine="tc")
    assert e.tc_status() == 0
    assert_out(out, case["out"], f"tc engine {net} {mode} B={B}")


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["simt", "tc"])
@pytest.mark.parametrize("net,mode,p,B", FWD_SIMT)
def test_per_layer_forward_exact(engines, backend, net, mode, p, B):
    e = engines[net]
    case = exact_case(net, B, SEED, mode, 1, p)
    if backend == "simt":
        print(f"[simt paths] {net} B={B}: {_fmt_paths(simt_paths(net, B))}")
    x, mu = _f32(case["x"]), _f32(case["mu"])
    e.set_gemm_backend(backend)
    try:
        if mode == "det":
            out = e.forward(x, "det", theta=mu, p_dropout=p, noise=_noise(case))
        elif mode == "ws":
            out = e.forward(x, "ws", wsamp=_wsamp(case), S=1)
        else:
            out = e.forward(x, "flipout", theta=mu, wsamp=_wsamp(case), noise=_noise(case))
    finally:
        e.set_gemm_backend("simt")
    assert e.gemm_status() == 0
    assert_out(out, case["out"], f"per-layer {backend} {net} {mode} p={p} B={B}")


# ---------------------------------------------------------------------------------------------------------- 4. gradients
def _depth(net):
    return {"inception": 5, "linear": 5, "conv": 4}[net]


def kappa(net, backend, B):
    """per layer: |g - g_ref| <= kappa A.  First-order error analysis of the backward with an exact forward:
    * the tail: dL/do from the fp32 outputs, the 1/B or 1/(540 B) loss scale and the softplus derivative, <= 32 u of the
      tail's term magnitude (the seed of the magnitude pass, `_dL_do`);
    * fp32 accumulation, any order (split-K, atomics, Chan merges): a sum of n terms errs by <= (n - 1) u sum|terms|.  The
      input-gradient sums of every layer above (Cout kh kw terms each) compound into the operand of the weight-gradient sum
      of B Hout Wout (+ 1) terms;
    * operand rounding (r = u_op per rounding, 2^-10 TF32, 2^-8 bf16): one for each gradient operand a GEMM reads and one
      for each gradient stored between levels, i.e. 2 per level of the deepest path plus 2 for the weight-gradient GEMM.
    u = 2^-24."""
    r = {"simt": 0.0, "tc": U_TF32, "fused": U_BF16}[backend]
    dx_sum = sum(co * kh * kw for (_, _, _, _, co, kh, kw, _, _, dx) in OPS[net] if dx)
    return {l: r * (2 * _depth(net) + 2) + U32 * (32 + dx_sum + B * ho * wo + 1)
            for (l, _, _, _, _, _, _, ho, wo, _) in OPS[net]}


def _dL_do(kind, out, y, B):
    """dL/do [B,2] from the kernel's own fp32 outputs (float64; the head's d out / d o = 1 - exp(-out), 0 at the floor) and
    its term magnitude: the scale channel's 1/var - d^2/var^2 (HNN) and 1 - r^2 (ELBO) cancel, so the kernel's fp32 tail
    errs relative to |1/var| + |d^2/var^2| resp. 1 + r^2, not to their difference"""
    out = out.detach().double().cpu().clone().requires_grad_(True)
    y = y.double()
    loc, sc = out[:, 0].detach(), out[:, 1].detach()
    if kind == "hnn":
        loss = F.gaussian_nll_loss(out[:, 0], y, out[:, 1] ** 2)
        var = (sc * sc).clamp_min(1e-6)
        d = loc - y
        mag = torch.stack([d.abs() / var, (1.0 / var + d * d / var**2) * sc], 1) / B
    else:  # the ELBO's likelihood part: c N / B NLL_sum, c = 1 / (N 540)
        loss = O.heteroskedastic_nll_sum(out, y) / (540.0 * B)
        s = F.softplus(sc)
        r = (y - loc) / s
        mag = torch.stack([r.abs() / s, (1.0 + r * r) / s * torch.sigmoid(sc)], 1) / (540.0 * B)
    (g,) = torch.autograd.grad(loss, out)
    o = out.detach()
    dsp = torch.where(o > 1e-9, -torch.expm1(-o), torch.zeros_like(o))
    return g * dsp, mag * dsp


def grad_ref(case, do, sc=0, mu=None):
    """float64 backward from dL/do through the oracle's graph: dict of grad_mu (grad), grad_sigma (ws / flipout)"""
    net, mode, p, s = case["net"], case["mode"], case["p"], case["scen"][sc]
    mu = (case["mu"] if mu is None else mu).clone().requires_grad_(True)
    sg = case["sigma"].clone().requires_grad_(True)
    rec = {}
    O.run_net(net, case["x"], _passes(net, mode, mu, sg, case["eps"][sc], s.get("flip"), rec), _drop(net, p, s.get("masks", {})))
    o = rec[len(O.net_layers(net)) - 1]
    if mode == "det":
        (gm,) = torch.autograd.grad(o, mu, grad_outputs=do)
        return dict(grad=gm)
    gm, gs = torch.autograd.grad(o, (mu, sg), grad_outputs=do)
    return dict(grad_mu=gm, grad_sigma=gs)


def grad_mag(case, do_mag, sc=0):
    """the magnitude pass: A = sum |terms| of every gradient entry (same gates, routes and dropout scaling as the value pass)"""
    net, mode, p, s = case["net"], case["mode"], case["p"], case["scen"][sc]
    layers = O.net_layers(net)
    pre = case["pre"][sc]
    mu, eps, sg = case["mu"], case["eps"][sc], case["sigma"]
    w = mu if mode in ("det", "flipout") else mu + sg * eps
    aw = w.abs().clone().requires_grad_(True)
    ad = (sg * eps).abs().clone().requires_grad_(True) if mode == "flipout" else None
    a_ = O.unflatten(aw, net)
    d_ = O.unflatten(ad, net) if ad is not None else None
    cap = {}

    def lay(i, inp):
        L = layers[i]
        z = inp.detach().abs() + (inp - inp.detach())
        m = O._op(L, z, a_[i][0], a_[i][1])
        if d_ is not None:
            m = m + O._op(L, z, d_[i][0], None)
        v = pre[i].detach() + (m - m.detach())
        cap[i] = v
        return v

    O.run_net(net, case["x"], lay, _drop(net, p, s.get("masks", {})))
    grads = torch.autograd.grad(cap[len(layers) - 1], [t for t in (aw, ad) if t is not None], grad_outputs=do_mag)
    if mode == "det":
        return dict(grad=grads[0])
    # grad_sigma = eps * (the perturbation path's gradient); eps = 0 on the biases
    return dict(grad_mu=grads[0], grad_sigma=eps.abs() * grads[-1])


def kl_grads(case):
    c = 1.0 / (KW["dataset_size"] * 540.0)
    mu, sg = case["mu"], case["sigma"]
    return dict(grad_mu=c * (mu - KW["prior_loc"]) / KW["prior_scale"] ** 2,
                grad_sigma=c * (-1.0 / sg + sg / KW["prior_scale"] ** 2))


def _layer_slices(net):
    sites = O.site_table(net)
    return [(i, slice(sites[2 * i][2], sites[2 * i + 1][2] + L.cout)) for i, L in enumerate(O.net_layers(net))]


STATS = {}


def check_grads(got, ref, mag, kl, net, backend, B, tag, assert_ok=True):
    """|g - kl - g_ref| <= kappa A + 8 u |kl| per entry (the analytic KL term: c = 1 / (N 540), the difference, the product,
    the quotient and the final sum, <= 5 roundings); prints max / median err / (kappa A) per layer; returns the entries
    that fail.  Only asserted checks enter the summary."""
    ks = kappa(net, backend, B)
    failing = {}
    for name in ref:
        g = got[name].detach().double().cpu()
        k_ = kl[name] if kl is not None else torch.zeros_like(g)
        err = (g - k_ - ref[name]).abs()
        for i, sl in _layer_slices(net):
            bound = ks[i] * mag[name][sl] + 8 * U32 * k_[sl].abs()
            ratio = err[sl] / bound.clamp_min(1e-300)
            ratio = torch.where(bound > 0, ratio, torch.where(err[sl] > 0, torch.full_like(ratio, math.inf), ratio))
            live = mag[name][sl] > 0  # entries with at least one non-zero term
            n_live, n_ref = int(live.sum()), int((ref[name][sl] != 0).sum())
            mx = ratio.max().item()
            if n_live == 0:  # nothing downstream reads this layer here: 0 against 0, not a check
                print(f"[{tag}] {name} layer {i}: empty (no non-zero term in {live.numel()} entries), err {err[sl].max().item():.1e}")
            else:
                md = ratio[live].median().item()
                if assert_ok:
                    s = STATS.setdefault((backend, net, name, i), [0.0, []])
                    s[0] = max(s[0], mx)
                    s[1].append(md)
                print(f"[{tag}] {name} layer {i}: {n_live}/{live.numel()} live entries ({n_ref} non-zero), max err/(kA) "
                      f"{mx:.2e}, median {md:.2e} (kappa {ks[i]:.2e})")
            bad = torch.nonzero(ratio > 1).flatten() + sl.start
            if len(bad):
                failing.setdefault(name, []).extend(bad.tolist())
    if assert_ok:
        assert not failing, (tag, {k: (len(v), v[:6]) for k, v in failing.items()})
    return failing


def _step(e, kind, p, case, backend):
    x, y, mu = _f32(case["x"]), _f32(case["y"]), _f32(case["mu"])
    e.set_gemm_backend(backend)
    try:
        if kind == "hnn":
            got = e.hnn_step(x, y, mu, p, _noise(case))
            return dict(out=got["out"], grad=got["grad"])
        got = e.elbo_step(x, y, mu, _f32(case["sigma"]), mode=kind, guide="normal", noise=_noise(case), **KW)
        return dict(out=got["out"][0], grad_mu=got["grad_mu"], grad_sigma=got["grad_sigma"])
    finally:
        e.set_gemm_backend("simt")


@pytest.mark.gpu
@pytest.mark.parametrize("net,kind,p,backend,B", STEPS)
def test_step_out_exact_and_grads_bounded(engines, net, kind, p, backend, B):
    e = engines[net]
    case = _case_for_step(net, kind, p, B)
    got = _step(e, kind, p, case, backend)
    assert e.tc_status() == 0 and e.gemm_status() == 0
    tag = f"step {backend} {net} {kind} p={p} B={B}"
    if backend == "simt":
        print(f"[simt paths] {net} B={B}: {_fmt_paths(simt_paths(net, B))}")
    assert_out(got["out"], case["out"][0], tag)
    do, do_mag = _dL_do(kind, got["out"], case["y"], B)
    check_grads(got, grad_ref(case, do), grad_mag(case, do_mag), kl_grads(case) if kind != "hnn" else None, net, backend, B, tag)


# ---------------------------------------------------------------------------------------------------------- member-batched
def _members(kind, M, B):
    return [_case_for_step("inception", kind, 0.0, B, member=m) for m in range(M)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,M,B", ENSEMBLE)
def test_ensemble_steps_exact(engines, kind, M, B):
    """hnn_step_ensemble / elbo_step_ensemble on the fused back-end, each member with its own sparsity pattern"""
    got, cases = _ensemble_step(engines["inception"], kind, M, B)
    for m, case in enumerate(cases):
        _check_member(got, case, m, kind, B, f"ensemble {kind} M={M} member {m} B={B}")


def _ensemble_step(e, kind, M, B, order=None):
    cases = _members(kind, M, B)
    run = [cases[j] for j in (order or range(M))]
    x = torch.stack([c["x"] for c in run]).float().to(DEV)
    y = torch.stack([c["y"] for c in run]).float().to(DEV)
    mu = torch.stack([c["mu"] for c in run]).float().to(DEV)
    e.set_gemm_backend("fused")
    try:
        if kind == "hnn":
            g = e.hnn_step_ensemble(x, y, mu, 0.0, None)
            got = [dict(out=g["out"][m], grad=g["grad"][m]) for m in range(M)]
        else:
            sg = torch.stack([c["sigma"] for c in run]).float().to(DEV)
            dicts = []
            for c in run:
                d = {"weight_eps": c["eps"][0]}
                d.update(c["scen"][0].get("flip", {}))
                dicts.append(d)
            g = e.elbo_step_ensemble(x, y, mu, sg, mode=kind, guide="normal", noise=injected_to_engine("inception", dicts, B, DEV), **KW)
            got = [dict(out=g["out"][m, 0], grad_mu=g["grad_mu"][m], grad_sigma=g["grad_sigma"][m]) for m in range(M)]
    finally:
        e.set_gemm_backend("simt")
    assert e.tc_status() == 0
    return got, cases


def _check_member(got, case, m, kind, B, tag, assert_ok=True):
    worst, bad_w = check_out(got[m]["out"], case["out"][0], tag)
    print(f"[{tag}] worst {worst:.1f} ulp")
    do, do_mag = _dL_do(kind, got[m]["out"], case["y"], B)
    failing = check_grads(got[m], grad_ref(case, do), grad_mag(case, do_mag), kl_grads(case) if kind != "hnn" else None,
                          "inception", "fused", B, tag, assert_ok=assert_ok)
    if assert_ok:
        assert not bad_w, (tag, bad_w[:8], worst)
    return bad_w, failing


@pytest.mark.gpu
@pytest.mark.parametrize("M", [3, 5])
def test_predict_moments_ensemble_exact(engines, M):
    """predict_moments_ensemble (Inception, tc, S = 2 weight draws per member): every member's moments against its own
    exact outputs"""
    e = engines["inception"]
    S, B = 2, 129
    cases = [exact_case("inception", B, SEED, "ws", S, 0.0, m) for m in range(M)]  # one batch x, own theta per member
    x = _f32(cases[0]["x"])
    mu = torch.stack([c["mu"] for c in cases]).float().to(DEV)
    sg = torch.stack([c["sigma"] for c in cases]).float().to(DEV)
    eps = torch.cat([c["eps"] for c in cases]).float().to(DEV)
    from bayesrul_b200 import Noise
    got = e.predict_moments_ensemble(x, mu, sg, S=S, noise=Noise(weight_eps=eps), engine="tc")
    assert e.tc_status() == 0
    for m in range(M):
        _check_moments([t[m] for t in got], cases[m]["out"], f"predict_moments_ensemble M={M} member {m}")


# ---------------------------------------------------------------------------------------------------------- 3. moments
def moments_bounds(out):
    """float64 moments of the exact per-sample outputs [S,B,2] and their bounds.  The fp32 Welford update and Chan merge
    of S samples each commit <= 4 roundings per sample to the mean and <= 6 to M2 (|err| <= 4 S u max|x| resp.
    <= 8 S u max|x|^2, the merges included); the outputs carry <= OUT_ULPS ulps of softplus error."""
    S = out.shape[0]
    loc, sc = out[..., 0], out[..., 1]
    es = OUT_ULPS * U32
    mloc, msc2 = loc.abs().amax(0), (sc * sc).amax(0)
    pred = loc.mean(0)
    ep = loc.var(0) if S > 1 else torch.full_like(pred, math.nan)
    al = (sc * sc).mean(0)
    b_pred = (es + 4 * S * U32) * mloc + 1e-30
    b_al = (2 * es + 8 * S * U32) * msc2 + 1e-30
    b_ep = (2 * es + 8 * S * U32) * mloc**2 * (S / max(S - 1, 1)) * 2 + 1e-30
    std = (al + (ep if S > 1 else 0.0)).sqrt()
    b_std = ((b_al + (b_ep if S > 1 else 0.0)) / (2 * std.clamp_min(1e-30)) + 2 * U32 * std)
    return [(pred, b_pred), (std, b_std), (ep, b_ep), (al, b_al)]


def _check_moments(got, out, tag):
    S = out.shape[0]
    for (ref, bound), g, k in zip(moments_bounds(out), got, ("pred", "std", "ep_var", "al_var")):
        g = g.detach().double().cpu()
        if k in ("ep_var", "std") and S == 1:  # the unbiased variance of one sample, as torch's var(0)
            assert torch.isnan(g).all(), (tag, f"{k} must be NaN at S = 1")
            continue
        r = ((g - ref).abs() / bound)
        print(f"[{tag}] {k}: max err/bound {r.max().item():.2e}, median {r.median().item():.2e}")
        assert (r <= 1).all(), (tag, k, int((r > 1).sum()), r.max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("net,engine,S", MOMENTS)
def test_predict_moments_bounded(engines, net, engine, S):
    from bayesrul_b200 import Noise
    e = engines[net]
    case = exact_case(net, B_MOM, SEED, "ws", S)
    got = e.predict_moments(_f32(case["x"]), _f32(case["mu"]), _f32(case["sigma"]), S=S, noise=Noise(weight_eps=_f32(case["eps"])),
                            engine=engine)
    assert e.tc_status() == 0
    _check_moments(got, case["out"], f"predict_moments {net} {engine} S={S}")


# ---------------------------------------------------------------------------------------------------------- 5. controls
@pytest.mark.gpu
def test_control_moved_nonzero(engines):
    """one non-zero of layer 10 (Inception fc) moved by one position for the kernel only: the forward check names exactly the
    windows the move changes, and the gradient check flags the moved weight's row"""
    e, B = engines["inception"], 129
    case = _case_for_step("inception", "hnn", 0.0, B)
    (_, shape, wo) = O.site_table("inception")[20]
    mu = case["mu"].clone()
    W = mu[wo: wo + shape[0] * shape[1]].view(shape)
    for row, col in torch.nonzero(W).tolist():  # the first non-zero whose move changes some window
        col2 = col + 1 if col + 1 < shape[1] and W[row, col + 1] == 0 else col - 1
        W[row, col2], W[row, col] = W[row, col], 0.0
        moved = dict(case, mu=mu)
        expect = check_out(oracle(moved)["out"][0], case["out"][0], "control moved (oracle)")[1]
        if expect:
            break
        W[row, col], W[row, col2] = W[row, col2], 0.0
    got = _step(e, "hnn", 0.0, moved, "simt")
    _, bad = check_out(got["out"], case["out"][0], "control moved")
    print(f"[control moved] fc row {row}: column {col} -> {col2}; flagged windows {bad[:10]}.. ({len(bad)}), "
          f"changed windows {len(expect)}")
    assert expect and bad == expect
    do, do_mag = _dL_do("hnn", got["out"], case["y"], B)
    failing = check_grads(got, grad_ref(case, do), grad_mag(case, do_mag), None, "inception", "simt", B, "control moved",
                          assert_ok=False)
    # with dL/do taken from the kernel's outputs, the moved weight shows where its unit's activation is read: the head's
    # weight column of fc unit `row` (and, below, the branches that produce fc inputs col / col2)
    (_, hshape, ho) = O.site_table("inception")[22]
    head = sorted({(j - ho) % hshape[1] for j in failing.get("grad", []) if ho <= j < ho + hshape[0] * hshape[1]})
    print(f"[control moved] gradient check flags head columns {head}, {len(failing.get('grad', []))} entries in all")
    assert head == [row]


@pytest.mark.gpu
def test_control_dropped_window(engines):
    """the reference drops the last window of a ragged batch (B = 257): the gradient check flags it"""
    e, B = engines["inception"], 257
    case = _case_for_step("inception", "hnn", 0.0, B)
    got = _step(e, "hnn", 0.0, case, "fused")
    do, do_mag = _dL_do("hnn", got["out"], case["y"], B)
    do_ref = do.clone()
    do_ref[-1] = 0.0
    failing = check_grads(got, grad_ref(case, do_ref), grad_mag(case, do_mag), None, "inception", "fused", B, "control dropped",
                          assert_ok=False)
    print(f"[control dropped] {len(failing.get('grad', []))} gradient entries flagged")
    assert failing.get("grad")


@pytest.mark.gpu
def test_control_swapped_members(engines):
    """members 0 and 1 swapped in the member-batched call: both are flagged, member 2 is not"""
    got, cases = _ensemble_step(engines["inception"], "hnn", 3, 129, order=[1, 0, 2])
    for m, case in enumerate(cases):
        bad_w, failing = _check_member(got, case, m, "hnn", 129, f"control swapped member {m}", assert_ok=False)
        print(f"[control swapped] member {m}: {len(bad_w)} windows, {len(failing.get('grad', []))} gradient entries flagged")
        assert (bool(bad_w) and bool(failing)) == (m < 2), m
