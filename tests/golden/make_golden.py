"""Generate tests/golden/*.npz from the reference's OWN code.

    python tests/golden/make_golden.py <path of the reference's `bayesrul` package directory>

Imports (read-only) <bayesrul>/models/nets/{inception,conv,linear}.py (with a stub
`torchinfo`), models/deepens.py and utils/miscellaneous.py, runs them on seeded inputs and stores
inputs + outputs.  Nothing from the reference is copied into the repo; the fixtures are the
reference's numerical behaviour.  The parameter-sized inputs (theta, ws_eps) and the LRT noise are
stored as a SHA-256 of their values and sigma as its constant, which keeps every fixture small:
tests/helpers.load_golden regenerates them from the same seeds and checks each against its digest.
TyXe / Pyro are not importable, so for the LRT / Flipout / weight-sampling fixtures the reference
nets are executed with `torch.nn.functional.{conv1d,conv2d,linear}` patched by the published
per-call rule (SURVEY Appendix A.3/A.4) -- this pins the *composition* (which call sees which
tensor, in which order) on the reference's module code, while the per-call rule itself stays
"parity unpinned".
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

if len(sys.argv) != 2:
    sys.exit(__doc__)
REF = sys.argv[1]
OUT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
from tests.helpers import golden_digest  # noqa: E402


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


sys.modules.setdefault("torchinfo", types.SimpleNamespace(summary=lambda *a, **k: None))
inception = _load("ref_inception", f"{REF}/models/nets/inception.py")
conv = _load("ref_conv", f"{REF}/models/nets/conv.py")
linear = _load("ref_linear", f"{REF}/models/nets/linear.py")
misc = _load("ref_misc", f"{REF}/utils/miscellaneous.py")
deepens = _load("ref_deepens", f"{REF}/models/deepens.py")


def build(net, dropout=0.0):
    if net == "inception":
        return inception.Inception(30, 18, dropout=dropout)
    if net == "conv":
        return conv.Conv(30, 18, dropout=dropout)
    return linear.Linear(30, 18, dropout=dropout, out_size=2)


def flat(m):
    return torch.cat([p.detach().flatten() for _, p in m.named_parameters()])


def load_flat(m, theta):
    off = 0
    with torch.no_grad():
        for _, p in m.named_parameters():
            n = p.numel()
            p.copy_(theta[off: off + n].reshape(p.shape))
            off += n


class FixedMask(nn.Module):
    """Stands in for nn.Dropout: applies a recorded Bernoulli mask with 1/keep scaling."""

    def __init__(self, p, store, gen):
        super().__init__()
        self.p, self.store, self.gen = p, store, gen

    def forward(self, t):
        keep = 1.0 - self.p
        m = (torch.rand(t.shape, generator=self.gen) < keep).to(t.dtype)
        self.store.append(m)
        return t * m / keep


def swap_dropout(module, store, gen):
    for name, child in list(module.named_children()):
        if isinstance(child, nn.Dropout):
            setattr(module, name, FixedMask(child.p, store, gen))
        else:
            swap_dropout(child, store, gen)


class Patched:
    """Patch F.conv1d / F.conv2d / F.linear for the duration of one reference-net forward."""

    def __init__(self, rule):
        self.rule, self.calls = rule, 0

    def __enter__(self):
        self.orig = {k: getattr(F, k) for k in ("conv1d", "conv2d", "linear")}
        for k, fn in self.orig.items():
            def wrapper(x, w, b=None, *a, _fn=fn, **kw):
                i = self.calls
                self.calls += 1
                return self.rule(i, lambda xx, ww, bb: _fn(xx, ww, bb, *a, **kw), x, w, b)
            setattr(F, k, wrapper)
            setattr(torch.nn.functional, k, wrapper)
        return self

    def __exit__(self, *exc):
        for k, fn in self.orig.items():
            setattr(F, k, fn)


def main():
    torch.manual_seed(12345)
    g = torch.Generator().manual_seed(777)
    B, S = 6, 5
    for net in ("inception", "conv", "linear"):
        m = build(net).eval()
        m.apply(misc.weights_init)
        theta = flat(m)
        names = [n for n, _ in m.named_parameters()]
        shapes = [tuple(p.shape) for _, p in m.named_parameters()]
        x = torch.randn(B, 30, 18, generator=g)
        fx = {"theta_sha256": np.array(golden_digest(theta)), "x": x.numpy(), "names": np.array(names),
              "shapes": np.array([str(s) for s in shapes])}
        with torch.no_grad():
            fx["out_det"] = m(x).numpy()

        # ---- MC dropout (A4): reference net built with dropout, masks recorded in call order
        p = 0.241437
        md = build(net, dropout=p)
        md.train()
        load_flat(md, theta)
        masks = []
        swap_dropout(md, masks, torch.Generator().manual_seed(99))
        with torch.no_grad():
            fx["out_drop"] = md(x).numpy()
        fx["drop_p"] = np.float64(p)
        fx["names_dropout_variant"] = np.array([n for n, _ in md.named_parameters()])
        for j, mk in enumerate(masks):
            fx[f"drop_mask_call{j}"] = mk.numpy()

        # ---- weight sampling predict (A7/A11/A12): W_s loaded into the reference module
        sigma = torch.full_like(theta, 0.05)
        eps = torch.randn(S, theta.numel(), generator=g)
        outs = []
        with torch.no_grad():
            for s in range(S):
                load_flat(m, theta + sigma * eps[s])
                outs.append(m(x))
            load_flat(m, theta)
        out = torch.stack(outs)
        loc, scale = out[:, :, 0], out[:, :, 1]
        ep_var = loc.var(0)
        al_var = (scale**2).mean(0)
        fx.update(sigma_value=sigma[0].numpy(), ws_eps_sha256=np.array(golden_digest(eps)), out_ws=out.numpy(),
                  ep_var=ep_var.numpy(), al_var=al_var.numpy(), std=al_var.add(ep_var).sqrt().numpy(),
                  pred=loc.mean(0).numpy())

        # ---- LRT (A5): per-call rule of SURVEY A.3 patched into the reference forward
        off, lay_w = 0, []
        for nme, prm in m.named_parameters():
            lay_w.append((off, prm.numel()))
            off += prm.numel()
        lrt_eps, sig_list = [], []

        def lrt_rule(i, fn, xx, ww, bb):
            sw = sigma[lay_w[2 * i][0]: lay_w[2 * i][0] + lay_w[2 * i][1]].reshape(ww.shape)
            sb = sigma[lay_w[2 * i + 1][0]: lay_w[2 * i + 1][0] + lay_w[2 * i + 1][1]]
            mean = fn(xx, ww, bb)
            var = fn(xx * xx, sw * sw, sb * sb)
            e = torch.randn(mean.shape, generator=g)
            lrt_eps.append(e)
            return mean + var.sqrt() * e

        with torch.no_grad(), Patched(lrt_rule):
            fx["out_lrt"] = m(x).numpy()
        fx["lrt_eps_shapes"] = np.array([str(tuple(e.shape)) for e in lrt_eps])
        fx["lrt_eps_sha256"] = np.array([golden_digest(e) for e in lrt_eps])

        # ---- Flipout (A6): per-call rule of SURVEY A.4
        w_s = theta + sigma * eps[0]
        fin, fout = [], []

        def fo_rule(i, fn, xx, ww, bb):
            wsamp = w_s[lay_w[2 * i][0]: lay_w[2 * i][0] + lay_w[2 * i][1]].reshape(ww.shape)
            bsamp = w_s[lay_w[2 * i + 1][0]: lay_w[2 * i + 1][0] + lay_w[2 * i + 1][1]]
            cin = xx.shape[1] if xx.dim() > 2 else xx.shape[-1]
            s_in = (torch.rand(xx.shape[0], cin, generator=g) > 0.5).float() * 2 - 1
            s_out = (torch.rand(xx.shape[0], ww.shape[0], generator=g) > 0.5).float() * 2 - 1
            fin.append(s_in)
            fout.append(s_out)
            mean = fn(xx, ww, None)
            pert = fn(xx * s_in.reshape(s_in.shape + (1,) * (xx.dim() - 2)), wsamp - ww, None)
            sh = (1,) * (mean.dim() - 2)
            return mean + pert * s_out.reshape(s_out.shape + sh) + bsamp.reshape((1, -1) + sh)

        with torch.no_grad(), Patched(fo_rule):
            fx["out_flipout"] = m(x).numpy()
        for i in range(len(fin)):
            fx[f"flip_in_call{i}"] = fin[i].numpy()
            fx[f"flip_out_call{i}"] = fout[i].numpy()
        np.savez_compressed(os.path.join(OUT, f"{net}.npz"), **fx)
        print(net, "P =", theta.numel(), "calls:", len(lrt_eps), "dropout sites:", len(masks))

    # ---- deep ensemble (A14): the reference function itself
    import pandas as pd
    rng = np.random.default_rng(5)
    M, n = 5, 64
    mu_m = rng.normal(50, 10, (M, n)).astype(np.float32)
    sd_m = rng.uniform(0.5, 5, (M, n)).astype(np.float32)
    labels = rng.uniform(0, 100, n).astype(np.float32)
    df = pd.concat([pd.DataFrame(dict(model=f"HNN_{k:03d}", preds=mu_m[k], stds=sd_m[k], labels=labels))
                    for k in range(M)])
    de = deepens.deep_ensemble(df)
    np.savez_compressed(os.path.join(OUT, "deep_ensemble.npz"), mu_m=mu_m, sigma_m=sd_m,
                        preds=de.preds.values, stds=de.stds.values)

    # ---- weights_init statistics (per-layer std of the reference initialiser)
    stats = {}
    for net in ("inception", "conv", "linear"):
        torch.manual_seed(1)
        m = build(net)
        m.apply(misc.weights_init)
        stats[net] = np.array([p.detach().std().item() for _, p in m.named_parameters()])
    np.savez_compressed(os.path.join(OUT, "weights_init_std.npz"), **stats)
    print("done")


if __name__ == "__main__":
    main()
