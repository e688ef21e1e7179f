"""Range of every MMA operand of the DCGAN refinement chain, as FP16 would see it.

The tensor-core chain stores the operands of its GEMM passes as FP16: the same 10-bit mantissa as the TF32 values
they replace, so FP16 holds them exactly as long as they lie in its normal range [2^-14, 65504].  This tool runs the
CPU oracle (oracle/graph_refiner.py) with the bench's weights over all refinement steps and reports, for every
operand tensor of every pass:

  * amax (max |x|) over all steps, and the margin log2(65504 / amax) to FP16's largest finite value;
  * the share of nonzero values below 2^-14 (FP16 subnormals or zero);
  * for the data-gradients, the same after the per-sample power-of-two scale the head applies: the chain's gradient is
    linear in d loss / d logit (dl = sigmoid(logit) - 1) per sample, so the head multiplies dl by 2^e_b with
    |dl| * 2^e_b in [1, 2) and the policy step divides it out again.

    python tools/fp16_range.py [--arch dcgan64_l1 dcgan32_l1] [--batch 16] [--steps 50]
"""
from __future__ import annotations

import argparse
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "collaborative-gan-sampling_b200"))

from cgs import nets as N                       # noqa: E402
from cgs import synthetic as S                  # noqa: E402
from oracle import nets as onets                # noqa: E402
from oracle import graph_refiner as gr          # noqa: E402

FP16_MAX = 65504.0
FP16_MIN_NORMAL = 2.0 ** -14


class Stat:
    def __init__(self):
        self.amax = 0.0
        self.nz = 0
        self.small = 0

    def add(self, t):
        a = t.detach().abs().reshape(-1).double()
        nz = a[a > 0]
        self.amax = max(self.amax, float(a.max()) if a.numel() else 0.0)
        self.nz += int(nz.numel())
        self.small += int((nz < FP16_MIN_NORMAL).sum())

    def row(self, name):
        margin = math.log2(FP16_MAX / self.amax) if self.amax > 0 else float("inf")
        share = self.small / self.nz if self.nz else 0.0
        return "| %s | %.3g | %.1f | %.2e |" % (name, self.amax, margin, share)


def step_tensors(h, arch, w):
    """One evaluation at feature h: acts[i] = input of layer i of the chain (G tail + D without the head),
    grads[i] = d sum(loss) / d (pre-activation output of layer i), dl [B]."""
    layers = arch["gtail"] + arch["d"][:-1]
    head = arch["d"][-1]
    x = h.detach().clone().requires_grad_(True)
    acts, pres = [], []
    cur = x
    for L in layers:
        acts.append(cur)
        scope = "generator" if L in arch["gtail"] else "discriminator"
        p = "%s/%s/" % (scope, L["name"])
        if L["type"] == "conv":
            pre = onets.conv2d_same(cur, onets._t(w, p + "w"), onets._t(w, p + "biases"))
        else:
            pre = onets.deconv2d_same(cur, onets._t(w, p + "w"), onets._t(w, p + "biases"))
        if L["bn"]:
            q = "%s/%s/" % (scope, L["bn"])
            pre = onets.batch_norm(pre, onets._t(w, q + "gamma"), onets._t(w, q + "beta"),
                                   onets._t(w, q + "moving_mean"), onets._t(w, q + "moving_variance"), "inference")
        pre.retain_grad()
        pres.append(pre)
        cur = onets.activation(pre, L["act"])
    p = "discriminator/%s/" % head["name"]
    logit = cur.reshape(cur.shape[0], -1) @ onets._t(w, p + "Matrix") + onets._t(w, p + "bias")
    gr.loss_refine(logit).sum().backward()
    return acts, [t.grad for t in pres], logit.detach().reshape(-1)


def chain_factors(logit):
    """Per-sample factors that turn the oracle's gradient into the chain's, unscaled and scaled.  The head kernel
    computes dl = sigmoid(l) - 1 in FP32, which is exactly 0 from l ~ 17 on (autograd's -sigmoid(-l) is not), and
    scales it by 2^e_b so that |dl| * 2^e_b lies in [1, 2) (e_b = 0 where dl == 0)."""
    l = logit.numpy().astype(np.float32)
    dl_chain = (np.float32(1) / (np.float32(1) + np.exp(-l)) - np.float32(1)).astype(np.float32)
    dl_oracle = -1.0 / (1.0 + np.exp(l.astype(np.float64)))
    _, e = np.frexp(dl_chain)
    e = np.where(dl_chain == 0, 1, e)
    plain = dl_chain / dl_oracle
    return torch.from_numpy(plain.astype(np.float32)), torch.from_numpy((plain * np.ldexp(1.0, 1 - e)).astype(np.float32))


def analyse(arch_name, batch, steps, gain=2.5, seed=2019, rate=0.1):
    arch = onets.get_arch(arch_name)
    w = S.init_weights(arch, seed=seed, gain=gain)
    h0 = torch.from_numpy(S.proposal_features(arch, batch, seed=3))
    layers = arch["gtail"] + arch["d"][:-1]
    names = [L["name"] for L in layers]
    # every step's feature: the oracle's own trace (momentum, the bench's rate)
    o = gr.build_refiner(h0, arch, w, steps, rate, return_trace=True)
    feats = [h0] + [t["feature"] for t in o["trace"]]
    st = {}
    def stat(key):
        return st.setdefault(key, Stat())
    for h in feats:
        acts, grads, logit = step_tensors(h, arch, w)
        plain, scaled = chain_factors(logit)
        view = lambda f, t: f.view(-1, *([1] * (t.dim() - 1)))
        for i, a in enumerate(acts):
            if a.shape[-1] > 4:                       # image-like tensors stay FP32
                stat("act %s input" % names[i]).add(a)
        for i, g in enumerate(grads):
            # d loss / d pre(i) is the A operand of layer i's data-gradient pass
            if g.shape[-1] > 4:
                stat("grad %s output" % names[i]).add(g * view(plain, g))
                stat("grad %s output, scaled" % names[i]).add(g * view(scaled, g))
    # the matrices the chain converts to FP16: packed, BN folded, TF32 rounded (cgs.nets.PackedNet)
    wstat, nstat = Stat(), Stat()
    for L in layers:
        scope = "generator" if L in arch["gtail"] else "discriminator"
        wf, wb, _ = N.pack_layer(L, *N.fold_layer(L, scope, w))
        if L["cin"] > 4 and L["cout"] > 4:
            wstat.add(N.round_tf32(wf))
            wstat.add(N.round_tf32(wb))
        elif L["cin"] > 4:                            # G's last deconv: the narrow edge kernel's forward matrix
            nstat.add(N.round_tf32(wf))
        else:                                         # D's first conv: the narrow edge kernel's data-gradient matrix
            nstat.add(N.round_tf32(wb))
    print("\n### %s, B=%d, K=%d (gain %.1f, seed %d)\n" % (arch_name, batch, steps, gain, seed))
    print("| tensor | amax | log2(65504 / amax) | nonzero share < 2^-14 |")
    print("|---|---|---|---|")
    for k, v in st.items():
        print(v.row(k))
    print(wstat.row("packed weights of the GEMM layers (BN folded, TF32 rounded)"))
    print(nstat.row("packed weights of the narrow image-edge passes (TF32 rounded; FP16 inside edge_narrow_tc)"))
    logit = o["optimal_logit"]
    print("\nlogits: best mean %.2f, max %.2f" % (float(logit.mean()), float(logit.max())))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--arch", nargs="+", default=["dcgan64_l1", "dcgan32_l1"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    for a in args.arch:
        analyse(a, args.batch, args.steps)


if __name__ == "__main__":
    main()
