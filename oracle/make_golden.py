"""Generate tests/golden/*.npz (TEST INFRASTRUCTURE).  Needs a checkout of the original project (/root/reference, or
the directory CGS_REFERENCE_ROOT names):

    python -m oracle.make_golden

* sampling_ref.npz   -- outputs of the reference's OWN sampling/{policy,rejector,idpsampler,refiner_cpu}.py
                        (imported with the shims of oracle/ref_shims.py) on seeded inputs: these PIN the oracle.
* graph_refiner.npz  -- outputs of the oracle's torch restatement of sampling/collaborator.py on seeded inputs
                        (parity unpinned by the reference: it ships no vectors and TF 1.13 cannot run here).
* reference_cases.npz -- outputs of the reference's OWN sampling/{policy,rejector,idpsampler}.py on the fixed-seed cases
                        of tests/test_oracle_vs_reference.py and tests/test_fillup_cpu.py (oracle/ref_cases.py).
* refine2d_scores.npz -- the MLP scores behind sampling_ref.npz's 2-D refiner runs, recorded on the host that made
                        them (`python -m oracle.make_golden refine2d` records only these).
Weights are regenerated from their seed; a checksum is stored to catch initialiser drift.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

from . import graph_refiner as gr
from . import nets, ref_cases, ref_shims, sampling_np

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def sampling_ref():
    ref = ref_shims.load_reference_sampling()
    rng = np.random.RandomState(20191)
    g = {}
    # ---- DRS: three consecutive calls (state carried), fp32 and fp64 scores, shift 100 / 60 / None
    for tag, dt in (("f32", np.float32), ("f64", np.float64)):
        R = ref.rejector.Rejector()
        smax = np.amax(rng.beta(2, 5, size=128).astype(dt))
        R.set_score_max(smax)
        g["drs_%s_smax" % tag] = np.asarray(smax)
        g["drs_%s_M0" % tag] = np.asarray(R.D_tilde_M)
        for call, sp in enumerate((100.0, 60.0, None)):
            n = (777, 1000, 33)[call]
            sig = rng.beta(2, 5, size=(n, 1)).astype(dt)
            if call == 1:
                sig[5] = 0.9999        # above the running max: App. A9 collapse
            samples = np.arange(n, dtype=np.float32).reshape(n, 1)
            np.random.seed(900 + call)
            good = R.sampling(samples, sig, shift_percent=sp)
            np.random.seed(900 + call)
            u = np.random.rand(n)
            g["drs_%s_%d_sig" % (tag, call)] = sig
            g["drs_%s_%d_u" % (tag, call)] = u
            g["drs_%s_%d_accepted_rows" % (tag, call)] = good[:, 0].astype(np.int64)
            g["drs_%s_%d_M" % (tag, call)] = np.asarray(R.D_tilde_M)
    # ---- MH: T in {0,5,20}, burn-in {0,3}, three consecutive calls
    for tag, dt in (("f32", np.float32), ("f64", np.float64)):
        for T, B in ((0, 0), (5, 3), (20, 0)):
            S = ref.idpsampler.IndependenceSampler(T=T, B=B)
            d0 = np.mean(rng.beta(2, 5, size=100).astype(dt))
            S.set_score_curr(d0)
            key = "mh_%s_T%d_B%d" % (tag, T, B)
            g[key + "_d0"] = np.asarray(d0)
            for call in range(3):
                n = (1500, 1, 700)[call]
                sig = rng.beta(2, 5, size=(n, 1)).astype(dt)
                samples = np.arange(n, dtype=np.float32).reshape(n, 1)
                np.random.seed(300 + call)
                good = S.sampling(samples, sig)
                np.random.seed(300 + call)
                u = np.random.rand(n)
                g["%s_%d_sig" % (key, call)] = sig
                g["%s_%d_u" % (key, call)] = u
                g["%s_%d_emit" % (key, call)] = good.reshape(-1).astype(np.int64)
                g["%s_%d_d" % (key, call)] = np.asarray(np.squeeze(S.d_curr), dtype=np.float64)
                g["%s_%d_cnt" % (key, call)] = np.asarray(S.cnt_chain)
    # ---- policy: 5 steps of each method on a [200,2] array
    for method in ("sgd", "momentum", "ladam"):
        P = ref.policy.PolicyAdaptive(0.1, method)
        theta = (rng.randn(200, 2) * 3).astype(np.float32)
        g["policy_%s_theta0" % method] = theta.copy()
        for it in range(5):
            grad = (rng.randn(200, 2) * 10 ** rng.uniform(-6, 0, size=(200, 1))).astype(np.float32)
            loss = (rng.rand(200) - 0.5).astype(np.float32)
            P.apply_gradient(theta, grad, loss)
            g["policy_%s_%d_grad" % (method, it)] = grad
            g["policy_%s_%d_loss" % (method, it)] = loss
            g["policy_%s_%d_theta" % (method, it)] = theta.copy()
    # ---- 2-D refiner: the reference's refiner_cpu over the oracle MLP (FakeSession shim)
    ws = nets.init_mlp2d(64, 6, seed=2019, gain=1.5)
    g["r2d_mlp_checksum"] = np.asarray(sum(float(np.abs(k).sum() + np.abs(b).sum()) for k, b in ws))
    data = ref.Datasets.ToyDataset("Imbal-8Gaussians", scale=10, ratio=0.9)
    for K, n in ((10, 300), (50, 1000)):
        args = types.SimpleNamespace(rollout_steps=K, rollout_rate=0.1, rollout_method="ladam")
        Rf = ref.refiner_cpu.Refiner(args)
        Rf.set_env(ref_shims.FakeGan, ref_shims.FakeSession(ws), data)
        x0 = (rng.randn(n, 2) * 4).astype(np.float32)
        np.random.seed(77)
        real = data.next_batch(n)
        np.random.seed(77)
        out = Rf.manipulate_sample(x0, "deterministic")
        key = "r2d_K%d" % K
        g[key + "_x0"] = x0
        g[key + "_real"] = real.astype(np.float32)
        g[key + "_out"] = out
    np.savez_compressed(os.path.join(OUT, "sampling_ref.npz"), **g)
    return len(g)


def graph_ref():
    g = {}
    for name, B, K, gain in (("mnist", 4, 3, 3.0), ("dcgan32_l2", 2, 2, 2.5), ("dcgan64_l1", 2, 2, 2.5)):
        arch = nets.get_arch(name)
        w = nets.scale_weights_for_signal(arch, nets.init_weights(arch, seed=2019), gain)
        g[name + "_wsum"] = np.asarray(sum(float(np.abs(v).sum()) for v in w.values()))
        h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(11)))
        o = gr.build_refiner(h0, arch, w, K, 0.1)
        g[name + "_h0"] = h0.numpy()
        g[name + "_refined"] = o["refined"].numpy()
        g[name + "_optimal_logit"] = o["optimal_logit"].numpy()
        g[name + "_default_logit"] = o["default_logit"].numpy()
        g[name + "_optimal_step"] = o["optimal_step"].numpy()
        g[name + "_final_feature"] = o["final_feature"].numpy()
        g[name + "_cfg"] = np.asarray([B, K, gain])
    np.savez_compressed(os.path.join(OUT, "graph_refiner.npz"), **g)
    return len(g)


def reference_cases():
    g = ref_cases.record(ref_shims.load_reference_sampling())
    np.savez_compressed(ref_cases.GOLDEN, **g)
    return len(g)


def refine2d_scores():
    """The MLP scores the reference's 2-D refiner was fed at every step of sampling_ref.npz's r2d_* runs.

    The oracle MLP runs in float32 on torch-CPU, whose last bits depend on the host's BLAS kernel and thread count, so
    the recorded r2d_*_out reproduce only on a host like the one that made them.  Run on such a host (checked below),
    this stores what the MLP returned there; the test replays it, which pins the refinement loop on any host.  The
    loop treats rows independently, so the K=50 run keeps a seeded sample of its rows (the file stays small)."""
    gold = np.load(os.path.join(OUT, "sampling_ref.npz"))
    ws = nets.init_mlp2d(64, 6, seed=2019, gain=1.5)
    g = {}
    for K, n_rows in ((10, None), (50, 200)):
        key = "r2d_K%d" % K
        calls = []

        def score(x):
            calls.append(nets.mlp2d_sigmoid_saliency(x, ws))
            return calls[-1]
        real_sig, _ = nets.mlp2d_sigmoid_saliency(gold[key + "_real"], ws)
        o = sampling_np.refine_2d(gold[key + "_x0"], score, np.mean(real_sig), K, 0.1, "ladam")
        if not np.array_equal(o["optimal_batch"], gold[key + "_out"]):
            raise RuntimeError("this host's float32 MLP does not reproduce %s_out: record on the host that made it" % key)
        n = len(gold[key + "_x0"])
        rows = np.arange(n) if n_rows is None else np.sort(np.random.RandomState(K).choice(n, n_rows, replace=False))
        g[key + "_rows"] = rows
        g[key + "_real_mean"] = np.asarray(np.mean(real_sig))
        g[key + "_sig"] = np.stack([s[rows] for s, _ in calls])
        g[key + "_sal"] = np.stack([a[rows] for _, a in calls])
    np.savez_compressed(os.path.join(OUT, "refine2d_scores.npz"), **g)
    return len(g)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if sys.argv[1:] != ["refine2d"]:          # `refine2d`: only re-record the scores (no reference checkout needed)
        print("sampling_ref.npz:", sampling_ref(), "arrays")
        print("graph_refiner.npz:", graph_ref(), "arrays")
        print("reference_cases.npz:", reference_cases(), "arrays")
    print("refine2d_scores.npz:", refine2d_scores(), "arrays")
