"""What the reference's own sampling modules return on the fixed-seed cases of ``tests/test_oracle_vs_reference.py`` and
``tests/test_fillup_cpu.py``.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Each ``*_case`` function builds a test's inputs from its seeds;
each ``*_reference`` function runs the reference (``ref`` = ``ref_shims.load_reference_sampling()``) on them and returns
its outputs.  ``record`` collects every case under flat keys; ``oracle/make_golden.py`` stores that as
``tests/golden/reference_cases.npz``, which the tests compare the oracle with wherever no checkout of the original is
present.  The reference's own arithmetic runs only where the original is checked out; none of it is restated here.
"""
from __future__ import annotations

import os

import numpy as np

from . import fillup_np as F
from . import ref_shims

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "reference_cases.npz")

DTYPES = {"f32": np.float32, "f64": np.float64}
DRS_SHIFTS = (100.0, 60.0, None, 100.0, 12.5)
MH_CHAINS = ((0, 0), (1, 0), (5, 2), (20, 0), (20, 5))
MH_SIZES = (900, 1, 333, 64)
POLICY_METHODS = ("sgd", "momentum", "ladam")
FILLUP_KINDS = ("rejection", "hastings")


def drs_case(dt):
    """(score_max, samples [1000,2], [(sig [1000,1], shift_percent)] per call)."""
    rng = np.random.RandomState(1)
    smax = np.amax(rng.beta(2, 5, size=200).astype(dt))
    samples = rng.randn(1000, 2).astype(np.float32)
    calls = []
    for call, sp in enumerate(DRS_SHIFTS):
        sig = rng.beta(2, 5, size=(1000, 1)).astype(dt)
        if call == 3:
            sig[17] = 1.0 - 1e-9
        calls.append((sig, sp))
    return smax, samples, calls


def drs_reference(ref, dt):
    smax, samples, calls = drs_case(dt)
    R = ref.rejector.Rejector()
    R.set_score_max(smax)
    out = {"M0": np.asarray(R.D_tilde_M)}
    for call, (sig, sp) in enumerate(calls):
        np.random.seed(call)
        out["%d_good" % call] = np.asarray(R.sampling(samples, sig, shift_percent=sp))
        out["%d_M" % call] = np.asarray(R.D_tilde_M)
    return out


def mh_case(dt, T, B):
    """(initial score, [(sig [n,1], samples [n,3])] per call)."""
    rng = np.random.RandomState(T + 7 * B)
    d0 = np.mean(rng.beta(2, 5, size=64).astype(dt))
    calls = []
    for n in MH_SIZES:
        sig = rng.beta(2, 5, size=(n, 1)).astype(dt)
        calls.append((sig, rng.randn(n, 3).astype(np.float32)))
    return d0, calls


def mh_reference(ref, dt, T, B):
    d0, calls = mh_case(dt, T, B)
    S = ref.idpsampler.IndependenceSampler(T=T, B=B)
    S.set_score_curr(d0)
    out = {"d0": np.asarray(S.d_curr), "cnt0": np.asarray(S.cnt_chain)}
    for call, (sig, samples) in enumerate(calls):
        np.random.seed(call)
        out["%d_good" % call] = np.asarray(S.sampling(samples, sig))
        out["%d_d" % call] = np.asarray(np.squeeze(S.d_curr), dtype=np.float64)
        out["%d_cnt" % call] = np.asarray(S.cnt_chain)
    return out


def policy_case():
    """(theta [100,2], [(grad, loss)] per step)."""
    rng = np.random.RandomState(5)
    theta = (rng.randn(100, 2)).astype(np.float32)
    steps = []
    for _ in range(4):
        g = rng.randn(100, 2).astype(np.float32) * 1e-3
        steps.append((g, (rng.rand(100) - .5).astype(np.float32)))
    return theta, steps


def policy_reference(ref, method):
    theta, steps = policy_case()
    P = ref.policy.PolicyAdaptive(0.1, method)
    out = {}
    for i, (g, l) in enumerate(steps):
        P.apply_gradient(theta, g, l)
        out["%d_theta" % i] = theta.copy()
    try:
        ref.policy.PolicyAdaptive(0.1, "nope").apply_gradient(theta, theta)
        out["unknown_method_raises"] = np.asarray(False)
    except NotImplementedError:
        out["unknown_method_raises"] = np.asarray(True)
    return out


def fillup_stream(seed, dim=3):
    rng = np.random.RandomState(seed)

    def propose(n):
        x = rng.randn(n, dim).astype(np.float32)
        s = rng.beta(2, 5, size=(n, 1)).astype(np.float32)
        return x, s
    return propose


def fillup_run(kind, rejector_cls, sampler_cls):
    """nsgan fill-up loop (oracle/fillup_np.py) over the given sampler classes, eval size 200, batches of 32."""
    propose = fillup_stream(3)
    base_x, base_s = propose(200)
    np.random.seed(11)
    if kind == "rejection":
        smp = rejector_cls()
        smp.set_score_max(np.float32(0.9))
        return F.fill_up_nsgan(base_x, base_s, propose, lambda x, s: smp.sampling(x, s, shift_percent=100.0), 200, 32,
                               store_guard="running")
    smp = sampler_cls(T=3)
    smp.set_score_curr(np.float32(0.3))
    return F.fill_up_nsgan(base_x, base_s, propose, smp.sampling, 200, 32, store_guard="batch")


def fillup_reference(ref, kind):
    r = fillup_run(kind, ref.rejector.Rejector, ref.idpsampler.IndependenceSampler)
    return {k: np.asarray(r[k]) for k in ("samples", "cnt", "cnt_propose", "n_backfilled")}


def cases():
    """(name, function, args) of every recorded case."""
    out = [("drs_%s" % t, drs_reference, (dt,)) for t, dt in DTYPES.items()]
    out += [("mh_%s_T%d_B%d" % (t, T, B), mh_reference, (dt, T, B)) for t, dt in DTYPES.items() for T, B in MH_CHAINS]
    out += [("policy_%s" % m, policy_reference, (m,)) for m in POLICY_METHODS]
    out += [("fillup_%s" % k, fillup_reference, (k,)) for k in FILLUP_KINDS]
    return out


def record(ref):
    """Every case's reference outputs under '<case>__<output>' keys."""
    g = {}
    for name, fn, args in cases():
        for k, v in fn(ref, *args).items():
            g[name + "__" + k] = v
    return g


def expected(name):
    """The reference's outputs for case ``name``: computed where the original is checked out, else the ones stored in
    GOLDEN; None when neither is available."""
    fn, args = {n: (f, a) for n, f, a in cases()}[name]
    if ref_shims.reference_available():
        return fn(ref_shims.load_reference_sampling(), *args)
    if not os.path.exists(GOLDEN):
        return None
    with np.load(GOLDEN) as g:
        return {k.split("__", 1)[1]: g[k] for k in g.files if k.split("__", 1)[0] == name}
