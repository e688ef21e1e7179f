"""Oracle vs the reference's own modules: executed in place where the original project is checked out, else through
the outputs oracle/make_golden.py recorded from it (tests/golden/reference_cases.npz, see oracle/ref_cases.py)."""
import types

import numpy as np
import pytest

from oracle import nets as onets
from oracle import ref_cases as rc
from oracle import ref_shims
from oracle import sampling_np as snp


@pytest.fixture(scope="module")
def ref():
    if not ref_shims.reference_available():
        pytest.skip(ref_shims.SKIP_REASON)
    return ref_shims.load_reference_sampling()


def expected(name):
    out = rc.expected(name)
    if out is None:
        pytest.skip(ref_shims.SKIP_REASON + " and no recorded outputs (python -m oracle.make_golden)")
    return out


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_drs_bit_exact(dt):
    exp = expected("drs_%s" % ("f32" if dt == np.float32 else "f64"))
    _, samples, calls = rc.drs_case(dt)
    m = exp["M0"][()]
    for call, (sig, sp) in enumerate(calls):
        np.random.seed(call)
        acc, m = snp.drs_accept(sig, np.random.rand(1000), m, shift_percent=sp)
        assert np.array_equal(samples[acc], exp["%d_good" % call])
        assert float(m) == float(exp["%d_M" % call])


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("T,B", [(0, 0), (1, 0), (5, 2), (20, 0), (20, 5)])
def test_mh_bit_exact_with_carried_state(dt, T, B):
    exp = expected("mh_%s_T%d_B%d" % ("f32" if dt == np.float32 else "f64", T, B))
    _, calls = rc.mh_case(dt, T, B)
    d, cnt = exp["d0"][()], int(exp["cnt0"])
    for call, (sig, samples) in enumerate(calls):
        n = len(sig)
        np.random.seed(call)
        emit, d, cnt, _ = snp.mh_chain(sig, np.random.rand(n), d, cnt, T, B)
        got = samples[emit] if len(emit) else np.zeros((0,), np.float32)
        assert np.array_equal(got.astype(np.float32), exp["%d_good" % call])
        assert cnt == int(exp["%d_cnt" % call]) and float(np.squeeze(d)) == float(exp["%d_d" % call])


def test_mh_uniform_stream_equals_rand():
    np.random.seed(3)
    a = np.array([np.random.uniform(0, 1) for _ in range(50)])
    np.random.seed(3)
    assert np.array_equal(a, np.random.rand(50))


@pytest.mark.parametrize("method", ["sgd", "momentum", "ladam"])
def test_policy_bit_exact(method):
    exp = expected("policy_%s" % method)
    b, steps = rc.policy_case()
    st = snp.policy_new_state()
    for i, (g, l) in enumerate(steps):
        snp.policy_step(method, b, g, st, 0.1, l)
        assert np.array_equal(exp["%d_theta" % i], b)
    assert bool(exp["unknown_method_raises"])
    with pytest.raises(NotImplementedError):
        snp.policy_step("nope", b, b, snp.policy_new_state(), 0.1)


@pytest.mark.parametrize("mode", ["deterministic", "probabilistic"])
def test_refiner_cpu_bit_exact(ref, mode):
    ws = onets.init_mlp2d(64, 6, seed=4, gain=1.5)
    sess = ref_shims.FakeSession(ws)
    data = ref.Datasets.ToyDataset("Imbal-8Gaussians", scale=10, ratio=0.9)
    K, n = 12, 400
    Rf = ref.refiner_cpu.Refiner(types.SimpleNamespace(rollout_steps=K, rollout_rate=0.1, rollout_method="ladam"))
    Rf.set_env(ref_shims.FakeGan, sess, data)
    x0 = (np.random.RandomState(0).randn(n, 2) * 4).astype(np.float32)
    np.random.seed(9)
    out = Rf.manipulate_sample(x0, mode)
    assert sess.calls == K + 2                       # K+2 host<->runtime crossings per call (SURVEY 3.2)
    np.random.seed(9)
    real = data.next_batch(n)
    rs, _ = onets.mlp2d_sigmoid_saliency(real.astype(np.float32), ws)
    idx = np.random.randint(K + 1, size=n) if mode == "probabilistic" else None
    o = snp.refine_2d(x0, lambda x: onets.mlp2d_sigmoid_saliency(x, ws), np.mean(rs), K, 0.1, "ladam", idx)
    exp = o["probabilistic"] if mode == "probabilistic" else o["optimal_batch"]
    assert out.dtype == exp.dtype and np.array_equal(out, exp)
