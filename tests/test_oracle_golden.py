"""Oracle vs the committed golden vectors (runs anywhere, no reference tree and no GPU needed).

tests/golden/sampling_ref.npz was produced by the reference's OWN sampling/*.py (oracle/make_golden.py), so these
tests pin the oracle: decisions / indices / state bit-for-bit, policy updates bit-for-bit."""
import os

import numpy as np
import pytest

from oracle import nets as onets
from oracle import sampling_np as snp

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "sampling_ref.npz"))


@pytest.mark.parametrize("tag", ["f32", "f64"])
def test_drs_matches_reference_vectors(gold, tag):
    m = snp.drs_score_max(gold["drs_%s_smax" % tag])
    assert float(m) == float(gold["drs_%s_M0" % tag])
    for call, sp in enumerate((100.0, 60.0, None)):
        sig, u = gold["drs_%s_%d_sig" % (tag, call)], gold["drs_%s_%d_u" % (tag, call)]
        acc, m = snp.drs_accept(sig, u, m, shift_percent=sp)
        assert np.array_equal(np.nonzero(acc)[0], gold["drs_%s_%d_accepted_rows" % (tag, call)])
        assert float(m) == float(gold["drs_%s_%d_M" % (tag, call)])


@pytest.mark.parametrize("tag,dt", [("f32", np.float32), ("f64", np.float64)])
@pytest.mark.parametrize("T,B", [(0, 0), (5, 3), (20, 0)])
def test_mh_matches_reference_vectors(gold, tag, dt, T, B):
    key = "mh_%s_T%d_B%d" % (tag, T, B)
    d, cnt = dt(gold[key + "_d0"]), 1
    for call in range(3):
        sig, u = gold["%s_%d_sig" % (key, call)], gold["%s_%d_u" % (key, call)]
        emit, d, cnt, _ = snp.mh_chain(sig, u, d, cnt, T, B)
        assert np.array_equal(emit, gold["%s_%d_emit" % (key, call)])
        assert float(np.squeeze(d)) == float(gold["%s_%d_d" % (key, call)])
        assert cnt == int(gold["%s_%d_cnt" % (key, call)])


@pytest.mark.parametrize("method", ["sgd", "momentum", "ladam"])
def test_policy_matches_reference_vectors(gold, method):
    theta = gold["policy_%s_theta0" % method].copy()
    state = snp.policy_new_state()
    for it in range(5):
        snp.policy_step(method, theta, gold["policy_%s_%d_grad" % (method, it)], state, 0.1,
                        gold["policy_%s_%d_loss" % (method, it)])
        assert np.array_equal(theta, gold["policy_%s_%d_theta" % (method, it)])


@pytest.mark.parametrize("K", [10, 50])
def test_refine2d_matches_reference_vectors(gold, K):
    """The reference refined these rows with the oracle MLP's float32 scores, whose last bits depend on the host's BLAS
    (kernel and thread count).  The scores it was fed are stored (oracle/make_golden.py refine2d_scores) and replayed,
    so the refinement loop is pinned bit for bit on any host; the MLP must reproduce them to float32 accuracy."""
    ws = onets.init_mlp2d(64, 6, seed=2019, gain=1.5)
    assert float(gold["r2d_mlp_checksum"]) == sum(float(np.abs(k).sum() + np.abs(b).sum()) for k, b in ws)
    key = "r2d_K%d" % K
    fed = np.load(os.path.join(GOLD, "refine2d_scores.npz"))
    rows, sig, sal = fed[key + "_rows"], fed[key + "_sig"], fed[key + "_sal"]
    n = len(gold[key + "_x0"])
    real_sig, _ = onets.mlp2d_sigmoid_saliency(gold[key + "_real"], ws)
    assert np.isclose(np.mean(real_sig), fed[key + "_real_mean"], rtol=1e-6, atol=0)
    calls = []

    def replay(x):
        i = len(calls)
        calls.append(i)
        s, a = onets.mlp2d_sigmoid_saliency(x, ws)
        a = a * np.float32(len(rows) / n)           # the saliency carries 1/rows fed; the reference fed all n
        np.testing.assert_allclose(s, sig[i], rtol=1e-5, atol=0)
        np.testing.assert_allclose(a, sal[i], rtol=1e-4, atol=1e-4 * float(np.abs(sal[i]).max()))
        return sig[i], sal[i]
    o = snp.refine_2d(gold[key + "_x0"][rows], replay, fed[key + "_real_mean"], K, 0.1, "ladam")
    assert len(calls) == K + 1 == len(sig)
    assert np.array_equal(o["optimal_batch"], gold[key + "_out"][rows])


def test_graph_refiner_fixture_is_reproducible():
    """The conv-path fixture is oracle output (parity unpinned by the reference); check it regenerates."""
    import torch
    from oracle import graph_refiner as gr
    g = np.load(os.path.join(GOLD, "graph_refiner.npz"))
    arch = onets.get_arch("mnist")
    B, K, gain = g["mnist_cfg"]
    w = onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=2019), float(gain))
    assert abs(sum(float(np.abs(v).sum()) for v in w.values()) - float(g["mnist_wsum"])) < 1e-6 * float(g["mnist_wsum"])
    o = gr.build_refiner(torch.from_numpy(g["mnist_h0"]), arch, w, int(K), 0.1)
    assert np.abs(o["refined"].numpy() - g["mnist_refined"]).max() <= 1e-5
    assert np.array_equal(o["optimal_step"].numpy(), g["mnist_optimal_step"])
