"""GPU parity for the 2-D path: fused MLP score / refine kernel vs the pinned numpy oracle."""
import types

import numpy as np
import pytest
import torch

from oracle import nets as onets
from oracle import sampling_np as snp

pytestmark = pytest.mark.gpu

SCALE = 10.0   # synthetic/run_shaping.sh:2  (--scale 10)


class _Data:
    def __init__(self, pts):
        self.pts = pts

    def next_batch(self, n):
        return self.pts[:n]


@pytest.mark.parametrize("nlayers", [6, 3])
def test_score_matches_oracle(cgs_lib, cuda_device, nlayers):
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(64, nlayers, seed=3)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(0)
    for n in (1, 63, 1000):
        x = (rng.randn(n, 2) * 4).astype(np.float32)
        sig_ref, sal_ref = onets.mlp2d_sigmoid_saliency(x, ws)
        sig, sal = mlp.score(x, want_saliency=True)
        assert np.abs(sig.cpu().numpy() - sig_ref).max() <= 2e-6
        assert np.abs(sal.cpu().numpy() - sal_ref).max() <= 2e-5 * np.abs(sal_ref).max()


@pytest.mark.parametrize("method,K,n", [("ladam", 50, 1000), ("ladam", 10, 257), ("momentum", 20, 500), ("sgd", 5, 64)])
def test_refine_matches_oracle(cgs_lib, cuda_device, method, K, n):
    from sampling.refiner_cpu import MlpSpec, Refiner
    ws = onets.init_mlp2d(64, 6, seed=2019, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(1)
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    real = (rng.randn(n, 2) * 3).astype(np.float32)
    real_sig, _ = onets.mlp2d_sigmoid_saliency(real, ws)
    rate = 0.1 if method == "ladam" else 50.0
    o = snp.refine_2d(x0, lambda x: onets.mlp2d_sigmoid_saliency(x, ws), np.mean(real_sig), K, rate, method)
    args = types.SimpleNamespace(rollout_steps=K, rollout_rate=rate, rollout_method=method)
    ref = Refiner(args)
    ref.set_env(mlp, None, _Data(real))
    out = ref.manipulate_sample(x0, "deterministic")
    assert out.dtype == np.float32 and out.shape == (n, 2)
    err = np.abs(out - o["optimal_batch"]).max()
    same_step = np.mean(ref.optimal_step.cpu().numpy() == o["optimal_step"])
    moved = np.abs(o["optimal_batch"] - x0).max()
    print(method, K, n, "max-abs err %.3e  moved %.3f  same optimal_step %.4f" % (err, moved, same_step))
    # BASELINE.md §5: max-abs <= 1e-4 * scale, identical optimal_step for >= 99.9 % of samples
    ok = np.abs(out - o["optimal_batch"]).max(axis=1) <= 1e-4 * SCALE
    assert ok.mean() >= 0.999
    assert same_step >= 0.999 - 1.0 / n


def test_probabilistic_returns_float64_trajectory_rows(cgs_lib, cuda_device):
    from sampling.refiner_cpu import MlpSpec, Refiner
    ws = onets.init_mlp2d(64, 6, seed=1, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(4)
    n, K = 300, 8
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    real = (rng.randn(n, 2) * 3).astype(np.float32)
    real_sig, _ = onets.mlp2d_sigmoid_saliency(real, ws)
    np.random.seed(11)
    idx = np.random.randint(K + 1, size=n)
    o = snp.refine_2d(x0, lambda x: onets.mlp2d_sigmoid_saliency(x, ws), np.mean(real_sig), K, 0.1, "ladam", idx)
    ref = Refiner(types.SimpleNamespace(rollout_steps=K, rollout_rate=0.1, rollout_method="ladam"))
    ref.set_env(mlp, None, _Data(real))
    np.random.seed(11)
    out = ref.manipulate_sample(x0, "probabilistic")
    assert out.dtype == np.float64
    assert np.abs(out - o["probabilistic"]).max() <= 1e-4 * SCALE
    with pytest.raises(NotImplementedError):
        ref.manipulate_sample(x0, "greedy")


@pytest.mark.parametrize("method,K,n,nlayers", [("ladam", 50, 10000, 6), ("momentum", 7, 97, 6), ("sgd", 3, 1, 3),
                                                ("ladam", 5, 20001, 2), ("ladam", 4, 300, 8)])
def test_split_refine_kernel_is_bit_identical(cgs_lib, cuda_device, method, K, n, nlayers):
    """The split form (four threads per point, 16-wide layer slices exchanged through shared memory) accumulates every
    element in the order of the one-thread form (DEBUG_MLP2D_ONE_THREAD selects the latter): same bits for the best
    point, its loss and step, and the whole trajectory -- at the benchmark size, ragged sizes, a single point, more
    than 96 points per CTA round, the shallowest and the deepest MLP."""
    from cgs import lib as L
    from sampling.refiner_cpu import MlpSpec, Refiner
    ws = onets.init_mlp2d(64, nlayers, seed=7, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(2)
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    real = (rng.randn(max(n, 8), 2) * 3).astype(np.float32)
    rate = 0.1 if method == "ladam" else 50.0

    def run(flags):
        with L.debug_flags(flags):
            ref = Refiner(types.SimpleNamespace(rollout_steps=K, rollout_rate=rate, rollout_method=method))
            ref.set_env(mlp, None, _Data(real))
            np.random.seed(3)
            det = ref.manipulate_sample(x0, "deterministic")
            step, loss = ref.optimal_step.cpu().numpy().copy(), ref.optimal_loss.cpu().numpy().copy()
            np.random.seed(3)
            prob = ref.manipulate_sample(x0, "probabilistic")          # reads the full trajectory
            return det, step, loss, prob

    a, b = run(0), run(L.DEBUG_MLP2D_ONE_THREAD)
    for u, v in zip(a, b):
        assert np.array_equal(np.asarray(u), np.asarray(v))
