"""GPU parity for the cluster form of the 2-D MLP kernels (csrc/mlp2d_cluster.cu): hidden widths other than 64 against
the pinned numpy oracle, and the cluster form at nhidden = 64 against the one-SM kernels bit for bit."""
import types

import numpy as np
import pytest

from oracle import nets as onets
from oracle import sampling_np as snp

pytestmark = pytest.mark.gpu

SCALE = 10.0   # synthetic/run_shaping.sh:2  (--scale 10)


class _Data:
    def __init__(self, pts):
        self.pts = pts

    def next_batch(self, n):
        return self.pts[:n]


@pytest.mark.parametrize("nh", [16, 128, 208, 256])
@pytest.mark.parametrize("nlayers", [2, 3, 6, 8])
def test_wide_score_matches_oracle(cgs_lib, cuda_device, nh, nlayers):
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(nh, nlayers, seed=3)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(0)
    for n in (1, 63, 1000):
        x = (rng.randn(n, 2) * 4).astype(np.float32)
        sig_ref, sal_ref = onets.mlp2d_sigmoid_saliency(x, ws)
        sig, sal = mlp.score(x, want_saliency=True)
        assert np.abs(sig.cpu().numpy() - sig_ref).max() <= 2e-6
        assert np.abs(sal.cpu().numpy() - sal_ref).max() <= 2e-5 * np.abs(sal_ref).max()


def _sigmoid_saliency_f64(x, ws):
    """onets.mlp2d_sigmoid_saliency with FP64 accumulation, rounded to FP32 at the end: the reference trajectory of
    test_wide_refine_matches_oracle, which no FP32 summation order favours."""
    import torch
    import torch.nn.functional as F
    xt = torch.from_numpy(np.asarray(x, np.float64)).requires_grad_(True)
    net = xt
    for i, (k, b) in enumerate(ws):
        net = net @ torch.from_numpy(k.astype(np.float64)) + torch.from_numpy(b.astype(np.float64))
        if i < len(ws) - 1:
            net = torch.relu(net)
    (g,) = torch.autograd.grad(F.softplus(-net).mean(), xt)
    return torch.sigmoid(net).detach().numpy().astype(np.float32), g.numpy().astype(np.float32)


def _refiner(mlp, method, K, rate, real):
    from sampling.refiner_cpu import Refiner
    ref = Refiner(types.SimpleNamespace(rollout_steps=K, rollout_rate=rate, rollout_method=method))
    ref.set_env(mlp, None, _Data(real))
    return ref


@pytest.mark.parametrize("nh,method,K,n,nlayers", [(256, "ladam", 50, 1000, 6), (128, "momentum", 20, 500, 6),
                                                   (48, "sgd", 5, 64, 3), (256, "ladam", 4, 300, 8)])
def test_wide_refine_matches_oracle(cgs_lib, cuda_device, nh, method, K, n, nlayers):
    """Against the oracle's refine_2d run with FP64 accumulation, with the bars of BASELINE.md §5, or with what the
    pinned FP32 oracle itself reaches against that run where that is less.  At nh = 256, ladam K = 50 a few points
    are so sensitive to summation order that correct FP32 evaluations part by more than the bar: the pinned oracle
    misses it on 3 of the 1000 points (up to 1.2e-2), and the same oracle over the same net with its hidden units
    stored in another order misses it on 0 to 2 points (up to 3.4e-2).  The kernel is held to the oracle's own
    count plus one point; every other case here is well conditioned and keeps the plain bar."""
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(nh, nlayers, seed=2019, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(1)
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    real = (rng.randn(n, 2) * 3).astype(np.float32)
    real_sig, _ = onets.mlp2d_sigmoid_saliency(real, ws)
    rate = 0.1 if method == "ladam" else 50.0
    o = snp.refine_2d(x0, lambda x: _sigmoid_saliency_f64(x, ws), np.mean(real_sig), K, rate, method)
    o32 = snp.refine_2d(x0, lambda x: onets.mlp2d_sigmoid_saliency(x, ws), np.mean(real_sig), K, rate, method)
    ref = _refiner(mlp, method, K, rate, real)
    out = ref.manipulate_sample(x0, "deterministic")
    assert out.dtype == np.float32 and out.shape == (n, 2)
    # BASELINE.md §5: max-abs <= 1e-4 * scale, identical optimal_step for >= 99.9 % of samples
    bar = 1e-4 * SCALE
    ok = np.abs(out - o["optimal_batch"]).max(axis=1) <= bar
    ok32 = np.abs(o32["optimal_batch"] - o["optimal_batch"]).max(axis=1) <= bar
    same_step = np.mean(ref.optimal_step.cpu().numpy() == o["optimal_step"])
    same_step32 = np.mean(o32["optimal_step"] == o["optimal_step"])
    print(nh, method, K, n, "within the bar: kernel %d, FP32 oracle %d of %d; same optimal_step: kernel %.4f, FP32 "
          "oracle %.4f" % (ok.sum(), ok32.sum(), n, same_step, same_step32))
    assert ok.mean() >= min(0.999, ok32.mean()) - 1.0 / n
    assert same_step >= min(0.999, same_step32) - 1.0 / n


def test_wide_probabilistic_returns_float64_trajectory_rows(cgs_lib, cuda_device):
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(256, 6, seed=1, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(4)
    n, K = 300, 8
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    real = (rng.randn(n, 2) * 3).astype(np.float32)
    real_sig, _ = onets.mlp2d_sigmoid_saliency(real, ws)
    np.random.seed(11)
    idx = np.random.randint(K + 1, size=n)
    o = snp.refine_2d(x0, lambda x: onets.mlp2d_sigmoid_saliency(x, ws), np.mean(real_sig), K, 0.1, "ladam", idx)
    ref = _refiner(mlp, "ladam", K, 0.1, real)
    np.random.seed(11)
    out = ref.manipulate_sample(x0, "probabilistic")
    assert out.dtype == np.float64
    assert np.abs(out - o["probabilistic"]).max() <= 1e-4 * SCALE


@pytest.mark.parametrize("method,K,n,nlayers", [("ladam", 50, 10000, 6), ("momentum", 7, 97, 6), ("sgd", 3, 1, 3),
                                                ("ladam", 5, 20001, 2), ("ladam", 4, 300, 8)])
def test_cluster_form_is_bit_identical_at_64(cgs_lib, cuda_device, method, K, n, nlayers):
    """At nhidden = 64 the cluster form (DEBUG_MLP2D_CLUSTER) accumulates every element in the order of the one-SM
    kernels: same bits for the best point, its loss and step, the whole trajectory, and the score, logit and saliency."""
    import ctypes as C

    import torch
    from cgs import lib as L
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(64, nlayers, seed=7, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(2)
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    real = (rng.randn(max(n, 8), 2) * 3).astype(np.float32)
    rate = 0.1 if method == "ladam" else 50.0
    xt = torch.from_numpy(x0).to(cuda_device)

    def run(flags):
        with L.debug_flags(flags):
            ref = _refiner(mlp, method, K, rate, real)
            np.random.seed(3)
            det = ref.manipulate_sample(x0, "deterministic")
            step, loss = ref.optimal_step.cpu().numpy().copy(), ref.optimal_loss.cpu().numpy().copy()
            np.random.seed(3)
            prob = ref.manipulate_sample(x0, "probabilistic")          # reads the full trajectory
            sig = torch.empty(n, device=cuda_device)
            logit = torch.empty(n, device=cuda_device)
            sal = torch.empty(n, 2, device=cuda_device)
            L.check(L.load().cgs_mlp2d_score(C.byref(mlp.desc), L.ptr(xt), n, 3 * n, L.ptr(sig), L.ptr(logit),
                                             L.ptr(sal), L.stream_ptr()))
            sig_only = torch.empty(n, device=cuda_device)
            L.check(L.load().cgs_mlp2d_score(C.byref(mlp.desc), L.ptr(xt), n, 3 * n, L.ptr(sig_only), None, None,
                                             L.stream_ptr()))
            torch.cuda.synchronize()
            return det, step, loss, prob, sig.cpu().numpy(), logit.cpu().numpy(), sal.cpu().numpy(), \
                sig_only.cpu().numpy()

    a, b = run(0), run(L.DEBUG_MLP2D_CLUSTER)
    for u, v in zip(a, b):
        assert np.array_equal(np.asarray(u), np.asarray(v))


def test_wide_refine_is_batch_invariant(cgs_lib, cuda_device):
    """Each point's result depends on nothing but the point and n_mean: one call of 10^4 points and two calls of
    5000 with the same n_mean give the same bits."""
    import torch
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(256, 6, seed=5, gain=1.5)
    mlp = MlpSpec(ws, cuda_device)
    rng = np.random.RandomState(6)
    n = 10000
    x0 = (rng.randn(n, 2) * 4).astype(np.float32)
    ref = _refiner(mlp, "ladam", 10, 0.1, None)
    whole = ref.manipulate_sample(x0, "deterministic", n_mean=n, real_sigmoid_mean=0.5)
    step_whole = ref.optimal_step.cpu().numpy().copy()
    parts, steps = [], []
    for h in (slice(0, n // 2), slice(n // 2, n)):
        parts.append(ref.manipulate_sample(x0[h], "deterministic", n_mean=n, real_sigmoid_mean=0.5))
        steps.append(ref.optimal_step.cpu().numpy().copy())
    torch.cuda.synchronize()
    assert np.array_equal(whole, np.concatenate(parts))
    assert np.array_equal(step_whole, np.concatenate(steps))


@pytest.mark.parametrize("nh", [40, 272, 512])
def test_unsupported_widths_raise(cgs_lib, cuda_device, nh):
    from sampling.refiner_cpu import MlpSpec
    mlp = MlpSpec(onets.init_mlp2d(nh, 3, seed=0), cuda_device)
    x = np.zeros((4, 2), np.float32)
    with pytest.raises(NotImplementedError):
        mlp.score(x)
    with pytest.raises(NotImplementedError):
        _refiner(mlp, "ladam", 2, 0.1, None).manipulate_sample(x, real_sigmoid_mean=0.5)


def test_malformed_layers_raise(cgs_lib, cuda_device):
    from sampling.refiner_cpu import MlpSpec
    ws = onets.init_mlp2d(128, 4, seed=0)
    bad_kernel = list(ws)
    bad_kernel[2] = (ws[2][0][:, :64], ws[2][1])                 # 128 -> 64 in the middle
    bad_bias = list(ws)
    bad_bias[3] = (ws[3][0], np.zeros(2, np.float32))           # two biases for one output
    bad_input = list(ws)
    bad_input[0] = (np.zeros((3, 128), np.float32), ws[0][1])   # 3-D input
    for layers, name in ((bad_kernel, "layer 2"), (bad_bias, "layer 3"), (bad_input, "layer 0")):
        with pytest.raises(ValueError, match=name):
            MlpSpec(layers, cuda_device)
