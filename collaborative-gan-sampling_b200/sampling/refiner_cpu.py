"""Drop-in for the reference's ``sampling/refiner_cpu.py`` (host-loop refiner of the 2-D path).

Same names as ``sampling/refiner_cpu.py:6-81``: ``Refiner(args)`` (``args.rollout_steps / rollout_rate /
rollout_method``), ``set_env(gan, sess, data)``, ``manipulate_sample(fake_batch, mode='deterministic')``.
The reference crosses host<->TF K+2 times per call; here the whole K-step loop is ONE kernel
(``cgs_refine_mlp2d``).  ``gan`` must expose the discriminator MLP weights (``MlpSpec`` below, or any object
with a ``d_mlp`` attribute holding one); ``sess`` is accepted for signature compatibility and ignored;
``data.next_batch(n)`` is called exactly as the reference does (refiner_cpu.py:22), so it consumes
``np.random`` identically.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

try:
    from . import _paths  # noqa: F401
    from .policy import PolicyAdaptive
except ImportError:
    import _paths  # noqa: F401
    from policy import PolicyAdaptive
from cgs import lib as L
from cgs import runtime as R


class MlpSpec:
    """The 2-D discriminator MLP of synthetic/GAN.py:28-37 as device tensors.

    ``layers`` = [(kernel [in,out], bias [out]), ...] in TF ``tf.layers.dense`` layout, first 2->nhidden,
    last nhidden->1.
    """

    def __init__(self, layers, device=None):
        dev = torch.device(device) if device is not None else R.require_cuda()
        self.device = dev
        self.nlayers = len(layers)
        self.nhidden = int(np.asarray(layers[0][0]).shape[1]) if not isinstance(layers[0][0], torch.Tensor) \
            else int(layers[0][0].shape[1])
        self.tensors = []
        self.desc = L.MlpDesc()
        self.desc.nlayers = self.nlayers
        self.desc.nhidden = self.nhidden
        if self.nlayers > L.MLP_MAX_LAYERS:
            raise NotImplementedError("at most %d layers" % L.MLP_MAX_LAYERS)
        # the kernels read every layer at the shape nlayers and nhidden imply: check it before they do
        nh = self.nhidden
        for i, (k, b) in enumerate(layers):
            want = (2 if i == 0 else nh, 1 if i == self.nlayers - 1 else nh)
            ks, bs = tuple(np.shape(k)), tuple(np.shape(b))
            if ks != want or bs != want[1:]:
                raise ValueError("layer %d: kernel %s and bias %s, expected %s and %s" % (i, ks, bs, want, want[1:]))
        for i, (k, b) in enumerate(layers):
            kt, _ = R.to_device(k, torch.float32, dev)
            bt, _ = R.to_device(b, torch.float32, dev)
            self.tensors += [kt, bt]
            self.desc.weights[i] = kt.data_ptr()
            self.desc.biases[i] = bt.data_ptr()

    def score(self, x, n_mean=None, want_saliency=False):
        """(fake_sigmoid [N,1], fake_saliency [N,2] | None) for a batch -- synthetic/GAN.py:108-111."""
        xt, _ = R.to_device(x, torch.float32, self.device)
        n = xt.shape[0]
        sig = torch.empty(n, 1, dtype=torch.float32, device=self.device)
        sal = torch.empty(n, 2, dtype=torch.float32, device=self.device) if want_saliency else None
        L.check(L.load().cgs_mlp2d_score(C.byref(self.desc), L.ptr(xt), n, int(n_mean or n), L.ptr(sig), None,
                                         L.ptr(sal), L.stream_ptr()))
        return sig, sal


def _mlp_of(gan):
    if isinstance(gan, MlpSpec):
        return gan
    if hasattr(gan, "d_mlp"):
        return gan.d_mlp
    raise TypeError("gan must be an MlpSpec or expose one as .d_mlp (the TF graph handles of the reference "
                    "cannot be fused into a kernel)")


class Refiner():
    def __init__(self, args):
        self.forward_steps = args.rollout_steps
        self.step_size = args.rollout_rate
        self.method = args.rollout_method
        self.policy = PolicyAdaptive(self.step_size, self.method)
        self.optimal_step = None
        self.optimal_loss = None

    def set_env(self, gan, sess, data):
        self.sess = sess
        self.gan = gan
        self.data = data

    def manipulate_sample(self, fake_batch, mode='deterministic', n_mean=None, real_sigmoid_mean=None):
        if mode not in ('deterministic', 'probabilistic'):
            raise NotImplementedError                                   # refiner_cpu.py:81
        mlp = _mlp_of(self.gan)
        lib = L.load()
        x, x_np = R.to_device(fake_batch, torch.float32, mlp.device)
        n = x.shape[0]
        if real_sigmoid_mean is None:
            # real reference (refiner_cpu.py:22-23); the mean is taken on the host in FP32 like np.mean
            real_batch = self.data.next_batch(n)
            real_sig, _ = mlp.score(np.asarray(real_batch, dtype=np.float32))
            real_sigmoid_mean = np.mean(real_sig.cpu().numpy())
        cfg = L.Refine2dCfg()
        cfg.steps = int(self.forward_steps)
        cfg.policy = self.policy.config()
        cfg.n_mean = int(n_mean or n)
        cfg.real_sigmoid_mean = float(real_sigmoid_mean)
        best_x = torch.empty_like(x)
        best_loss = torch.empty(n, dtype=torch.float32, device=x.device)
        best_step = torch.empty(n, dtype=torch.float32, device=x.device)
        traj = None
        if mode == 'probabilistic':
            traj = torch.empty(n, cfg.steps + 1, 3, dtype=torch.float32, device=x.device)
        L.check(lib.cgs_refine_mlp2d(C.byref(mlp.desc), C.byref(cfg), L.ptr(x), n, L.ptr(best_x), L.ptr(best_loss),
                                     L.ptr(best_step), L.ptr(traj), L.stream_ptr()))
        self.policy.reset_moving_average()                               # refiner_cpu.py:69
        self.optimal_step, self.optimal_loss = best_step, best_loss
        if mode == 'probabilistic':
            indices_batch = np.random.randint(self.forward_steps + 1, size=n)      # refiner_cpu.py:72
            idx = torch.from_numpy(indices_batch).to(x.device)
            picked = traj[torch.arange(n, device=x.device), idx, :2].to(torch.float64)   # refiner_cpu.py:73-75
            return R.back(picked, x_np)
        return R.back(best_x, x_np)
