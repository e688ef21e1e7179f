"""Small end-to-end run of the image path for compute-sanitizer (memcheck / racecheck): every round-2 kernel once --
class-fused tcgen05 tiles (forced), tcgen05 edge kernels on the s2d layout, device-side early exit, graph replay."""
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "collaborative-gan-sampling_b200"))
import torch
from cgs import lib as L, nets as N, synthetic as S
from sampling.collaborator import Refiner

lib = L.load()
dev = torch.device("cuda", 0)
# default rules / class-fused tiles whenever legal / class fusion + M-tile pairs / CTA pairs (cta_group::2) whenever legal
FUSE, MPAIR, CPAIR = L.DEBUG_FORCE_FUSION, L.DEBUG_FORCE_MTILE_PAIRS, L.DEBUG_FORCE_CTA_PAIRS
for flags, name, B, thr in ((0, "dcgan64_l1", 5, None), (FUSE, "dcgan64_l1", 5, None), (FUSE, "dcgan32_l2", 6, None),
                            (FUSE | MPAIR, "dcgan64_l3", 3, 0.0), (MPAIR, "dcgan32_l4", 4, None),
                            (FUSE | CPAIR, "dcgan64_l1", 5, None), (CPAIR, "dcgan32_l2", 7, 0.0),
                            (CPAIR | MPAIR | L.DEBUG_NO_FUSION, "dcgan64_l2", 9, None),
                            (FUSE, "mnist", 20, 0.1)):
    with L.debug_flags(flags):
        arch = N.get_arch(name)
        spec = N.NetSpec(arch, S.init_weights(arch, gain=3.0 if name == "mnist" else 2.5), dev)
        r = Refiner(3, 0.1)
        r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        r.early_exit_logit = thr
        h0 = torch.from_numpy(S.proposal_features(arch, B, seed=1)).to(dev)
        x = r.build_refiner(h0)
        torch.cuda.synchronize()
    print(flags, name, "ok", tuple(x.shape), float(r.optimal_logit.mean()))
# 2-D refinement: split form (four threads per point, named barriers) and the one-thread form
import types
import numpy as np
from sampling.refiner_cpu import MlpSpec, Refiner as Refiner2d


class _Data:
    def __init__(self, pts):
        self.pts = pts

    def next_batch(self, n):
        return self.pts[:n]


rng = np.random.RandomState(0)
mlp = MlpSpec(S.init_mlp2d(64, 6, seed=3, gain=1.5), dev)
for flags, n in ((0, 333), (0, 20000), (L.DEBUG_MLP2D_ONE_THREAD, 333)):
    with L.debug_flags(flags):
        r2 = Refiner2d(types.SimpleNamespace(rollout_steps=4, rollout_rate=0.1, rollout_method="ladam"))
        r2.set_env(mlp, None, _Data((rng.randn(n, 2) * 3).astype(np.float32)))
        out = r2.manipulate_sample((rng.randn(n, 2) * 4).astype(np.float32), "probabilistic")
    print(flags, "2-D", n, "ok", out.shape)
print("launches", lib.cgs_launch_count())
