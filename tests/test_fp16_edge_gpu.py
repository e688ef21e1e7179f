"""The image-edge passes of the FP16 operand chain (DESIGN.md §2, §4.1c).

In an FP16 chain the 64-channel tensors on the narrow side of the image-edge layers are FP16 too: G's last hidden
activation, read by the narrow forward pass (edge_narrow_tc's FP16 form), and d loss / d (D's first conv output), read
by the narrow data-gradient pass; the wide data-gradient pass reads its derivative operand (G's last hidden
activation) as FP16.  The refined feature stays FP32, so a one-layer G tail keeps the TF32 form for its narrow forward
pass.  The reference is the TF32 operand chain (CGS_DEBUG_TF32_OPERANDS), with the K = 50 TF32 tolerances of
tests/test_k50_parity_gpu.py.
"""
import numpy as np
import pytest
import torch

from oracle import graph_refiner as gr
from oracle import nets as onets
from parity_metrics import k50_metrics

pytestmark = pytest.mark.gpu

TOL = dict(img_rel_l2=1e-2, img_max_abs=0.4, logit_frac=0.02, logit_floor=0.05, step=0.95)


def _setup(name, B, seed=2):
    from cgs import nets as N
    arch = N.get_arch(name)
    w = onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=9), 2.5)
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(seed)))
    return arch, w, h0


def _refiner(arch, w, dev, K):
    from cgs import nets as N
    from sampling.collaborator import Refiner
    spec = N.NetSpec(arch, w, dev, math="tf32")
    ref = Refiner(K, 0.1, "momentum")
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    return ref


def _refine(arch, w, h0, dev, flags, K=50, exit_logit=None):
    from cgs import lib as L
    with L.debug_flags(flags):
        ref = _refiner(arch, w, dev, K)
        ref.early_exit_logit = exit_logit
        x = ref.build_refiner(h0.to(dev), None, "deterministic")
        torch.cuda.synchronize()
    return dict(refined=x.cpu().numpy(), optimal_logit=ref.optimal_logit.cpu().numpy(),
                optimal_step=ref.optimal_step.cpu().numpy(), default_logit=ref.default_logit.cpu().numpy())


def _narrow_forms(arch, w, h0, dev, flags):
    """Parameter type of every edge_narrow_tc_kernel launch of a K = 1 refinement, in launch order."""
    from cgs import lib as L
    with L.debug_flags(flags):
        ref = _refiner(arch, w, dev, 1)
        ref.build_refiner(h0.to(dev))
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            ref.build_refiner(h0.to(dev))
            torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                 and "edge_narrow_tc_kernel" in e.name), key=lambda e: e.time_range.start)
    return ["fp16" if "NarrowTc16Params" in e.name else "tf32" for e in ev]


@pytest.mark.parametrize("name,flags,expect", [
    ("dcgan64_l1", 0, ["fp16", "fp16", "fp16"]),                    # forward, data-gradient, forward
    ("dcgan64_l4", 0, ["tf32", "fp16", "tf32"]),                    # narrow forward over the FP32 refined feature
    ("dcgan64_l1", "TF32_OPERANDS", ["tf32", "tf32", "tf32"]),
])
def test_narrow_kernel_form(cgs_lib, cuda_device, name, flags, expect):
    from cgs import lib as L
    arch, w, h0 = _setup(name, 4)
    assert _narrow_forms(arch, w, h0, cuda_device, getattr(L, "DEBUG_" + flags) if flags else 0) == expect


@pytest.mark.parametrize("name,B", [("dcgan32_l1", 64), ("dcgan64_l1", 32), ("dcgan64_l4", 32)])
def test_fp16_edge_chain_matches_tf32_chain_at_k50(cgs_lib, cuda_device, name, B):
    from cgs import lib as L
    arch, w, h0 = _setup(name, B)
    ref = _refine(arch, w, h0, cuda_device, L.DEBUG_TF32_OPERANDS)
    got = _refine(arch, w, h0, cuda_device, 0)
    assert any(not np.array_equal(got[k], ref[k]) for k in got)
    m = k50_metrics(ref, got, onets.get_arch(name), w)
    print(name, m)
    assert m["img_rel_l2"] <= TOL["img_rel_l2"] and m["img_max_abs"] <= TOL["img_max_abs"], m
    assert m["optimal_logit_max_abs"] <= max(TOL["logit_floor"], TOL["logit_frac"] * abs(m["logit_gain_mean_ref"])), m
    assert m["optimal_step_agree"] >= TOL["step"], m
    assert m["logit_gain_mean_ref"] > 1.0


@pytest.mark.parametrize("name,B", [("dcgan32_l1", 4), ("dcgan64_l1", 3), ("dcgan64_l3", 3), ("dcgan64_l4", 3)])
def test_forward_logits_and_grad_fp16_edge(cgs_lib, cuda_device, name, B):
    """One forward + data-gradient chain against the CPU oracle, held to the single-pass TF32 bars of
    tests/test_conv_gpu.py (gradient rel-L2 8e-2, logits 1.5e-2)."""
    arch, w, _ = _setup(name, B)
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(1)))
    logit_ref, grad_ref, _ = gr.forward_logits_and_grad(h0, arch, w)
    logit, grad = _refiner(arch, w, cuda_device, 1).compute_forward_logits_and_grad(h0.to(cuda_device))
    g, gref = grad.cpu().double().numpy(), grad_ref.double().numpy()
    rel = float(np.linalg.norm(g - gref) / np.linalg.norm(gref))
    lerr = float(np.abs(logit.cpu().numpy() - logit_ref.numpy()).max())
    print(name, "grad rel %.2e logit %.2e" % (rel, lerr))
    assert rel <= 8e-2
    assert lerr <= 1.5e-2 * max(1.0, float(np.abs(logit_ref.numpy()).max()))


def test_early_exit_on_the_fp16_edge_chain(cgs_lib, cuda_device):
    """Device-side compaction on DCGAN-64 ℓ1: the same rows leave, and the kept states match the TF32 chain."""
    from cgs import lib as L
    arch, w, h0 = _setup("dcgan64_l1", 32, seed=4)
    plain = _refine(arch, w, h0, cuda_device, L.DEBUG_TF32_OPERANDS, K=20)
    thr = float(np.median(plain["optimal_logit"]))
    ref = _refine(arch, w, h0, cuda_device, L.DEBUG_TF32_OPERANDS, K=20, exit_logit=thr)
    got = _refine(arch, w, h0, cuda_device, 0, K=20, exit_logit=thr)
    gain = float(np.mean(ref["optimal_logit"] - ref["default_logit"]))
    assert gain > 0.5
    d = np.abs(got["optimal_logit"] - ref["optimal_logit"])
    assert float(d.max()) <= max(0.05, 0.02 * gain), d
    assert np.mean((got["optimal_logit"] >= thr) == (ref["optimal_logit"] >= thr)) >= 0.95
    e = np.linalg.norm(got["refined"] - ref["refined"]) / np.linalg.norm(ref["refined"])
    assert e <= 1e-2, e


@pytest.mark.parametrize("name", ["dcgan64_l1", "dcgan64_l4"])
def test_fp16_edge_chain_is_shard_invariant(cgs_lib, cuda_device, name):
    """A batch refined whole equals its two halves refined separately, bit for bit: no result depends on which other
    rows share a launch (the per-sample gradient scale, the band tiles of the edge kernels, the GEMM row tiles)."""
    arch, w, h0 = _setup(name, 24, seed=5)
    whole = _refine(arch, w, h0, cuda_device, 0, K=6)
    halves = [_refine(arch, w, h, cuda_device, 0, K=6) for h in (h0[:12], h0[12:])]
    for k in whole:
        assert np.array_equal(whole[k], np.concatenate([halves[0][k], halves[1][k]])), k
