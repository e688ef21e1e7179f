"""FP16 operands in the DCGAN refinement chain (choose_operand_type, DESIGN.md §2).

The chain's GEMM layers run kind::f16 over FP16 operands, with the head's per-sample power-of-two gradient scale; the
TF32 path stays reachable through CGS_DEBUG_TF32_OPERANDS and is the reference here.  FP16 holds the TF32-rounded
values exactly inside its normal range, so the two paths differ like two TF32 runs with different rounding ties and
accumulation orders: the K=50 TF32 tolerances of tests/test_k50_parity_gpu.py apply.
"""
import numpy as np
import pytest
import torch

from oracle import nets as onets
from parity_metrics import k50_metrics

pytestmark = pytest.mark.gpu

TOL = dict(img_rel_l2=1e-2, img_max_abs=0.4, logit_frac=0.02, logit_floor=0.05, step=0.95)


def _setup(name, B, seed=2):
    from cgs import nets as N
    arch = N.get_arch(name)
    w = onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=9), 3.0 if name == "mnist" else 2.5)
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(seed)))
    return arch, w, h0


def _refine(arch, w, h0, dev, flags, K=50, exit_logit=None):
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    spec = N.NetSpec(arch, w, dev, math="tf32")
    with L.debug_flags(flags):
        ref = Refiner(K, 0.1, "momentum")
        ref.early_exit_logit = exit_logit
        ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        x = ref.build_refiner(h0.to(dev), None, "deterministic")
        torch.cuda.synchronize()
    return dict(refined=x.cpu().numpy(), optimal_logit=ref.optimal_logit.cpu().numpy(),
                optimal_step=ref.optimal_step.cpu().numpy(), default_logit=ref.default_logit.cpu().numpy())


@pytest.mark.parametrize("name,B", [("dcgan32_l1", 64), ("dcgan64_l1", 32)])
def test_fp16_chain_matches_tf32_chain_at_k50(cgs_lib, cuda_device, name, B):
    from cgs import lib as L
    arch, w, h0 = _setup(name, B)
    ref = _refine(arch, w, h0, cuda_device, L.DEBUG_TF32_OPERANDS)
    got = _refine(arch, w, h0, cuda_device, 0)
    # the chain did take FP16 operands: two TF32 runs would be bit-identical
    assert any(not np.array_equal(got[k], ref[k]) for k in got)
    m = k50_metrics(ref, got, onets.get_arch(name), w)
    print(name, m)
    assert m["img_rel_l2"] <= TOL["img_rel_l2"] and m["img_max_abs"] <= TOL["img_max_abs"], m
    assert m["optimal_logit_max_abs"] <= max(TOL["logit_floor"], TOL["logit_frac"] * abs(m["logit_gain_mean_ref"])), m
    assert m["optimal_step_agree"] >= TOL["step"], m
    assert m["logit_gain_mean_ref"] > 1.0


def test_scaled_gradient_survives_a_saturated_logit(cgs_lib, cuda_device):
    """Rows whose logit is so large that d loss / d logit is 2^-24 .. 2^-14 (logit ~10 .. 16.6): unscaled, their FP16
    gradient chain would lie in FP16's subnormals or flush to zero; with the per-sample scale it matches the TF32 path
    as closely as an ordinary row does.  Features along the path from two proposals to their refined optimum under
    the bench's weights (DCGAN-64, logits up to ~38 after 50 steps)."""
    from cgs import lib as L
    from cgs import nets as N
    from cgs import synthetic as S
    from sampling.collaborator import Refiner
    arch = N.get_arch("dcgan64_l1")
    spec = N.NetSpec(arch, S.init_weights(arch, seed=2019, gain=2.5), cuda_device, math="tf32")
    h0 = torch.from_numpy(S.proposal_features(arch, 2, seed=3)).to(cuda_device)
    r = Refiner(50, 0.1, "momentum")
    r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    r.build_refiner(h0, None, "deterministic", keep_optimal_feature=True)
    alphas = torch.linspace(0.0, 1.2, 96, device=cuda_device).view(1, -1, 1, 1, 1)
    feats = (h0.unsqueeze(1) + alphas * (r.optimal_feature - h0).unsqueeze(1)).reshape(-1, *h0.shape[1:]).contiguous()

    def grad(flags):
        with L.debug_flags(flags):
            q = Refiner(1, 0.1)
            q.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
            lg, g = q.compute_forward_logits_and_grad(feats)
            torch.cuda.synchronize()
        return lg.cpu().double(), g.cpu().double().reshape(feats.shape[0], -1)

    lg_ref, g_ref = grad(L.DEBUG_TF32_OPERANDS)
    lg, g = grad(0)
    dl = (torch.sigmoid(lg_ref.float()) - 1.0).abs().double()
    tiny = (dl > 0) & (dl <= 2.0 ** -14)
    normal = dl > 0.05
    assert int(tiny.sum()) >= 3 and int(normal.sum()) >= 3, (lg_ref.min(), lg_ref.max())
    rel = (g - g_ref).norm(dim=1) / g_ref.norm(dim=1).clamp_min(1e-300)
    print("saturated rows: logit %.1f..%.1f, rel-L2 max %.2e (ordinary rows %.2e)"
          % (float(lg_ref[tiny].min()), float(lg_ref[tiny].max()), float(rel[tiny].max()), float(rel[normal].max())))
    assert bool((g_ref[tiny].norm(dim=1) > 0).all())
    assert float(rel[tiny].max()) <= max(5e-2, 2.0 * float(rel[normal].max()))
    assert float((lg - lg_ref).abs().max()) <= 2e-2 * max(1.0, float(lg_ref.abs().max()))


def test_early_exit_on_the_fp16_chain(cgs_lib, cuda_device):
    """Device-side compaction with FP16 operands: the same rows leave, and the kept states match the TF32 chain."""
    from cgs import lib as L
    arch, w, h0 = _setup("dcgan32_l1", 48, seed=4)
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


@pytest.mark.parametrize("name", ["mnist", "dcgan48_l1"])
def test_chains_without_fp16_operands_are_unchanged(cgs_lib, cuda_device, name):
    """MNIST (fc layers, pitched image) and a 48-pixel DCGAN (pitched image) keep TF32 operands: the knob changes
    nothing, bit for bit."""
    from cgs import lib as L
    arch, w, h0 = _setup(name, 8)
    a = _refine(arch, w, h0, cuda_device, 0, K=5)
    b = _refine(arch, w, h0, cuda_device, L.DEBUG_TF32_OPERANDS, K=5)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
