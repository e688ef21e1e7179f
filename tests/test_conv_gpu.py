"""GPU parity for the image path: per-layer forward / data-gradient and the K-step refinement vs the FP32 oracle.

Tolerances (BASELINE.md §5): FP32 SIMT mode is compared at 2e-5 relative (summation order only); the TF32
tensor-core mode at rel-L2 <= 1e-3 per layer pass (10-bit mantissa operands, FP32 accumulation).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import graph_refiner as gr
from oracle import nets as onets

pytestmark = pytest.mark.gpu

TOL = {"fp32": 2e-5, "tf32": 1e-3}


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def pad_c(x, cs):
    out = np.zeros(x.shape[:-1] + (cs,), np.float32)
    out[..., :x.shape[-1]] = x
    return out


def _refine(spec, h0, flags, K=3):
    """K refinement steps of h0 under the CGS_DEBUG knobs `flags`: (refined, optimal_logit, current_feature,
    optimal_step)."""
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    with L.debug_flags(flags):
        r = Refiner(K, 0.1)
        r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        x = r.build_refiner(h0)
        torch.cuda.synchronize()
        return x.clone(), r.optimal_logit.clone(), r.current_feature.clone(), r.optimal_step.clone()


@pytest.fixture
def general_lowering(cgs_lib):
    """Route the image-edge passes through the general tcgen05 lowerings (DEBUG_EDGE_GENERAL) for one test."""
    from cgs import lib as L
    with L.debug_flags(L.DEBUG_EDGE_GENERAL):
        yield


@pytest.mark.parametrize("arch_name,B", [("mnist", 5), ("mnist", 67), ("dcgan64_l2", 2)])
def test_edge_layers_general_lowering(cgs_lib, cuda_device, general_lowering, arch_name, B):
    """The tcgen05 window / scatter lowerings stay covered although the fused edge kernels are the default."""
    test_layers_forward_backward(cgs_lib, cuda_device, arch_name, B, "tf32")


@pytest.fixture
def forced_fusion(cgs_lib):
    """Class-fused tcgen05 tiles whenever they are legal (DEBUG_FORCE_FUSION), whatever the tile count."""
    from cgs import lib as L
    with L.debug_flags(L.DEBUG_FORCE_FUSION):
        yield


@pytest.mark.parametrize("arch_name,B", [("dcgan32_l1", 3), ("dcgan32_l2", 40), ("dcgan64_l2", 9), ("dcgan64_l1", 2)])
def test_layers_class_fused_tiles(cgs_lib, cuda_device, forced_fusion, arch_name, B):
    """The class-fused instances of the transposed-type passes (one A tile per shift feeds all parity classes) against
    the oracle, at batches where the launcher would otherwise pick one class per tile."""
    test_layers_forward_backward(cgs_lib, cuda_device, arch_name, B, "tf32")


@pytest.mark.parametrize("arch_name,B,gain", [("dcgan32_l2", 6, 2.5), ("dcgan64_l1", 3, 2.5), ("dcgan32_l2", 600, 2.5),
                                               ("dcgan32_l1", 1024, 2.5)])   # the last two: several tiles per CTA
def test_class_fusion_is_bit_identical(cgs_lib, cuda_device, arch_name, B, gain):
    """Fused tiles accumulate every class in the same (tap, channel block) order as the one-class tiles, so the choice
    (which depends on the tile count, i.e. on the batch) never changes a bit: shard invariance is preserved."""
    from cgs import lib as L
    arch, w, spec = _make(arch_name, 5, gain, cuda_device, "tf32")
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(4))).to(cuda_device)

    fused, plain = _refine(spec, h0, L.DEBUG_FORCE_FUSION), _refine(spec, h0, L.DEBUG_NO_FUSION)
    assert all(torch.equal(a, b) for a, b in zip(fused, plain))


@pytest.mark.parametrize("arch_name,B,gain", [("mnist", 40, 3.0), ("mnist", 300, 3.0), ("dcgan32_l2", 7, 2.5), ("dcgan64_l1", 3, 2.5),
                                               ("dcgan32_l1", 1024, 2.5)])
def test_m_tile_pairs_are_bit_identical(cgs_lib, cuda_device, arch_name, B, gain):
    """Two M tiles per CTA sharing the weight atoms (DEBUG_FORCE_MTILE_PAIRS forces them, DEBUG_NO_MTILE_PAIRS forbids
    them): every accumulator sees the same MMA sequence, so the results are bit-identical, incl. odd tile counts
    (half-empty last pair) and several pairs per CTA."""
    from cgs import lib as L
    arch, w, spec = _make(arch_name, 5, gain, cuda_device, "tf32")
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(4))).to(cuda_device)

    # class fusion off in both: pairs everywhere legal
    paired = _refine(spec, h0, L.DEBUG_FORCE_MTILE_PAIRS | L.DEBUG_NO_FUSION)
    single = _refine(spec, h0, L.DEBUG_NO_MTILE_PAIRS | L.DEBUG_NO_FUSION)
    assert all(torch.equal(a, b) for a, b in zip(paired, single))
    default = _refine(spec, h0, 0)
    assert all(torch.equal(a, b) for a, b in zip(default, single))


@pytest.mark.parametrize("arch_name,B,gain", [("dcgan32_l2", 7, 2.5), ("dcgan64_l1", 3, 2.5), ("dcgan64_l3", 5, 2.5),
                                               ("dcgan32_l1", 1024, 2.5), ("dcgan32_l2", 601, 2.5)])
def test_cta_pairs_are_bit_identical(cgs_lib, cuda_device, arch_name, B, gain):
    """CTA pairs (cluster of two, tcgen05 cta_group::2, M = 256; DEBUG_FORCE_CTA_PAIRS forces them, DEBUG_NO_CTA_PAIRS
    forbids them): every accumulator row sees the same K order as in a single-CTA tile, so the results are
    bit-identical -- with class-fused tiles and 256-wide tiles, odd tile counts (the pair's second tile past the batch)
    and several units per pair."""
    from cgs import lib as L
    arch, w, spec = _make(arch_name, 5, gain, cuda_device, "tf32")
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(4))).to(cuda_device)

    paired = _refine(spec, h0, L.DEBUG_FORCE_CTA_PAIRS | L.DEBUG_FORCE_FUSION)   # class fusion forced in both
    single = _refine(spec, h0, L.DEBUG_NO_CTA_PAIRS | L.DEBUG_FORCE_FUSION)
    assert all(torch.equal(a, b) for a, b in zip(paired, single))
    default = _refine(spec, h0, 0)
    assert all(torch.equal(a, b) for a, b in zip(default, single))
    # M-tile pairs INSIDE CTA pairs (units of four M tiles; class fusion off so the 128-wide passes take them)
    quad = _refine(spec, h0, L.DEBUG_FORCE_CTA_PAIRS | L.DEBUG_FORCE_MTILE_PAIRS | L.DEBUG_NO_FUSION)
    assert all(torch.equal(a, b) for a, b in zip(quad, single))


@pytest.mark.parametrize("math", ["fp32", "tf32"])
@pytest.mark.parametrize("arch_name,B", [("mnist", 5), ("mnist", 67), ("dcgan32_l1", 3), ("dcgan64_l2", 2), ("dcgan64_l2", 9)])
def test_layers_forward_backward(cgs_lib, cuda_device, arch_name, B, math):
    from cgs import nets as N
    _layer_parity(cgs_lib, cuda_device, N.get_arch(arch_name), B, math)


@pytest.mark.parametrize("win", [31, 63])
def test_odd_width_image_layer(cgs_lib, cuda_device, win):
    """An image-input conv whose width is odd has no space-to-depth form: cgs_layer_forward must not take the s2d
    tcgen05 edge kernel for it (its output rows would be read W / 2 pixels wide) and still match the oracle."""
    from cgs import nets as N
    arch = N.get_arch("mnist")
    arch["d"] = [dict(arch["d"][0], hin=32, win=win)] + arch["d"][1:]   # k = 4: pad 1, 16 x (win + 1) / 2 outputs
    _layer_parity(cgs_lib, cuda_device, arch, 3, "tf32", names={"d_conv1"})


def _layer_parity(cgs_lib, cuda_device, arch, B, math, names=None):
    """cgs_layer_forward / cgs_layer_backward of every GEMM layer of `arch` (or of the layers in `names`) vs the
    oracle."""
    from cgs import lib as L
    from cgs import nets as N
    w = onets.init_weights(arch, seed=11)
    spec = N.NetSpec(arch, w, cuda_device, math=math)
    rng = np.random.RandomState(1)
    chain = [("generator", l, spec.gtail.layer_desc(i)) for i, l in enumerate(arch["gtail"])] + \
            [("discriminator", l, spec.d.layer_desc(i)) for i, l in enumerate(arch["d"][:-1])]
    worst = {}
    for scope, layer, desc in chain:
        if names is not None and layer["name"] not in names:
            continue
        cin, cout = layer["cin"], layer["cout"]
        shp = (B, cin) if layer["type"] == "fc" else (B, layer["hin"], layer["win"], cin)
        x = rng.standard_normal(shp).astype(np.float32)
        xt = torch.from_numpy(x).requires_grad_(True)
        y = onets.run_layers(xt, [layer], scope, w, "inference")
        dy = rng.standard_normal(tuple(y.shape)).astype(np.float32)
        # gradient w.r.t. the layer's PRE-activation output is what the backward GEMM consumes
        ypre = onets.run_layers(xt, [dict(layer, act="none")], scope, w, "inference")
        (dx,) = torch.autograd.grad((ypre * torch.from_numpy(dy)).sum(), xt)
        cs_in, cs_out = N.cstride(cin), N.cstride(cout)
        x_dev = torch.from_numpy(pad_c(x, cs_in)).to(cuda_device)
        y_dev = torch.full(tuple(y.shape[:-1]) + (cs_out,), float("nan"), device=cuda_device)
        ws = torch.empty(int(cgs_lib.cgs_layer_workspace_bytes(C.byref(desc), B)), dtype=torch.uint8, device=cuda_device)
        L.check(cgs_lib.cgs_layer_forward(C.byref(desc), L.MATH_IDS[math], B, L.ptr(x_dev), L.ptr(y_dev), L.ptr(ws),
                                          ws.numel(), L.stream_ptr()))
        torch.cuda.synchronize()
        got = y_dev.cpu().numpy()
        e = rel_l2(got[..., :cout], y.detach().numpy())
        worst[layer["name"] + ".fwd"] = e
        assert e <= TOL[math], (layer["name"], "fwd", e)
        assert np.all(got[..., cout:] == 0), "padding channels must stay zero"
        dy_dev = torch.from_numpy(pad_c(dy, cs_out)).to(cuda_device)
        dx_dev = torch.full(tuple(x.shape[:-1]) + (cs_in,), float("nan"), device=cuda_device)
        L.check(cgs_lib.cgs_layer_backward(C.byref(desc), L.MATH_IDS[math], B, L.ptr(dy_dev), L.ptr(dx_dev), None, 0,
                                           L.ptr(ws), ws.numel(), L.stream_ptr()))
        torch.cuda.synchronize()
        gotg = dx_dev.cpu().numpy()
        e = rel_l2(gotg[..., :cin], dx.numpy())
        worst[layer["name"] + ".bwd"] = e
        assert e <= TOL[math], (layer["name"], "bwd", e)
    print(arch["name"], math, {k: "%.2e" % v for k, v in worst.items()})


def _make(arch_name, seed, gain, cuda_device, math="fp32"):
    from cgs import nets as N
    arch = N.get_arch(arch_name)
    w = onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=seed), gain)
    return arch, w, N.NetSpec(arch, w, cuda_device, math=math)


@pytest.mark.parametrize("math", ["fp32", "tf32"])
@pytest.mark.parametrize("arch_name,B,gain", [("mnist", 6, 3.0), ("dcgan32_l1", 4, 2.5), ("dcgan64_l3", 3, 2.5)])
def test_forward_logits_and_grad(cgs_lib, cuda_device, arch_name, B, gain, math):
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make(arch_name, 5, gain, cuda_device, math)
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(1)))
    logit_ref, grad_ref, img_ref = gr.forward_logits_and_grad(h0, arch, w)
    ref = Refiner(1, 0.1)
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    logit, grad = ref.compute_forward_logits_and_grad(h0.to(cuda_device))
    img, logit2 = ref.feature_to_image(h0.to(cuda_device))
    tol = 5e-5 if math == "fp32" else 3e-3
    gtol = tol if math == "fp32" else 8e-2     # TF32: ReLU masks of near-zero units flip -> gradient rel-L2 ~ sqrt(flip rate)
    ltol = tol if math == "fp32" else 1.5e-2
    print(arch_name, math, "logit", logit_ref.numpy(), "err", np.abs(logit.cpu().numpy() - logit_ref.numpy()).max(),
          "grad rel", rel_l2(grad.cpu().numpy(), grad_ref.numpy()), "img rel", rel_l2(img.cpu().numpy(), img_ref.numpy()))
    assert rel_l2(img.cpu().numpy(), img_ref.numpy()) <= tol
    assert np.abs(logit.cpu().numpy() - logit_ref.numpy()).max() <= ltol * max(1.0, np.abs(logit_ref.numpy()).max())
    assert rel_l2(grad.cpu().numpy(), grad_ref.numpy()) <= gtol
    assert np.array_equal(logit.cpu().numpy(), logit2.cpu().numpy())


@pytest.mark.parametrize("math", ["fp32", "tf32"])
@pytest.mark.parametrize("arch_name,B,K,method,gain", [("mnist", 6, 5, "momentum", 3.0), ("mnist", 3, 3, "sgd", 3.0),
                                                        ("dcgan32_l2", 4, 4, "momentum", 2.5),
                                                        ("dcgan64_l1", 2, 3, "momentum", 2.5),
                                                        # refinement at the last map: the policy step is fused into the
                                                        # wide image-edge pass (edge_wide_tc EPI_UPDATE in TF32 mode)
                                                        ("dcgan32_l4", 5, 3, "momentum", 2.5), ("dcgan64_l4", 2, 2, "sgd", 2.5),
                                                        # 24-pixel rows at the image edge: no tcgen05 edge kernel takes
                                                        # them, the chain keeps the pitched image layout
                                                        ("dcgan48_l1", 2, 3, "momentum", 2.5)])
def test_build_refiner_matches_oracle(cgs_lib, cuda_device, arch_name, B, K, method, gain, math):
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make(arch_name, 9, gain, cuda_device, math)
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(2)))
    o = gr.build_refiner(h0, arch, w, K, 0.1, method=method)
    ref = Refiner(K, 0.1, method)
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    out = ref.build_refiner(h0.to(cuda_device), None, "deterministic", keep_optimal_feature=True)
    tol = 1e-4 if math == "fp32" else 1e-2          # DESIGN.md §2: K-step images rel-L2 <= 1e-2 in TF32 mode
    e_img = rel_l2(out.cpu().numpy(), o["refined"].numpy())
    e_logit = np.abs(ref.optimal_logit.cpu().numpy() - o["optimal_logit"].numpy()).max()
    e_feat = rel_l2(ref.current_feature.cpu().numpy(), o["final_feature"].numpy())
    print(arch_name, math, "default", o["default_logit"].numpy(), "optimal", o["optimal_logit"].numpy(), "steps",
          o["optimal_step"].numpy(), "| img rel %.2e logit abs %.2e final feature rel %.2e" % (e_img, e_logit, e_feat))
    ltol = tol if math == "fp32" else 2e-2          # DESIGN.md §2: logits within 2 % (of max(1, |logit|)) in TF32 mode
    assert e_img <= tol and e_feat <= tol
    assert e_logit <= ltol * max(1.0, np.abs(o["optimal_logit"].numpy()).max())
    assert np.abs(ref.default_logit.cpu().numpy() - o["default_logit"].numpy()).max() <= ltol * 2
    if math == "fp32":
        assert np.array_equal(ref.optimal_step.cpu().numpy(), o["optimal_step"].numpy())
    else:
        assert (ref.optimal_step.cpu().numpy() == o["optimal_step"].numpy()).mean() >= 0.5   # ties between near-equal steps
    assert rel_l2(ref.optimal_feature.cpu().numpy(), o["optimal_feature"].numpy()) <= tol


def test_probabilistic_mode_and_clip(cgs_lib, cuda_device):
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make("mnist", 9, 3.0, cuda_device)
    B, K = 7, 4
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(3)))
    idx = np.array([0, 1, 2, 3, 4, 4, 0])        # value K keeps the proposal (collaborator.py:77,81-83)
    o = gr.build_refiner(h0, arch, w, K, 0.1, mode="probabilistic", prob_indices=idx)
    ref = Refiner(K, 0.1)
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    out = ref.build_refiner(h0.to(cuda_device), None, "probabilistic", prob_indices=idx)
    assert rel_l2(out.cpu().numpy(), o["refined"].numpy()) <= 1e-4
    assert np.array_equal(ref.optimal_step.cpu().numpy(), o["optimal_step"].numpy())
    # clipping (collaborator.py:69-70); a zero bound disables it (truthiness test, sic)
    ref2 = Refiner(K, 0.1)
    ref2.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    ref2.set_constraints(0.05, 0.8)
    o2 = gr.build_refiner(h0, arch, w, K, 0.1, vmin=0.05, vmax=0.8)
    out2 = ref2.build_refiner(h0.to(cuda_device), None)
    assert rel_l2(out2.cpu().numpy(), o2["refined"].numpy()) <= 1e-4
    assert float(ref2.current_feature.max()) <= 0.8 + 1e-6 and float(ref2.current_feature.min()) >= 0.05 - 1e-6
    with pytest.raises(TypeError):
        r3 = Refiner(K, 0.1, "ladam")
        r3.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        r3.build_refiner(h0.to(cuda_device), None)
    with pytest.raises(NotImplementedError):
        ref.build_refiner(h0.to(cuda_device), None, "greedy")


def test_cuda_graph_replay_is_bit_identical(cgs_lib, cuda_device):
    """cuda_graph=True replays the captured K-step launch sequence: same bits as eager launches, call after call."""
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make("mnist", 9, 3.0, cuda_device, "tf32")
    eager = Refiner(4, 0.1)
    graph = Refiner(4, 0.1, cuda_graph=True)
    for r in (eager, graph):
        r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    for seed in (1, 2, 3):
        h0 = torch.relu(torch.randn(33, *arch["feature_shape"], generator=torch.Generator().manual_seed(seed))).to(cuda_device)
        a = eager.build_refiner(h0)
        b = graph.build_refiner(h0)
        assert torch.equal(a, b) and torch.equal(eager.optimal_logit, graph.optimal_logit)
        assert torch.equal(eager.optimal_step, graph.optimal_step) and torch.equal(eager.current_feature, graph.current_feature)


def test_launch_and_lowering_knobs_do_not_change_results(cgs_lib, cuda_device):
    """Programmatic dependent launch (DEBUG_PDL_ON) and where the split-K partial sums are added (head kernel or a
    separate reduce kernel, DEBUG_NO_HEAD_PARTIALS) change nothing: bit-identical.  The fc split-K lowering (off with
    DEBUG_NO_FC_SPLIT), the fused edge kernels (off with DEBUG_EDGE_GENERAL) and their pairing into one kernel (off with
    DEBUG_NO_EDGE_PAIR) only change summation order or nothing at all: same refined batch within the TF32 tolerance and
    the same best step for nearly every sample."""
    from cgs import lib as L
    arch, w, spec = _make("mnist", 5, 3.0, cuda_device, "tf32")
    h0 = torch.relu(torch.randn(40, *arch["feature_shape"], generator=torch.Generator().manual_seed(4))).to(cuda_device)

    base = _refine(spec, h0, 0, K=5)
    for same in (L.DEBUG_PDL_ON, L.DEBUG_NO_HEAD_PARTIALS):  # PDL; separate split-K reduce kernel instead of the head's
        assert all(torch.equal(a, b) for a, b in zip(base, _refine(spec, h0, same, K=5))), same
    # DEBUG_NO_EDGE_PAIR: the two edge pairs as four separate kernels
    for flags in (L.DEBUG_NO_FC_SPLIT, L.DEBUG_EDGE_GENERAL, L.DEBUG_NO_EDGE_PAIR, L.DEBUG_NO_FC_SPLIT | L.DEBUG_EDGE_GENERAL):
        x, logit, _, step = _refine(spec, h0, flags, K=5)
        assert rel_l2(x.cpu().numpy(), base[0].cpu().numpy()) <= 1e-2
        assert float((logit - base[1]).abs().max()) <= 1.5e-2
        assert float((step == base[3]).float().mean()) >= 0.9


def test_mnist_layer2_and_chunked_batches(cgs_lib, cuda_device, monkeypatch):
    """Refinement at the [14,14,64] map (G-tail = last deconv only) and chunked refinement of over-size batches."""
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make("mnist_l2", 4, 3.0, cuda_device, "fp32")
    h0 = torch.relu(torch.randn(5, *arch["feature_shape"], generator=torch.Generator().manual_seed(7)))
    o = gr.build_refiner(h0, arch, w, 3, 0.1)
    ref = Refiner(3, 0.1)
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    out = ref.build_refiner(h0.to(cuda_device), keep_optimal_feature=True)
    assert rel_l2(out.cpu().numpy(), o["refined"].numpy()) <= 1e-4
    assert np.array_equal(ref.optimal_step.cpu().numpy(), o["optimal_step"].numpy())
    full_logit, full_feat = ref.optimal_logit.clone(), ref.current_feature.clone()
    monkeypatch.setattr(Refiner, "_max_rows_per_launch", lambda self: 2)     # force 3 chunks (2 + 2 + 1)
    out2 = ref.build_refiner(h0.to(cuda_device), keep_optimal_feature=True)
    assert torch.equal(out, out2) and torch.equal(full_logit, ref.optimal_logit)
    assert torch.equal(full_feat, ref.current_feature) and ref.optimal_feature.shape[0] == 5


@pytest.mark.parametrize("arch_name,B,K,thr", [("mnist", 12, 6, -0.2), ("mnist", 40, 8, 0.1), ("dcgan32_l2", 6, 4, -1.0)])
def test_early_exit_compaction_matches_oracle(cgs_lib, cuda_device, arch_name, B, K, thr):
    """Opt-in early exit (README.md:13): samples D already classifies as real leave the batch (ordered compaction of
    feature / momentum rows); every sample's result equals the oracle's frozen-at-exit semantics, and an unreachable
    threshold reproduces the reference's best-of-K bit for bit."""
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make(arch_name, 9, 3.0 if arch_name == "mnist" else 2.5, cuda_device, "fp32")
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(2)))
    o = gr.build_refiner(h0, arch, w, K, 0.1, exit_logit=thr)
    assert 0 < int(o["done"].sum()) <= B                      # the case actually exercises exits
    ref = Refiner(K, 0.1)
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    ref.early_exit_logit = thr
    out = ref.build_refiner(h0.to(cuda_device), keep_optimal_feature=True)
    assert np.array_equal(ref.optimal_step.cpu().numpy(), o["optimal_step"].numpy())
    ee_logit, ee_feat, ee_img = ref.optimal_logit.clone(), ref.current_feature.clone(), out.clone()
    # FP32 SIMT vs torch-CPU over K chained steps: summation-order noise is amplified by the dynamics
    assert rel_l2(out.cpu().numpy(), o["refined"].numpy()) <= 5e-4
    assert np.abs(ee_logit.cpu().numpy() - o["optimal_logit"].numpy()).max() <= 1e-3
    assert rel_l2(ee_feat.cpu().numpy(), o["final_feature"].numpy()) <= 5e-4
    assert rel_l2(ref.optimal_feature.cpu().numpy(), o["optimal_feature"].numpy()) <= 5e-4
    # disabled-in-effect == reference behaviour, bit for bit
    plain = Refiner(K, 0.1)
    plain.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    a = plain.build_refiner(h0.to(cuda_device))
    # samples that never exit are untouched by the compaction of the others: bit-identical to the plain run
    stay = ~o["done"].to(cuda_device)
    if bool(stay.any()):
        assert torch.equal(ee_img[stay], a[stay]) and torch.equal(ee_logit[stay], plain.optimal_logit[stay])
        assert torch.equal(ee_feat[stay], plain.current_feature[stay])
    # the device-side compaction has no host synchronisation: the whole K loop is CUDA-graph capturable and the
    # replay gives the same bits as the eager launches, call after call
    gref = Refiner(K, 0.1, cuda_graph=True)
    gref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    gref.early_exit_logit = thr
    for _ in range(2):
        gout = gref.build_refiner(h0.to(cuda_device), keep_optimal_feature=True)
        assert torch.equal(gout, ee_img) and torch.equal(gref.optimal_logit, ee_logit)
        assert torch.equal(gref.current_feature, ee_feat) and torch.equal(gref.optimal_step, ref.optimal_step)
        assert torch.equal(gref.optimal_feature, ref.optimal_feature)
    ref.early_exit_logit = 1e30
    b = ref.build_refiner(h0.to(cuda_device))
    assert torch.equal(a, b) and torch.equal(plain.optimal_logit, ref.optimal_logit)
    assert torch.equal(plain.current_feature, ref.current_feature)


@pytest.mark.parametrize("arch_name,B,K", [("dcgan32_l2", 37, 5), ("dcgan64_l2", 11, 4)])
def test_early_exit_is_identical_across_tile_lowerings(cgs_lib, cuda_device, arch_name, B, K):
    """Device-side early exit under every tcgen05 tile lowering (TF32 mode): class-fused tiles, M-tile pairs, CTA pairs
    and M-tile pairs inside CTA pairs all read the live-image count and schedule tiles from it; units whose second /
    third / fourth M tile lies past the live images must neither be stored nor disturb the others.  Same bits as the
    plain one-tile-per-CTA lowering, eager and replayed as a CUDA graph."""
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make(arch_name, 9, 2.5, cuda_device, "tf32")
    h0 = torch.relu(torch.randn(B, *arch["feature_shape"], generator=torch.Generator().manual_seed(6))).to(cuda_device)
    probe = Refiner(K // 2, 0.1)
    probe.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    probe.build_refiner(h0)
    thr = float(torch.median(probe.optimal_logit))            # about half of the batch has left by step K / 2

    def run(flags, graph):
        with L.debug_flags(flags):
            r = Refiner(K, 0.1, cuda_graph=graph)
            r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
            r.early_exit_logit = thr
            x = r.build_refiner(h0, keep_optimal_feature=True)
            torch.cuda.synchronize()
            return x.clone(), r.optimal_logit.clone(), r.current_feature.clone(), r.optimal_step.clone(), r.optimal_feature.clone()

    plain = run(L.DEBUG_NO_FUSION | L.DEBUG_NO_MTILE_PAIRS | L.DEBUG_NO_CTA_PAIRS, False)   # the one-tile-per-CTA lowering
    steps = plain[3].cpu().numpy()
    assert 0 < (steps < K).sum()                               # some samples did stop early
    for flags in (L.DEBUG_FORCE_FUSION, L.DEBUG_FORCE_MTILE_PAIRS | L.DEBUG_NO_FUSION, L.DEBUG_FORCE_CTA_PAIRS | L.DEBUG_FORCE_FUSION,
                  L.DEBUG_FORCE_CTA_PAIRS | L.DEBUG_FORCE_MTILE_PAIRS | L.DEBUG_NO_FUSION, 0):
        for graph in (False, True):
            got = run(flags, graph)
            assert all(torch.equal(a, b) for a, b in zip(got, plain)), (flags, graph)


def test_programmatic_dependent_launch_is_bit_identical_at_scale(cgs_lib, cuda_device):
    """At batches where the refinement loop switches programmatic dependent launch on by itself (average pass >= 12
    GFLOP: DCGAN-64 from 157 rows) the kernels' set-up overlaps the previous kernel's drain; every kernel waits for its
    predecessor before touching activation memory, so the bits equal those of plain stream order (DEBUG_PDL_OFF),
    eager and replayed as a CUDA graph."""
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make("dcgan64_l1", 5, 2.5, cuda_device, "tf32")
    h0 = torch.relu(torch.randn(208, *arch["feature_shape"], generator=torch.Generator().manual_seed(8))).to(cuda_device)

    def run(flags, graph):
        with L.debug_flags(flags):
            r = Refiner(3, 0.1, cuda_graph=graph)
            r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
            outs = []
            for _ in range(2):
                x = r.build_refiner(h0)
                torch.cuda.synchronize()
                outs.append((x.clone(), r.optimal_logit.clone(), r.current_feature.clone(), r.optimal_step.clone()))
            assert all(torch.equal(a, b) for a, b in zip(*outs))
            return outs[0]

    plain = run(L.DEBUG_PDL_OFF, False)
    for flags, graph in ((0, False), (0, True), (L.DEBUG_PDL_ON, True)):
        assert all(torch.equal(a, b) for a, b in zip(run(flags, graph), plain)), (flags, graph)


def test_prefetch_overlaps_upload_and_changes_nothing(cgs_lib, cuda_device):
    """`Refiner.prefetch` uploads the next proposal batch on a side stream; `build_refiner` orders itself after the copy.
    Same bits as handing the host array over directly, also when the prefetch is issued while another batch is being
    refined and with graph replay."""
    from cgs import nets as N
    from sampling.collaborator import Refiner
    arch, w, spec = _make("dcgan32_l1", 5, 2.5, cuda_device, "tf32")
    g = torch.Generator().manual_seed(3)
    batches = [torch.relu(torch.randn(9, *arch["feature_shape"], generator=g)).pin_memory() for _ in range(3)]
    for graph in (False, True):
        r = Refiner(3, 0.1, cuda_graph=graph)
        r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        direct = []
        for h in batches:
            x = r.build_refiner(h.numpy())
            direct.append((torch.from_numpy(x), r.optimal_logit.clone().cpu()))
        staged = r.prefetch(batches[0])
        for i in range(3):
            nxt = r.prefetch(batches[i + 1]) if i + 1 < 3 else None      # issued before batch i is refined
            x = r.build_refiner(staged)
            assert isinstance(x, torch.Tensor) and x.is_cuda
            assert torch.equal(x.cpu(), direct[i][0]) and torch.equal(r.optimal_logit.cpu(), direct[i][1])
            staged = nxt
