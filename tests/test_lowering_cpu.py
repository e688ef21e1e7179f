"""Host-side lowering + weight packing, checked on the CPU against the oracle's TF-semantics layers."""
import numpy as np
import pytest
import torch

from oracle import nets as onets

import emulate


def _arches():
    return ["mnist", "dcgan32_l1", "dcgan64_l3"]


def test_arch_builders_agree(cgs_lib):
    from cgs import nets as N
    for name in _arches() + ["dcgan64_l1", "dcgan64_l4", "dcgan32_l2"]:
        assert N.get_arch(name) == onets.get_arch(name)


@pytest.mark.parametrize("arch_name", _arches())
def test_layer_forward_and_dgrad_lowering(cgs_lib, arch_name):
    from cgs import nets as N
    arch = N.get_arch(arch_name)
    w = onets.init_weights(arch, seed=7)
    rng = np.random.RandomState(0)
    B = 2
    for scope, layers in (("generator", arch["gtail"]), ("discriminator", arch["d"])):
        for layer in layers:
            if layer["type"] == "fc" and layer["cout"] == 1:
                continue
            wf, bf = N.fold_layer(layer, scope, w)
            w_fwd, w_bwd, bias = N.pack_layer(layer, wf, bf)
            cin, cout = layer["cin"], layer["cout"]
            if layer["type"] == "fc":
                x = rng.standard_normal((B, cin)).astype(np.float32)
            else:
                x = rng.standard_normal((B, layer["hin"], layer["win"], cin)).astype(np.float32)
            # oracle forward (pre-activation, BN inference) and its data-gradient
            xt = torch.from_numpy(x).requires_grad_(True)
            Lnoact = dict(layer, act="none")
            y = onets.run_layers(xt, [Lnoact], scope, w, "inference")
            dy = torch.from_numpy(rng.standard_normal(tuple(y.shape)).astype(np.float32))
            (dx,) = torch.autograd.grad((y * dy).sum(), xt)
            # replay forward
            cs_in, cs_out = N.cstride(cin), N.cstride(cout)
            hin, win = (layer["hin"], layer["win"]) if layer["type"] != "fc" else (1, 1)
            xp = np.zeros((B, hin, win, cs_in))
            xp[..., :cin] = x.reshape(B, hin, win, cin)
            acc = emulate.layer_pass(layer, False, B, xp, w_fwd.numpy())
            got = acc[..., :cout] + bias.numpy()[:cout]
            ref = y.detach().numpy().reshape(got.shape)
            assert np.abs(got - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max()), (layer["name"], "fwd")
            assert np.all(acc[..., cout:] == 0)
            # replay backward
            hout, wout = (y.shape[1], y.shape[2]) if layer["type"] != "fc" else (1, 1)
            dyp = np.zeros((B, hout, wout, cs_out))
            dyp[..., :cout] = dy.numpy().reshape(B, hout, wout, cout)
            gacc = emulate.layer_pass(layer, True, B, dyp, w_bwd.numpy())
            gref = dx.numpy().reshape(B, hin, win, cin)
            assert np.abs(gacc[..., :cin] - gref).max() <= 1e-4 * max(1.0, np.abs(gref).max()), (layer["name"], "bwd")


def test_multiply_high_division_is_exact():
    """csrc/conv_gemm.cuh fast_div: n // d == (n * ceil(2^64 / d)) >> 64 for every 32-bit n (magic 0 encodes d == 1).
    The persistent tile index of every GEMM / edge kernel is decomposed with it, so it must be exact, not close."""
    import random
    rng = random.Random(7)
    ds = [1, 2, 3, 4, 7, 8, 14, 25, 49, 98, 147, 148, 196, 1024, 1568, 2048, 65535, 65536, 1 << 20, (1 << 31) - 1]
    ds += [rng.randrange(1, 1 << 31) for _ in range(200)]
    for d in ds:
        magic = 0 if d <= 1 else ((1 << 64) - 1) // d + 1
        ns = [0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, (1 << 31) - 1, (1 << 32) - 1] + [rng.randrange(0, 1 << 32) for _ in range(200)]
        for n in ns:
            if n < 0 or n >= (1 << 32):
                continue
            got = n if magic == 0 else (n * magic) >> 64
            assert got == n // d, (n, d)


@pytest.mark.parametrize("arch_name", ["dcgan32_l1", "dcgan64_l1", "mnist"])
def test_class_fusion_plan_and_cta_pair_split(cgs_lib, arch_name):
    """Host logic of the class-fused tiles and of their split over a CTA pair (csrc/conv_gemm.cu build_fusion), checked
    without a GPU: every (class, tap) of a group appears exactly once, at the shift of its tap and with the K atom the
    weight packing gave it; each class meets its taps in packing order (so fused and one-class tiles accumulate in the
    same order); runs are adjacent slots with one accumulate state and at most 256 columns; the two CTAs of a pair
    fetch complementary halves of every run, each exactly once, into distinct half-atom slots."""
    from cgs import nets as N
    arch = N.get_arch(arch_name)
    fused = 0
    for layer in arch["gtail"] + arch["d"][:-1]:
        for backward in (False, True):
            plan = emulate.fusion_plan(layer, backward, 4)
            p = emulate.gemm_params(layer, backward, 4)
            transposed = p["os"] == 2 and p["nclasses"] == 4 and p["cblocks"] > 0 and not p["window"]
            if plan is None:
                # only k = 5 transposed-type passes with N <= 128 are ever fused
                assert not (transposed and layer["k"] == 5 and p["N"] <= 128), layer["name"]
                continue
            fused += 1
            assert transposed and layer["k"] == 5
            cb = p["cblocks"]
            assert plan["ns"] == (4 if p["N"] <= 64 else 2) and len(plan["groups"]) == (1 if plan["ns"] == 4 else 2)
            seen_classes = []
            for G in plan["groups"]:
                cls = G["cls"][:G["ncls"]]
                assert G["ncls"] == plan["ns"]
                seen_classes += cls
                if plan["ns"] == 2:
                    assert p["cls"][cls[0]]["oy0"] % 2 == p["cls"][cls[1]]["oy0"] % 2
                shifts = plan["shifts"][G["shift0"]:G["shift0"] + G["nshifts"]]
                assert len({(s["dy"], s["dx"]) for s in shifts}) == len(shifts)
                covered = {c: [] for c in cls}          # class -> K atoms in the order of the walk
                touched = set()
                for s in shifts:
                    n = s["ncls"]
                    slots = s["slot"][:n]
                    assert slots == sorted(set(slots)) and 1 <= n <= G["ncls"]
                    for q, slot in enumerate(slots):
                        g = p["cls"][cls[slot]]
                        taps = [t for t in range(g["ntaps"]) if (g["dy"][t], g["dx"][t]) == (s["dy"], s["dx"])]
                        assert len(taps) == 1, (layer["name"], s["dy"], s["dx"])
                        assert s["katom0"][q] == (g["k0"] + taps[0] * cb * 32) // 32
                        covered[cls[slot]].append(s["katom0"][q])
                    # runs: a partition of the listed slots into ranges of adjacent slots with one accumulate state
                    i = 0
                    for r in range(s["nrun"]):
                        s0, ln = s["run_slot"][r], s["run_len"][r]
                        assert slots[i:i + ln] == list(range(s0, s0 + ln)) and ln * p["N"] <= 256
                        assert {slot in touched for slot in slots[i:i + ln]} == {bool(s["run_acc"][r])}
                        # CTA pair: the run's B rows are its atoms back to back, split in the middle
                        pieces = [(i + j // 2, j % 2) for j in range(2 * ln)]          # (entry, half)
                        for rank in (0, 1):
                            mine = pieces[rank * ln:(rank + 1) * ln]
                            got = [(s["pc_slot"][rank][i + j], s["pc_half"][rank][i + j], s["pc_katom"][rank][i + j])
                                   for j in range(ln)]
                            assert got == [(s0 + j, half, s["katom0"][e]) for j, (e, half) in enumerate(mine)]
                        i += ln
                    assert i == n
                    for rank in (0, 1):
                        assert len(set(s["pc_slot"][rank][:n])) == n            # distinct half-atom slots per CTA
                    both = sorted((s["pc_katom"][r][q], s["pc_half"][r][q]) for r in (0, 1) for q in range(n))
                    assert both == sorted((k, h) for k in s["katom0"][:n] for h in (0, 1))
                    touched |= set(slots)
                for c in cls:
                    g = p["cls"][c]
                    assert covered[c] == [g["k0"] // 32 + t * cb for t in range(g["ntaps"])], (layer["name"], c)
            assert sorted(seen_classes) == [0, 1, 2, 3]
    assert (fused > 0) == (arch_name != "mnist")


@pytest.mark.parametrize("arch_name", ["mnist", "mnist_l2", "dcgan32_l1", "dcgan32_l2", "dcgan32_l3", "dcgan32_l4",
                                       "dcgan64_l1", "dcgan64_l2", "dcgan64_l3", "dcgan64_l4", "dcgan48_l1"])
def test_chain_layout_follows_the_operand_rule(cgs_lib, arch_name):
    """cgs_debug_chain_layout against DESIGN.md §2's rule, without a GPU.  DCGAN-32 / -64 chains take FP16 operands:
    every tensor is FP16 except the refined feature act[0], the image and its gradient (s2d) and the head input act[n];
    so a one-layer G tail runs layer 0's narrow pass over FP32 (its TF32 form).  MNIST and DCGAN-48 (no tcgen05 edge
    kernel takes 24-pixel rows: pitched image) and every chain under DEBUG_TF32_OPERANDS are FP32 throughout."""
    import chain_ref as R
    from cgs import lib as L
    from cgs import nets as N
    arch = N.get_arch(arch_name)
    spec = N.NetSpec(arch, onets.init_weights(arch, seed=3), "cpu")
    f16_arch = arch_name.startswith(("dcgan32", "dcgan64"))
    for flags in (0, L.DEBUG_TF32_OPERANDS):
        with L.debug_flags(flags):
            lay = R.chain_layout(spec.gtail.desc, spec.d.desc)
        n, ng = lay["n"], lay["n_gtail"]
        assert (n, ng) == (len(arch["gtail"]) + len(arch["d"]) - 1, len(arch["gtail"]))
        assert lay["img_mode"] == (R.S2D if f16_arch else R.PITCHED)
        f16 = f16_arch and not flags
        assert lay["f16"] == f16
        for kind, i, t in [("act", i, t) for i, t in enumerate(lay["act"])] + \
                          [("grad", i, t) for i, t in enumerate(lay["grad"]) if t is not None]:
            fp32 = i == ng or (kind == "act" and i in (0, n))
            assert t["fp16"] == (f16 and not fp32), (kind, i)
            image = i == ng
            assert t["layout"] == (lay["img_mode"] if image else R.DENSE), (kind, i)
            assert t["C"] <= 4 if image else t["C"] >= 32
            assert t["elems"] >= t["H"] * t["W"] * t["C"]
        if arch_name == "dcgan64_l4":                      # layer 0 = G's last deconv, reading the FP32 feature
            assert ng == 1 and not lay["act"][0]["fp16"] and lay["grad"][2]["fp16"] == f16
