"""Every pass of the refinement chain, alone, bit for bit against an exact FP64 reference (tests/chain_ref.py).

Weights, biases and inputs lie on coarse binary grids, so every FP32 accumulation of a pass is exact whatever the
lowering; each pass runs through cgs_debug_chain_pass exactly as a refinement call runs it (route, FP16 / TF32
operands, layouts, fused epilogue) and its stored result must equal the reference's epilogue of the exact value,
rounded as the pass stores it.  Only tanh / tanh' keep an allowance (2 FP32 ulp; 1 ulp of the stored format), and the
head's sigmoid (expf) where its result sits next to a power of two.  One line per (arch, operands, pass, B, knob).
"""
import numpy as np
import pytest
import torch

import chain_ref as R

pytestmark = pytest.mark.gpu

ARCHES = ["dcgan32_l1", "dcgan64_l1", "dcgan64_l2", "dcgan64_l4", "mnist", "dcgan48_l1"]
# batches at which the launcher takes M-tile pairs and CTA pairs on its own
BIG = {"dcgan32_l1": 600, "dcgan64_l1": 200, "dcgan64_l2": 200, "dcgan64_l4": 200, "mnist": 300, "dcgan48_l1": 200}
W_BITS, X_BITS = 4, 5
_NETS = {}


def _net(name, dev):
    if name not in _NETS:
        _NETS[name] = R.ChainNet(name, dev, seed=ARCHES.index(name) + 1)
    return _NETS[name]


def _operands(which):
    from cgs import lib as L
    return {"default": 0, "tf32": L.DEBUG_TF32_OPERANDS}[which]


def _compare(got, exp, tanh_like, t, rounded):
    """Elementwise acceptance: equal values, or for tanh / tanh' results within 2 FP32 ulp (1 ulp of FP16 / TF32 when
    the value is stored in that format)."""
    ok = got == exp
    if tanh_like:
        if t["fp16"]:
            ok |= R.within_fp16_ulp(got, exp)
        elif rounded:
            e32 = np.asarray(exp, np.float32)
            ok |= np.abs(got - exp) <= np.spacing(np.abs(e32)).astype(np.float64) * 2 ** 13
        else:
            ok |= R.ulps_fp32(got, exp) <= 2
    return ok


def _run_pass(cn, lay, i, backward, B, rng, tag, x=None, x_exact=None, aux_val=None):
    """Run pass (i, backward), i < n, on grid inputs; returns '' or a mismatch report.  x / x_exact: the input as
    stored and the value the exact reference uses (FP32 operands that are not TF32-exact)."""
    dev = cn.device
    n, ng = lay["n"], lay["n_gtail"]
    _, l = cn.layers[i]
    if not backward:
        tin, tout = lay["act"][i], lay["act"][i + 1]
    else:
        tin, tout = lay["grad"][i + 1], (lay["grad"][i] if i > 0 else lay["act"][0])
    if x is None:
        x = R.grid(rng, R.dense_shape(tin, B), X_BITS, 2.0)
    if x_exact is None:
        x_exact = x
    xin = R.to_chain(x, tin, dev)
    out = R.empty_chain(tout, B, dev)
    aux = aux32 = None
    if backward and i > 0:
        taux = lay["act"][i]
        aux_v = R.grid(rng, R.dense_shape(taux, B), X_BITS, 1.0) if aux_val is None else aux_val
        aux, aux32 = R.to_chain(aux_v, taux, dev), aux_v.astype(np.float32)
    val, bound = cn.exact_pass(i, backward, x_exact, R.dense_shape(lay["act"][i], B))
    v32 = R.exact_f32(val.reshape(R.dense_shape(tout, B)), bound.reshape(R.dense_shape(tout, B)), W_BITS + X_BITS)
    if not backward:
        e = R.act_fwd(v32, l["act"])
        rounded = not tout["fp16"] and i + 1 not in (ng, n)
        tanh_like = l["act"] == "tanh"
    elif i > 0:
        act = cn.layers[i - 1][1]["act"]
        e = R.act_bwd(v32, aux32, act)
        rounded, tanh_like = not tout["fp16"], act == "tanh"
    else:
        e, rounded, tanh_like = v32, False, False
    exp = R.store(e, tout, rounded)
    cn.run(B, i, backward, xin, out, aux=aux)
    got = R.from_chain(out, tout, B)
    rep = R.mismatch_report(got, exp, _compare(got, exp, tanh_like, tout, rounded))
    print("%s pass %d %s %s -> %s: %s" % (tag, i, "dgrad" if backward else "fwd", R.describe(tin), R.describe(tout),
                                          "exact" if not rep else "MISMATCH " + rep))
    return rep


def _all_passes(cn, B, flags, tag, seed):
    from cgs import lib as L
    rng = np.random.RandomState(seed)
    fails = []
    with L.debug_flags(flags):
        lay = cn.layout()
        for i in range(lay["n"]):
            for backward in (False, True):
                rep = _run_pass(cn, lay, i, backward, B, rng, tag)
                if rep:
                    fails.append("pass %d %s: %s" % (i, "dgrad" if backward else "fwd", rep))
    return fails


@pytest.mark.parametrize("name", ARCHES)
def test_packed_weights_are_the_grid_filters(cgs_lib, cuda_device, name):
    _net(name, cuda_device).check_packing()


@pytest.mark.parametrize("B", [1, 3, 37, "big"])
@pytest.mark.parametrize("operands", ["default", "tf32"])
@pytest.mark.parametrize("name", ARCHES)
def test_every_pass_is_exact(cgs_lib, cuda_device, name, operands, B):
    B = BIG[name] if B == "big" else B
    cn = _net(name, cuda_device)
    fails = _all_passes(cn, B, _operands(operands), "%s %s B=%d knob=none" % (name, operands, B), seed=B)
    assert not fails, "\n".join(fails)


KNOBS = ["FORCE_FUSION", "NO_FUSION", "FORCE_MTILE_PAIRS|NO_FUSION", "FORCE_CTA_PAIRS|FORCE_FUSION",
         "FORCE_CTA_PAIRS|FORCE_MTILE_PAIRS|NO_FUSION", "NO_FC_SPLIT", "EDGE_GENERAL|TF32_OPERANDS"]


@pytest.mark.parametrize("knob", KNOBS)
@pytest.mark.parametrize("name,B", [("dcgan32_l1", 37), ("dcgan64_l1", 37), ("mnist", 37), ("dcgan64_l4", 5)])
def test_lowering_knobs_are_exact(cgs_lib, cuda_device, name, B, knob):
    """Each lowering knob against the exact reference, not only against the other lowerings."""
    from cgs import lib as L
    flags = 0
    for k in knob.split("|"):
        flags |= getattr(L, "DEBUG_" + k)
    fails = _all_passes(_net(name, cuda_device), B, flags, "%s B=%d knob=%s" % (name, B, knob), seed=7)
    assert not fails, "\n".join(fails)


STEPS = {"raw": None, "momentum_first": ("momentum", 1, 0), "momentum": ("momentum", 0, 0), "sgd": ("sgd", 0, 0),
         "clip": ("momentum", 0, 1)}


@pytest.mark.parametrize("step", list(STEPS))
@pytest.mark.parametrize("name", ["dcgan32_l1", "dcgan64_l1", "dcgan64_l4"])
def test_per_sample_gradient_scale(cgs_lib, cuda_device, name, step):
    """Layer 0's data-gradient pass of an FP16 chain removes 2^gexp[b] per sample, raw or inside the fused policy step.
    A distinct exponent per sample, so that a wrong sample index in a tile that spans 32 (DCGAN-32) or 8 (DCGAN-64)
    samples, or in the wide edge kernel's step (dcgan64_l4), changes the result."""
    from cgs import lib as L
    cn = _net(name, cuda_device)
    B = 37
    rng = np.random.RandomState(11)
    lay = cn.layout()
    assert lay["f16"]
    tin, tf = lay["grad"][1], lay["act"][0]
    gexp = (7 * np.arange(B)) % 25
    x = R.grid(rng, R.dense_shape(tin, B), X_BITS, 2.0)
    val, bound = cn.exact_pass(0, True, x, R.dense_shape(tf, B))
    v32 = R.exact_f32(val, bound, W_BITS + X_BITS)
    g32 = (v32 * np.exp2(-gexp.astype(np.float64)).reshape(-1, 1, 1, 1)).astype(np.float32)   # exact
    feat = rng.standard_normal(R.dense_shape(tf, B)).astype(np.float32)
    mom = (0.1 * rng.standard_normal(R.dense_shape(tf, B))).astype(np.float32)
    gexp_t = torch.from_numpy(gexp.astype(np.int32)).to(cuda_device)
    if STEPS[step] is None:
        out = R.empty_chain(tf, B, cuda_device)
        cn.run(B, 0, True, R.to_chain(x, tin, cuda_device), out, gexp=gexp_t)
        checks = [("gradient", R.from_chain(out, tf, B), g32.astype(np.float64))]
    else:
        method, first, clip = STEPS[step]
        cfg = L.RefineCfg(steps=1, rate=0.1, method=L.POLICY_IDS[method], alpha=0.9, mode=0, clip=clip, vmin=-0.5,
                          vmax=0.5, math=0)
        fbuf, mbuf = R.to_chain(feat, tf, cuda_device), R.to_chain(mom, tf, cuda_device)
        cn.run(B, 0, True, R.to_chain(x, tin, cuda_device), fbuf, gexp=gexp_t, cfg=cfg, mom=mbuf, first=first)
        theta, m = R.policy(cfg, feat, g32, mom, first)
        checks = [("feature", R.from_chain(fbuf, tf, B), theta.astype(np.float64))]
        if method == "momentum":
            checks.append(("momentum", R.from_chain(mbuf, tf, B), m.astype(np.float64)))
    for what, got, exp in checks:
        rep = R.mismatch_report(got, exp)
        print("%s default B=%d pass 0 dgrad step=%s %s: %s" % (name, B, step, what, "exact" if not rep else rep))
        assert not rep, (what, rep)


def _range_net(name, layer, dev, filt):
    """A grid net whose layer `layer` has the weights filt(shape, rng) (TF layout) and no bias."""
    arch = R.grid_arch(name)
    w = R.grid_weights(arch, np.random.RandomState(3))
    scope, l = ([("generator", x) for x in arch["gtail"]] + [("discriminator", x) for x in arch["d"][:-1]])[layer]
    key = "%s/%s/w" % (scope, l["name"])
    w[key] = filt(w[key].shape, np.random.RandomState(4)).astype(np.float32)
    w[key[:-1] + "biases"][:] = 0.0
    return R.ChainNet(name, dev, weights=w)


def _sign_per_output(shape, rng, unit):
    """Data-gradient of a conv: output channel = input channel ci (axis 2); a sign per ci, magnitudes on unit * Z."""
    s = np.where(np.arange(shape[2]) % 2 == 0, 1.0, -1.0).reshape(1, 1, -1, 1)
    return s * rng.randint(0, 17, size=shape) / 16.0 * unit


def _fp16_gradient_pass(cn, B, dy, bits, tag):
    """D's d_h2 data-gradient of DCGAN-64 l1 (FP16 in, FP16 out), derivative operand positive (act' = 1)."""
    lay = cn.layout()
    i = 6
    assert lay["grad"][i]["fp16"] and lay["grad"][i + 1]["fp16"]
    tin, tout, taux = lay["grad"][i + 1], lay["grad"][i], lay["act"][i]
    val, bound = cn.exact_pass(i, True, dy, R.dense_shape(taux, B))
    v32 = R.exact_f32(val, bound, bits)
    out = R.empty_chain(tout, B, cn.device)
    cn.run(B, i, True, R.to_chain(dy, tin, cn.device), out, aux=R.to_chain(np.ones(R.dense_shape(taux, B)), taux, cn.device))
    got, exp = R.from_chain(out, tout, B), R.fp16_rn_satfinite(v32).astype(np.float64)
    rep = R.mismatch_report(got, exp)
    print("%s: %s" % (tag, "exact" if not rep else rep))
    return v32, got, rep


def test_fp16_outputs_saturate(cgs_lib, cuda_device):
    """Exact results beyond +-65504 store +-65504 (satfinite), never inf; the others RN-even."""
    cn = _range_net("dcgan64_l1", 6, cuda_device, lambda s, r: _sign_per_output(s, r, 1.0))
    B = 9
    rng = np.random.RandomState(5)
    dy = np.concatenate([rng.randint(0, 2 ** b + 1, size=(1, 8, 8, 256)) for b in range(B)]).astype(np.float64)
    v32, got, rep = _fp16_gradient_pass(cn, B, dy, W_BITS, "dcgan64_l1 default B=9 pass 6 dgrad saturation")
    assert (v32 > R.FP16_MAX).sum() > 100 and (v32 < -R.FP16_MAX).sum() > 100 and (np.abs(v32) < 2048).sum() > 100
    assert np.all(np.isfinite(got))
    assert not rep, rep


def test_fp16_subnormal_inputs_and_outputs(cgs_lib, cuda_device):
    """FP16 subnormal operands (2^-24 Z below 2^-14) are multiplied exactly, and results in (0, 2^-14) are stored as
    RN-even FP16 subnormals."""
    cn = _range_net("dcgan64_l1", 6, cuda_device, lambda s, r: _sign_per_output(s, r, 1.0))
    B = 8
    rng = np.random.RandomState(6)
    keep = rng.rand(B, 8, 8, 256) < 1.0 / 64
    dy = np.concatenate([rng.randint(0, 2 ** (b + 1), size=(1, 8, 8, 256)) for b in range(B)]) * keep * 2.0 ** -24
    assert ((dy > 0) & (dy < 2.0 ** -14)).sum() > 1000
    v32, got, rep = _fp16_gradient_pass(cn, B, dy, W_BITS + 24, "dcgan64_l1 default B=8 pass 6 dgrad subnormals")
    sub = (np.abs(v32) > 0) & (np.abs(v32) < 2.0 ** -14)
    assert sub.sum() > 1000 and (np.abs(v32) >= 2.0 ** -14).sum() > 100
    assert not rep, rep


@pytest.mark.parametrize("backward", [False, True])
def test_narrow_fp16_form_rounds_its_weights_to_nearest(cgs_lib, cuda_device, backward):
    """The FP16 form of edge_narrow_tc converts its FP32 weights in its prologue; like every FP16 operand of the chain
    they are rounded to nearest even.  Weights below FP16's normal range make the rounding visible."""
    name, i = "dcgan64_l1", (3 if not backward else 4)      # G's last deconv forward / D's first conv data-gradient
    cn = _range_net(name, i, cuda_device,
                    lambda s, r: r.randint(-2047, 2048, size=s) * 2.0 ** -30)
    lay = cn.layout()
    B = 3
    rng = np.random.RandomState(8)
    tin = lay["act"][i] if not backward else lay["grad"][i + 1]
    tout = lay["act"][i + 1] if not backward else lay["grad"][i]
    assert tin["fp16"] and not tout["fp16"]
    x = R.grid(rng, R.dense_shape(tin, B), X_BITS, 2.0)
    scope, l = cn.layers[i]
    key = "%s/%s/w" % (scope, l["name"])
    w16 = cn.w[key].astype(np.float16).astype(np.float64)               # RN-even to FP16 subnormals
    assert not np.array_equal(w16, cn.w[key])
    w64 = dict(cn.w64)
    w64[key] = torch.from_numpy(w16).to(cuda_device)
    saved, cn.w64 = cn.w64, w64
    try:
            val, bound = cn.exact_pass(i, backward, x, R.dense_shape(lay["act"][i], B))
    finally:
        cn.w64 = saved
    v32 = R.exact_f32(val, bound, 24 + X_BITS)
    out = R.empty_chain(tout, B, cuda_device)
    aux = R.to_chain(np.zeros(R.dense_shape(lay["act"][i], B)), lay["act"][i], cuda_device) if backward else None
    cn.run(B, i, backward, R.to_chain(x, tin, cuda_device), out, aux=aux)
    got = R.from_chain(out, tout, B)
    if backward:                                   # tanh'(0) = 1, then the image gradient is rounded to TF32
        exp = R.tf32_rna(v32).astype(np.float64)
        ok = got == exp
    else:                                          # bias 0: tanh of the exact value
        exp = np.tanh(val).astype(np.float32).astype(np.float64)
        ok = R.ulps_fp32(got, exp) <= 2
    rep = R.mismatch_report(got, exp, ok)
    print("%s default B=%d pass %d %s subnormal-FP16 weights: %s" % (name, B, i, "dgrad" if backward else "fwd",
                                                                    "exact" if not rep else rep))
    assert not rep, rep


@pytest.mark.parametrize("operands", ["default", "tf32"])
@pytest.mark.parametrize("name", ["dcgan64_l1", "dcgan64_l4", "mnist"])
def test_fp32_operands_are_truncated_to_tf32(cgs_lib, cuda_device, name, operands):
    """The two MMAs that read FP32 values which are not TF32-exact -- layer 0's forward pass over the refined feature and
    D's first conv over the image -- see each operand truncated to TF32 (its low 13 mantissa bits dropped), not
    rounded: the results equal the exact reference over the truncated operands."""
    from cgs import lib as L
    cn = _net(name, cuda_device)
    B = 5
    rng = np.random.RandomState(9)
    with L.debug_flags(_operands(operands)):
        lay = cn.layout()
        fails = []
        for i in (0, lay["n_gtail"]):
            t = lay["act"][i]
            assert not t["fp16"]
            g = R.grid(rng, R.dense_shape(t, B), X_BITS, 2.0 if i == 0 else 1.0)
            x = R.off_tf32(rng, g).astype(np.float64)
            assert np.array_equal(R.trunc_tf32(x), g) and not np.array_equal(x, g)
            rep = _run_pass(cn, lay, i, False, B, rng, "%s %s B=%d knob=none off-TF32 input" % (name, operands, B),
                            x=x, x_exact=g)
            if rep:
                fails.append("pass %d fwd: %s" % (i, rep))
    assert not fails, "\n".join(fails)


HEAD_LOGITS = [0.0, -20.0, -23.5, -40.0, 17.0, 18.25, 40.0] + [s * 2.0 ** k for k in range(-9, 5) for s in (1, -1)]


@pytest.mark.parametrize("operands", ["default", "tf32"])
@pytest.mark.parametrize("name", ["dcgan64_l1", "dcgan32_l1", "mnist"])
def test_head(cgs_lib, cuda_device, name, operands):
    """head_kernel: the logit bit-exact; gexp exact (|dl| * 2^gexp in [1, 2), 0 for dl = 0) except where |dl| is within
    4 ulp of a power of two (expf); dpre within 1 ulp (FP16 or TF32) of the value of dl * 2^gexp * w * act'."""
    from cgs import lib as L
    cn = _net(name, cuda_device)
    rng = np.random.RandomState(10)
    with L.debug_flags(_operands(operands)):
        lay = cn.layout()
        n = lay["n"]
        tf, td = lay["act"][n], lay["grad"][n]
        target = np.array(HEAD_LOGITS + list(R.grid(rng, (19,), 9, 16.0)))
        B = len(target)
        wh = cn.head_w()
        bias = float(cn.w["discriminator/%s/bias" % cn.head["name"]][0])
        f = R.grid(rng, (B, wh.size), X_BITS, 2.0)
        f[:, 0] = 0.0
        f[:, 0] = target - (f @ wh + bias)                      # wh[0] == 1: every logit lands on its target
        logit64 = f @ wh + bias
        assert np.array_equal(logit64, target) and float((np.abs(f) @ np.abs(wh)).max()) < 2.0 ** (24 - 9)
        dpre = R.empty_chain(td, B, cuda_device)
        logits = torch.full((B,), float("nan"), device=cuda_device)
        gexp = torch.full((B,), -99, dtype=torch.int32, device=cuda_device)
        cn.run(B, n, True, R.to_chain(f, tf, cuda_device), dpre, aux=logits, gexp=gexp)
    got_logit = logits.cpu().numpy().astype(np.float64)
    l32 = target.astype(np.float32)
    dl = (np.float32(1) / (np.float32(1) + np.exp(-l32)) - np.float32(1)).astype(np.float32)
    dl64 = -1.0 / (1.0 + np.exp(target))
    e = np.where(dl != 0, 1 - np.frexp(dl)[1], 0)
    p2 = np.exp2(np.round(np.log2(np.maximum(np.abs(dl64), 1e-300))))
    near = np.abs(np.abs(dl64) - p2) <= 4 * np.spacing(p2.astype(np.float32)).astype(np.float64)
    act = cn.layers[n - 1][1]["act"]
    scaled = td["fp16"]
    dls = (dl * np.exp2(e if scaled else 0).astype(np.float32)).astype(np.float32)
    o = R.act_bwd(dls.reshape(-1, 1) * wh.astype(np.float32).reshape(1, -1), f.astype(np.float32), act)
    got = R.from_chain(dpre, td, B).reshape(B, -1)
    if scaled:
        exp = R.fp16_rn_satfinite(o).astype(np.float64)
        ok = R.within_fp16_ulp(got, exp)
        got_e = gexp.cpu().numpy()
    else:
        exp = R.tf32_rna(o).astype(np.float64)
        ok = np.abs(got - exp) <= np.spacing(np.abs(exp).astype(np.float32)).astype(np.float64) * 2 ** 13
        got_e = e
    ok[near] = True
    checks = [("logit", R.mismatch_report(got_logit.reshape(-1, 1), target.reshape(-1, 1))),
              ("gexp", R.mismatch_report(np.where(near, e, got_e).reshape(-1, 1), e.reshape(-1, 1))),
              ("dpre", R.mismatch_report(got, exp, ok))]
    zero = target >= 17
    assert np.all(dl[zero] == 0)
    assert np.all(got[zero] == 0) and np.all(np.isfinite(got)), "dl = 0 must give an all-zero dpre"
    if scaled:
        assert np.all(got_e[zero] == 0) and got_e[target == 0][0] == 1 and np.all(got_e[target <= -20] == 0)
    for what, rep in checks:
        print("%s %s B=%d head %s: %s" % (name, operands, B, what, "exact" if not rep else rep))
    assert not any(rep for _, rep in checks), checks
