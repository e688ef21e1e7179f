"""Exact references for single passes of the refinement chain (test helper, not product code).

The weights, biases and inputs of a pass are put on coarse binary grids (w in 2^-4 Z, x in 2^-5 Z, ...).  Then every
product and every partial sum of the pass is an FP32 number, in any order, as long as sum |w * x| < 2^(24 - a - b) for
grids 2^-a and 2^-b: the FP32 accumulator of any lowering equals the FP64 value.  The expected output of a pass is
therefore its epilogue applied to that exact value, rounded the way the pass stores it (FP16: RN-even, satfinite; TF32
`round_out`: RNA, `cgs.nets.round_tf32`; FP32: as is), and the comparison is exact.

  * `ChainNet`: a grid-weight spec of an architecture with BN removed (`fold_layer` is then the identity and the
    packed FP32 / TF32 / FP16 matrices hold the grid values unchanged), its chain layout and a runner for one pass
    (`cgs_debug_chain_pass`);
  * `to_chain` / `from_chain`: dense FP64 tensors <-> the chain's buffers (FP32 or FP16; dense NHWC, s2d, pitched);
  * `exact_pass`: the FP64 value of a pass (`oracle.nets.run_layers`, autograd for the data-gradient) and the bound
    sum |w * x| per output element that makes it exact;
  * rounding and epilogue models; `mismatch_report` names the first mismatch and counts them per row and column.
"""
import ctypes as C

import numpy as np
import torch

from cgs import lib as L
from cgs import nets as N
from oracle import nets as onets
from oracle import sampling_np

DENSE, S2D, PITCHED = 0, 1, 2              # cgs_debug_chain_layout layouts
LAYOUT_NAMES = {DENSE: "dense", S2D: "s2d", PITCHED: "pitched"}
FP16_MAX = 65504.0
SLOPE = {"relu": 0.0, "lrelu": 0.2, "none": 1.0}


# ------------------------------------------------------------------------------------------------ chain layout
def chain_layout(gtail_desc, d_desc, math=L.MATH_TF32_TENSOR):
    """Decoded cgs_debug_chain_layout under the current CGS_DEBUG knobs."""
    lib = L.load()
    n = L.check(lib.cgs_debug_chain_layout(C.byref(gtail_desc), C.byref(d_desc), math, None, 0))
    buf = np.zeros(n, np.int32)
    L.check(lib.cgs_debug_chain_layout(C.byref(gtail_desc), C.byref(d_desc), math, buf.ctypes.data, n))
    v = buf.tolist()
    keys = ("fp16", "layout", "H", "W", "C", "cs", "pitch", "elems")
    nl = v[0]
    ents = [dict(zip(keys, v[4 + 8 * i:12 + 8 * i])) for i in range(2 * nl + 1)]
    return dict(n=nl, n_gtail=v[1], img_mode=v[2], f16=v[3], act=ents[:nl + 1], grad=[None] + ents[nl + 1:])


def describe(t):
    return "%s %s %dx%dx%d" % ("fp16" if t["fp16"] else "fp32", LAYOUT_NAMES[t["layout"]], t["H"], t["W"], t["C"])


# ------------------------------------------------------------------------------------------------ converters
def dense_shape(t, B):
    return (B, t["H"], t["W"], t["C"])


def to_chain(x, t, device):
    """Dense [B, H, W, C] values -> the chain's buffer [B, elems] of tensor `t` (zeros in padding channels and
    margins).  The values must be exact in the buffer's type."""
    x = np.asarray(x, np.float64)
    B, H, W, Cc = x.shape[0], t["H"], t["W"], t["C"]
    x = x.reshape(B, H, W, Cc)
    if t["layout"] == DENSE:
        buf = np.zeros((B, H, W, t["cs"]))
        buf[..., :Cc] = x
    elif t["layout"] == PITCHED:
        buf = np.zeros((B, H, W + 8, 4))
        buf[:, :, 2:2 + W, :Cc] = x
    else:                                   # [B][H/2][W/2][py][px][4]
        buf = np.zeros((B, H // 2, W // 2, 2, 2, 4))
        buf[..., :Cc] = x.reshape(B, H // 2, 2, W // 2, 2, Cc).transpose(0, 1, 3, 2, 4, 5)
    flat = np.zeros((B, t["elems"]))
    flat[:, :buf[0].size] = buf.reshape(B, -1)
    a = flat.astype(np.float16 if t["fp16"] else np.float32)
    assert np.array_equal(a.astype(np.float64), flat), "input not exact in %s" % describe(t)
    return torch.from_numpy(a).to(device)


def empty_chain(t, B, device):
    """An output buffer of tensor `t`, filled with NaN so that an element the pass does not write cannot pass."""
    return torch.full((B, t["elems"]), float("nan"), dtype=torch.float16 if t["fp16"] else torch.float32, device=device)


def from_chain(buf, t, B):
    """The chain's buffer of tensor `t` -> dense [B, H, W, C] float64."""
    a = buf.detach().cpu().numpy().astype(np.float64).reshape(B, -1)
    H, W, Cc = t["H"], t["W"], t["C"]
    if t["layout"] == DENSE:
        return a[:, :H * W * t["cs"]].reshape(B, H, W, t["cs"])[..., :Cc]
    if t["layout"] == PITCHED:
        return a[:, :H * (W + 8) * 4].reshape(B, H, W + 8, 4)[:, :, 2:2 + W, :Cc]
    s = a[:, :H * W * 4].reshape(B, H // 2, W // 2, 2, 2, 4).transpose(0, 1, 3, 2, 4, 5)
    return s.reshape(B, H, W, 4)[..., :Cc]


# ------------------------------------------------------------------------------------------------ grids
def grid(rng, shape, bits, maxabs):
    """Uniform values of 2^-bits Z in [-maxabs, maxabs]."""
    q = int(round(maxabs * 2 ** bits))
    return rng.randint(-q, q + 1, size=shape).astype(np.float64) / 2 ** bits


def off_tf32(rng, x):
    """x (TF32-exact FP32 values) with random bits below the TF32 mantissa set where x != 0: truncating the operand to
    TF32 gives x back, rounding it to nearest does not in about half of the cases."""
    x32 = np.asarray(x, np.float32)
    low = rng.randint(1, 0x2000, size=x32.shape).astype(np.int32)
    return np.where(x32 != 0, (x32.view(np.int32) | low).view(np.float32), x32)


def trunc_tf32(x):
    x32 = np.ascontiguousarray(x, np.float32)
    return (x32.view(np.int32) & ~0x1FFF).view(np.float32)


def grid_arch(name):
    """The architecture with every BN removed: packing is then the identity on the weight values."""
    arch = N.get_arch(name)
    return dict(arch, gtail=[dict(l, bn=None) for l in arch["gtail"]], d=[dict(l, bn=None) for l in arch["d"]])


def grid_weights(arch, rng, bits=4, maxabs=1.0):
    """TF-layout weights and biases on 2^-bits Z; the head's first weight is 1 (tests place logits through it)."""
    w = {}
    for scope, layers in (("generator", arch["gtail"]), ("discriminator", arch["d"])):
        for l in layers:
            p = "%s/%s/" % (scope, l["name"])
            if l["type"] == "conv":
                w[p + "w"] = grid(rng, (l["k"], l["k"], l["cin"], l["cout"]), bits, maxabs)
            elif l["type"] == "deconv":
                w[p + "w"] = grid(rng, (l["k"], l["k"], l["cout"], l["cin"]), bits, maxabs)
            else:
                w[p + "Matrix"] = grid(rng, (l["cin"], l["cout"]), bits, maxabs)
            w[p + ("bias" if l["type"] == "fc" else "biases")] = grid(rng, (l["cout"],), bits, maxabs)
    head = "discriminator/%s/" % arch["d"][-1]["name"]
    w[head + "Matrix"][0, 0] = 1.0
    w[head + "bias"][:] = 0.25
    return {k: v.astype(np.float32) for k, v in w.items()}


# ------------------------------------------------------------------------------------------------ the net
class ChainNet:
    """Grid weights of one architecture, packed for the library, and one-pass launches of its refinement chain."""

    def __init__(self, name, device, seed=0, weights=None):
        self.arch = grid_arch(name)
        self.name = name
        self.device = device
        self.w = weights if weights is not None else grid_weights(self.arch, np.random.RandomState(seed))
        self.spec = N.NetSpec(self.arch, self.w, device, math="tf32")
        self.layers = [("generator", l) for l in self.arch["gtail"]] + [("discriminator", l) for l in self.arch["d"][:-1]]
        self.head = self.arch["d"][-1]
        self.w64 = {k: torch.from_numpy(np.asarray(v, np.float64)).to(device) for k, v in self.w.items()}
        self.wabs = {k: v.abs() for k, v in self.w64.items()}
        self._ws = None

    def layout(self):
        return chain_layout(self.spec.gtail.desc, self.spec.d.desc)

    def head_w(self):
        return self.w["discriminator/%s/Matrix" % self.head["name"]][:, 0].astype(np.float64)

    def check_packing(self):
        """The packed matrices of every GEMM layer hold the grid filters, permuted by cgs_pack_map, unchanged: FP32
        `w_fwd` / `w_bwd` and their FP16 copies `w16_*`."""
        for i, (scope, l) in enumerate(self.layers):
            net = self.spec.gtail if scope == "generator" else self.spec.d
            li = [x["name"] for x in net.layers].index(l["name"])
            wf, bf = N.fold_layer(l, scope, self.w)
            ref_f, ref_b, bias = N.pack_layer(l, wf, bf)
            d = net.layer_desc(li)
            for ptr, rows, cols, ref, ptr16 in ((d.w_fwd, d.rows_fwd, d.kcols_fwd, ref_f, d.w16_fwd),
                                                 (d.w_bwd, d.rows_bwd, d.kcols_bwd, ref_b, d.w16_bwd)):
                got = _tensor_at(net, ptr, torch.float32, rows * cols).view(rows, cols).cpu()
                assert torch.equal(got, ref), (l["name"], "packed FP32 weights")
                if ptr16:
                    got16 = _tensor_at(net, ptr16, torch.float16, rows * cols).view(rows, cols).cpu()
                    assert torch.equal(got16.float(), ref), (l["name"], "packed FP16 weights")
            # the packed matrix is the TF filter permuted by cgs_pack_map (gather layout)
            if L.load().cgs_pass_layout(C.byref(d), 0) == 0 and l["type"] != "fc":
                ky, kx, ch = N.pack_map(l, False)
                valid = (ky >= 0) & (ch < l["cin"])
                filt = wf if l["type"] == "conv" else wf.permute(0, 1, 3, 2)            # [k, k, cin, cout]
                expect = filt[ky.clamp(min=0), kx.clamp(min=0), ch.clamp(max=l["cin"] - 1), :] * valid.view(-1, 1)
                assert torch.equal(ref_f, expect.t()), (l["name"], "pack map")

    def workspace(self, B):
        lib = L.load()
        n = int(lib.cgs_refine_workspace_bytes(C.byref(self.spec.gtail.desc), C.byref(self.spec.d.desc), B))
        if self._ws is None or self._ws.numel() < n:
            self._ws = torch.empty(n, dtype=torch.uint8, device=self.device)
        return self._ws

    def run(self, B, layer, backward, inp, out, aux=None, gexp=None, cfg=None, mom=None, first=0):
        lib = L.load()
        ws = self.workspace(B)
        L.check(lib.cgs_debug_chain_pass(C.byref(self.spec.gtail.desc), C.byref(self.spec.d.desc), L.MATH_TF32_TENSOR,
                                         B, layer, int(backward), L.ptr(inp), L.ptr(out), L.ptr(aux), L.ptr(gexp),
                                         C.byref(cfg) if cfg is not None else None, L.ptr(mom), int(first),
                                         L.ptr(ws), ws.numel(), L.stream_ptr()))
        torch.cuda.synchronize()

    def exact_pass(self, i, backward, x, in_shape):
        """FP64 value of pass (i, backward) on the dense input x: forward, the pre-activation output with bias;
        data-gradient, d sum(pre * x) / d (layer input), in_shape the dense shape of that input.  Returns (value,
        bound), bound = sum |w * x| (+ |bias|) per output element."""
        scope, l = self.layers[i]
        lin = dict(l, act="none", bn=None)
        xt = torch.from_numpy(np.asarray(x, np.float64)).to(self.device)

        def run(w, xv):
            if not backward:
                return onets.run_layers(xv, [lin], scope, w, "inference")
            z = torch.zeros(in_shape, dtype=torch.float64, device=self.device, requires_grad=True)
            pre = onets.run_layers(z, [lin], scope, w, "inference")
            (g,) = torch.autograd.grad((pre * xv.reshape(pre.shape)).sum(), z)
            return g

        val = run(self.w64, xt)
        bound = run(self.wabs, xt.abs())
        return val.detach().cpu().numpy(), bound.detach().cpu().numpy()


def _tensor_at(net, ptr, dtype, numel):
    for t in net.tensors:
        if t.data_ptr() == ptr and t.dtype == dtype and t.numel() == numel:
            return t
    raise KeyError("no packed tensor at %#x" % ptr)


# ------------------------------------------------------------------------------------------------ rounding models
def exact_f32(v, bound, bits):
    """v (FP64) as FP32, after checking the exactness condition: every partial sum on 2^-bits Z below 2^(24 - bits)."""
    limit = 2.0 ** (24 - bits)
    assert float(np.max(bound, initial=0.0)) < limit, "sum |w x| = %g breaks exact FP32 accumulation (< %g)" % (
        float(np.max(bound)), limit)
    v32 = np.asarray(v, np.float64).astype(np.float32)
    assert np.array_equal(v32.astype(np.float64), v)
    return v32


def fp16_rn_satfinite(v32):
    """cvt.rn.satfinite.f16.f32: round to nearest even, +-65504 instead of inf."""
    v32 = np.asarray(v32, np.float32)
    with np.errstate(over="ignore"):
        h = v32.astype(np.float16)
    return np.where(np.isinf(h) & np.isfinite(v32), np.copysign(np.float16(FP16_MAX), v32), h).astype(np.float16)


def tf32_rna(v32):
    return N.round_tf32(torch.from_numpy(np.ascontiguousarray(v32, np.float32))).numpy()


def store(v32, t, round_out):
    """What a pass stores for the FP32 epilogue result v32 into tensor t."""
    if t["fp16"]:
        return fp16_rn_satfinite(v32).astype(np.float64)
    return (tf32_rna(v32) if round_out else np.asarray(v32, np.float32)).astype(np.float64)


def act_fwd(v32, act):
    """Epilogue FWD after the bias: max(v, slope * v) in FP32 (tanh: the caller allows ulps)."""
    v32 = np.asarray(v32, np.float32)
    if act == "tanh":
        return np.tanh(v32.astype(np.float64)).astype(np.float32)
    return np.maximum(v32, v32 * np.float32(SLOPE[act]))


def act_bwd(a32, x0, act):
    """Epilogue BWD: a * act'(x0), x0 the forward output (FP32 arithmetic; tanh: a * (1 - x0 * x0))."""
    a32, x0 = np.asarray(a32, np.float32), np.asarray(x0, np.float32)
    if act == "tanh":
        return a32 * (np.float32(1) - x0 * x0)
    return a32 * np.where(x0 > 0, np.float32(1), np.float32(SLOPE[act]))


def policy(cfg, feature, grad32, mom, first):
    """The fused policy step (sampling/policy.py:27-37 via the pinned oracle, then collaborator.py:69-70's clip)."""
    theta = np.array(feature, np.float32)
    method = "sgd" if cfg.method == L.POLICY_SGD else "momentum"
    state = {"momentum": None if first or method == "sgd" else np.array(mom, np.float32)}
    sampling_np.policy_step(method, theta, np.asarray(grad32, np.float32), state, cfg.rate, alpha=cfg.alpha)
    if cfg.clip:
        theta = np.minimum(np.maximum(theta, np.float32(cfg.vmin)), np.float32(cfg.vmax))
    return theta, state["momentum"]


def ulps_fp32(got, exp):
    exp32 = np.asarray(exp, np.float32)
    return np.abs(np.asarray(got, np.float64) - exp32.astype(np.float64)) / np.spacing(np.abs(exp32)).astype(np.float64)


def within_fp16_ulp(got, exp, n=1):
    e16 = np.asarray(exp, np.float16)
    return np.abs(np.asarray(got, np.float64) - e16.astype(np.float64)) <= n * np.spacing(np.abs(e16)).astype(np.float64)


# ------------------------------------------------------------------------------------------------ report
def mismatch_report(got, exp, ok=None):
    """'' when every element matches, else: count, first (b, y, x, c) with both values, counts per row and column."""
    got = np.asarray(got, np.float64)
    exp = np.asarray(exp, np.float64)
    if got.ndim == 2:
        got, exp = got[:, None, None, :], exp[:, None, None, :]
        ok = None if ok is None else ok[:, None, None, :]
    if ok is None:
        ok = (got == exp) | (np.isnan(got) & np.isnan(exp))
    bad = np.argwhere(~ok)
    if not len(bad):
        return ""
    b, y, x, c = bad[0]
    rows = np.bincount(bad[:, 1], minlength=got.shape[1])
    cols = np.bincount(bad[:, 2], minlength=got.shape[2])
    return ("%d of %d elements differ; first (b, y, x, c) = (%d, %d, %d, %d): got %r, expected %r; per row %s; per "
            "column %s" % (len(bad), ok.size, b, y, x, c, got[b, y, x, c], exp[b, y, x, c],
                           {int(i): int(n) for i, n in enumerate(rows) if n}, {int(i): int(n) for i, n in enumerate(cols) if n}))
