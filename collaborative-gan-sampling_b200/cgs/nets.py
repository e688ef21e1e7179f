"""Network specs for the image path: architecture descriptions, BN folding and weight packing.

A *spec* replaces the graph-building callables the reference hands to ``Refiner.set_env``
(``nsgan/GAN.py:172-180``): it is an architecture description plus packed device weights.

Weight interchange format (input of :func:`pack_network`) = the reference's TF variables by name and layout
(``nsgan/ops.py:38-46,49-62,75-79,19-26``):
  ``<scope>/<layer>/w``        conv   [kh, kw, Cin, Cout]     deconv [kh, kw, Cout, Cin]
  ``<scope>/<layer>/biases``   [Cout]
  ``<scope>/<layer>/Matrix``   linear [in, out]   ``<scope>/<layer>/bias`` [out]
  ``<scope>/<bn>/gamma|beta|moving_mean|moving_variance``  [C]
with scope ``generator`` / ``discriminator`` (``nsgan/GAN.py:62,75``).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import lib as L

BN_EPS = 1e-5   # nsgan/ops.py:23


def conv_out_size_same(size, stride):          # nsgan/ops.py:28-29
    return int(math.ceil(float(size) / float(stride)))


def arch_mnist_infogan(layer=1):
    """infoGAN-MNIST nets of nsgan/GAN.py:59-101.  layer=1 splits at the [7,7,128] map exactly like the reference
    (GAN.py:87-101); layer=2 refines the [14,14,64] map that feeds the last deconv instead."""
    if layer not in (1, 2):
        raise ValueError("layer must be 1 or 2")
    gtail = [
        dict(type="deconv", name="g_dc3", k=4, cin=128, cout=64, hin=7, win=7, bn="g_bn3", act="relu"),
        dict(type="deconv", name="g_dc4", k=4, cin=64, cout=1, hin=14, win=14, bn=None, act="tanh"),
    ][layer - 1:]
    return {
        "name": "mnist_infogan" if layer == 1 else "mnist_infogan_l2",
        "feature_shape": [7, 7, 128] if layer == 1 else [14, 14, 64],
        "image_shape": [28, 28, 1],
        # proposal head = nsgan/GAN.py:87-92 input_to_feature (BN inference); only used to produce proposals from z
        "z_dim": 62,
        "head": [
            dict(type="fc", name="g_fc1", cin=62, cout=1024, bn="g_bn1", act="relu"),
            dict(type="fc", name="g_fc2", cin=1024, cout=6272, bn="g_bn2", act="relu"),
        ] + ([dict(type="deconv", name="g_dc3", k=4, cin=128, cout=64, hin=7, win=7, bn="g_bn3", act="relu")]
             if layer == 2 else []),
        "head_reshape": [7, 7, 128],
        "gtail": gtail,
        "d": [
            dict(type="conv", name="d_conv1", k=4, cin=1, cout=64, hin=28, win=28, bn=None, act="lrelu"),
            dict(type="conv", name="d_conv2", k=4, cin=64, cout=128, hin=14, win=14, bn="d_bn2", act="lrelu"),
            dict(type="fc", name="d_fc3", cin=6272, cout=1024, bn="d_bn3", act="lrelu"),
            dict(type="fc", name="d_fc4", cin=1024, cout=1, bn=None, act="none"),
        ],
    }


def arch_dcgan(size=64, layer=1, gf=64, df=64, c_dim=3, k=5):
    """DCGAN generator tail from activation map ``layer`` (1..4) + discriminator (SURVEY.md App. B; upstream
    carpedm20/DCGAN-tensorflow shapes, k=5 s=2 defaults of nsgan/ops.py:37,48)."""
    if not 1 <= layer <= 4:
        raise ValueError("layer must be 1..4")
    sizes = [size]
    for _ in range(4):
        sizes.append(conv_out_size_same(sizes[-1], 2))
    gsz = [sizes[4], sizes[3], sizes[2], sizes[1], size]
    gch = [gf * 8, gf * 4, gf * 2, gf, c_dim]
    gtail = []
    for i in range(layer - 1, 4):
        last = i == 3
        gtail.append(dict(type="deconv", name="g_h%d" % (i + 1), k=k, cin=gch[i], cout=gch[i + 1], hin=gsz[i],
                          win=gsz[i], bn=None if last else "g_bn%d" % (i + 1), act="tanh" if last else "relu"))
    dch = [c_dim, df, df * 2, df * 4, df * 8]
    dsz = [size, sizes[1], sizes[2], sizes[3], sizes[4]]
    d = [dict(type="conv", name="d_h%d_conv" % i, k=k, cin=dch[i], cout=dch[i + 1], hin=dsz[i], win=dsz[i],
              bn=None if i == 0 else "d_bn%d" % i, act="lrelu") for i in range(4)]
    d.append(dict(type="fc", name="d_h4_lin", cin=sizes[4] * sizes[4] * df * 8, cout=1, bn=None, act="none"))
    # proposal head (upstream DCGAN generator up to the refined map): linear -> reshape -> bn0 -> relu [-> deconvs]
    head = [dict(type="fc", name="g_h0_lin", cin=100, cout=gsz[0] * gsz[0] * gch[0], bn="g_bn0", bn_channels=gch[0],
                 act="relu")]
    for i in range(layer - 1):
        head.append(dict(type="deconv", name="g_h%d" % (i + 1), k=k, cin=gch[i], cout=gch[i + 1], hin=gsz[i], win=gsz[i],
                         bn="g_bn%d" % (i + 1), act="relu"))
    return {"name": "dcgan%d_l%d" % (size, layer),
            "feature_shape": [gsz[layer - 1], gsz[layer - 1], gch[layer - 1]],
            "image_shape": [size, size, c_dim], "z_dim": 100, "head": head, "head_reshape": [gsz[0], gsz[0], gch[0]],
            "gtail": gtail, "d": d}


def get_arch(name):
    if name in ("mnist", "mnist_infogan"):
        return arch_mnist_infogan()
    if name in ("mnist_l2", "mnist_infogan_l2"):
        return arch_mnist_infogan(2)
    if name.startswith("dcgan"):
        size, _, layer = name[len("dcgan"):].partition("_l")
        return arch_dcgan(int(size), int(layer or 1))
    raise KeyError(name)


def cstride(c):
    return (c + 3) & ~3


def _as_t(v):
    return v.detach().to("cpu", torch.float32) if isinstance(v, torch.Tensor) else torch.from_numpy(np.asarray(v, np.float32))


def fold_layer(layer, scope, weights, fold_bn=True):
    """Inference-mode BN folded into the layer: returns (W_tf_layout_scaled, bias_folded).  fold_bn=False: the layer's
    own (W, bias), for a batch-statistic BN applied after it."""
    p = "%s/%s/" % (scope, layer["name"])
    if layer["type"] == "fc":
        w, b = _as_t(weights[p + "Matrix"]).clone(), _as_t(weights[p + "bias"]).clone()
    else:
        w, b = _as_t(weights[p + "w"]).clone(), _as_t(weights[p + "biases"]).clone()
    if layer["bn"] and fold_bn:
        q = "%s/%s/" % (scope, layer["bn"])
        s = _as_t(weights[q + "gamma"]).double() / torch.sqrt(_as_t(weights[q + "moving_variance"]).double() + BN_EPS)
        t = _as_t(weights[q + "beta"]).double() - _as_t(weights[q + "moving_mean"]).double() * s
        if layer.get("bn_channels"):            # BN applied after an NHWC reshape of a linear output: tile per channel
            rep = layer["cout"] // layer["bn_channels"]
            s, t = s.repeat(rep), t.repeat(rep)
        if layer["type"] == "conv":
            w = (w.double() * s.view(1, 1, 1, -1)).float()
        elif layer["type"] == "deconv":
            w = (w.double() * s.view(1, 1, -1, 1)).float()
        else:
            w = (w.double() * s.view(1, -1)).float()
        b = (b.double() * s + t).float()
    return w, b


def _padded_cin(layer):
    """fc inputs are padded with zeros to a multiple of 32 (one K atom), e.g. z_dim 62 -> 64, 100 -> 128."""
    return (layer["cin"] + 31) // 32 * 32 if layer["type"] == "fc" else layer["cin"]


def _layer_desc(layer):
    d = L.LayerDesc()
    d.type = L.LAYER_IDS[layer["type"]]
    d.k = layer.get("k", 1)
    d.cin, d.cout = _padded_cin(layer), layer["cout"]
    d.hin, d.win = layer.get("hin", 1), layer.get("win", 1)
    d.act = L.ACT_IDS[layer["act"]]
    return d


def pack_map(layer, backward):
    """(ky, kx, ch) int64 tensors for every K index of the packed matrix (cgs_pack_map, host only)."""
    lib = L.load()
    d = _layer_desc(layer)
    n = L.check(lib.cgs_pack_map(C.byref(d), int(backward), None, None, None, 0))
    ky = np.empty(n, np.int32)
    kx = np.empty(n, np.int32)
    ch = np.empty(n, np.int32)
    L.check(lib.cgs_pack_map(C.byref(d), int(backward), ky.ctypes.data, kx.ctypes.data, ch.ctypes.data, n))
    return torch.from_numpy(ky).long(), torch.from_numpy(kx).long(), torch.from_numpy(ch).long()


def pack_layer(layer, w, b):
    """Folded TF-layout weights -> (w_fwd [cout, Kf], w_bwd [cin, Kb] or None, bias [cstride(cout)])."""
    cin, cout = _padded_cin(layer), layer["cout"]
    if cin != layer["cin"]:                    # zero rows for the padded fc inputs
        w = torch.cat([w, torch.zeros(cin - layer["cin"], cout)], dim=0)
    bias = torch.zeros(cstride(cout))
    bias[:cout] = b
    if layer["type"] == "fc" and cout == 1:
        return w.t().contiguous(), None, bias           # head: [1, cin] row vector, used in both directions

    def gather(ky, kx, ch, reduce_is_cin):
        nred = cin if reduce_is_cin else cout
        valid = (ky >= 0) & (ch < nred)
        kyc, kxc, chc = ky.clamp(min=0), kx.clamp(min=0), ch.clamp(max=nred - 1)
        if layer["type"] == "fc":
            m = w[chc, :] if reduce_is_cin else w[:, chc].t()          # [K, cout] / [K, cin]
        elif layer["type"] == "conv":                                   # [kh,kw,Cin,Cout]
            m = w[kyc, kxc, chc, :] if reduce_is_cin else w[kyc, kxc, :, chc]
        else:                                                           # deconv [kh,kw,Cout,Cin]
            m = w[kyc, kxc, :, chc] if reduce_is_cin else w[kyc, kxc, chc, :]
        m = m * valid.view(-1, 1).to(m.dtype)
        return m.t().contiguous()                                       # [rows, K]

    def scatter(small_is_cout):
        """rows = (ky*k + kx)*4 + small channel, K = the large channel count (cgs_pass_layout == 1)."""
        k = layer["k"]
        if layer["type"] == "deconv":            # [kh,kw,Cout,Cin], forward: small = cout, reduce over cin
            m = w                                 # [k,k,cout,cin]
        else:                                    # conv [kh,kw,Cin,Cout], backward: small = cin, reduce over cout
            m = w                                 # [k,k,cin,cout]
        small, big = m.shape[2], m.shape[3]
        out = torch.zeros(k, k, 4, big)
        out[:, :, :small, :] = m
        return out.reshape(k * k * 4, big).contiguous()

    def window():
        """rows = large channel, K index = ky*32 + kx*4 + small channel (cgs_pass_layout == 2)."""
        k = layer["k"]
        small, big = w.shape[2], w.shape[3]                # conv [k,k,cin,cout] fwd / deconv [k,k,cout,cin] bwd
        out = torch.zeros(big, k, 8, 4)
        out[:, :, :k, :small] = w.permute(3, 0, 1, 2)
        return out.reshape(big, k * 32).contiguous()

    lib = L.load()
    d = _layer_desc(layer)
    kinds = {0: None, 1: scatter, 2: window}
    lf, lb = lib.cgs_pass_layout(C.byref(d), 0), lib.cgs_pass_layout(C.byref(d), 1)
    w_fwd = gather(*pack_map(layer, False), True) if lf == 0 else (scatter(True) if lf == 1 else window())
    w_bwd = gather(*pack_map(layer, True), False) if lb == 0 else (scatter(False) if lb == 1 else window())
    return w_fwd, w_bwd, bias


FP16_MAX = 65504.0


def round_tf32(t):
    """Round-to-nearest (ties away, like cvt.rna.tf32.f32) to a 10-bit mantissa, so that the tensor core's operand
    truncation is exact instead of a systematic shrink."""
    i = t.contiguous().view(torch.int32)
    r = ((i + 0x1000) & ~0x1FFF).view(torch.float32)
    return torch.where(torch.isfinite(t), r, t)


class PackedNet:
    """A chain of packed layers resident on one device + the cgs_net_desc that points at them.

    fold_bn=False packs the layers without their BN (training mode): ``bn_desc`` (cgs_batchnorm_desc) then points at
    device copies of every BN's gamma / beta, which the library applies with the statistics of the batch."""

    def __init__(self, layers, scope, weights, device, math="tf32", fold_bn=True):
        if len(layers) > L.MAX_LAYERS:
            raise ValueError("too many layers")
        self.layers = [dict(l) for l in layers]
        self.scope = scope
        self.device = torch.device(device)
        self.tensors = []
        self.desc = L.NetDesc()
        self.desc.n_layers = len(layers)
        self.bn_desc = None
        if not fold_bn:
            self.bn_desc = L.BatchnormDesc()
            self.bn_desc.n_layers = len(layers)
        for i, layer in enumerate(layers):
            w, b = fold_layer(layer, scope, weights, fold_bn)
            if not fold_bn and layer["bn"]:
                q = "%s/%s/" % (scope, layer["bn"])
                gamma, beta = (_as_t(weights[q + k]).to(self.device) for k in ("gamma", "beta"))
                self.tensors += [gamma, beta]
                self.bn_desc.gamma[i], self.bn_desc.beta[i] = gamma.data_ptr(), beta.data_ptr()
            wf, wb, bias = pack_layer(layer, w, b)
            if math == "tf32" and wb is not None:       # GEMM layers only; the 1-logit head stays FP32
                wf, wb = round_tf32(wf), round_tf32(wb)
            d = _layer_desc(layer)
            wf = wf.to(self.device)
            bias = bias.to(self.device)
            self.tensors += [wf, bias]
            d.w_fwd, d.rows_fwd, d.kcols_fwd = wf.data_ptr(), wf.shape[0], wf.shape[1]
            d.bias = bias.data_ptr()
            if wb is not None:
                wb = wb.to(self.device)
                self.tensors.append(wb)
                d.w_bwd, d.rows_bwd, d.kcols_bwd = wb.data_ptr(), wb.shape[0], wb.shape[1]
                if math == "tf32" and fold_bn and max(float(wf.abs().max()), float(wb.abs().max())) <= FP16_MAX:
                    # FP16 copies of the TF32-rounded matrices (the same values: same 10-bit mantissa, inside FP16's
                    # range); whether a chain runs on them is the library's decision (choose_operand_type)
                    wf16, wb16 = wf.half(), wb.half()
                    self.tensors += [wf16, wb16]
                    d.w16_fwd, d.w16_bwd = wf16.data_ptr(), wb16.data_ptr()
            self.desc.layers[i] = d

    def layer_desc(self, i):
        return self.desc.layers[i]


class NetSpec:
    """What ``Refiner.set_env`` receives in place of the reference's TF callables."""

    def __init__(self, arch, weights, device="cuda", role=None, math="tf32"):
        """math='tf32': tensor-core path (weights pre-rounded to TF32); math='fp32': exact-FP32 SIMT path."""
        if math not in L.MATH_IDS:
            raise ValueError("math must be 'tf32' or 'fp32'")
        self.arch = arch
        self.math = math
        self.device = torch.device(device)
        self.gtail = PackedNet(arch["gtail"], "generator", weights, self.device, math)
        self.d = PackedNet(arch["d"], "discriminator", weights, self.device, math)
        self.role = role
        self._weights = weights
        self._d_batch = None

    @property
    def d_batch(self):
        """D packed for training-mode BN (``discriminator_spec(spec, is_training=True)``): unfolded weights and the
        BN parameters, packed on first use; ``d`` (inference mode, BN folded) is unchanged."""
        if self._d_batch is None:
            self._d_batch = PackedNet(self.arch["d"], "discriminator", self._weights, self.device, self.math, fold_bn=False)
        return self._d_batch

    @classmethod
    def from_variables(cls, arch, variables, device="cuda", math="tf32", layout="tf"):
        """Build a spec from an externally produced name -> array mapping (SURVEY.md §8 f3): Saver decorations are
        stripped, ``layout='torch'`` converts PyTorch-ordered kernels, and every variable is checked against the
        architecture (missing names / wrong layouts raise with the offending name)."""
        from . import weights as W
        v = W.normalize_names(variables)
        if layout == "torch":
            v = W.from_torch_layout(arch, v)
        elif layout != "tf":
            raise ValueError("layout must be 'tf' or 'torch'")
        return cls(arch, W.validate(arch, v), device, math=math)

    @classmethod
    def from_npz(cls, arch, path, device="cuda", math="tf32", layout="tf"):
        """Spec from an ``.npz`` of the reference's TF variables (``cgs.weights`` says how to dump a checkpoint)."""
        from . import weights as W
        return cls.from_variables(arch, W.load_npz(path), device, math=math, layout=layout)

    @property
    def feature_shape(self):
        return tuple(self.arch["feature_shape"])

    @property
    def image_shape(self):
        return tuple(self.arch["image_shape"])


class _Role:
    """View of a NetSpec playing one of the two set_env roles (discriminator / feature_to_data)."""

    def __init__(self, spec, role, is_training=False):
        self.spec, self.role, self.is_training = spec, role, bool(is_training)


def discriminator_spec(spec, is_training=False):
    """``partial(self.discriminator, is_training=..., reuse=True)`` (nsgan/GAN.py:175).  False (the default): BN in
    inference mode, folded into the weights.  True: the reference's mode, BN with the statistics of the batch being
    refined and the gradient through them (the moving averages are not updated)."""
    return _Role(spec, "discriminator", is_training)


def feature_to_data_spec(spec):
    return _Role(spec, "feature_to_data")


def loss_refine(logits=None):
    """Marker for the only refinement loss the reference uses: un-reduced BCE-with-ones (nsgan/GAN.py:176-177)."""
    raise NotImplementedError("loss_refine is a marker object; the CUDA path fuses softplus(-logit) and its gradient")


loss_refine.is_bce_with_ones = True


class ProposalHead:
    """z -> refined activation map on the device: ``input_to_feature`` of nsgan/GAN.py:87-92 (fc+BN+relu x2) or the
    DCGAN generator up to the refined layer (linear, reshape, bn0, relu[, deconvs]); BN in inference mode, folded.
    Runs the same gathered-GEMM kernel as the refinement loop (SURVEY.md §8 f2)."""

    def __init__(self, arch, weights, device="cuda", math="tf32"):
        self.arch = arch
        self.math = math
        self.device = torch.device(device)
        self.net = PackedNet(arch["head"], "generator", weights, self.device, math)
        self._ws = None

    def __call__(self, z):
        import ctypes as C
        lib = L.load()
        zt = z if isinstance(z, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(z, dtype=np.float32))
        x = zt.to(self.device, torch.float32)
        B = x.shape[0]
        for i, layer in enumerate(self.net.layers):
            d = self.net.layer_desc(i)
            if layer["type"] == "fc":
                x = x.reshape(B, -1)
                if x.shape[1] != d.cin:
                    x = torch.nn.functional.pad(x, (0, d.cin - x.shape[1]))
                y = torch.empty(B, cstride(layer["cout"]), dtype=torch.float32, device=self.device)
            else:
                if x.dim() == 2:
                    x = x.reshape(B, *self.arch["head_reshape"])
                y = torch.empty(B, layer["hin"] * 2, layer["win"] * 2, cstride(layer["cout"]), dtype=torch.float32,
                                device=self.device)
            nbytes = int(lib.cgs_layer_workspace_bytes(C.byref(d), B))
            if self._ws is None or self._ws.numel() < nbytes:
                self._ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=self.device)
            L.check(lib.cgs_layer_forward(C.byref(d), L.MATH_IDS[self.math], B, L.ptr(x.contiguous()), L.ptr(y),
                                          L.ptr(self._ws), self._ws.numel(), L.stream_ptr()))
            x = y
        return x.reshape(B, *self.arch["feature_shape"])
