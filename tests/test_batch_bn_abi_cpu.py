"""Training-mode discriminator, host side: the ctypes mirror of cgs_batchnorm_desc has the C layout, and the workspace
query sizes and refuses batch-BN chains without a GPU."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "cgs.h"
int main(void) {
  printf("%zu %zu %zu %zu\n", sizeof(cgs_batchnorm_desc), offsetof(cgs_batchnorm_desc, n_layers),
         offsetof(cgs_batchnorm_desc, gamma), offsetof(cgs_batchnorm_desc, beta));
  return 0;
}
"""


def test_batchnorm_desc_layout_matches_the_header(tmp_path):
    from cgs import lib as L
    src = tmp_path / "probe.c"
    src.write_text(PROBE)
    exe = tmp_path / "probe"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size, n_off, g_off, b_off = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert C.sizeof(L.BatchnormDesc) == size
    assert (L.BatchnormDesc.n_layers.offset, L.BatchnormDesc.gamma.offset, L.BatchnormDesc.beta.offset) == (n_off, g_off, b_off)
    assert L.load().cgs_version() == 1


def _spec(arch):
    from cgs import nets as N
    from oracle import nets as onets
    return N.NetSpec(arch, onets.init_weights(arch, seed=1), "cpu")


def test_workspace_adds_the_pre_bn_tensors(cgs_lib):
    """DCGAN-64 l1 at B = 1024: the three BN layers' pre-BN outputs (16x16x128, 8x8x256, 4x4x512 per sample) are
    about 235 MB on top of the inference-mode workspace; a null descriptor is the plain query."""
    from cgs import nets as N
    spec = _spec(N.get_arch("dcgan64_l1"))
    g, d, db = C.byref(spec.gtail.desc), C.byref(spec.d.desc), spec.d_batch
    B = 1024
    plain = cgs_lib.cgs_refine_workspace_bytes(g, d, B)
    assert cgs_lib.cgs_refine_workspace_bytes_bn(g, d, None, B) == plain
    extra = cgs_lib.cgs_refine_workspace_bytes_bn(g, C.byref(db.desc), C.byref(db.bn_desc), B) - plain
    pre = 4 * B * (16 * 16 * 128 + 8 * 8 * 256 + 4 * 4 * 512)
    assert pre <= extra <= pre + (4 << 20), (extra, pre)
    assert 230e6 < pre < 240e6


def test_unfolded_packing_leaves_the_inference_packing_alone(cgs_lib):
    import torch
    from cgs import nets as N
    spec = _spec(N.get_arch("mnist"))
    before = [t.clone() for t in spec.d.tensors]
    db = spec.d_batch
    assert all(torch.equal(a, b) for a, b in zip(before, spec.d.tensors))
    assert spec.d.bn_desc is None and db.bn_desc.n_layers == 4
    assert [bool(db.bn_desc.gamma[i]) for i in range(4)] == [False, True, True, False]   # d_bn2, d_bn3


@pytest.mark.parametrize("where", ["image_edge", "head", "layer_count"])
def test_unsupported_batch_bn_layers_are_refused(cgs_lib, where):
    from cgs import lib as L
    from cgs import nets as N
    spec = _spec(N.get_arch("mnist"))
    db = spec.d_batch
    bn = L.BatchnormDesc()
    C.memmove(C.byref(bn), C.byref(db.bn_desc), C.sizeof(bn))
    j = {"image_edge": 0, "head": 3, "layer_count": 1}[where]
    bn.gamma[j], bn.beta[j] = bn.gamma[1], bn.beta[1]
    if where == "layer_count":
        bn.n_layers = 3
    n = cgs_lib.cgs_refine_workspace_bytes_bn(C.byref(spec.gtail.desc), C.byref(db.desc), C.byref(bn), 8)
    assert n == 0
    msg = L.last_error()
    assert {"image_edge": "image-edge", "head": "head", "layer_count": "layers"}[where] in msg, msg
