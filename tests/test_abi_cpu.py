"""The C-ABI library builds, loads and exports every symbol include/cgs.h declares; host-only calls work without
a GPU; compute calls fail loudly (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "cgs.h")).read()
    return sorted(set(re.findall(r"CGS_API[^;(]*?\b(cgs_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(cgs_lib):
    from cgs import lib
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(cgs_lib, n), n
    assert set(lib.EXPORTED_SYMBOLS) <= set(names) | {"cgs_debug_trace"}
    assert cgs_lib.cgs_version() == 1


def declared_debug_flags():
    text = open(os.path.join(ROOT, "include", "cgs.h")).read()
    body = re.search(r"enum cgs_debug_flag \{(.*?)\};", text, re.S).group(1)
    return {name: int(v) for name, v in re.findall(r"\bCGS_(DEBUG_[A-Z0-9_]+)\s*=\s*(\d+)", body)}


def test_debug_flags_mirror_the_header():
    from cgs import lib
    flags = declared_debug_flags()
    assert len(flags) >= 20 and len(set(flags.values())) == len(flags)
    assert all(v & (v - 1) == 0 for v in flags.values())          # one bit each
    mirrored = {n: getattr(lib, n) for n in dir(lib) if n.startswith("DEBUG_") and isinstance(getattr(lib, n), int)}
    assert mirrored == flags


def test_sass_is_blackwell_native():
    import subprocess
    so = os.path.join(ROOT, "collaborative-gan-sampling_b200", "cgs", "libcgs.so")
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    assert "sm_100a" in sass or "SM100" in sass.upper()
    # tcgen05 MMAs / TMA loads / TMEM loads / commits, and the CTA-pair (cta_group::2) forms with multicast commits
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM", "UTCBAR", "UTCHMMA.2CTA", "UTMALDG.4D.2CTA", "UTCBAR.2CTA.MULTICAST"):
        assert mnemonic in sass, mnemonic


def test_host_only_entry_points(cgs_lib):
    from cgs import lib as L, nets as N
    arch = N.get_arch("dcgan64_l1")
    for layer in arch["gtail"] + arch["d"][:-1]:
        for bw in (0, 1):
            d = N._layer_desc(layer)
            layout = cgs_lib.cgs_pass_layout(C.byref(d), bw)
            assert layout in (0, 1, 2)
            if layout == 0:
                ky, kx, ch = N.pack_map(layer, bw)
                assert len(ky) % 32 == 0 and int(ky.max()) < layer.get("k", 1)
    bad = N._layer_desc(dict(type="conv", name="x", k=7, cin=64, cout=64, hin=8, win=8, act="relu"))
    assert cgs_lib.cgs_pack_map(C.byref(bad), 0, None, None, None, 0) == L.CGS_ERR_UNSUPPORTED
    assert b"kernel size" in cgs_lib.cgs_last_error()
    assert cgs_lib.cgs_drs_workspace_bytes(1000) > 8000 and cgs_lib.cgs_mh_workspace_bytes(1000) > 12000


@pytest.mark.skipif(torch.cuda.is_available(), reason="only meaningful on the GPU-less build box")
def test_no_cpu_fallback():
    from cgs import lib as L
    from sampling.idpsampler import IndependenceSampler
    from sampling.policy import PolicyAdaptive
    from sampling.rejector import Rejector
    with pytest.raises(RuntimeError):
        Rejector().sampling(np.zeros((4, 2), np.float32), np.full((4, 1), .5, np.float32))
    with pytest.raises(RuntimeError):
        IndependenceSampler().sampling(np.zeros((4, 2), np.float32), np.full((4, 1), .5, np.float32))
    with pytest.raises(RuntimeError):
        PolicyAdaptive(0.1, "sgd").apply_gradient(np.zeros((4, 2), np.float32), np.zeros((4, 2), np.float32))
    # the raw ABI refuses as well
    cfg = L.PolicyCfg()
    rc = L.load().cgs_policy_step(C.byref(cfg), None, None, None, None, None, None, 1, 1, 1, None)
    assert rc == L.CGS_ERR_CUDA and b"CPU" in L.load().cgs_last_error()


def test_synthetic_init_matches_oracle_init(cgs_lib):
    from cgs import nets as N, synthetic as S
    from oracle import nets as onets
    arch = N.get_arch("mnist")
    a, b = S.init_weights(arch, seed=5, gain=2.0), onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=5), 2.0)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    for (k1, b1), (k2, b2) in zip(S.init_mlp2d(seed=3), onets.init_mlp2d(seed=3)):
        assert np.array_equal(k1, k2) and np.array_equal(b1, b2)
