"""Import the reference's own ``sampling/*.py`` (numpy code) from a checkout of the original project.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  The original project is
not part of this repository; it is taken from ``/root/reference`` unless
``CGS_REFERENCE_ROOT`` names another checkout.  This module is used by
``oracle/make_golden.py`` (fixture generation) and by ``-m "not gpu"`` tests,
which fall back to the outputs make_golden stored when no checkout is present.

Shims (SURVEY.md §8c), none of which touches the reference's arithmetic:
  1. ``np.float = float``  -- ``sampling/rejector.py:12,18`` use the alias that
     numpy >= 1.24 removed.
  2. a stub ``tensorflow`` module -- ``sampling/policy.py:3`` imports it at top
     level; the numpy branches (``policy.py:26-51,61``) never touch ``tf``.
  3. ``FakeSession`` / ``FakeGan`` -- serve ``fake_sigmoid`` / ``fake_saliency``
     (``synthetic/GAN.py:108-111``) for ``sampling/refiner_cpu.py:23,27,52``
     from an FP32 torch-CPU copy of the 2-D discriminator MLP.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("CGS_REFERENCE_ROOT", "/root/reference")
SKIP_REASON = "no checkout of the original project (/root/reference or CGS_REFERENCE_ROOT)"


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "sampling", "rejector.py"))


_CACHE: dict = {}


def load_reference_sampling():
    """Return a namespace with the reference's policy/rejector/idpsampler/refiner_cpu modules."""
    if "ns" in _CACHE:
        return _CACHE["ns"]
    if not reference_available():
        raise RuntimeError(SKIP_REASON)
    if not hasattr(np, "float"):
        np.float = float  # shim 1
    if "tensorflow" not in sys.modules:
        sys.modules["tensorflow"] = types.ModuleType("tensorflow")  # shim 2
    sdir = os.path.join(REFERENCE_ROOT, "sampling")
    ddir = os.path.join(REFERENCE_ROOT, "synthetic")
    ns = types.SimpleNamespace()
    saved = {k: sys.modules.get(k) for k in ("policy", "rejector", "idpsampler", "refiner_cpu", "Datasets")}
    sys.path.insert(0, sdir)
    sys.path.insert(0, ddir)
    try:
        for name in ("policy", "rejector", "idpsampler", "refiner_cpu", "Datasets"):
            sys.modules.pop(name, None)
            mod = importlib.import_module(name)
            src = os.path.realpath(mod.__file__)
            assert src.startswith(os.path.realpath(REFERENCE_ROOT)), src
            setattr(ns, name, mod)
    finally:
        sys.path.remove(sdir)
        sys.path.remove(ddir)
        # do not leave the reference's flat module names shadowing the product's drop-ins
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    _CACHE["ns"] = ns
    return ns


class FakeGan:
    """Stands in for ``synthetic/GAN.py``'s graph handles (keys only)."""
    fake_samples = "fake_samples"
    fake_sigmoid = "fake_sigmoid"
    fake_saliency = "fake_saliency"


class FakeSession:
    """``sess.run([..], feed_dict={gan.fake_samples: x})`` served by the oracle MLP (shim 3)."""

    def __init__(self, mlp_weights):
        from . import nets
        self._w = mlp_weights
        self._nets = nets
        self.calls = 0

    def run(self, fetches, feed_dict):
        self.calls += 1
        x = np.asarray(feed_dict[FakeGan.fake_samples], dtype=np.float32)
        sig, sal = self._nets.mlp2d_sigmoid_saliency(x, self._w)
        table = {FakeGan.fake_sigmoid: sig, FakeGan.fake_saliency: sal}
        if isinstance(fetches, (list, tuple)):
            return [table[f] for f in fetches]
        return table[fetches]
