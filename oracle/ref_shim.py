"""Import the UNMODIFIED reference: a drscotthawley/flocoder checkout named by ``FLOCODER_REFERENCE``, else one
placed (git-ignored) at ``oracle/_ref``.

TEST INFRASTRUCTURE ONLY.  The reference is not part of this repository, so
nothing that must run from the repository alone (``-m gpu`` tests, ``smoke()``,
``bench.py``) may call this; it is used to (a) prove the restatement in
``oracle/`` equal to the real thing and (b) generate the frozen vectors under
``tests/golden/``.  Without a checkout the tests that import it skip.

The reference's ``flocoder.sampling`` imports plotting/metrics/codec packages at
module level that are not installed here (SURVEY.md section 8c).  They carry no
arithmetic on the sampling path, so empty stand-in modules are registered
before the import; no reference file is touched.
"""
from __future__ import annotations

import os
import sys
import types
import warnings

REFERENCE_ROOT = os.environ.get("FLOCODER_REFERENCE") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "flocoder", "unet.py"))


def _stub(name: str, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    try:
        __import__(name)
        return sys.modules[name]
    except Exception:
        pass
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def load():
    """Returns (flocoder.unet, flocoder.sampling) of the reference checkout."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REFERENCE_ROOT} (set FLOCODER_REFERENCE or place one at oracle/_ref)")
    _stub("omegaconf", OmegaConf=object)
    _stub("matplotlib")
    _stub("matplotlib.pyplot")
    _stub("matplotlib.gridspec")
    _stub("torchmetrics")
    _stub("torchmetrics.image")
    _stub("torchmetrics.image.fid", FrechetInceptionDistance=object)
    _stub("geomloss", SamplesLoss=object)
    _stub("vector_quantize_pytorch", VectorQuantize=object, ResidualVQ=object)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import flocoder.unet as ref_unet          # noqa: E402
        import flocoder.sampling as ref_sampling  # noqa: E402
    return ref_unet, ref_sampling


def reference_euler(model, x0, sample_N, cond=None, eps=1e-3):
    """The legacy Euler recurrence (legacy/train_sd_flowers.py:50-67) driven through the
    reference model.  The legacy script itself cannot be imported (it runs a training job
    at import time and draws its own noise/cond from globals), so only its three-line
    recurrence is replayed here around the *reference* ``Unet``."""
    import torch
    with torch.no_grad():
        x = x0.detach().clone()
        dt = 1.0 / sample_N
        for i in range(sample_N):
            num_t = i / sample_N * (1 - eps) + eps
            t = torch.ones(x0.shape[0]) * num_t
            x = x.detach().clone() + model(x, t * 999, cond) * dt
    return x
