"""log_likelihood without a GPU: the generic composition against the closed form of a linear flow, argument errors before
the model is called, and the argument checks of flo_unet_jvp / flo_integrate_divergence."""
import ctypes
import math

import pytest
import torch

from flocoder_b200 import _lib, sampling


class Linear(torch.nn.Module):
    """v(x, t) = A x with a fixed diagonal A over a 2x2x2 latent (float64)."""

    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(5)
        self.a = torch.nn.Parameter((torch.rand(2, 2, 2, generator=g, dtype=torch.float64) - 0.5))
        self.calls = 0

    def forward(self, x, time, cond=None):
        self.calls += 1
        return self.a * x


def latents(b=3):
    return torch.randn(b, 2, 2, 2, generator=torch.Generator().manual_seed(1), dtype=torch.float64)


def test_linear_flow_matches_the_closed_form():
    """x_t = e^{A(t-1)} x_1 backwards to t = 0, and log p_1(x_1) = log N(e^{-A} x_1) - tr A; Rademacher probes give the
    trace of a diagonal Jacobian exactly."""
    m, x1 = Linear(), latents()
    g = torch.Generator().manual_seed(2)
    logp, noise, nfe = sampling.log_likelihood(m, x1, n_steps=50, n_probes=2, generator=g)
    a = m.a.detach()
    z = torch.exp(-a) * x1
    want = -0.5 * z.flatten(1).pow(2).sum(1) - 4 * math.log(2 * math.pi) - a.sum()
    assert nfe == 4 * 49 and m.calls == 2 * nfe
    assert logp.dtype == torch.float64 and logp.shape == (3,)
    assert float((noise - z).abs().max()) < 1e-8
    assert float((logp - want).abs().max()) < 1e-8


def test_noise_is_invert_latents_and_probes_may_be_given():
    m, x1 = Linear(), latents()
    probes = torch.randint(0, 2, (3,) + tuple(x1.shape), generator=torch.Generator().manual_seed(4)).double() * 2 - 1
    logp, noise, nfe = sampling.log_likelihood(m, x1, n_steps=7, probes=probes)
    inv, nfe_inv = sampling.invert_latents(m, x1, n_steps=7, method="rk4")
    assert torch.equal(noise, inv) and nfe == nfe_inv
    logp3, _, _ = sampling.log_likelihood(m, x1, n_steps=7, probes=probes, n_probes=3)
    assert torch.equal(logp, logp3)


@pytest.mark.parametrize("kw, what", [
    (dict(probes=torch.ones(2, 3, 2, 2, 3)), "probes must be"),
    (dict(probes=torch.ones(3, 2, 2, 2)), "probes must be"),
    (dict(n_probes=0), "n_probes"),
    (dict(n_probes=1.5), "n_probes"),
    (dict(n_probes=2, probes=torch.ones(3, 3, 2, 2, 2)), "disagrees"),
    (dict(n_steps=1), "n_steps"),
    (dict(n_steps=2.5), "n_steps"),
])
def test_argument_errors_raise_before_the_model_is_called(kw, what):
    m = Linear()
    with pytest.raises(ValueError, match=what):
        sampling.log_likelihood(m, latents(), **kw)
    assert m.calls == 0


def test_c_abi_argument_checks_need_no_device():
    L = _lib.lib()
    buf = (ctypes.c_float * 4)()
    div = (ctypes.c_double * 4)()
    ts = (ctypes.c_float * 2)(1.0, 0.0)
    p = ctypes.cast(buf, ctypes.c_void_p)

    def integ(y=p, ts_=ts, n_ts=2, probes=p, n_p=1, d=ctypes.cast(div, ctypes.c_void_p), b=1, h=None):
        return L.flo_integrate_divergence(h, y, ts_, n_ts, 999.0, None, probes, n_p, d, b, None)

    for kw, what in [(dict(n_p=0), "probe"), (dict(n_p=65535), "probe"), (dict(n_ts=1), "time points"), (dict(b=0), "batch"), (dict(), "NULL"),
                     (dict(h=p, y=None), "NULL"), (dict(h=p, ts_=None), "NULL"), (dict(h=p, probes=None), "NULL"),
                     (dict(h=p, d=None), "NULL")]:
        assert integ(**kw) == _lib.FLO_ERR_INVALID and what in L.flo_last_error().decode(), kw

    def jvp(x=p, t=p, dx=p, n_p=1, v=p, dv=p, b=1, h=None):
        return L.flo_unet_jvp(h, x, t, None, dx, n_p, v, dv, b, None)

    for kw, what in [(dict(n_p=0), "tangent"), (dict(n_p=65535), "tangent"), (dict(b=0), "batch"), (dict(), "NULL"), (dict(h=p, x=None), "NULL"),
                     (dict(h=p, dx=None), "NULL"), (dict(h=p, v=None), "NULL"), (dict(h=p, dv=None), "NULL")]:
        assert jvp(**kw) == _lib.FLO_ERR_INVALID and what in L.flo_last_error().decode(), kw
    with pytest.raises(ValueError, match="NULL"):
        _lib.check(jvp(), "flo_unet_jvp")
