"""RK45 sampling without a GPU: the legacy composition for foreign models (scipy's ``solve_ivp`` on the host) against
``solve_ivp`` called directly, argument errors before anything runs, and the C ABI's argument checks."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.integrate import solve_ivp

from flocoder_b200 import sampling


class Toy(torch.nn.Module):
    """A foreign velocity model: anything callable as ``model(x, time, cond=None)`` with parameters."""

    def __init__(self, n_classes=0):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self.w = torch.nn.Parameter(torch.randn(4, 4, generator=g) * 0.5)
        self.emb = torch.nn.Parameter(torch.randn(max(n_classes, 1), 4, generator=g))
        self.calls = 0

    def forward(self, x, time, cond=None):
        self.calls += 1
        v = torch.einsum("oc,bchw->bohw", self.w, torch.tanh(x)) + torch.sin(time / 999 * 3)[:, None, None, None]
        if cond and cond.get("class_cond") is not None:
            v = v + self.emb[cond["class_cond"]][:, :, None, None]
        return v


SHAPE = (3, 4, 5, 6)


def direct(model, y0, t0, cond=None, cfg=0.0, rtol=1e-5, atol=1e-5):
    def fun(t, yf):
        x = torch.from_numpy(yf).float().reshape(SHAPE)
        tv = torch.ones(SHAPE[0]) * t * 999
        v = model(x, tv, cond=cond)
        if cfg and cond and cond.get("class_cond") is not None:
            v_nc = model(x, tv, cond={**cond, "class_cond": None})
            v = v_nc + cfg * (v - v_nc)
        return v.detach().double().numpy().ravel()
    return solve_ivp(fun, (t0, 1.0), y0.double().numpy().ravel(), method="RK45", rtol=rtol, atol=atol)


@pytest.mark.parametrize("case", ["plain", "cfg", "init"])
def test_foreign_model_is_solve_ivp(case):
    m = Toy(n_classes=5)
    y0 = torch.randn(SHAPE, generator=torch.Generator().manual_seed(1))
    cond, cfg, init, t0 = None, 3.0, None, 0.0
    if case == "cfg":
        cond = {"class_cond": torch.tensor([0, 3, 4])}
    if case == "init":
        init = torch.randn(SHAPE, generator=torch.Generator().manual_seed(2))
        t0 = float(sampling.warp_time(torch.tensor(0.3)))
    with torch.no_grad():
        got, nfe = sampling.generate_latents(m, SHAPE, method="rk45", n_steps=7, cond=cond, cfg_strength=cfg, source=y0,
                                             init_latents=init, init_strength=0.3)
        start = y0 if init is None else (1 - 0.3) * y0 + 0.3 * init
        sol = direct(m, start, t0, cond, cfg)
    assert sol.success and nfe == sol.nfev and (nfe - 2) % 6 == 0
    assert np.array_equal(got.double().numpy().ravel(), sol.y[:, -1].astype(np.float32).astype(np.float64))
    assert 0.0 < t0 < 1.0 if init is not None else t0 == 0.0


def test_tolerances_are_passed_through():
    m = Toy()
    y0 = torch.randn(SHAPE, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        _, loose = sampling.generate_latents_rk45(m, SHAPE, source=y0, rtol=1e-3, atol=1e-3)
        _, tight = sampling.generate_latents_rk45(m, SHAPE, source=y0, rtol=1e-7, atol=1e-7)
        assert loose == direct(m, y0, 0.0, rtol=1e-3, atol=1e-3).nfev
    assert tight > loose


@pytest.mark.parametrize("kwargs", [dict(rtol=0.0), dict(rtol=-1e-5), dict(atol=-1e-9), dict(max_steps=0), dict(max_steps=2.5),
                                    dict(init_latents=torch.zeros(SHAPE), init_strength=1.0)])
def test_argument_errors_raise_before_anything_runs(kwargs):
    m = Toy()
    with pytest.raises(ValueError):
        sampling.generate_latents_rk45(m, SHAPE, **kwargs)
    assert m.calls == 0


def test_max_steps_is_a_runtime_error():
    m = Toy()
    with pytest.raises(RuntimeError, match="max_steps"):
        sampling.generate_latents_rk45(m, SHAPE, source=torch.randn(SHAPE), rtol=1e-9, atol=1e-9, max_steps=2)


def test_sharded_sampler_does_not_offer_rk45():
    from flocoder_b200 import dist
    with pytest.raises(ValueError, match="RK45"):
        dist.generate_latents_sharded(Toy(), SHAPE, sampler=sampling.generate_latents_rk45, source=torch.randn(SHAPE))


@pytest.mark.parametrize("args, what", [
    ((0.0, 1.0, 0.0, 1e-5), "rtol"), ((0.0, 1.0, 1e-5, -1.0), "atol"), ((1.0, 1.0, 1e-5, 1e-5), "t0"),
    ((0.5, 0.2, 1e-5, 1e-5), "t0"), ((0.0, float("nan"), 1e-5, 1e-5), "t0")])
def test_c_abi_argument_checks_need_no_device(args, what):
    from flocoder_b200 import _lib
    L = _lib.lib()
    counts = (ctypes.c_int * 3)()
    t0, t1, rtol, atol = args
    rc = L.flo_integrate_rk45(None, None, t0, t1, rtol, atol, 999.0, None, 0.0, 100, counts, 1, None)
    assert rc == _lib.FLO_ERR_INVALID and what in L.flo_last_error().decode()
    rc = L.flo_integrate_rk45(None, None, 0.0, 1.0, 1e-5, 1e-5, 999.0, None, 0.0, 0, counts, 1, None)
    assert rc == _lib.FLO_ERR_INVALID and "max_steps" in L.flo_last_error().decode()
    rc = L.flo_integrate_rk45(None, None, 0.0, 1.0, 1e-5, 1e-5, 999.0, None, 0.0, 100, counts, 1, None)
    assert rc == _lib.FLO_ERR_INVALID and "NULL" in L.flo_last_error().decode()
