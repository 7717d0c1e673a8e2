"""invert_latents without a GPU: the generic composition for foreign models against a hand loop of ``rk4_step`` over the
reversed grid and against ``solve_ivp`` on ``(1, t0)`` called directly, argument errors before anything runs, and the
argument checks of the reverse C exports."""
import ctypes
from functools import partial

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
        if cond and cond.get("mask_cond") is not None:
            v = v * cond["mask_cond"]
        return v


SHAPE = (3, 4, 5, 6)


def data(seed=1):
    return torch.randn(SHAPE, generator=torch.Generator().manual_seed(seed))


def conds():
    mask = torch.rand(SHAPE, generator=torch.Generator().manual_seed(9))
    return {"plain": (None, 0.0), "cfg": ({"class_cond": torch.tensor([0, 3, 4])}, 3.0),
            "mask": ({"mask_cond": mask}, 0.0)}


def direct(model, y0, t0, t1, cond=None, cfg=0.0, rtol=1e-5, atol=1e-5):
    """solve_ivp on y0.ravel() with the velocity the samplers feed it: fl32(t) * 999 as the time, CFG on the host."""
    shape = tuple(y0.shape)

    def fun(t, yf):
        x = torch.from_numpy(yf).float().reshape(shape)
        tv = torch.ones(shape[0]) * t * 999
        v = model(x, tv, cond=cond)
        if cfg and cond and cond.get("class_cond") is not None:
            v_nc = model(x, tv, cond={**cond, "class_cond": None})
            v = v_nc + cfg * (v - v_nc)
        return v.detach().double().numpy().ravel()
    return solve_ivp(fun, (t0, t1), y0.double().numpy().ravel(), method="RK45", rtol=rtol, atol=atol)


def as_f32(sol):
    return sol.y[:, -1].astype(np.float32).astype(np.float64)


@pytest.mark.parametrize("init_strength", [0.0, 0.3])
@pytest.mark.parametrize("case", list(conds()))
def test_foreign_rk4_is_a_hand_loop_over_the_reversed_grid(case, init_strength):
    m = Toy(n_classes=5)
    cond, cfg = conds()[case]
    y = data()
    with torch.no_grad():
        got, nfe = sampling.invert_latents(m, y, n_steps=9, cond=cond, cfg_strength=cfg, init_strength=init_strength)
        n = 9 if init_strength == 0 else max(1, int(9 * (1 - init_strength)))
        ts = sampling.warp_time(torch.linspace(init_strength, 1.0, n)).flip(0)
        assert float(ts[0]) == 1.0 and ts[-1] == sampling.warp_time(torch.tensor(init_strength))
        t_vec = torch.zeros(SHAPE[0])
        f = partial(sampling.v_func_cfg, m, cond, cfg, t_vec)
        want = y
        for i in range(len(ts) - 1):
            want = sampling.rk4_step(f, want, ts[i], ts[i + 1] - ts[i])
    assert torch.equal(got, want)
    assert nfe == 4 * (n - 1)


def test_rk4_grid_at_zero_strength_is_the_sampling_grid():
    """invert_latents' grid at init_strength 0 is generate_latents_rk4's, so a generate -> invert round trip retraces it."""
    for n in (1, 2, 7, 50, 200):
        ts, k = sampling._rk4_grid(n, 0.0)
        assert k == n and torch.equal(ts, sampling.time_grid(n))
        assert torch.equal(sampling._rk4_grid(n)[0], ts)


@pytest.mark.parametrize("init_strength", [0.0, 0.3])
@pytest.mark.parametrize("case", list(conds()))
def test_foreign_rk45_is_solve_ivp_backwards(case, init_strength):
    m = Toy(n_classes=5)
    cond, cfg = conds()[case]
    y = data(2)
    t0 = float(sampling.warp_time(torch.tensor(init_strength)))
    with torch.no_grad():
        got, nfe = sampling.invert_latents(m, y, cond=cond, cfg_strength=cfg, method="rk45", init_strength=init_strength)
        sol = direct(m, y, 1.0, t0, cond, cfg)
    assert sol.success and sol.t[-1] == t0 and nfe == sol.nfev and (nfe - 2) % 6 == 0
    assert np.array_equal(got.double().numpy().ravel(), as_f32(sol))


@pytest.mark.parametrize("case", list(conds()))
def test_foreign_rk45_per_sample_is_solve_ivp_on_each_sample(case):
    m = Toy(n_classes=5)
    cond, cfg = conds()[case]
    y = data(3) * torch.tensor([0.5, 1.0, 1.5])[:, None, None, None]
    with torch.no_grad():
        got, nfe = sampling.invert_latents(m, y, cond=cond, cfg_strength=cfg, method="rk45", per_sample=True)
        assert nfe.dtype == torch.int64 and nfe.shape == (SHAPE[0],)
        for i in range(SHAPE[0]):
            sol = direct(m, y[i:i + 1], 1.0, 0.0, sampling._sample_cond(cond, i), cfg)
            assert sol.success and int(nfe[i]) == sol.nfev
            assert np.array_equal(got[i:i + 1].double().numpy().ravel(), as_f32(sol))


def test_round_trip_on_a_foreign_model_shrinks_with_n_steps():
    m = Toy()
    x0 = data(4)
    errs = []
    with torch.no_grad():
        for n in (10, 40):
            x1, _ = sampling.generate_latents_rk4(m, SHAPE, n_steps=n, source=x0)
            back, _ = sampling.invert_latents(m, x1, n_steps=n)
            errs.append(float((back - x0).norm() / x0.norm()))
    assert errs[1] < errs[0] < 1e-2


@pytest.mark.parametrize("kwargs", [dict(rtol=0.0), dict(rtol=-1e-5), dict(atol=-1e-9), dict(max_steps=0),
                                    dict(max_steps=2.5), dict(init_strength=1.0), dict(init_strength=-0.1),
                                    dict(method="euler"), dict(n_steps=0), dict(n_steps=2.5)])
@pytest.mark.parametrize("method", ["rk4", "rk45"])
def test_argument_errors_raise_before_anything_runs(kwargs, method):
    if method == "rk45" and "n_steps" in kwargs:
        pytest.skip("n_steps is ignored by RK45")
    m = Toy()
    with pytest.raises(ValueError):
        sampling.invert_latents(m, data(), **{"method": method, **kwargs})
    assert m.calls == 0


def test_rk45_ignores_n_steps():
    m = Toy()
    y = data(5)
    with torch.no_grad():
        want, nfe = sampling.invert_latents(m, y, method="rk45")
        for n in (None, 10 ** 12):
            got, nfe2 = sampling.invert_latents(m, y, n_steps=n, method="rk45")
            assert torch.equal(got, want) and nfe2 == nfe


def test_max_steps_is_a_runtime_error():
    m = Toy()
    with pytest.raises(RuntimeError, match="max_steps"):
        sampling.invert_latents(m, data(), method="rk45", rtol=1e-9, atol=1e-9, max_steps=2)


@pytest.mark.parametrize("export", ["flo_integrate_rk45_reverse", "flo_integrate_rk45_per_sample_reverse"])
@pytest.mark.parametrize("args, what", [
    ((1.0, 0.0, 0.0, 1e-5), "rtol"), ((1.0, 0.0, -1e-5, 1e-5), "rtol"), ((1.0, 0.0, 1e-5, -1.0), "atol"),
    ((1.0, 1.0, 1e-5, 1e-5), "t1 < t0"), ((0.2, 0.5, 1e-5, 1e-5), "t1 < t0"), ((1.0, float("nan"), 1e-5, 1e-5), "t1 < t0"),
    ((float("nan"), 0.0, 1e-5, 1e-5), "t1 < t0"), ((float("inf"), 0.0, 1e-5, 1e-5), "t1 < t0")])
def test_reverse_c_abi_argument_checks_need_no_device(export, args, what):
    from flocoder_b200 import _lib
    L = _lib.lib()
    fn = getattr(L, export)
    counts = (ctypes.c_int * 3)()
    t0, t1, rtol, atol = args
    rc = fn(None, None, t0, t1, rtol, atol, 999.0, None, 0.0, 100, counts, 1, None)
    assert rc == _lib.FLO_ERR_INVALID and what in L.flo_last_error().decode()
    with pytest.raises(ValueError, match=what.split()[0]):
        _lib.check(rc, export)
    rc = fn(None, None, 1.0, 0.0, 1e-5, 1e-5, 999.0, None, 0.0, 0, counts, 1, None)
    assert rc == _lib.FLO_ERR_INVALID and "max_steps" in L.flo_last_error().decode()
    with pytest.raises(ValueError, match="max_steps"):
        _lib.check(rc, export)
    rc = fn(None, None, 1.0, 0.0, 1e-5, 1e-5, 999.0, None, 0.0, 100, counts, 1, None)
    assert rc == _lib.FLO_ERR_INVALID and "NULL" in L.flo_last_error().decode()


def test_forward_c_exports_still_refuse_a_descending_interval():
    from flocoder_b200 import _lib
    L = _lib.lib()
    counts = (ctypes.c_int * 3)()
    for fn in (L.flo_integrate_rk45, L.flo_integrate_rk45_per_sample):
        rc = fn(None, None, 1.0, 0.0, 1e-5, 1e-5, 999.0, None, 0.0, 100, counts, 1, None)
        assert rc == _lib.FLO_ERR_INVALID and "need finite t0 < t1" in L.flo_last_error().decode()
