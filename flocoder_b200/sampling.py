"""Drop-in for the integrator half of ``flocoder/sampling.py`` (lines 23-146).

Same function names, argument order, defaults and return values as the reference:
``warp_time``, ``rk4_step``, ``v_func_cfg``, ``generate_latents_rk4``, ``generate_latents``
(+ the legacy ``euler_sampler``, ``legacy/train_sd_flowers.py:50-67``, and ``generate_latents_rk45``, the adaptive
Dormand-Prince sampler the reference's ``method='rk45'`` dispatch names, with scipy's ``solve_ivp`` semantics), and
``invert_latents``, which runs the same ODE backwards from data latents to noise, and ``log_likelihood``, the model's
density of data latents by the instantaneous change of variables along that inversion.

When ``model`` is a :class:`flocoder_b200.unet.Unet` the whole trajectory runs inside the
C-ABI call ``flo_integrate``: stage times, the four U-Net evaluations per interval, the
classifier-free-guidance combine and the RK4 axpy/state update are all device-side (the RK
combination is the epilogue of the last convolution), with no per-evaluation host sync.  The
reference's per-evaluation ``.item()`` / ``empty_cache()`` / ``synchronize()`` calls
(``sampling.py:60,64-67``) carry no arithmetic and are not reproduced.

For any other callable ``model`` the functions keep the reference's generic semantics
(plain tensor algebra on whatever device the tensors live on) so ``rk4_step`` and
``v_func_cfg`` stay usable as building blocks; that generic composition is reference
behaviour for foreign models, not a fallback for ours.
"""
from __future__ import annotations

import math
import random
from functools import partial

import torch

from . import _lib
from .unet import Unet

__all__ = ["warp_time", "rk4_step", "v_func_cfg", "generate_latents_rk4", "generate_latents_rk45", "generate_latents",
           "invert_latents", "log_likelihood", "euler_sampler", "time_grid", "g2rgb", "decode_latents", "sampler"]


def warp_time(t, dt=None, s=.5):
    """Parametric time warp, ``sampling.py:23-33`` (s=.5 -> 2t^3-3t^2+2t)."""
    if s < 0 or s > 1.5:
        raise ValueError(f"s={s} is out of bounds.")
    tw = 4 * (1 - s) * t ** 3 + 6 * (s - 1) * t ** 2 + (3 - 2 * s) * t
    if dt:   # same operator precedence as the reference's derivative branch (sampling.py:32)
        return tw, dt * 12 * (1 - s) * t ** 2 + 12 * (s - 1) * t + (3 - 2 * s)
    return tw


@torch.no_grad()
def rk4_step(f, y, t, dt, debug=False):
    """One classic RK4 step for an arbitrary velocity function ``f(y, t)`` (``sampling.py:37-48``)."""
    k1 = f(y, t)
    t_mid = t + dt / 2
    k2 = f(y + dt * k1 / 2, t_mid)
    k3 = f(y + dt * k2 / 2, t_mid)
    k4 = f(y + dt * k3, t + dt)
    return y + (dt / 6) * (k1 + 2 * k2 + 2 * k3 + k4)


@torch.no_grad()
def v_func_cfg(model, cond, cfg_strength, t_vec_template, x, t, t_scale=999, debug=False):
    """Velocity with optional classifier-free guidance (``sampling.py:51-76``)."""
    t_vec_template.fill_(float(t))
    t_vec = t_vec_template
    v = model(x, t_vec * t_scale, cond=cond)
    if cond and cond.get("class_cond") is not None and cfg_strength:
        cond_no_class = dict(cond)
        cond_no_class["class_cond"] = None
        v_no_class = model(x, t_vec * t_scale, cond=cond_no_class)
        v = v_no_class + cfg_strength * (v - v_no_class)
    return v


def time_grid(n_steps, start=0.0, device=None, dtype=torch.float32):
    """The grid ``generate_latents_rk4`` integrates over: linspace then ALWAYS ``warp_time``
    (``sampling.py:102,109,111`` -- ``if warp_time:`` tests the function object)."""
    return warp_time(torch.linspace(start, 1.0, n_steps, device=device, dtype=dtype))


def _rk4_grid(n_steps, init_strength=None):
    """``(warped fp32 CPU grid, interval count n_steps)`` of :func:`generate_latents_rk4`: ``linspace(0, 1, n_steps)``, or
    with ``init_latents`` ``linspace(s, 1, max(1, int(n_steps * (1 - s))))`` for ``s = init_strength``
    (``sampling.py:102-111``); :func:`invert_latents` runs the same grid backwards."""
    if init_strength is None:
        ts = torch.linspace(0, 1, n_steps, device="cpu", dtype=torch.float32)
    else:
        n_steps = max(1, int(n_steps * (1.0 - init_strength)))
        ts = torch.linspace(init_strength, 1.0, n_steps, device="cpu", dtype=torch.float32)
    return warp_time(ts), n_steps


def _device_dtype(model):
    p = next(model.parameters())
    return p.device, p.dtype


def _class_ids(model, cond):
    cls = Unet.split_cond(cond)
    if cls is not None and not model.class_condition:
        cls = None
    return cls


@torch.no_grad()
def generate_latents_rk4(model, shape, n_steps=50, cond=None, cfg_strength=3.0, source=None,
                         init_latents=None, init_strength=0.0, jitter_strength=0, debug=False):
    """RK4 sampling over the warped grid (``sampling.py:79-122``).  Returns ``(latents, nfe)``
    with ``nfe = n_steps*4`` exactly as the reference reports it (it over-counts by 4)."""
    device, dtype = _device_dtype(model)
    y = source if source is not None else torch.randn(shape, device=device, dtype=dtype)
    if init_latents is None:
        ts, n_steps = _rk4_grid(n_steps)
        jitter_strength = 0
    else:
        y = (1 - init_strength) * y + init_strength * init_latents
        ts, n_steps = _rk4_grid(n_steps, init_strength)
    nfe = n_steps * 4

    if not isinstance(model, Unet):
        # foreign model: the reference's generic composition (sampling.py:112-119)
        ts_d = ts.to(device=device, dtype=dtype)
        t_vec = torch.zeros(shape[0], device=device, dtype=dtype)
        v_func = partial(v_func_cfg, model, cond, cfg_strength, t_vec)
        for i in range(len(ts_d) - 1):
            y = rk4_step(v_func, y, ts_d[i], ts_d[i + 1] - ts_d[i])
            if random.random() < 0.1 and jitter_strength > 0:
                y += torch.randn_like(y) * jitter_strength * (1 - ts_d[i])
        return y, nfe

    # ---- B200 fast path: the whole trajectory is one C-ABI call ----
    b, c, h, w = y.shape
    eng = model.engine(h, w)
    out_dtype = y.dtype
    state = y.to(device=eng.device, dtype=torch.float32).contiguous()
    if state.data_ptr() == y.data_ptr():
        state = state.clone()                      # never integrate in place on the caller's tensor
    cls = _class_ids(model, cond)
    cfg = float(cfg_strength) if (cls is not None and cfg_strength) else 0.0
    eng.set_mask(model.mask_of(cond), b)           # inpainting: the same mask for every evaluation (sampling.py:63,73)
    grid = ts.tolist()
    if len(grid) >= 2:
        if jitter_strength > 0:
            # stochastic jitter needs a host decision per interval (sampling.py:118-119)
            for i in range(len(grid) - 1):
                eng.integrate(state, grid[i:i + 2], _lib.FLO_RK4, class_ids=cls, cfg_strength=cfg)
                if random.random() < 0.1:
                    state += torch.randn_like(state) * jitter_strength * (1 - grid[i])
        else:
            eng.integrate(state, grid, _lib.FLO_RK4, class_ids=cls, cfg_strength=cfg)
    return state.to(out_dtype), nfe


def _rk45_t0(init_latents, init_strength):
    """First point of the grid :func:`generate_latents_rk4` would use: ``warp_time(0) = 0``, or the fp32
    ``warp_time(init_strength)`` with ``init_latents``."""
    if init_latents is None:
        return 0.0
    return float(warp_time(torch.tensor(float(init_strength), dtype=torch.float32)))


def _solve_ivp_rk45(model, y, cond, cfg_strength, t0, rtol, atol, max_steps, what="", t1=1.0):
    """The legacy composition for a foreign model: ``solve_ivp`` on the host over ``y.ravel()``, one model call per stage,
    from ``t0`` to ``t1`` (either direction).  Returns ``(state at t1, nfev)``; ``what`` names the problem in the errors
    (e.g. ``"sample 3 "``)."""
    import numpy as np
    from scipy.integrate import solve_ivp
    t_vec = torch.zeros(y.shape[0], device=y.device, dtype=y.dtype)
    calls = [0]

    def fun(t, yf):
        calls[0] += 1
        if calls[0] > 2 + 6 * max_steps:
            raise RuntimeError(f"RK45 {what}used max_steps={max_steps} attempts and stopped at t={t}")
        x = torch.from_numpy(np.ascontiguousarray(yf)).to(device=y.device, dtype=y.dtype).reshape(y.shape)
        return v_func_cfg(model, cond, cfg_strength, t_vec, x, t).double().cpu().numpy().ravel()

    sol = solve_ivp(fun, (t0, t1), y.double().cpu().numpy().ravel(), method="RK45", rtol=rtol, atol=atol)
    if sol.status != 0:
        raise RuntimeError(f"RK45 {what}failed at t={sol.t[-1]}: {sol.message}")
    return torch.from_numpy(sol.y[:, -1]).reshape(y.shape).to(device=y.device, dtype=y.dtype), int(sol.nfev)


def _check_rk45_args(rtol, atol, max_steps):
    if not rtol > 0:
        raise ValueError(f"rtol must be > 0, got {rtol}")
    if not atol >= 0:
        raise ValueError(f"atol must be >= 0, got {atol}")
    if int(max_steps) != max_steps or max_steps < 1:
        raise ValueError(f"max_steps must be a positive integer, got {max_steps}")


def _sample_cond(cond, i):
    """``cond`` for sample ``i`` alone: the per-sample tensors (``class_cond``, ``mask_cond``) cut to ``[i:i+1]``."""
    if cond is None:
        return None
    out = dict(cond)
    for key in ("class_cond", "mask_cond"):
        if out.get(key) is not None:
            out[key] = out[key][i:i + 1]
    return out


@torch.no_grad()
def generate_latents_rk45(model, shape, cond=None, cfg_strength=3.0, source=None, init_latents=None, init_strength=0.0,
                          rtol=1e-5, atol=1e-5, max_steps=10000, per_sample=False):
    """Adaptive Dormand-Prince 5(4) from ``t0`` to ``t1 = 1``: ``scipy.integrate.solve_ivp(fun, (t0, 1), y0.ravel(),
    method='RK45', rtol=rtol, atol=atol)`` as the legacy RK45 samplers call it.  Returns ``(latents, nfe)`` with
    ``nfe`` = scipy's ``nfev`` (``2 + 6 * attempts``).

    * ``t0`` is the first point of the warped grid :func:`generate_latents_rk4` would use: 0, or
      ``warp_time(init_strength)`` after the same ``y = (1-s)*noise + s*init_latents`` mix.
    * The model sees ``torch.ones(B) * t * 999`` in fp32 at every stage time ``t``; class conditioning and
      classifier-free guidance follow :func:`v_func_cfg`, the inpainting mask applies to every evaluation.
    * The whole batch is ONE ODE system with one step size, and the error norm is the RMS over all ``B*C*H*W``
      elements, so a sample's trajectory (and the step count) depends on the rest of its batch -- the legacy
      behaviour of calling ``solve_ivp`` on the flattened batch.

    With ``per_sample=True`` every sample is its own problem, ``solve_ivp(fun_i, (t0, 1), y0[i].ravel(), 'RK45')``,
    with its own step size, accept / reject decisions and error norm (the RMS over its ``C*H*W`` elements), so its result
    does not depend on the rest of the batch; ``nfe`` is then a CPU int64 tensor ``[B]`` of each sample's ``nfev``, and
    ``max_steps`` counts each sample's attempts.  Everything else is as above.

    For a :class:`~flocoder_b200.unet.Unet` the integration runs on the device (``flo_integrate_rk45``, or
    ``flo_integrate_rk45_per_sample`` with one controller per sample while the batch shares every evaluation: stage
    inputs, error norms and step-size control are kernels; the host waits once per attempt of six evaluations).  Any
    other callable keeps the legacy composition: ``solve_ivp`` on the host, calling the model once per stage (per sample,
    on ``x[i:i+1]`` with ``cond`` cut to that sample).  A step size below scipy's minimum step, or more than ``max_steps``
    attempts, raises RuntimeError (naming the sample with ``per_sample``)."""
    _check_rk45_args(rtol, atol, max_steps)
    if init_latents is not None and not 0.0 <= init_strength < 1.0:
        raise ValueError(f"init_strength must be in [0, 1) with init_latents (t0 = warp_time(init_strength) < 1), "
                         f"got {init_strength}")
    device, dtype = _device_dtype(model)
    y = source if source is not None else torch.randn(shape, device=device, dtype=dtype)
    if init_latents is not None:
        y = (1 - init_strength) * y + init_strength * init_latents
    t0 = _rk45_t0(init_latents, init_strength)

    if not isinstance(model, Unet):
        # foreign model: the legacy composition -- scipy on the host, one model call per stage
        return _rk45_foreign(model, y, cond, cfg_strength, t0, 1.0, rtol, atol, max_steps, per_sample)

    b, c, h, w = y.shape
    eng = model.engine(h, w)
    out_dtype = y.dtype
    state = y.to(device=eng.device, dtype=torch.float32).contiguous()
    if state.data_ptr() == y.data_ptr():
        state = state.clone()                      # never integrate in place on the caller's tensor
    cls = _class_ids(model, cond)
    cfg = float(cfg_strength) if (cls is not None and cfg_strength) else 0.0
    eng.set_mask(model.mask_of(cond), b)
    if per_sample:
        counts = eng.integrate_rk45_per_sample(state, t0, 1.0, rtol=rtol, atol=atol, class_ids=cls, cfg_strength=cfg,
                                               max_steps=int(max_steps))
        return state.to(out_dtype), counts[:, 0].clone()
    nfe, _, _ = eng.integrate_rk45(state, t0, 1.0, rtol=rtol, atol=atol, class_ids=cls, cfg_strength=cfg,
                                   max_steps=int(max_steps))
    return state.to(out_dtype), nfe


def _rk45_foreign(model, y, cond, cfg_strength, t0, t1, rtol, atol, max_steps, per_sample):
    """:func:`_solve_ivp_rk45` on the whole batch, or with ``per_sample`` on every sample alone (``nfe`` a CPU int64 ``[B]``)."""
    if not per_sample:
        return _solve_ivp_rk45(model, y, cond, cfg_strength, t0, rtol, atol, max_steps, t1=t1)
    outs, nfe = [], torch.zeros(y.shape[0], dtype=torch.int64)
    for i in range(y.shape[0]):
        out_i, nfe[i] = _solve_ivp_rk45(model, y[i:i + 1], _sample_cond(cond, i), cfg_strength, t0, rtol, atol,
                                        max_steps, what=f"sample {i} ", t1=t1)
        outs.append(out_i)
    return torch.cat(outs, dim=0) if outs else y.clone(), nfe


@torch.no_grad()
def invert_latents(model, latents, n_steps=50, cond=None, cfg_strength=3.0, method="rk4", init_strength=0.0, rtol=1e-5,
                   atol=1e-5, max_steps=10000, per_sample=False):
    """Integrate data latents back towards noise: the sampling ODE run backwards from ``t = 1`` down to
    ``t0 = warp_time(init_strength)`` (``t0 = 0`` by default, where the sampler draws its noise).  Returns
    ``(state at t0, nfe)``.

    Uses: encode a real latent (e.g. from ``codec.encode``) to the noise that generates it; measure a model's round-trip
    error (generate, invert, compare); or invert partway, to ``t0 > 0``, and integrate forward again from there with other
    conditioning -- the deterministic counterpart of the ``init_latents`` mixing of the forward samplers.

    * ``method="rk4"``: classic RK4 over the grid :func:`generate_latents_rk4` uses with ``init_latents`` and this
      ``init_strength`` (at 0 the plain sampling grid of ``n_steps`` points), traversed from 1 down to ``t0``: negative
      ``dt`` in every step.  ``nfe`` is the true count ``4 * (len(grid) - 1)``, NOT the ``n_steps * 4`` the forward
      sampler reports after the reference.
    * ``method="rk45"``: adaptive Dormand-Prince with scipy's step-size control, ``solve_ivp(fun, (1, t0), y.ravel(),
      method='RK45', rtol=rtol, atol=atol)``; ``nfe`` as :func:`generate_latents_rk45` reports it (an int, or with
      ``per_sample=True`` a CPU int64 ``[B]`` of each sample's own ``solve_ivp`` count).  ``n_steps`` is then ignored.
    * Classifier-free guidance and the inpainting mask (``cond``) apply to every evaluation, as in the forward samplers.

    For a :class:`~flocoder_b200.unet.Unet` the whole inversion runs on the device (``flo_integrate`` over the descending
    grid, ``flo_integrate_rk45_reverse`` / ``flo_integrate_rk45_per_sample_reverse``).  Any other callable gets the
    generic composition: :func:`rk4_step` with negative ``dt``, or ``solve_ivp`` on the host (per sample with
    ``per_sample``).  Argument errors raise ValueError before the model is called."""
    if method not in ("rk4", "rk45"):
        raise ValueError(f"method must be 'rk4' or 'rk45', got {method!r}")
    _check_rk45_args(rtol, atol, max_steps)
    if not 0.0 <= init_strength < 1.0:
        raise ValueError(f"init_strength must be in [0, 1) (t0 = warp_time(init_strength) < 1), got {init_strength}")
    if method == "rk4" and (int(n_steps) != n_steps or n_steps < 1):
        raise ValueError(f"n_steps must be a positive integer, got {n_steps}")
    y = latents
    if method == "rk4":                               # RK45 ignores n_steps
        grid = _rk4_grid(int(n_steps), init_strength)[0].flip(0)     # 1 -> warp_time(init_strength)
    t0 = float(warp_time(torch.tensor(float(init_strength), dtype=torch.float32)))   # generate_latents_rk45's t0

    if not isinstance(model, Unet):
        if method == "rk45":
            return _rk45_foreign(model, y, cond, cfg_strength, 1.0, t0, rtol, atol, max_steps, per_sample)
        device, dtype = _device_dtype(model)
        ts_d = grid.to(device=device, dtype=dtype)
        t_vec = torch.zeros(y.shape[0], device=device, dtype=dtype)
        v_func = partial(v_func_cfg, model, cond, cfg_strength, t_vec)
        for i in range(len(ts_d) - 1):
            y = rk4_step(v_func, y, ts_d[i], ts_d[i + 1] - ts_d[i])
        return y, 4 * (len(grid) - 1)

    b, c, h, w = y.shape
    eng = model.engine(h, w)
    out_dtype = y.dtype
    state = y.to(device=eng.device, dtype=torch.float32).contiguous()
    if state.data_ptr() == y.data_ptr():
        state = state.clone()                      # never integrate in place on the caller's tensor
    cls = _class_ids(model, cond)
    cfg = float(cfg_strength) if (cls is not None and cfg_strength) else 0.0
    eng.set_mask(model.mask_of(cond), b)
    if method == "rk4":
        if len(grid) >= 2:
            eng.integrate(state, grid.tolist(), _lib.FLO_RK4, class_ids=cls, cfg_strength=cfg)
        return state.to(out_dtype), 4 * (len(grid) - 1)
    kw = dict(rtol=rtol, atol=atol, class_ids=cls, cfg_strength=cfg, max_steps=int(max_steps), reverse=True)
    if per_sample:
        counts = eng.integrate_rk45_per_sample(state, 1.0, t0, **kw)
        return state.to(out_dtype), counts[:, 0].clone()
    nfe, _, _ = eng.integrate_rk45(state, 1.0, t0, **kw)
    return state.to(out_dtype), nfe


def _check_likelihood_args(latents, n_steps, n_probes, probes):
    """The probe count ``P`` of :func:`log_likelihood`; ValueError for anything it cannot run."""
    if latents.dim() != 4:
        raise ValueError(f"latents must be [B,C,H,W], got {tuple(latents.shape)}")
    if int(n_steps) != n_steps or n_steps < 2:
        raise ValueError(f"n_steps must be an integer >= 2, got {n_steps}")
    if n_probes is not None and (int(n_probes) != n_probes or n_probes < 1):
        raise ValueError(f"n_probes must be a positive integer, got {n_probes}")
    if probes is None:
        return 1 if n_probes is None else int(n_probes)
    if probes.dim() != 5 or tuple(probes.shape[1:]) != tuple(latents.shape) or probes.shape[0] < 1:
        raise ValueError(f"probes must be [P,{','.join(map(str, latents.shape))}], got {tuple(probes.shape)}")
    if n_probes is not None and int(n_probes) != probes.shape[0]:
        raise ValueError(f"n_probes={n_probes} disagrees with the {probes.shape[0]} probes given")
    return probes.shape[0]


def _divergence_foreign(model, y, grid, cond, probes):
    """The generic composition for any callable: RK4 over ``grid`` (the arithmetic of :func:`rk4_step`) with, at every
    stage, ``d = mean_p probe_p . (J v probe_p)`` from ``torch.func.jvp`` of ``model(x, t * 999, cond)``, accumulated with
    the same RK4 weights in fp64.  Returns ``(state at grid[-1], div)``."""
    device, dtype = _device_dtype(model)
    ts = grid.to(device=device, dtype=dtype)
    t_vec = torch.zeros(y.shape[0], device=device, dtype=dtype)
    div = torch.zeros(y.shape[0], dtype=torch.float64, device=device)
    eps = probes.to(device=device, dtype=dtype)

    def f(x, t):
        t_vec.fill_(float(t))
        fn = lambda xx: model(xx, t_vec * 999, cond=cond)            # noqa: E731
        v, d = None, torch.zeros(y.shape[0], dtype=torch.float64, device=device)
        for e in eps:
            v, jv = torch.func.jvp(fn, (x,), (e,))
            d += (e * jv).double().flatten(1).sum(1)
        return v, d / eps.shape[0]

    for i in range(len(ts) - 1):
        t, dt = ts[i], ts[i + 1] - ts[i]
        k1, d1 = f(y, t)
        t_mid = t + dt / 2
        k2, d2 = f(y + dt * k1 / 2, t_mid)
        k3, d3 = f(y + dt * k2 / 2, t_mid)
        k4, d4 = f(y + dt * k3, t + dt)
        y = y + (dt / 6) * (k1 + 2 * k2 + 2 * k3 + k4)
        div += float(dt) / 6 * (d1 + 2 * d2 + 2 * d3 + d4)
    return y, div


@torch.no_grad()
def log_likelihood(model, latents, n_steps=50, cond=None, n_probes=None, probes=None, generator=None):
    """Log-density ``log p(x)`` of data latents under the flow, in nats, by the instantaneous change of variables
    ``d/dt log p_t(x_t) = -div v(x_t, t)``.  Returns ``(logp, noise, nfe)``.

    * The latents are integrated back to ``noise`` with the RK4 of :func:`invert_latents` (``init_strength = 0``: the
      warped sampling grid of ``n_steps >= 2`` points from 1 down to 0), and ``div v`` is integrated alongside with the same
      RK4 weights, estimated at every stage by Hutchinson's ``mean_p probe_p . (J_x v probe_p)`` with exact Jacobian-vector
      products.
    * ``logp = -|noise|^2 / 2 - (D/2) ln(2 pi) + div`` per sample, ``D = C*H*W`` and ``div`` the integral from 1 to 0 of
      ``div v dt``: fp64 ``[B]`` on ``latents.device``.  Bits per dimension are ``-logp / (D ln 2)``.
    * Probes are fixed over the whole trajectory: ``probes`` ``[P,B,C,H,W]``, or ``n_probes`` (default 1) Rademacher +-1
      draws from ``generator``.  Given both, ``n_probes`` must equal ``P``.  More probes lower the estimator's variance;
      the ``D`` basis vectors scaled by ``sqrt(D)`` give the exact trace.
    * ``cond={'class_cond': ids}`` gives ``log p(x | class)``; there is no guidance.  ``nfe = 4 * (n_steps - 1)`` velocity
      evaluations, each carrying ``P`` Jacobian-vector products.

    For a :class:`~flocoder_b200.unet.Unet` the whole trajectory runs on the device (``flo_integrate_divergence``: the fp32
    path; NotImplementedError for 16-bit models, ``mask_cond`` and more than 256 pixels).  Any other callable gets the
    generic composition with ``torch.func.jvp`` in the model's dtype.  Argument errors raise ValueError before the model is
    called."""
    n_tan = _check_likelihood_args(latents, n_steps, n_probes, probes)
    b, c, h, w = latents.shape
    if probes is None:
        gen_device = generator.device if generator is not None else torch.device("cpu")
        probes = torch.randint(0, 2, (n_tan, b, c, h, w), generator=generator, device=gen_device).mul_(2).sub_(1)
    grid = _rk4_grid(int(n_steps), 0.0)[0].flip(0)                  # invert_latents' grid: 1 -> 0
    nfe = 4 * (len(grid) - 1)
    if not isinstance(model, Unet):
        noise, div = _divergence_foreign(model, latents, grid, cond, probes)
    else:
        model.check_jvp_supported(h, w)
        eng = model.engine(h, w)
        state = latents.to(device=eng.device, dtype=torch.float32).contiguous()
        if state.data_ptr() == latents.data_ptr():
            state = state.clone()                      # never integrate in place on the caller's tensor
        eps = probes.to(device=eng.device, dtype=torch.float32).contiguous()
        div = eng.integrate_divergence(state, grid.tolist(), eps, class_ids=_class_ids(model, cond))
        noise = state.to(latents.dtype)
    z = noise.double().flatten(1)
    d = c * h * w
    logp = -0.5 * (z * z).sum(1) - 0.5 * d * math.log(2 * math.pi) + div.to(z.device)
    return logp.to(latents.device), noise, nfe


@torch.no_grad()
def generate_latents(model, shape, method="rk4", n_steps=50, cond=None, cfg_strength=3.0, device=None,
                     source=None, init_latents=None, init_strength=0.0, debug=False):
    """Dispatch (``sampling.py:128-146``).  ``method='rk45'`` runs :func:`generate_latents_rk45` (the reference's
    branch calls that name, which it no longer defines) with its default tolerances; ``n_steps`` is then ignored."""
    if device is None:
        device = next(model.parameters()).device
    if method == "rk45":
        return generate_latents_rk45(model, shape, cond, cfg_strength, source=source, init_latents=init_latents,
                                     init_strength=init_strength)
    return generate_latents_rk4(model, shape, n_steps, cond, cfg_strength, source=source,
                                init_latents=init_latents, init_strength=init_strength)


@torch.no_grad()
def euler_latents(model, shape, sample_N, cond=None, source=None, eps=1e-3):
    """The legacy Euler recurrence with the result left on the model's device (what :func:`euler_sampler` and the
    sharded / benchmark callers share).  Returns ``(x, nfe=N)``."""
    dev, dtype = _device_dtype(model)
    x = source if source is not None else torch.randn(shape, device=dev, dtype=dtype)
    dt = 1.0 / sample_N
    times = [i / sample_N * (1 - eps) + eps for i in range(sample_N)]
    if not isinstance(model, Unet):
        x = x.detach().clone()
        for num_t in times:
            t = torch.ones(shape[0], device=x.device, dtype=x.dtype) * num_t
            x = x.detach().clone() + model(x, t * 999, cond) * dt
        return x, sample_N
    b, c, h, w = x.shape
    eng = model.engine(h, w)
    out_dtype = x.dtype
    state = x.to(device=eng.device, dtype=torch.float32).contiguous().clone()
    cls = _class_ids(model, cond)
    eng.set_mask(model.mask_of(cond), b)
    # the legacy loop feeds fl32(num_t) (ones*num_t in fp32) and multiplies the velocity by fl32(dt)
    ts32 = torch.tensor(times, dtype=torch.float64).to(torch.float32).tolist()
    eng.integrate(state, ts32, _lib.FLO_EULER_LEGACY, dt=dt, class_ids=cls, cfg_strength=0.0)
    return state.to(out_dtype), sample_N


@torch.no_grad()
def euler_sampler(model, shape, sample_N, device=None, cond=None, source=None, eps=1e-3):
    """Legacy fixed-step Euler (``legacy/train_sd_flowers.py:43,50-67``): ``dt = 1/N``,
    ``t_i = i/N*(1-eps)+eps``, ``x <- x + model(x, t_i*999, cond)*dt``.  Returns ``(x, nfe=N)``.

    ``cond`` and ``source`` are explicit here (the legacy script drew both from globals); like
    the legacy function the result is returned on the CPU."""
    x, nfe = euler_latents(model, shape, sample_N, cond=cond, source=source, eps=eps)
    return x.cpu(), nfe


# --------------------------------------------------------------------------------------------------
# The immediate caller of the path (SURVEY.md section 8(f), N1): sampler() = conditioning set-up +
# generate_latents + chunked decode through a user-supplied codec.  The codec itself (SD-VAE / VQGAN) is out
# of scope: any object with .encode(images) / .decode(latents) / .parameters() works.
# --------------------------------------------------------------------------------------------------
def g2rgb(gf_img, keep_gray=False):
    """Grayscale piano-roll -> quantised RGB (``metrics.py:319-327``): value >= .75 -> red, within .25 of .5 -> green,
    else black; ``keep_gray`` gives a black/white image thresholded at .5.  3-channel input passes through."""
    if gf_img.shape[-3] == 3:
        return gf_img
    g = gf_img.squeeze(-3)
    if keep_gray:
        return (g > 0.5).float().unsqueeze(-3).repeat(1, 3, 1, 1)
    red = (g >= 0.75).float()
    green = ((g - 0.5).abs() < 0.25).float()
    return torch.stack([red, green, torch.zeros_like(g)], dim=-3)


def decode_latents(codec, latents, is_midi=False, keep_gray=False, device=None, chunk_size=128, debug=False):
    """Decode in chunks of ``chunk_size`` (``sampling.py:169-183``): each chunk goes to the codec's device, is decoded,
    optionally mapped through :func:`g2rgb`, parked on the host, and the concatenation returns to ``latents.device``."""
    if device is None:
        try:
            device = next(codec.parameters()).device
        except (StopIteration, AttributeError, TypeError):
            device = latents.device
    out = []
    for i in range(0, latents.shape[0], chunk_size):
        img = codec.decode(latents[i:i + chunk_size].to(device))
        if is_midi:
            img = g2rgb(img, keep_gray=keep_gray)
        out.append(img.cpu())
    return torch.cat(out, dim=0).to(latents.device)


@torch.no_grad()
def sampler(model, codec, method="rk4", batch_size=256, n_steps=100, cond=None, n_classes=0, latent_shape=(4, 16, 16),
            cfg_strength=3.0, is_midi=False, keep_gray=False, device=None, source=None, init_image=None,
            init_strength=0.0, debug=False):
    """``sampling.py:187-229``: returns ``(pred_latents, decoded, nfe)``.

    * ``cond`` is a dict (``None`` is treated as ``{}``; the reference would raise on ``None``).  Without a
      ``class_cond`` and with ``n_classes > 0`` it draws 10 random classes and tiles them ``batch_size // 10`` times
      (one class per grid column, ``sampling.py:217-218``); an existing ``class_cond`` / ``mask_cond`` / ``source`` is
      cut to ``batch_size``.
    * ``init_image`` (a path, a PIL image or a ``[C,H,W]`` / ``[1,C,H,W]`` float tensor in [0,1]) is encoded by the codec
      and repeated over the batch; integration then starts at ``t = init_strength`` (``sampling.py:104-109``).
    """
    if device is None:
        device = next(model.parameters()).device
    codec_device = next(codec.parameters()).device
    assert device == codec_device, f"sampler, device mismatch: device = {device}, but  codec_device {codec_device}"
    cond = {} if cond is None else cond

    init_latents = None
    if init_image is not None:
        if isinstance(init_image, str):
            from PIL import Image
            init_image = Image.open(init_image)
        if not torch.is_tensor(init_image):
            from torchvision.transforms import ToTensor       # what the reference uses (sampling.py:11,208)
            init_image = ToTensor()(init_image)
        img = init_image if init_image.dim() == 4 else init_image.unsqueeze(0)
        init_latents = codec.encode(img.to(device))
        if init_latents.shape[0] == 1 and batch_size > 1:
            init_latents = init_latents.repeat(batch_size, 1, 1, 1)

    shape = (batch_size,) + tuple(latent_shape)
    if source is not None:
        source = source[:batch_size]
    if cond.get("class_cond") is None and n_classes > 0:
        cond["class_cond"] = torch.randint(n_classes, (10,)).repeat(batch_size // 10).to(device)
    elif cond.get("class_cond") is not None:
        cond["class_cond"] = cond["class_cond"][:batch_size]
    if cond.get("mask_cond") is not None:
        cond["mask_cond"] = cond["mask_cond"][:batch_size]

    pred_latents, nfe = generate_latents(model, shape, method, n_steps, cond, cfg_strength, device=device, source=source,
                                         init_latents=init_latents, init_strength=init_strength)
    decoded = decode_latents(codec, pred_latents, is_midi, keep_gray, device=device)
    return pred_latents, decoded, nfe
