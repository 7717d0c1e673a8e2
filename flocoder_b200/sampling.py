"""Drop-in for the integrator half of ``flocoder/sampling.py`` (lines 23-146).

Same function names, argument order, defaults and return values as the reference:
``warp_time``, ``rk4_step``, ``v_func_cfg``, ``generate_latents_rk4``, ``generate_latents``
(+ the legacy ``euler_sampler``, ``legacy/train_sd_flowers.py:50-67``, and ``generate_latents_rk45``, the adaptive
Dormand-Prince sampler the reference's ``method='rk45'`` dispatch names, with scipy's ``solve_ivp`` semantics).

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

import random
from functools import partial

import torch

from . import _lib
from .unet import Unet

__all__ = ["warp_time", "rk4_step", "v_func_cfg", "generate_latents_rk4", "generate_latents_rk45", "generate_latents",
           "euler_sampler", "time_grid", "g2rgb", "decode_latents", "sampler"]


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
        ts = torch.linspace(0, 1, n_steps, device="cpu", dtype=torch.float32)
        jitter_strength = 0
    else:
        y = (1 - init_strength) * y + init_strength * init_latents
        n_steps = max(1, int(n_steps * (1.0 - init_strength)))
        ts = torch.linspace(init_strength, 1.0, n_steps, device="cpu", dtype=torch.float32)
    ts = warp_time(ts)
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


@torch.no_grad()
def generate_latents_rk45(model, shape, cond=None, cfg_strength=3.0, source=None, init_latents=None, init_strength=0.0,
                          rtol=1e-5, atol=1e-5, max_steps=10000):
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

    For a :class:`~flocoder_b200.unet.Unet` the integration runs on the device (``flo_integrate_rk45``: stage inputs,
    error norm and step-size control are kernels; the host waits once per attempt of six evaluations).  Any other
    callable keeps the legacy composition: ``solve_ivp`` on the host, calling the model once per stage.  A step size
    below scipy's minimum step, or more than ``max_steps`` attempts, raises RuntimeError."""
    if not rtol > 0:
        raise ValueError(f"rtol must be > 0, got {rtol}")
    if not atol >= 0:
        raise ValueError(f"atol must be >= 0, got {atol}")
    if int(max_steps) != max_steps or max_steps < 1:
        raise ValueError(f"max_steps must be a positive integer, got {max_steps}")
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
        import numpy as np
        from scipy.integrate import solve_ivp
        t_vec = torch.zeros(y.shape[0], device=y.device, dtype=y.dtype)
        calls = [0]

        def fun(t, yf):
            calls[0] += 1
            if calls[0] > 2 + 6 * max_steps:
                raise RuntimeError(f"RK45 used max_steps={max_steps} attempts and stopped at t={t}")
            x = torch.from_numpy(np.ascontiguousarray(yf)).to(device=y.device, dtype=y.dtype).reshape(y.shape)
            return v_func_cfg(model, cond, cfg_strength, t_vec, x, t).double().cpu().numpy().ravel()

        sol = solve_ivp(fun, (t0, 1.0), y.double().cpu().numpy().ravel(), method="RK45", rtol=rtol, atol=atol)
        if sol.status != 0:
            raise RuntimeError(f"RK45 failed at t={sol.t[-1]}: {sol.message}")
        out = torch.from_numpy(sol.y[:, -1]).reshape(y.shape).to(device=y.device, dtype=y.dtype)
        return out, int(sol.nfev)

    b, c, h, w = y.shape
    eng = model.engine(h, w)
    out_dtype = y.dtype
    state = y.to(device=eng.device, dtype=torch.float32).contiguous()
    if state.data_ptr() == y.data_ptr():
        state = state.clone()                      # never integrate in place on the caller's tensor
    cls = _class_ids(model, cond)
    cfg = float(cfg_strength) if (cls is not None and cfg_strength) else 0.0
    eng.set_mask(model.mask_of(cond), b)
    nfe, _, _ = eng.integrate_rk45(state, t0, 1.0, rtol=rtol, atol=atol, class_ids=cls, cfg_strength=cfg,
                                   max_steps=int(max_steps))
    return state.to(out_dtype), nfe


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
