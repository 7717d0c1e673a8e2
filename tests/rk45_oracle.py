"""RK45 reference for the tests: ``scipy.integrate``'s RK45 stepped by hand over a velocity model, recording every
attempt's error norm (what decides accept / reject) next to scipy's own counts.

The model is called as the legacy RK45 samplers call it: the flattened batch is one ODE system, the time fed at stage time
``t`` is ``torch.ones(B) * t * 999`` in fp32, and classifier-free guidance is ``v_nc + cfg * (v_c - v_nc)``
(``sampling.py:51-76``).
"""
from __future__ import annotations

import numpy as np
import torch
from scipy.integrate import RK45


class _RecordingRK45(RK45):
    def __init__(self, *args, **kwargs):
        self.error_norms = []
        super().__init__(*args, **kwargs)

    def _estimate_error_norm(self, K, h, scale):
        norm = super()._estimate_error_norm(K, h, scale)
        self.error_norms.append(float(norm))
        return norm


def rk45_solve(model, y0, t0, t1, cond=None, cfg_strength=0.0, rtol=1e-5, atol=1e-5):
    """``solve_ivp(fun, (t0, t1), y0.ravel(), method='RK45', rtol=rtol, atol=atol)`` stepped by hand.

    ``model(x, time, cond=...)`` runs in the dtype of ``y0``.  Returns ``(latents, nfev, accepted, error_norms)``:
    the state at ``t1``, scipy's ``nfev``, the accepted step count and the error norm of every attempt in order
    (rejected attempts = ``len(error_norms) - accepted``)."""
    shape, dtype = tuple(y0.shape), y0.dtype
    b = shape[0]
    use_cfg = bool(cond) and cond.get("class_cond") is not None and bool(cfg_strength)
    cond_nc = None
    if use_cfg:
        cond_nc = dict(cond)
        cond_nc["class_cond"] = None

    def fun(t, yf):
        x = torch.from_numpy(np.ascontiguousarray(yf)).to(dtype).reshape(shape)
        tv = (torch.ones(b, dtype=torch.float32) * t * 999).to(dtype)
        with torch.no_grad():
            v = model(x, tv, cond=cond)
            if use_cfg:
                v_nc = model(x, tv, cond=cond_nc)
                v = v_nc + cfg_strength * (v - v_nc)
        return v.double().numpy().ravel()

    solver = _RecordingRK45(fun, t0, y0.double().numpy().ravel(), t1, rtol=rtol, atol=atol)
    accepted = 0
    while solver.status == "running":
        message = solver.step()
        if solver.status == "failed":
            raise RuntimeError(f"RK45 failed at t={solver.t}: {message}")
        accepted += 1
    y = torch.from_numpy(solver.y.copy()).reshape(shape).to(dtype)
    return y, solver.nfev, accepted, solver.error_norms
