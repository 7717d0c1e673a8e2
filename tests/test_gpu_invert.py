"""invert_latents on the device: reverse RK4 over the descending grid (``flo_integrate``) and reverse RK45
(``flo_integrate_rk45_reverse`` / ``flo_integrate_rk45_per_sample_reverse``) against the fp64 oracle run backwards, the
16-bit and layer-wise paths against the fp32 path's inversion, the generate -> invert round trip, and handle state.

* fp32 path: reverse RK4-50 within rel-L2 1e-5 + 4 e32 of the fp64 oracle's RK4 over the same reversed grid, e32 being the
  distance of the same oracle run with fp32 weights; reverse RK45 against scipy's RK45 on (1, t0) driving the fp64 oracle,
  with the count rule of test_gpu_rk45.py (counts claimed where every error norm is clear of 1) and the same bar, where
  4 e32 becomes the larger of it and the oracle's own RK45 error at the tolerance (check_rk45_vs_oracle says why).
* 16-bit paths: within BF16_FINAL_TOL of the fp32 path's inversion of the same latents, and bit-identical on repeat.
* round trip: generate with RK4, invert with RK4 over the same grid; the distance to the starting noise falls with n_steps."""
import os

import pytest
import torch

import oracle
from oracle.sampling_oracle import time_grid
from oracle.unet_oracle import OracleModel
from conftest import CONFIGS, GOLDEN_DIR, rel_l2
from rk45_oracle import rk45_solve
from test_gpu_rk45 import BF16_FINAL_TOL, FP32_TOL, NORM_MARGIN, cuda_model, noise, spec_for, state_dict

pytestmark = pytest.mark.gpu

# rel-L2 of generate(RK4-n) -> invert(RK4-n) to the starting noise on the fp32 path (flowers_sd, trained-like weights,
# B = 8), about three times the values measured
# (1.34e-6 and 3.58e-7 on an NVIDIA B200 at its 1000 W power limit): see test_round_trip_error_falls_with_n_steps
ROUND_TRIP_BOUND = {50: 4e-6, 200: 1e-6}


def inpaint_model(compute_dtype="fp32", layerwise=False):
    from flocoder_b200 import _lib
    from flocoder_b200.unet import Unet
    g = torch.load(os.path.join(GOLDEN_DIR, "inpaint_16.pt"), weights_only=False)
    torch.manual_seed(g["model_seed"])
    m = Unet(dim=g["dim"], channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True, compute_dtype=compute_dtype)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    if layerwise:
        m.engine_flags = _lib.FLO_FLAG_LAYERWISE
    return m.cuda().eval(), sd, spec_for(0, g["dim"])


def soft_mask(b):
    ramp = torch.linspace(-3, 3, 16)
    return torch.sigmoid(ramp[None, None, :, None] + ramp[None, None, None, :] * 0.5).expand(b, 4, 16, 16).contiguous()


def on_cuda(cond):
    return None if cond is None else {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in cond.items()}


def oracle_invert_rk4(sd, spec, y, n_steps, dtype, cond=None, cfg=0.0, init_strength=0.0):
    """The oracle's RK4 (sampling.py:37-76) over the fp32 warped grid of generate_latents_rk4 with init_strength,
    traversed from 1 down to warp_time(init_strength), in ``dtype``."""
    model = OracleModel({k: v.to(dtype) for k, v in sd.items()}, spec)
    if init_strength:
        ts = time_grid(max(1, int(n_steps * (1.0 - init_strength))), init_strength=init_strength)
    else:
        ts = time_grid(n_steps)
    ts = ts.flip(0).to(dtype)
    t_vec = torch.zeros(y.shape[0], dtype=dtype)
    c = None if cond is None else {k: (v.to(dtype) if torch.is_floating_point(v) else v) for k, v in cond.items()}
    y = y.to(dtype)
    with torch.no_grad():
        for i in range(len(ts) - 1):
            y = oracle.rk4_step(lambda x, t: oracle.v_func_cfg(model, c, cfg, t_vec, x, t), y, ts[i], ts[i + 1] - ts[i])
    return y


# ---------------------------------------------------------------------------------------------------------------------
# fp32 path against the fp64 oracle run backwards
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["plain", "cfg", "mask"])
def test_fp32_reverse_rk4_matches_the_fp64_oracle(case):
    from flocoder_b200 import sampling
    b, cond, cfg = 4, None, 0.0
    if case == "mask":
        m, sd, spec = inpaint_model()
        cond = {"mask_cond": soft_mask(b)}
    else:
        m, sd, spec = cuda_model(102, "fp32"), state_dict(102, True), spec_for(102)
        if case == "cfg":
            cond, cfg = {"class_cond": torch.tensor([0, 7, 101, 55])}, 3.0
    y = noise(b, 60)
    want = oracle_invert_rk4(sd, spec, y, 50, torch.float64, cond, cfg)
    e32 = rel_l2(oracle_invert_rk4(sd, spec, y, 50, torch.float32, cond, cfg), want)
    got, nfe = sampling.invert_latents(m, y.cuda(), n_steps=50, cond=on_cuda(cond), cfg_strength=cfg)
    e = rel_l2(got, want)
    print(f"{case}: reverse RK4-50 rel-L2 {e:.2e} (fp32 oracle {e32:.2e})")
    assert nfe == 4 * 49
    assert e <= FP32_TOL + 4 * e32


def check_rk45_vs_oracle(m, sd, spec, y, t0, init_strength=0.0, cond=None, cfg=0.0, tol=1e-5):
    """Reverse RK45 of the public function against scipy's RK45 on (1, t0) over the fp64 oracle.  Returns (robust, rejected).

    The bar is 1e-5 + max(4 e32, g).  g is the oracle's own RK45 error at this tolerance: its distance from the fp64 oracle's
    RK4-200 inversion over the same interval (which is ~1e-5 from the exact flow where RK4-50 is ~2e-3).  The device's fp32
    velocities are up to 1e-5 off per forward, the CPU fp32 oracle's 1e-7, and the error norms are differences of seven
    velocities, so on some nets the device takes the oracle's accept / reject decisions with step sizes a little apart, and
    lands elsewhere within the solution's own error.  Measured on a B200: stl_sd with equal counts 1.8e-4 from the oracle
    (e32 2.9e-6, g 7.7e-4; the device's RK4-50 inversion of the same inputs is 2.0e-7 from the oracle's), the inpainting net
    1.6e-3 (g 6.3e-3)."""
    from flocoder_b200 import sampling
    rk4_64 = oracle_invert_rk4(sd, spec, y, 200, torch.float64, cond, cfg, init_strength)
    want, nfev, accepted, norms = rk45_solve(OracleModel({k: v.double() for k, v in sd.items()}, spec), y.double(), 1.0,
                                             t0, cond=cond, cfg_strength=cfg, rtol=tol, atol=tol)
    g = rel_l2(want, rk4_64)
    y32, nfev32, _, norms32 = rk45_solve(OracleModel({k: v.float() for k, v in sd.items()}, spec), y.float(), 1.0, t0,
                                         cond=cond, cfg_strength=cfg, rtol=tol, atol=tol)
    e32 = rel_l2(y32, want)
    robust = nfev32 == nfev and len(norms32) == len(norms) and all(
        abs(a - 1.0) >= max(NORM_MARGIN, 10 * abs(a - b)) for a, b in zip(norms, norms32))
    got, nfe = sampling.invert_latents(m, y.cuda(), cond=on_cuda(cond), cfg_strength=cfg, method="rk45",
                                       init_strength=init_strength, rtol=tol, atol=tol)
    attempts = m.engine(16, 16).rk45_timing()[0]
    e = rel_l2(got, want)
    print(f"nfe {nfe} / {attempts} attempts (oracle {nfev} / {len(norms)}, fp32 oracle {nfev32}), counts claimed: {robust}, "
          f"final rel-L2 {e:.2e} (fp32 oracle {e32:.2e}, oracle RK45 vs RK4-200 {g:.2e})")
    if robust:
        assert (nfe, attempts) == (nfev, len(norms))
    assert e <= FP32_TOL + max(4 * e32, g)
    return robust, len(norms) - accepted


@pytest.mark.parametrize("name", list(CONFIGS))
def test_fp32_reverse_rk45_matches_scipy_on_the_fp64_oracle(name):
    n_classes = CONFIGS[name]
    m = cuda_model(n_classes, "fp32")
    robust, _ = check_rk45_vs_oracle(m, state_dict(n_classes, True), spec_for(n_classes), noise(4, 61 + n_classes), 0.0)
    if name == "flowers_sd":
        assert robust, "flowers_sd is where equal counts are claimed"


def test_fp32_reverse_rk45_with_cfg_partway_and_with_a_mask():
    from flocoder_b200 import sampling
    m = cuda_model(102, "fp32")
    s = 0.3
    t0 = float(sampling.warp_time(torch.tensor(s)))
    check_rk45_vs_oracle(m, state_dict(102, True), spec_for(102), noise(4, 62), t0, init_strength=s,
                         cond={"class_cond": torch.tensor([3, 9, 0, 77])}, cfg=3.0)
    mi, sd, spec = inpaint_model()
    check_rk45_vs_oracle(mi, sd, spec, noise(4, 63), 0.0, cond={"mask_cond": soft_mask(4)})


def test_fp32_reverse_rk45_per_sample_matches_scipy_on_each_sample():
    from flocoder_b200 import sampling
    sd, spec = state_dict(102, True), spec_for(102)
    m = cuda_model(102, "fp32")
    y = noise(3, 64) * torch.tensor([0.5, 1.0, 1.5])[:, None, None, None]
    got, nfe = sampling.invert_latents(m, y.cuda(), method="rk45", per_sample=True)
    assert nfe.dtype == torch.int64 and nfe.shape == (3,)
    m64 = OracleModel({k: v.double() for k, v in sd.items()}, spec)
    m32 = OracleModel({k: v.float() for k, v in sd.items()}, spec)
    claimed = 0
    for i in range(3):
        want, nfev, _, norms = rk45_solve(m64, y[i:i + 1].double(), 1.0, 0.0)
        y32, nfev32, _, norms32 = rk45_solve(m32, y[i:i + 1].float(), 1.0, 0.0)
        robust = nfev32 == nfev and len(norms32) == len(norms) and all(
            abs(a - 1.0) >= max(NORM_MARGIN, 10 * abs(a - b)) for a, b in zip(norms, norms32))
        e, e32 = rel_l2(got[i], want[0]), rel_l2(y32, want)
        print(f"sample {i}: nfe {int(nfe[i])} (oracle {nfev}), counts claimed: {robust}, rel-L2 {e:.2e} (fp32 oracle {e32:.2e})")
        if robust:
            assert int(nfe[i]) == nfev
            claimed += 1
        assert e <= FP32_TOL + 4 * e32
    assert claimed > 0


@pytest.mark.parametrize("compute_dtype", ["fp32", "fp16"])
def test_b1_reverse_per_sample_equals_batched(compute_dtype):
    from flocoder_b200 import sampling
    m = cuda_model(102, compute_dtype)
    y = noise(1, 65).cuda()
    want, nfe = sampling.invert_latents(m, y, method="rk45")
    attempts = m.engine(16, 16).rk45_timing()[0]
    got, nfe_ps = sampling.invert_latents(m, y, method="rk45", per_sample=True)
    assert torch.equal(got, want)
    assert int(nfe_ps[0]) == nfe and m.engine(16, 16).rk45_timing()[0] == attempts


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit paths against the fp32 path's inversion
# ---------------------------------------------------------------------------------------------------------------------
_fp32_cache = {}


def invert(m, b, seed, method, cls=None, cfg=0.0):
    from flocoder_b200 import sampling
    cond = None if cls is None else {"class_cond": cls.cuda()}
    return sampling.invert_latents(m, noise(b, seed).cuda(), cond=cond, cfg_strength=cfg, method=method)


def check16(m, b, seed, method, cls=None, cfg=0.0, what=""):
    key = (b, seed, method, cls is not None, cfg)
    if key not in _fp32_cache:
        _fp32_cache[key] = invert(cuda_model(102, "fp32"), b, seed, method, cls, cfg)
    want, nfe32 = _fp32_cache[key]
    got, nfe = invert(m, b, seed, method, cls, cfg)
    e = rel_l2(got, want)
    print(f"{what} {method}: nfe {nfe} (fp32 path {nfe32}), rel-L2 {e:.2e}")
    assert e <= BF16_FINAL_TOL
    again, nfe2 = invert(m, b, seed, method, cls, cfg)
    assert nfe2 == nfe and torch.equal(again, got)


@pytest.mark.parametrize("method", ["rk4", "rk45"])
@pytest.mark.parametrize("B", [37, 256])
@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_inversion_vs_fp32_path(compute_dtype, B, method):
    check16(cuda_model(102, compute_dtype), B, 70 + B, method, what=f"{compute_dtype} B={B}")


@pytest.mark.parametrize("method", ["rk4", "rk45"])
@pytest.mark.parametrize("two_pass", [False, True])
def test_fused_inversion_cfg_routes(two_pass, method, monkeypatch):
    """B=150 with guidance 3: one 300-sample forward per evaluation (SF_CFG_2B), or the two-pass route (FLO_CFG_TWO_PASS)."""
    if two_pass:
        monkeypatch.setenv("FLO_CFG_TWO_PASS", "1")
    B = 150
    check16(cuda_model(102, "bf16"), B, 71, method, torch.arange(B) % 102, 3.0, what=f"bf16 cfg two_pass={two_pass}")


@pytest.mark.parametrize("method", ["rk4", "rk45"])
def test_layerwise_inversion_vs_fp32_path(method):
    from flocoder_b200 import _lib
    check16(cuda_model(102, "bf16", flags=_lib.FLO_FLAG_LAYERWISE), 37, 72, method, what="bf16 layer-wise B=37")


@pytest.mark.parametrize("per_sample", [False, True])
def test_layerwise_inpainting_inversion_vs_fp32_path(per_sample):
    from flocoder_b200 import sampling
    m, _, _ = inpaint_model("bf16", layerwise=True)
    ref, _, _ = inpaint_model("fp32")
    b = 37
    y = noise(b, 73).cuda()
    cond = {"mask_cond": soft_mask(b).cuda()}
    for method in ("rk4", "rk45"):
        kw = dict(cond=cond, method=method, per_sample=per_sample, rtol=1e-4, atol=1e-4)
        got, _ = sampling.invert_latents(m, y, **kw)
        want, _ = sampling.invert_latents(ref, y, **kw)
        e = rel_l2(got, want)
        print(f"bf16 layer-wise inpainting {method} per_sample={per_sample}: rel-L2 {e:.2e}")
        assert e <= BF16_FINAL_TOL
        again, _ = sampling.invert_latents(m, y, **kw)
        assert torch.equal(again, got)


# ---------------------------------------------------------------------------------------------------------------------
# round trip and handle state
# ---------------------------------------------------------------------------------------------------------------------
def test_round_trip_error_falls_with_n_steps():
    from flocoder_b200 import sampling
    m = cuda_model(102, "fp32")
    x0 = noise(8, 74).cuda()
    errs = {}
    for n in (50, 200):
        x1, _ = sampling.generate_latents_rk4(m, tuple(x0.shape), n_steps=n, source=x0)
        back, nfe = sampling.invert_latents(m, x1, n_steps=n)
        assert nfe == 4 * (n - 1)
        errs[n] = rel_l2(back, x0)
        print(f"round trip RK4-{n}: rel-L2 to the starting noise {errs[n]:.3e} (data rel-L2 {rel_l2(x1, x0):.3e})")
    assert errs[200] < errs[50]
    for n, bound in ROUND_TRIP_BOUND.items():
        assert errs[n] <= bound, f"RK4-{n} round trip {errs[n]:.3e} > {bound}"


@pytest.mark.parametrize("compute_dtype, cfg", [("bf16", 0.0), ("fp16", 3.0), ("fp32", 3.0)])
def test_forward_runs_after_reverse_runs_are_unchanged(compute_dtype, cfg):
    """reverse RK4 -> reverse RK45 -> reverse per-sample RK45, then forward RK45 (batched, per-sample) and RK4 on one
    handle: every forward run equals the same run on a fresh handle."""
    from flocoder_b200 import sampling
    B = 37
    cond = {"class_cond": (torch.arange(B) % 102).cuda()} if cfg else None
    x0 = noise(B, 75).cuda()
    kw = dict(cond=cond, cfg_strength=cfg, source=x0, rtol=1e-3, atol=1e-3)

    def forward_runs(m):
        return (sampling.generate_latents_rk45(m, (B, 4, 16, 16), **kw),
                sampling.generate_latents_rk45(m, (B, 4, 16, 16), per_sample=True, **kw),
                sampling.generate_latents_rk4(m, (B, 4, 16, 16), n_steps=6, cond=cond, cfg_strength=cfg, source=x0))

    fresh = forward_runs(cuda_model(102, compute_dtype))
    m = cuda_model(102, compute_dtype)
    inv = dict(cond=cond, cfg_strength=cfg, rtol=1e-3, atol=1e-3)
    sampling.invert_latents(m, x0, n_steps=6, **inv)
    sampling.invert_latents(m, x0, method="rk45", **inv)
    sampling.invert_latents(m, x0, method="rk45", per_sample=True, **inv)
    after = forward_runs(m)
    assert torch.equal(after[0][0], fresh[0][0]) and after[0][1] == fresh[0][1]
    assert torch.equal(after[1][0], fresh[1][0]) and torch.equal(after[1][1], fresh[1][1])
    assert torch.equal(after[2][0], fresh[2][0])
