"""RK45 on the device (``flo_integrate_rk45``) against scipy's RK45 driving the fp64 oracle, and the 16-bit paths against
the fp32 path.

* fp32 path: ``nfe`` and attempts equal to the oracle's where that can be claimed (below), final latents within rel-L2 1e-5 + 4 e32, where e32 is the
  distance from fp64 of the same oracle run with fp32 weights and velocities (the fp32 floor of the problem).
  Equal counts are claimed only where the problem allows it: every fp64 error norm is at least
  max(1e-3, 10 |n64 - n32|) away from 1, n32 being the fp32 oracle's norm of the same attempt, and both oracles agree on
  the counts.  On CPU the fp32 oracle moves some late norms by tens of percent at rtol 1e-5 on the midi_vqgan / stl_sd
  nets (0.845 -> 0.794), so there the step sequence is set by fp32 rounding and only the floor-relative bar applies;
  flowers_sd (norms move <= 1e-2) must meet the strict form.
* fused fp16 / bf16 (and the layer-wise flag): final latents within BF16_FINAL_TOL of the fp32 path's RK45 on the same
  inputs, bit-identical across runs, and an RK4 trajectory after an RK45 run on the same handle is bit-identical to the
  same trajectory on a fresh handle."""
import os

import pytest
import torch

from oracle.unet_oracle import OracleModel, UnetSpec, trained_like
from conftest import CONFIGS, GOLDEN_DIR, rel_l2, seeded_state_dict
from rk45_oracle import rk45_solve

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_FINAL_TOL = 1e-2          # final-latent bar of the 16-bit operand paths (BASELINE.json north_star)
NORM_MARGIN = 1e-3


def spec_for(n_classes, dim=16):
    return UnetSpec(dim=dim, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=n_classes)


_sd = {}


def state_dict(n_classes, trained):
    key = (n_classes, trained)
    if key not in _sd:
        sd = seeded_state_dict(n_classes)[1]
        _sd[key] = trained_like(sd) if trained else sd
    return _sd[key]


def cuda_model(n_classes, compute_dtype, trained=True, flags=0):
    from flocoder_b200.unet import Unet
    m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes, compute_dtype=compute_dtype)
    m.load_state_dict(state_dict(n_classes, trained))
    m.engine_flags = flags
    return m.cuda().eval()


def noise(b, seed):
    return torch.randn(b, 4, 16, 16, generator=torch.Generator().manual_seed(seed))


def check_vs_oracle(m, sd, spec, x0, t0, tol, cond=None, cfg=0.0, init=None, init_strength=0.0):
    """Returns (rejected attempts of the oracle, whether counts were claimed)."""
    from flocoder_b200 import sampling
    y0 = x0.double() if init is None else (1 - init_strength) * x0.double() + init_strength * init.double()
    want, nfev, accepted, norms = rk45_solve(OracleModel({k: v.double() for k, v in sd.items()}, spec), y0, t0, 1.0,
                                             cond=cond, cfg_strength=cfg, rtol=tol, atol=tol)
    y32, nfev32, _, norms32 = rk45_solve(OracleModel({k: v.float() for k, v in sd.items()}, spec), y0.float(), t0, 1.0,
                                         cond=cond, cfg_strength=cfg, rtol=tol, atol=tol)
    e32 = rel_l2(y32, want)
    robust = nfev32 == nfev and len(norms32) == len(norms) and all(
        abs(a - 1.0) >= max(NORM_MARGIN, 10 * abs(a - b)) for a, b in zip(norms, norms32))
    cond_d = None if cond is None else {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in cond.items()}
    got, nfe = sampling.generate_latents_rk45(m, tuple(x0.shape), cond=cond_d, cfg_strength=cfg, source=x0.cuda(),
                                              init_latents=None if init is None else init.cuda(),
                                              init_strength=init_strength, rtol=tol, atol=tol)
    eng = m.engine(16, 16)
    attempts = eng.rk45_timing()[0]
    rejected = len(norms) - accepted
    e = rel_l2(got, want)
    print(f"nfe {nfe} / {attempts} attempts (oracle {nfev} / {len(norms)}, fp32 oracle {nfev32}), counts claimed: {robust}, "
          f"final rel-L2 {e:.2e} (fp32 oracle {e32:.2e})")
    if robust:
        assert (nfe, attempts) == (nfev, len(norms)), f"device nfe {nfe} / {attempts} attempts, oracle {nfev} / {len(norms)}"
    assert e <= FP32_TOL + 4 * e32, f"final latents rel-L2 {e:.2e}, fp32 floor {e32:.2e}"
    return rejected, robust


# ---------------------------------------------------------------------------------------------------------------------
# fp32 path against scipy + the fp64 oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tol", [1e-5, 1e-3])
@pytest.mark.parametrize("trained", [False, True])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_fp32_rk45_matches_scipy_on_the_fp64_oracle(name, trained, tol):
    n_classes = CONFIGS[name]
    b = 4 + n_classes % 5                         # 6, 4, 4
    m = cuda_model(n_classes, "fp32", trained)
    rejected, robust = check_vs_oracle(m, state_dict(n_classes, trained), spec_for(n_classes), noise(b, b), 0.0, tol)
    if name == "flowers_sd":
        assert robust, "the flowers_sd cases are where equal counts are claimed"
        if tol == 1e-5:
            assert rejected > 0, "the tight-tolerance flowers_sd cases contain rejected attempts (the oracle shows 3)"


def test_fp32_rk45_class_conditioning_with_cfg():
    m = cuda_model(10, "fp32")
    cls = torch.tensor([0, 3, 9, 5, 1])
    check_vs_oracle(m, state_dict(10, True), spec_for(10), noise(5, 11), 0.0, 1e-5, cond={"class_cond": cls}, cfg=3.0)


def test_fp32_rk45_from_init_latents():
    from flocoder_b200 import sampling
    m = cuda_model(0, "fp32")
    t0 = float(sampling.warp_time(torch.tensor(0.3)))
    check_vs_oracle(m, state_dict(0, True), spec_for(0), noise(6, 12), t0, 1e-5, init=noise(6, 13), init_strength=0.3)


def test_fp32_rk45_inpainting_with_a_soft_mask():
    from flocoder_b200.unet import Unet
    g = torch.load(os.path.join(GOLDEN_DIR, "inpaint_16.pt"), weights_only=False)
    torch.manual_seed(g["model_seed"])
    m = Unet(dim=g["dim"], channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True, compute_dtype="fp32")
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.cuda().eval()
    b = 4
    ramp = torch.linspace(-3, 3, 16)
    mask = torch.sigmoid(ramp[None, None, :, None] + ramp[None, None, None, :] * 0.5).expand(b, 4, 16, 16).contiguous()
    check_vs_oracle(m, sd, spec_for(0, g["dim"]), noise(b, 14), 0.0, 1e-5, cond={"mask_cond": mask})


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit paths against the fp32 path
# ---------------------------------------------------------------------------------------------------------------------
_fp32_cache = {}


def fp32_rk45(b, seed, cls=None, cfg=0.0):
    from flocoder_b200 import sampling
    key = (b, seed, cls is not None, cfg)
    if key not in _fp32_cache:
        m = cuda_model(102, "fp32")
        cond = None if cls is None else {"class_cond": cls.cuda()}
        _fp32_cache[key] = sampling.generate_latents_rk45(m, (b, 4, 16, 16), cond=cond, cfg_strength=cfg,
                                                          source=noise(b, seed).cuda())
    return _fp32_cache[key]


def run16(m, b, seed, cls=None, cfg=0.0):
    from flocoder_b200 import sampling
    cond = None if cls is None else {"class_cond": cls.cuda()}
    return sampling.generate_latents_rk45(m, (b, 4, 16, 16), cond=cond, cfg_strength=cfg, source=noise(b, seed).cuda())


@pytest.mark.parametrize("B", [37, 300, 600])
@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_rk45_vs_fp32_path(compute_dtype, B):
    m = cuda_model(102, compute_dtype)
    got, nfe = run16(m, B, B)
    want, nfe32 = fp32_rk45(B, B)
    e = rel_l2(got, want)
    print(f"{compute_dtype} B={B}: nfe {nfe} (fp32 path {nfe32}), final rel-L2 {e:.2e}")
    assert e <= BF16_FINAL_TOL
    again, nfe2 = run16(m, B, B)
    assert nfe2 == nfe and torch.equal(again, got)


@pytest.mark.parametrize("two_pass", [False, True])
@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_rk45_cfg_routes(compute_dtype, two_pass, monkeypatch):
    """B=150: guidance as one 300-sample forward (SF_CFG_2B), or the conditional + combining two-pass route the planner takes
    when the last stage is N-split (forced here with FLO_CFG_TWO_PASS)."""
    B = 150
    if two_pass:
        monkeypatch.setenv("FLO_CFG_TWO_PASS", "1")
    m = cuda_model(102, compute_dtype)
    cls = torch.arange(B) % 102
    got, nfe = run16(m, B, 21, cls, 3.0)
    want, nfe32 = fp32_rk45(B, 21, cls, 3.0)
    e = rel_l2(got, want)
    print(f"{compute_dtype} cfg B={B} two_pass={two_pass}: nfe {nfe} (fp32 path {nfe32}), final rel-L2 {e:.2e}")
    assert e <= BF16_FINAL_TOL
    again, nfe2 = run16(m, B, 21, cls, 3.0)
    assert nfe2 == nfe and torch.equal(again, got)


def test_layerwise_rk45_vs_fp32_path():
    from flocoder_b200 import _lib
    m = cuda_model(102, "bf16", flags=_lib.FLO_FLAG_LAYERWISE)
    got, nfe = run16(m, 37, 37)
    want, nfe32 = fp32_rk45(37, 37)
    e = rel_l2(got, want)
    print(f"bf16 layer-wise B=37: nfe {nfe} (fp32 path {nfe32}), final rel-L2 {e:.2e}")
    assert e <= BF16_FINAL_TOL
    again, _ = run16(m, 37, 37)
    assert torch.equal(again, got)


@pytest.mark.parametrize("compute_dtype, cfg", [("bf16", 0.0), ("fp16", 3.0), ("fp32", 3.0)])
def test_rk4_after_rk45_on_one_handle_is_unchanged(compute_dtype, cfg):
    from flocoder_b200 import sampling
    B = 37
    cls = (torch.arange(B) % 102).cuda() if cfg else None
    cond = None if cls is None else {"class_cond": cls}
    x0 = noise(B, 5).cuda()
    fresh = cuda_model(102, compute_dtype)
    want, _ = sampling.generate_latents_rk4(fresh, (B, 4, 16, 16), n_steps=6, cond=cond, cfg_strength=cfg, source=x0)
    m = cuda_model(102, compute_dtype)
    sampling.generate_latents_rk45(m, (B, 4, 16, 16), cond=cond, cfg_strength=cfg, source=x0, rtol=1e-3, atol=1e-3)
    got, _ = sampling.generate_latents_rk4(m, (B, 4, 16, 16), n_steps=6, cond=cond, cfg_strength=cfg, source=x0)
    assert torch.equal(got, want)
