"""Unet.jvp and log_likelihood on the device (fp32 path) against the fp64 oracle.

* Unet.jvp: v and every dv[p] within the forward's 1e-5 rel-L2 of torch.func.jvp through the fp64 oracle, over configs that
  reach every nonlinear JVP kernel shape (class conditioning, 3 latent channels, dim 8 = 2 channels per group, two levels,
  non-square latents).
* Exact trace: with the D basis vectors as probes (scaled by sqrt(D) for log_likelihood), the diagonal of the device
  Jacobian and log_likelihood's divergence match the oracle's full Jacobian.
* End to end: log_likelihood's divergence against the generic composition on the fp64 OracleModel, and its noise against
  invert_latents.
* A sample's result does not depend on its batch and repeats bit for bit; the unsupported models are refused up front."""
import math

import pytest
import torch

from oracle.unet_oracle import OracleModel, UnetSpec, trained_like, unet_forward
from conftest import rel_l2

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5

# name: (dim, dim_mults, channels, n_classes, H, W)
JVP_CONFIGS = {
    "flowers_sd": (16, (1, 2, 4, 8), 4, 102, 16, 16),
    "midi_vqgan": (16, (1, 2, 4, 8), 4, 0, 16, 16),
    "rgb_latent": (16, (1, 2, 4, 8), 3, 0, 16, 16),
    "dim8": (8, (1, 2, 4, 8), 4, 0, 16, 16),
    "two_level": (16, (1, 2), 4, 0, 8, 8),
    "non_square": (16, (1, 2, 4, 8), 4, 0, 8, 16),
}
_models = {}


def model_for(name, compute_dtype="fp32", mask_cond=False):
    """(cuda Unet with trained-like weights, fp64 state dict, oracle spec, latent shape)."""
    from flocoder_b200.unet import Unet
    key = (name, compute_dtype, mask_cond)
    if key not in _models:
        dim, mults, ch, ncls, h, w = JVP_CONFIGS[name]
        torch.manual_seed(1234)
        m = Unet(dim=dim, channels=ch, dim_mults=list(mults), n_classes=ncls, mask_cond=mask_cond, compute_dtype=compute_dtype)
        sd = trained_like({k: v.detach().clone() for k, v in m.state_dict().items()})
        m.load_state_dict(sd)
        spec = UnetSpec(dim=dim, dim_mults=mults, channels=ch, groups=4, n_classes=ncls)
        _models[key] = (m.cuda().eval(), {k: v.double() for k, v in sd.items()}, spec, (ch, h, w))
    return _models[key]


def randn(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def rademacher(shape, seed):
    return torch.randint(0, 2, shape, generator=torch.Generator().manual_seed(seed)).float() * 2 - 1


def class_cond(n_classes, b):
    return {"class_cond": torch.arange(b) * 7 % n_classes} if n_classes else None


def on_cuda(cond):
    return None if cond is None else {k: v.cuda() for k, v in cond.items()}


@pytest.mark.parametrize("n_tan", [1, 3])
@pytest.mark.parametrize("name", list(JVP_CONFIGS))
def test_jvp_matches_forward_mode_through_the_fp64_oracle(name, n_tan):
    m, sd, spec, shape = model_for(name)
    b = 5
    x, dx = randn((b,) + shape, 1), randn((n_tan, b) + shape, 2)
    t = torch.linspace(0.1, 0.9, b, dtype=torch.float64) * 999
    cond = class_cond(spec.n_classes, b)
    tangents = dx[0] if n_tan == 1 else dx
    v, dv = m.jvp(x.cuda(), t.float().cuda(), tangents.cuda(), cond=on_cuda(cond))
    assert dv.shape == tangents.shape
    dv = dv.reshape((n_tan, b) + shape)
    f = lambda xx: unet_forward(sd, spec, xx, t, cond)      # noqa: E731
    for p in range(n_tan):
        want_v, want_dv = torch.func.jvp(f, (x.double(),), (dx[p].double(),))
        assert rel_l2(v, want_v) < FP32_TOL
        assert rel_l2(dv[p], want_dv) < FP32_TOL, (name, p, rel_l2(dv[p], want_dv))


def oracle_trace(sd, spec, x, t):
    """v and the exact trace of dv/dx per sample (fp64 Jacobian)."""
    v = unet_forward(sd, spec, x, t, None)
    tr = torch.zeros(x.shape[0], dtype=torch.float64)
    for i in range(x.shape[0]):
        jac = torch.autograd.functional.jacobian(lambda xx: unet_forward(sd, spec, xx, t[i:i + 1], None), x[i:i + 1])
        tr[i] = jac.reshape(x[0].numel(), x[0].numel()).diagonal().sum()
    return v, tr


def log_normal(z):
    z = z.double().flatten(1).cpu()
    return -0.5 * (z * z).sum(1) - 0.5 * z.shape[1] * math.log(2 * math.pi)


def test_basis_probes_give_the_exact_trace():
    from flocoder_b200 import sampling
    m, sd, spec, shape = model_for("two_level")
    b, d = 2, math.prod(shape)
    x = randn((b,) + shape, 3)
    basis = torch.eye(d).reshape((d, 1) + shape).expand((d, b) + shape).contiguous()
    t = torch.tensor([300.0, 700.0], dtype=torch.float64)
    _, dv = m.jvp(x.cuda(), t.float().cuda(), basis.cuda())
    diag = dv.reshape(d, b, d).diagonal(dim1=0, dim2=2).cpu()            # [b, d]: dv_p[b, p]
    for i in range(b):
        jac = torch.autograd.functional.jacobian(lambda xx: unet_forward(sd, spec, xx, t[i:i + 1], None), x[i:i + 1].double())
        assert rel_l2(diag[i], jac.reshape(d, d).diagonal()) < FP32_TOL

    # sqrt(D) e_p, p < D: E[eps eps^T] = I as for Rademacher probes, and the mean over p is exactly the trace
    logp, noise, nfe = sampling.log_likelihood(m, x.cuda(), n_steps=3, probes=(basis * math.sqrt(d)).cuda())
    assert nfe == 8
    # the oracle: RK4 over the same reversed grid in fp64, trace(jacobian) at every stage
    ts = sampling._rk4_grid(3, 0.0)[0].flip(0).double()
    y, div = x.double(), torch.zeros(b, dtype=torch.float64)
    for i in range(len(ts) - 1):
        t0, dt = ts[i], ts[i + 1] - ts[i]
        f = lambda xx, tt: oracle_trace(sd, spec, xx, torch.full((b,), float(tt) * 999, dtype=torch.float64))   # noqa: E731
        k1, d1 = f(y, t0)
        k2, d2 = f(y + dt * k1 / 2, t0 + dt / 2)
        k3, d3 = f(y + dt * k2 / 2, t0 + dt / 2)
        k4, d4 = f(y + dt * k3, t0 + dt)
        y = y + (dt / 6) * (k1 + 2 * k2 + 2 * k3 + k4)
        div += float(dt) / 6 * (d1 + 2 * d2 + 2 * d3 + d4)
    got = logp.cpu() - log_normal(noise)
    assert float(((got - div).abs() / div.abs()).max()) < FP32_TOL, (got, div)
    assert rel_l2(noise, y) < FP32_TOL


def test_end_to_end_matches_the_generic_composition_on_the_fp64_oracle():
    from flocoder_b200 import sampling
    m, sd, spec, shape = model_for("flowers_sd")
    b = 4
    x = randn((b,) + shape, 4)
    probes = rademacher((2, b) + shape, 5)
    cond = class_cond(spec.n_classes, b)
    logp, noise, nfe = sampling.log_likelihood(m, x.cuda(), n_steps=8, cond=on_cuda(cond), probes=probes.cuda())
    assert logp.dtype == torch.float64 and logp.device.type == "cuda" and nfe == 28
    want, want_noise, want_nfe = sampling.log_likelihood(OracleModel(sd, spec), x.double(), n_steps=8, cond=cond,
                                                         probes=probes.double())
    assert want_nfe == nfe
    got_div, want_div = logp.cpu() - log_normal(noise), want - log_normal(want_noise)
    assert float(((got_div - want_div).abs() / want_div.abs()).max()) < FP32_TOL, (got_div, want_div)
    inv, _ = sampling.invert_latents(m, x.cuda(), n_steps=8, cond=on_cuda(cond), cfg_strength=0.0, method="rk4")
    assert rel_l2(noise, inv) < 1e-6


def test_a_sample_does_not_depend_on_its_batch_and_repeats_exactly():
    from flocoder_b200 import sampling
    m, sd, spec, shape = model_for("flowers_sd")
    x = randn((7,) + shape, 6).cuda()
    probes = rademacher((2, 7) + shape, 7).cuda()
    cond = on_cuda(class_cond(spec.n_classes, 7))
    logp, noise, _ = sampling.log_likelihood(m, x, n_steps=6, cond=cond, probes=probes)
    one = {"class_cond": cond["class_cond"][3:4]}
    logp1, noise1, _ = sampling.log_likelihood(m, x[3:4], n_steps=6, cond=one, probes=probes[:, 3:4].contiguous())
    assert abs(float(logp[3] - logp1[0])) <= 1e-6 * abs(float(logp1[0]))
    assert rel_l2(noise[3:4], noise1) < 1e-6
    again, noise2, _ = sampling.log_likelihood(m, x, n_steps=6, cond=cond, probes=probes)
    assert torch.equal(logp, again) and torch.equal(noise, noise2)


@pytest.mark.parametrize("case", ["bf16", "fp16", "mask_cond", "32x32"])
def test_unsupported_models_are_refused_before_any_launch(case):
    from flocoder_b200 import sampling
    from flocoder_b200.unet import Unet
    shape = (4, 32, 32) if case == "32x32" else (4, 16, 16)
    if case == "mask_cond":
        m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True).cuda().eval()
    else:
        m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0,
                 compute_dtype=case if case in ("bf16", "fp16") else "fp32").cuda().eval()
    x = randn((2,) + shape, 8).cuda()
    t = torch.full((2,), 500.0, device="cuda")
    with pytest.raises(NotImplementedError):
        m.jvp(x, t, x)
    with pytest.raises(NotImplementedError):
        sampling.log_likelihood(m, x, n_steps=3)
    # the C entry points refuse the same handles before they allocate or launch anything
    eng = m.engine(shape[1], shape[2])
    n0 = eng.launch_count()
    with pytest.raises(NotImplementedError):
        eng.jvp(x, t, None, x[None].contiguous())
    with pytest.raises(NotImplementedError):
        eng.integrate_divergence(x.clone(), [1.0, 0.0], x[None].contiguous())
    assert eng.launch_count() == n0
