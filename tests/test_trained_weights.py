"""``oracle.trained_like``: the weights the GPU tests in test_gpu_trained_weights.py use, and why they are needed.

Default init sets every GroupNorm to gamma = 1, beta = 0 and gives nearly uniform attention softmaxes, so a kernel that
drops beta, reads gamma at the wrong channel or pairs values with the wrong pixel computes (almost) the default-init
numbers.  These CPU tests pin that the transform reaches every tensor it should, that the bug models above move their
own stage tensor far above the fp16 format floor with trained-like weights (and the GroupNorm ones not at all with
default weights), and that the format floors the GPU tolerances rest on stay where they are."""
import pytest
import torch

from oracle import ref_shim, unet_oracle
from oracle.unet_oracle import FP32, FUSED_BF16, FUSED_FP16, UnetSpec, trained_like, unet_forward
from conftest import CONFIGS, rel_l2, seeded_state_dict

AFFINE = (".norm.weight", ".norm.bias", ".to_out.1.weight", ".to_out.1.bias")


def spec_for(n_classes):
    return UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=n_classes)


def inputs(b, n_classes, seed):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(b, 4, 16, 16, generator=gen)
    t = torch.rand(b, generator=gen) * 999
    cond = {"class_cond": torch.randint(0, n_classes, (b,), generator=gen)} if n_classes else None
    return x, t, cond


def f64(sd):
    return {k: v.double() for k, v in sd.items()}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_transform_reaches_every_groupnorm_and_qkv(name):
    _, sd = seeded_state_dict(CONFIGS[name])
    tl = trained_like(sd)
    assert list(tl) == list(sd)
    gn = [k for k in sd if k.endswith(AFFINE)]
    qkv = [k for k in sd if k.endswith(".to_qkv.weight")]
    assert len(gn) == 110 and len(qkv) == 9
    for k in gn:
        assert torch.equal(sd[k], torch.ones_like(sd[k]) if k.endswith(".weight") else torch.zeros_like(sd[k])), k
        assert not (tl[k] == 1).any() and not (tl[k] == 0).any(), k
    spread = torch.cat([tl[k] - (1 if k.endswith(".weight") else 0) for k in gn])
    assert abs(float(spread.std()) - 0.3) < 0.03 and abs(float(spread.mean())) < 0.03
    for k in qkv:
        assert torch.equal(tl[k], sd[k] * 4.0), k
    for k in sd:
        if k not in gn and k not in qkv:
            assert torch.equal(tl[k], sd[k]), k
    # deterministic, new tensors, the same values for an fp64 copy
    again = trained_like(sd)
    assert all(torch.equal(tl[k], again[k]) for k in sd)
    assert all(tl[k].data_ptr() != sd[k].data_ptr() for k in sd)
    tl64 = trained_like(f64(sd))
    assert all(tl64[k].dtype == torch.float64 and torch.equal(tl64[k], tl[k].double()) for k in sd)
    assert not torch.equal(trained_like(sd, seed=4)[gn[0]], tl[gn[0]])


class _RollV:
    """Precision wrapper that pairs every value with the key of the previous pixel (v rolled by one pixel)."""

    def __init__(self, prec):
        self.prec = prec

    def op(self, t):
        return self.prec.op(t)

    def act(self, t):
        return self.prec.act(t)

    def qkv(self, t):
        q, k, v = self.prec.qkv(t).chunk(3, dim=1)
        return torch.cat((q, k, v.flatten(2).roll(1, dims=-1).view_as(v)), dim=1)


def _roll_v_in(prefix):
    real = unet_oracle.linear_attention

    def linear_attention(sd, p, x, prec):
        return real(sd, p, x, _RollV(prec) if p == prefix + ".fn.fn" else prec)
    return linear_attention


def _gn_bugs(sd):
    """(stage tensor, broken state dict) for the GroupNorm bug models."""
    zero_beta = dict(sd)
    zero_beta["mid_block1.block2.norm.bias"] = torch.zeros_like(sd["mid_block1.block2.norm.bias"])
    roll_gamma = dict(sd)
    w = sd["downs.3.2.fn.norm.weight"]
    roll_gamma["downs.3.2.fn.norm.weight"] = w.roll(w.numel() // 4)
    return {"beta zeroed in mid_block1.block2.norm (2x2)": ("mid_block1", zero_beta),
            "PreNorm gamma of downs.3.2 rolled by C/4": ("downs.3.2", roll_gamma)}


def _trace(sd, spec, x, t, cond, prec=FP32):
    tr = {}
    with torch.no_grad():
        unet_forward(sd, spec, x, t, cond, prec, tr)
    return tr


def test_bug_models_are_visible_with_trained_like_weights_only(monkeypatch):
    """Each bug model moves its own stage tensor by >= 20x the FUSED_FP16 oracle's error there (the floor the per-stage GPU
    comparison sits on) with trained-like weights; with default weights the GroupNorm bugs move nothing."""
    n = 0
    spec = spec_for(n)
    _, sd = seeded_state_dict(n)
    x, t, cond = inputs(8, n, seed=21)
    x64, t64 = x.double(), t.double()
    tl = trained_like(sd)
    clean = _trace(f64(tl), spec, x64, t64, cond)
    floor = _trace(tl, spec, x, t, cond, FUSED_FP16)
    cases = [(what, stage, _trace(f64(bad), spec, x64, t64, cond)) for what, (stage, bad) in _gn_bugs(tl).items()]
    with monkeypatch.context() as mp:
        mp.setattr(unet_oracle, "linear_attention", _roll_v_in("downs.2.2"))
        cases.append(("v rolled by one pixel in downs.2.2", "downs.2.2", _trace(f64(tl), spec, x64, t64, cond)))
    for what, stage, bad in cases:
        e_fmt = rel_l2(floor[stage], clean[stage])
        e_bug = rel_l2(bad[stage], clean[stage])
        print(f"{what:48s} at {stage:12s} bug {e_bug:.3e}  fp16 floor {e_fmt:.3e}")
        assert e_bug >= 20 * e_fmt, (what, e_bug, e_fmt)
    # default init: gamma = 1, beta = 0, so the same GroupNorm bugs leave every tensor bit-identical
    clean = _trace(f64(sd), spec, x64, t64, cond)
    for what, (stage, bad) in _gn_bugs(sd).items():
        bad = _trace(f64(bad), spec, x64, t64, cond)
        assert all(torch.equal(bad[k], clean[k]) for k in clean), what


@pytest.mark.parametrize("name", list(CONFIGS))
def test_format_floors_with_trained_like_weights(name):
    """The velocity error the 16-bit formats themselves cause (emulating oracles vs fp64), which the GPU tolerances scale:
    fp16 stays under the 2e-3 per-step bar with room for the kernels' own rounding, bf16 near 1e-2."""
    n = CONFIGS[name]
    spec = spec_for(n)
    _, sd = seeded_state_dict(n)
    tl = trained_like(sd)
    x, t, cond = inputs(8, n, seed=22)
    with torch.no_grad():
        want = unet_forward(f64(tl), spec, x.double(), t.double(), cond)
        e32 = rel_l2(unet_forward(tl, spec, x, t, cond), want)
        e16 = rel_l2(unet_forward(tl, spec, x, t, cond, FUSED_FP16), want)
        eb16 = rel_l2(unet_forward(tl, spec, x, t, cond, FUSED_BF16), want)
    print(name, "fp32", e32, "fused fp16", e16, "fused bf16", eb16)
    assert e32 <= 5e-6
    assert e16 <= 1.5e-3
    assert eb16 <= 1.2e-2          # 7.5e-3 / 8.0e-3 / 1.1e-2 (stl_sd, class-conditioned); the bf16 GPU tests use a ratio to it


@pytest.mark.skipif(not ref_shim.available(), reason="needs a flocoder reference checkout (oracle/_ref or FLOCODER_REFERENCE)")
@pytest.mark.parametrize("n_classes", [102, 0])
def test_restatement_equals_imported_reference_with_trained_like_weights(n_classes):
    ref_unet, _ = ref_shim.load()
    torch.manual_seed(99)
    ref = ref_unet.Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes).eval()
    sd = trained_like({k: v.detach().clone() for k, v in ref.state_dict().items()})
    ref.load_state_dict(sd)
    x, t, cond = inputs(3, n_classes, seed=23)
    with torch.no_grad():
        assert rel_l2(unet_forward(sd, spec_for(n_classes), x, t, cond), ref(x, t, cond)) < 2e-6
        ref64 = ref.double()
        got = unet_forward(f64(sd), spec_for(n_classes), x.double(), t.double(), cond)
        assert rel_l2(got, ref64(x.double(), t.double(), cond)) < 1e-12
