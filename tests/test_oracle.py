"""The CPU oracle pinned against the reference: (1) frozen outputs of the unmodified reference
(tests/golden, made by oracle/make_golden.py) and (2), where a reference checkout exists (oracle/_ref or FLOCODER_REFERENCE), the
imported reference itself on fresh inputs, fp32 and fp64."""
import pytest
import torch

import oracle
from oracle import ref_shim
from oracle.unet_oracle import OracleModel, UnetSpec, FP32, BF16_MATCHED, unet_forward
from conftest import CONFIGS, rel_l2, seeded_state_dict

SHAPE = (8, 4, 16, 16)


def spec_for(n_classes):
    return UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=n_classes)


@pytest.mark.parametrize("name", list(CONFIGS))
def test_forward_matches_golden(goldens, name):
    g = goldens[name]
    _, sd = seeded_state_dict(g["n_classes"])
    spec = spec_for(g["n_classes"])
    with torch.no_grad():
        v = unet_forward(sd, spec, g["x0"], g["fwd_t"])
        assert rel_l2(v, g["fwd_v"]) < 2e-6
        v = unet_forward(sd, spec, g["x0"], g["fwd_tvec"])
        assert rel_l2(v, g["fwd_v_tvec"]) < 2e-6
        if g["n_classes"] > 0:
            v = unet_forward(sd, spec, g["x0"], g["fwd_t"], cond={"class_cond": g["cls"]})
            assert rel_l2(v, g["fwd_v_cls"]) < 2e-6


@pytest.mark.parametrize("name", list(CONFIGS))
def test_integrators_match_golden(goldens, name):
    g = goldens[name]
    _, sd = seeded_state_dict(g["n_classes"])
    model = OracleModel(sd, spec_for(g["n_classes"]))
    x1, nfe = oracle.generate_latents_rk4(model, SHAPE, n_steps=10, source=g["x0"].clone())
    assert nfe == g["rk4_10_nfe"] == 40
    assert model.calls == 36                      # 9 intervals x 4 evaluations
    assert rel_l2(x1, g["rk4_10"]) < 2e-6
    x1, nfe = oracle.euler_sampler(model, SHAPE, 10, source=g["x0"])
    assert nfe == 10 and rel_l2(x1, g["euler_10"]) < 2e-6
    x1, nfe = oracle.generate_latents_rk4(model, SHAPE, n_steps=10, source=g["x0"].clone(),
                                          init_latents=g["init_latents"], init_strength=0.3)
    assert nfe == g["rk4_10_init03_nfe"] and rel_l2(x1, g["rk4_10_init03"]) < 2e-6
    if g["n_classes"] > 0:
        x1, _ = oracle.generate_latents_rk4(model, SHAPE, n_steps=10, cond={"class_cond": g["cls"]},
                                            cfg_strength=3.0, source=g["x0"].clone())
        assert rel_l2(x1, g["rk4_10_cfg3"]) < 2e-6
        x1, _ = oracle.generate_latents_rk4(model, SHAPE, n_steps=10, cond={"class_cond": g["cls"]},
                                            cfg_strength=0, source=g["x0"].clone())
        assert rel_l2(x1, g["rk4_10_cls_nocfg"]) < 2e-6


def test_rk4_50_matches_golden(goldens):
    g = goldens["midi_vqgan"]
    _, sd = seeded_state_dict(0)
    model = OracleModel(sd, spec_for(0))
    x1, nfe = oracle.generate_latents(model, SHAPE, method="rk4", n_steps=50, source=g["x0"].clone())
    assert nfe == 200 and model.calls == 196
    assert rel_l2(x1, g["rk4_50"]) < 5e-6


def test_time_grid_and_warp(goldens):
    ts = oracle.warp_time(torch.linspace(0, 1, 50))
    assert torch.equal(ts, goldens["flowers_sd"]["ts_50"])
    assert abs(float(ts[1]) - 0.039584) < 1e-6 and float(ts[-1]) == 1.0
    with pytest.raises(ValueError):
        oracle.warp_time(ts, s=1.6)
    with pytest.raises(ValueError):
        oracle.warp_time(ts, s=-0.1)
    tw, dtw = oracle.warp_time(torch.tensor(0.25), dt=0.1)
    assert abs(float(tw) - (2 * 0.25 ** 3 - 3 * 0.25 ** 2 + 2 * 0.25)) < 1e-7
    # derivative branch keeps the reference's operator precedence (sampling.py:32)
    assert abs(float(dtw) - (0.1 * 12 * 0.5 * 0.0625 + 12 * (-0.5) * 0.25 + 2.0)) < 1e-6
    stages = oracle.rk4_stage_times(ts)
    assert len(stages) == 196
    assert float(stages[-1][0]) == 1.0            # last stage time is exactly 1 (SURVEY appendix A)


def test_rk45_is_an_error():
    _, sd = seeded_state_dict(0)
    with pytest.raises(NameError):
        oracle.generate_latents(OracleModel(sd, spec_for(0)), SHAPE, method="rk45")


def test_bf16_matched_policy_is_close_but_not_equal():
    _, sd = seeded_state_dict(0)
    x = torch.randn(4, 4, 16, 16, generator=torch.Generator().manual_seed(1))
    t = torch.full((4,), 300.0)
    with torch.no_grad():
        a = unet_forward(sd, spec_for(0), x, t, prec=FP32)
        b = unet_forward(sd, spec_for(0), x, t, prec=BF16_MATCHED)
    e = rel_l2(b, a)
    assert 1e-4 < e < 2e-2, e      # SURVEY 8c: ~5e-3 per forward for bf16 GEMM operands


@pytest.mark.skipif(not ref_shim.available(), reason="needs a flocoder reference checkout (oracle/_ref or FLOCODER_REFERENCE)")
@pytest.mark.parametrize("n_classes", [102, 0])
def test_restatement_equals_imported_reference(n_classes):
    ref_unet, ref_sampling = ref_shim.load()
    torch.manual_seed(99)
    ref = ref_unet.Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes).eval()
    sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
    spec = spec_for(n_classes)
    x = torch.randn(3, 4, 16, 16, generator=torch.Generator().manual_seed(7))
    t = torch.tensor([0.0, 417.3, 999.0])
    cond = {"class_cond": torch.tensor([0, 5, 9])} if n_classes else None
    with torch.no_grad():
        assert rel_l2(unet_forward(sd, spec, x, t, cond), ref(x, t, cond)) < 2e-6
        # fp64: the restatement is the same function, not merely close in fp32
        ref64 = ref.double()
        sd64 = {k: v.double() for k, v in sd.items()}
        assert rel_l2(unet_forward(sd64, spec, x.double(), t.double(), cond), ref64(x.double(), t.double(), cond)) < 1e-12
        ref.float()
        x1_ref, nfe_ref = ref_sampling.generate_latents_rk4(ref, (3, 4, 16, 16), n_steps=6, cond=cond,
                                                            cfg_strength=2.0, source=x.clone())
        x1, nfe = oracle.generate_latents_rk4(OracleModel(sd, spec), (3, 4, 16, 16), n_steps=6, cond=cond,
                                              cfg_strength=2.0, source=x.clone())
    assert nfe == nfe_ref and rel_l2(x1, x1_ref) < 2e-6


@pytest.mark.skipif(not ref_shim.available(), reason="needs a flocoder reference checkout (oracle/_ref or FLOCODER_REFERENCE)")
def test_generic_dims_equal_reference():
    """A non-default shape (dim=32, 3 levels, 8 groups, 3 channels) to pin the wiring, not just one config."""
    ref_unet, _ = ref_shim.load()
    torch.manual_seed(5)
    ref = ref_unet.Unet(dim=32, channels=3, dim_mults=[1, 2, 2], resnet_block_groups=8, n_classes=0).eval()
    sd = {k: v.detach().clone() for k, v in ref.state_dict().items()}
    spec = UnetSpec(dim=32, dim_mults=(1, 2, 2), channels=3, groups=8, n_classes=0)
    x = torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(3))
    t = torch.tensor([10.0, 900.0])
    with torch.no_grad():
        assert rel_l2(unet_forward(sd, spec, x, t), ref(x, t)) < 2e-6


# ---- inpainting U-Net (mask_cond=True; SURVEY.md 8f N3): the oracle's mask branches against the frozen reference outputs ----
def inpaint_case(name):
    import os
    from conftest import GOLDEN_DIR
    from flocoder_b200.unet import Unet
    g = torch.load(os.path.join(GOLDEN_DIR, f"{name}.pt"), weights_only=False)
    torch.manual_seed(g["model_seed"])
    m = Unet(dim=g["dim"], channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    return g, sd, UnetSpec(dim=g["dim"], dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=0)


@pytest.mark.parametrize("name", ["inpaint_16", "midi_inpainting"])
def test_inpainting_forward_and_integrators_match_golden(name):
    g, sd, spec = inpaint_case(name)
    shape = tuple(g["x0"].shape)
    cond = {"mask_cond": g["mask_latents"]}
    with torch.no_grad():
        assert rel_l2(unet_forward(sd, spec, g["x0"], g["fwd_t"], cond=cond), g["fwd_v_mask"]) < 2e-6
        assert rel_l2(unet_forward(sd, spec, g["x0"], g["fwd_t"]), g["fwd_v_nomask"]) < 2e-6
        assert rel_l2(unet_forward(sd, spec, g["x0"], g["fwd_t"], cond={"mask_cond": torch.ones(shape)}), g["fwd_v_ones"]) < 2e-6
        assert rel_l2(unet_forward(sd, spec, g["x0"], g["fwd_t"], cond={"mask_cond": g["mask_half"]}), g["fwd_v_half"]) < 2e-6
    model = OracleModel(sd, spec)
    x1, _ = oracle.generate_latents_rk4(model, shape, n_steps=10, cond=cond, source=g["x0"].clone())
    assert rel_l2(x1, g["rk4_10_mask"]) < 2e-6
    x1, _ = oracle.euler_sampler(model, shape, 10, cond=cond, source=g["x0"])
    assert rel_l2(x1, g["euler_10_mask"]) < 2e-6
