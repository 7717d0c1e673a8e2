"""The CUDA paths with trained-like weights (``oracle.trained_like``: GroupNorm gamma / beta away from 1 / 0, sharp attention
softmaxes) against the oracle in float64.  Default init hides wrong GroupNorm affine reads and wrong key / value pairing
(tests/test_trained_weights.py shows both on the CPU); these tests run every kernel family with weights that expose them.

* fp32 path: <= 1e-5 per forward / per trajectory against fp64.
* fused fp16 / bf16 at the batch sizes that select the planner's variants, on a 16-sample slice: fp16 <= 2e-3 (worst sample
  3.2e-3); bf16 <= 1.15x the error of the bf16-emulating oracle on the same samples + 1e-4.
* per stage tensor: e_cuda <= 1.5 e_fmt + 1e-4, both against the fp64 trace, where e_fmt is the emulating oracle's error.
  A bug in one layer is far above this at its own stage but close to the bf16 floor in the final velocity."""
import pytest
import torch

import oracle
from oracle.unet_oracle import BF16_MATCHED, FP32, FUSED_BF16, FUSED_FP16, OracleModel, UnetSpec, trained_like, unet_forward
from conftest import CONFIGS, rel_l2, seeded_state_dict
from test_gpu_parity import _stage_activations

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
FP16_SLICE_TOL, FP16_SAMPLE_TOL = 2e-3, 3.2e-3


def spec_for(n_classes):
    return UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=n_classes)


def f64(sd):
    return {k: v.double() for k, v in sd.items()}


_weights, _models = {}, {}


def weights(n_classes):
    if n_classes not in _weights:
        _weights[n_classes] = trained_like(seeded_state_dict(n_classes)[1])
    return _weights[n_classes]


def cuda_model(n_classes, compute_dtype, layerwise=False):
    key = (n_classes, compute_dtype, layerwise)
    if key not in _models:
        from flocoder_b200 import _lib
        from flocoder_b200.unet import Unet
        m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes, compute_dtype=compute_dtype)
        m.load_state_dict(weights(n_classes))
        if layerwise:
            m.engine_flags = _lib.FLO_FLAG_LAYERWISE
        _models[key] = m.cuda().eval()
    return _models[key]


def inputs(b, n_classes, seed, channels=4, h=16, w=16):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(b, channels, h, w, generator=gen)
    t = torch.rand(b, generator=gen) * 999
    cls = torch.randint(0, n_classes, (b,), generator=gen) if n_classes else None
    return x, t, cls


def slice_idx(b):
    """First and last samples, ragged last groups, cluster and CTA boundaries: at most 16 samples."""
    return torch.tensor(sorted(i for i in {0, 1, 2, 7, 8, 95, 96, 97, b // 2, b // 2 + 1, b - 9, b - 8, b - 3, b - 2, b - 1, b // 3}
                               if 0 <= i < b))


def per_sample(a, ref):
    a, ref = a.double().cpu(), ref.double().cpu()
    return (a - ref).flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1)


# ---------------------------------------------------------------------------------------------------------------------
# fp32 path against fp64
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CONFIGS))
def test_fp32_forward_vs_fp64(name):
    n = CONFIGS[name]
    m = cuda_model(n, "fp32")
    x, t, cls = inputs(8, n, seed=31)
    conds = [None] + ([{"class_cond": cls}] if n else [])
    for cond in conds:
        with torch.no_grad():
            want = unet_forward(f64(weights(n)), spec_for(n), x.double(), t.double(), cond)
        got = m(x.cuda(), t.cuda(), None if cond is None else {"class_cond": cls.cuda()})
        e = rel_l2(got, want)
        print(name, "class ids" if cond else "no class ids", e)
        assert e <= FP32_TOL


def test_fp32_rk4_cfg_trajectory_vs_fp64():
    from flocoder_b200 import sampling
    n = 102
    m = cuda_model(n, "fp32")
    x, _, cls = inputs(4, n, seed=32)
    shape = tuple(x.shape)
    got, nfe = sampling.generate_latents_rk4(m, shape, n_steps=10, cond={"class_cond": cls.cuda()}, cfg_strength=3.0,
                                             source=x.cuda())
    want, nfe_ref = oracle.generate_latents_rk4(OracleModel(f64(weights(n)), spec_for(n)), shape, n_steps=10,
                                                cond={"class_cond": cls}, cfg_strength=3.0, source=x.double())
    assert nfe == nfe_ref
    e = rel_l2(got, want)
    print("fp32 RK4-10 cfg 3.0 vs fp64:", e)
    assert e <= FP32_TOL


FP32_SHAPES = {
    # name: (dim, channels, dim_mults, groups, latent (h, w), mask_cond)
    "inpaint_dim16": (16, 4, [1, 2, 4, 8], 4, (16, 16), True),
    "inpaint_dim8": (8, 4, [1, 2, 4, 8], 4, (8, 8), True),        # two channels per GroupNorm group (k_gn_any), 1x1 bottleneck
    "rgb_32x32_dim32": (32, 3, [1, 2, 4, 8], 4, (32, 32), False),  # GroupNorm(1, 32) over 32768 elements, tiled linear attention
    "dim64_16x16": (64, 4, [1, 2], 4, (16, 16), False),
    "three_channel_latents": (16, 3, [1, 2, 4, 8], 4, (16, 16), False),
    # groups per sample that are not powers of two: k_gn_any, and k_gn for GroupNorm(1, C) with 3 * 2^k channels
    "dim48_groups6": (48, 4, [1, 2, 4, 8], 6, (16, 16), False),
    "dim24_groups3": (24, 4, [1, 2, 4, 8], 3, (16, 16), False),
    "dim24_groups6": (24, 4, [1, 2, 4, 8], 6, (16, 16), False),     # 4-channel groups, 3 channel blocks per sample
    # planes that are not powers of two: k_gn_any at every level; 48x64 also runs the tiled linear attention at 3072 and
    # 768 pixels (48x48 is refused: linear attention at 24x24 = 576 pixels is neither <= 256 nor whole 256-pixel tiles)
    "12x12_mults124": (16, 4, [1, 2, 4], 4, (12, 12), False),
    "48x64_mults1248": (16, 4, [1, 2, 4, 8], 4, (48, 64), False),
    "16x8": (16, 4, [1, 2, 4, 8], 4, (16, 8), False),
    "8x32": (16, 4, [1, 2, 4, 8], 4, (8, 32), False),
    "mults13": (16, 4, [1, 3], 4, (16, 16), False),                 # 48 channels at the bottleneck: 12 per group
    "one_channel_latents": (16, 1, [1, 2, 4, 8], 4, (16, 16), False),
    "sixteen_channel_latents": (16, 16, [1, 2, 4, 8], 4, (16, 16), False),
}


def assert_plans(dim, channels, mults, groups, hw, compute_dtype, B, flags=0, mask_cond=False):
    """The shape is inside the envelope the planner accepts (tests/test_shape_envelope.py checks its kernels on the host)."""
    from flocoder_b200 import _lib
    _lib.describe_plan(_lib.make_cfg(dim, channels, mults, groups, 0, hw[0], hw[1], compute_dtype, 0, flags, mask_cond), B)


@pytest.mark.parametrize("shape_name", list(FP32_SHAPES))
def test_fp32_other_shapes_vs_fp64(shape_name):
    from flocoder_b200.unet import Unet
    dim, ch, mults, groups, (h, w), mask_cond = FP32_SHAPES[shape_name]
    assert_plans(dim, ch, mults, groups, (h, w), "fp32", 3, mask_cond=mask_cond)
    torch.manual_seed(41)
    m = Unet(dim=dim, channels=ch, dim_mults=mults, resnet_block_groups=groups, n_classes=0, mask_cond=mask_cond,
             compute_dtype="fp32")
    sd = trained_like({k: v.detach().clone() for k, v in m.state_dict().items()})
    m.load_state_dict(sd)
    m = m.cuda().eval()
    spec = UnetSpec(dim=dim, dim_mults=tuple(mults), channels=ch, groups=groups, n_classes=0)
    x, t, _ = inputs(3, 0, seed=42, channels=ch, h=h, w=w)
    cond = {"mask_cond": torch.rand(x.shape, generator=torch.Generator().manual_seed(43))} if mask_cond else None
    with torch.no_grad():
        want = unet_forward(f64(sd), spec, x.double(), t.double(), None if cond is None else {"mask_cond": cond["mask_cond"].double()})
    got = m(x.cuda(), t.cuda(), None if cond is None else {"mask_cond": cond["mask_cond"].cuda()})
    e = rel_l2(got, want)
    print(shape_name, e)
    assert e <= FP32_TOL


# ---------------------------------------------------------------------------------------------------------------------
# fused fp16 / bf16 at the planner's batch-size variants, on a 16-sample slice
# ---------------------------------------------------------------------------------------------------------------------
def _check_16bit(compute_dtype, got, want, fmt, what):
    e = rel_l2(got, want)
    worst = float(per_sample(got, want).max())
    if compute_dtype == "fp16":
        print(what, f"fp16 slice {e:.3e} worst sample {worst:.3e}")
        assert e <= FP16_SLICE_TOL and worst <= FP16_SAMPLE_TOL, (what, e, worst)
    else:
        e_fmt = rel_l2(fmt, want)
        print(what, f"bf16 slice {e:.3e} FUSED_BF16 oracle {e_fmt:.3e} ratio {e / e_fmt:.3f}")
        assert e <= 1.15 * e_fmt + 1e-4, (what, e, e_fmt)


@pytest.mark.parametrize("B", [5, 37, 300, 600])
@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_forward_slice_vs_fp64(compute_dtype, B):
    """B = 5 / 37: clusters of four, quarter tiles; 300: clusters of two, half tiles, the WIDE 4x4 chain; 600: no split, full
    tiles, the capped 4x4 instance."""
    n = 102
    m = cuda_model(n, compute_dtype)
    x, t, cls = inputs(B, n, seed=500 + B)
    idx = slice_idx(B)
    for use_cls in (False, True):
        got = m(x.cuda(), t.cuda(), {"class_cond": cls.cuda()} if use_cls else None).float().cpu()[idx]
        cond = {"class_cond": cls[idx]} if use_cls else None
        with torch.no_grad():
            want = unet_forward(f64(weights(n)), spec_for(n), x[idx].double(), t[idx].double(), cond)
            fmt = unet_forward(weights(n), spec_for(n), x[idx], t[idx], cond, FUSED_BF16) if compute_dtype == "bf16" else None
        assert torch.isfinite(got).all()
        _check_16bit(compute_dtype, got, want, fmt, f"B={B} {'class ids' if use_cls else 'no class ids'}")


@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_single_pass_cfg_slice_vs_fp64(compute_dtype):
    """B = 150 with guidance 3.0: 2B = 300 rows per evaluation through the single-pass CFG forward.  One RK4 interval (four
    guided evaluations), the resulting latents on a 16-sample slice against the fp64 trajectory of those samples."""
    from flocoder_b200 import sampling
    n, B = 102, 150
    m = cuda_model(n, compute_dtype)
    x, _, cls = inputs(B, n, seed=650)
    idx = slice_idx(B)
    got, _ = sampling.generate_latents_rk4(m, tuple(x.shape), n_steps=2, cond={"class_cond": cls.cuda()}, cfg_strength=3.0,
                                           source=x.cuda())
    shape = (len(idx),) + tuple(x.shape[1:])
    cond = {"class_cond": cls[idx]}
    want, _ = oracle.generate_latents_rk4(OracleModel(f64(weights(n)), spec_for(n)), shape, n_steps=2, cond=cond,
                                          cfg_strength=3.0, source=x[idx].double())
    fmt = None
    if compute_dtype == "bf16":
        fmt, _ = oracle.generate_latents_rk4(OracleModel(weights(n), spec_for(n), FUSED_BF16), shape, n_steps=2, cond=cond,
                                             cfg_strength=3.0, source=x[idx].clone())
    assert torch.isfinite(got).all()
    _check_16bit(compute_dtype, got.float().cpu()[idx], want, fmt, "B=150 cfg 3.0")


# ---------------------------------------------------------------------------------------------------------------------
# every stage tensor against the fp64 trace, bounded by the emulating oracle's error at the same tensor
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("compute_dtype,layerwise,B", [("fp16", False, 8), ("bf16", False, 8), ("fp16", False, 300),
                                                       ("bf16", False, 300), ("bf16", True, 8)])
def test_every_stage_tensor_within_the_format_floor(compute_dtype, layerwise, B):
    n = 102
    m = cuda_model(n, compute_dtype, layerwise)
    prec = BF16_MATCHED if layerwise else {"fp16": FUSED_FP16, "bf16": FUSED_BF16}[compute_dtype]
    x, t, cls = inputs(B, n, seed=700 + B)
    idx = slice_idx(B)
    ref, fmt = {}, {}
    with torch.no_grad():
        unet_forward(f64(weights(n)), spec_for(n), x[idx].double(), t[idx].double(), {"class_cond": cls[idx]}, FP32, ref)
        unet_forward(weights(n), spec_for(n), x[idx], t[idx], {"class_cond": cls[idx]}, prec, fmt)
    names = [k for k, v in ref.items() if v.dim() == 4]
    acts = _stage_activations(m, x.cuda(), t.cuda(), names, cls.cuda())
    assert len(acts) > 40
    rows, bad = [], []
    for name, a in acts.items():
        a = a[idx]
        f = fmt[name]
        # the kernel stores this tensor in 16 bits: the floor of reading it back includes that rounding
        if torch.equal(a, a.to(prec.dtype16).float()):
            f = f.to(prec.dtype16).float()
        e_cuda, e_fmt = rel_l2(a, ref[name]), rel_l2(f, ref[name])
        rows.append((name, e_cuda, e_fmt))
        if e_cuda > 1.5 * e_fmt + 1e-4:
            bad.append(f"{name}: cuda {e_cuda:.3e} > 1.5 x format {e_fmt:.3e} + 1e-4")
    for name, e_cuda, e_fmt in rows:
        print(f"{name:32s} cuda {e_cuda:.3e} format {e_fmt:.3e} ratio {e_cuda / max(e_fmt, 1e-30):.3f}")
    print("worst ratio", max((r[1] / max(r[2], 1e-30) for r in rows if r[1] > 1e-4), default=0.0))
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit shapes outside the BASELINE nets, on a 16-sample slice at B = 5 and 300
# ---------------------------------------------------------------------------------------------------------------------
SIXTEEN_BIT_SHAPES = {
    # name: (dim, channels, dim_mults, groups, latent (h, w), layer-wise)
    "groups1": (16, 4, [1, 2, 4, 8], 1, (16, 16), False),         # one group: no N-split of the GroupNorm chain steps
    "groups2": (16, 4, [1, 2, 4, 8], 2, (16, 16), False),
    "channels1": (16, 1, [1, 2, 4, 8], 4, (16, 16), False),
    "channels2": (16, 2, [1, 2, 4, 8], 4, (16, 16), False),
    "8x8_mults124": (16, 4, [1, 2, 4], 4, (8, 8), False),
    "4x64_mults124": (16, 4, [1, 2, 4], 4, (4, 64), False),      # 3-tile chain, transposed-K k_attn
    "16x8_mults124": (16, 4, [1, 2, 4], 4, (16, 8), False),
    "layerwise_channels8": (16, 8, [1, 2, 4, 8], 4, (16, 16), True),
    "layerwise_channels16": (16, 16, [1, 2, 4, 8], 4, (16, 16), True),
    "layerwise_dim32_groups8": (32, 4, [1, 2, 4, 8], 8, (16, 16), True),   # 4-channel groups: channel-block pairs, and k_gn
}
SIXTEEN_BIT_CASES = [(name, cd) for name, shape in SIXTEEN_BIT_SHAPES.items() for cd in (("bf16",) if shape[5] else ("fp16", "bf16"))]
_shape_models = {}


def shape_model(name, compute_dtype):
    from flocoder_b200 import _lib
    from flocoder_b200.unet import Unet
    key = (name, compute_dtype)
    if key not in _shape_models:
        dim, ch, mults, groups, _, layerwise = SIXTEEN_BIT_SHAPES[name]
        torch.manual_seed(51)
        m = Unet(dim=dim, channels=ch, dim_mults=mults, resnet_block_groups=groups, n_classes=0, compute_dtype=compute_dtype)
        sd = trained_like({k: v.detach().clone() for k, v in m.state_dict().items()})
        m.load_state_dict(sd)
        if layerwise:
            m.engine_flags = _lib.FLO_FLAG_LAYERWISE
        _shape_models[key] = (m.cuda().eval(), sd)
    return _shape_models[key]


@pytest.mark.parametrize("B", [5, 300])
@pytest.mark.parametrize("name,compute_dtype", SIXTEEN_BIT_CASES)
def test_16bit_other_shapes_slice_vs_fp64(name, compute_dtype, B):
    """Fused fp16 / bf16 within the _check_16bit bounds; the layer-wise bf16 path within 1.35x the error of the
    bf16-emulating oracle (BF16_MATCHED) + 2e-4."""
    from flocoder_b200 import _lib
    dim, ch, mults, groups, (h, w), layerwise = SIXTEEN_BIT_SHAPES[name]
    assert_plans(dim, ch, mults, groups, (h, w), compute_dtype, B, _lib.FLO_FLAG_LAYERWISE if layerwise else 0)
    m, sd = shape_model(name, compute_dtype)
    spec = UnetSpec(dim=dim, dim_mults=tuple(mults), channels=ch, groups=groups, n_classes=0)
    x, t, _ = inputs(B, 0, seed=800 + B, channels=ch, h=h, w=w)
    idx = slice_idx(B)
    got = m(x.cuda(), t.cuda()).float().cpu()[idx]
    assert torch.isfinite(got).all()
    with torch.no_grad():
        want = unet_forward(f64(sd), spec, x[idx].double(), t[idx].double(), None)
        fmt = None
        if compute_dtype == "bf16":
            fmt = unet_forward(sd, spec, x[idx], t[idx], None, BF16_MATCHED if layerwise else FUSED_BF16)
    if not layerwise:
        _check_16bit(compute_dtype, got, want, fmt, f"{name} B={B}")
        return
    e, e_fmt = rel_l2(got, want), rel_l2(fmt, want)
    print(name, f"B={B} layer-wise bf16 slice {e:.3e} BF16_MATCHED oracle {e_fmt:.3e} ratio {e / e_fmt:.3f}")
    assert e <= 1.35 * e_fmt + 2e-4, (name, B, e, e_fmt)
