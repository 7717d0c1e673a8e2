"""The inpainting U-Net (``mask_cond=True``) on the layer-wise bf16 tcgen05 route, host only (no GPU).

``compute_dtype="bf16"`` with ``FLO_FLAG_LAYERWISE`` plans every mask-fusion convolution, the 5x5 ``mask_fusion_conv.0``
included, onto k_conv_umma, with 16-channel bf16 mask pyramids.  Every other 16-bit mask route stays refused, and every
accepted shape plans only convolutions within k_conv_umma's preconditions."""
import itertools
import random
import re

import pytest

from flocoder_b200 import _lib
from test_shape_envelope import SMEM_MAX, plan_violations, pow2

LW = _lib.FLO_FLAG_LAYERWISE
MASK_OPS = ("mask_fusion_conv.0", "mask_fusion_conv.2", "mask_fusion_conv", "down_mask_fusions.0.0", "down_mask_fusions.1.0",
            "up_mask_fusions.0.0", "up_mask_fusions.1.0")


def cfg(dim=16, channels=4, mults=(1, 2, 4, 8), groups=4, hw=(16, 16), dtype="bf16", flags=LW, mask=True):
    return _lib.make_cfg(dim, channels, mults, groups, 0, hw[0], hw[1], dtype, 0, flags, mask_cond=mask)


@pytest.mark.parametrize("dim", [16, 32, 64])
def test_manifest_is_the_reference_state_dict(dim):
    from flocoder_b200.unet import Unet
    want = [(k, tuple(v.shape)) for k, v in Unet(dim=dim, channels=4, dim_mults=(1, 2, 4, 8), n_classes=0,
                                                  mask_cond=True).state_dict().items()]
    assert _lib.param_manifest(cfg(dim=dim)) == want


def conv_lines(text):
    return {m.group(1): line for line in text.splitlines() if (m := re.match(r" *\d+ conv +(\S+) ", line))}


@pytest.mark.parametrize("dim, hw", [(16, (16, 16)), (32, (16, 16)), (64, (8, 8))])   # dim 64 at 16x16: no GroupNorm(1, 64) kernel
def test_every_mask_op_has_a_tcgen05_tiling(dim, hw):
    text = _lib.describe_plan(cfg(dim=dim, hw=hw), 256)
    assert "\nfused:" not in text
    convs = conv_lines(text)
    for name in MASK_OPS:
        assert name in convs, name
        assert " | nb=" in convs[name] and "UNSUPPORTED" not in convs[name], convs[name]
    assert f" k=5 cin={dim}+16 cout={2 * dim} " in convs["mask_fusion_conv.0"]
    for name in ("down_mask_fusions.0.0", "up_mask_fusions.1.0"):
        assert "+16 " in convs[name] and "in1=mask_cond:" in convs[name]
    bufs = re.findall(r"buf +\d+ mask_cond:(\d) +C=(\d+) \d+x\d+ (\w+)", text)
    assert [b[0] for b in bufs] == ["0", "1", "2", "3"]
    assert all(c == "16" and t == "bf16" for _, c, t in bufs), bufs


def test_fp32_mask_plan_keeps_its_8_channel_fp32_pyramid():
    text = _lib.describe_plan(cfg(dtype="fp32", flags=0), 256)
    bufs = re.findall(r"buf +\d+ mask_cond:\d +C=(\d+) \d+x\d+ (\w+)", text)
    assert bufs == [("8", "f32")] * 4


@pytest.mark.parametrize("kwargs", [
    dict(dtype="bf16", flags=0),                    # default 16-bit route: fused stage kernels have no mask branches
    dict(dtype="bf16", flags=_lib.FLO_FLAG_NO_GRAPH),
    dict(dtype="fp16", flags=0),
    dict(dtype="fp16", flags=LW),
    dict(dim=8, hw=(8, 8)),                          # configs/midi_inpainting.yaml: dim % 16 != 0 stays fp32-only
    dict(channels=16),
])
def test_other_16bit_mask_routes_are_refused(kwargs):
    c = cfg(**kwargs)
    with pytest.raises(NotImplementedError, match="mask_cond|dim % 16"):
        _lib.param_manifest(c)
    with pytest.raises(NotImplementedError):
        _lib.describe_plan(c, 8)


def test_default_route_refusal_names_the_layerwise_route():
    with pytest.raises(NotImplementedError, match="mask_cond.*FLO_FLAG_LAYERWISE"):
        _lib.param_manifest(cfg(flags=0))


# ---------------------------------------------------------------------------------------------------------------------
# the accepted shape space of the new route
# ---------------------------------------------------------------------------------------------------------------------
DIMS = (16, 32, 48, 64)
GROUPS = (1, 2, 4, 8)
CHANNELS = (1, 3, 4, 8)
MULTS = ((1,), (1, 2), (1, 2, 4), (1, 2, 4, 8), (1, 1, 2, 2, 4))
LATENTS = ((16, 16), (8, 8), (16, 8), (8, 32), (4, 64), (12, 12), (4, 4), (2, 2), (32, 8))
BATCHES = (8, 300)


def conv_violations(text):
    """Every conv whose tcgen05 tiling is outside k_conv_umma's preconditions."""
    bad = []
    for name, line in conv_lines(text).items():
        f = re.search(r" (\d+)x(\d+) k=(\d+) cin=(\d+)\+(\d+) cout=(\d+) ", line)
        t = re.search(r"nb=(\d+) mt=(\d+) n_tile=(\d+) sbo=(\d+) S=\d+ stages=\d+ smem=(\d+) tmem=(\d+)", line)
        if f is None or t is None:
            bad.append(f"{name}: no tiling ({line[-80:]})")
            continue
        H, W, k, c0, c1, cout = map(int, f.groups())
        nb, mt, n_tile, sbo, smem, tmem = map(int, t.groups())
        pad = k // 2
        Hp, Wp = H + 2 * pad, W + 2 * pad
        a_bytes = (c0 + c1) // 8 * nb * Hp * Wp * 16
        if k % 2 == 0 or k > 5 or (c0 + c1) % 16 or cout % n_tile or n_tile % 16:
            bad.append(f"{name}: k={k} cin={c0}+{c1} cout={cout} n_tile={n_tile}")
        if a_bytes > smem or smem > SMEM_MAX:
            bad.append(f"{name}: A region {a_bytes} B, smem {smem} B")
        if not (pow2(tmem) and 32 <= tmem <= 512 and mt * n_tile <= tmem):
            bad.append(f"{name}: tmem {tmem} for {mt} x {n_tile}")
        if max(Wp, Hp, nb, c0 // 8, c1 // 8) > 256:             # TMA box dimensions
            bad.append(f"{name}: TMA box {Wp}x{Hp} nb={nb} ncb={c0 // 8}+{c1 // 8}")
        if sbo != 8 and (sbo != Wp or nb != 1 or H % 16 or W % 8):   # strip tiles: 16 rows x 8 columns of one sample
            bad.append(f"{name}: strip tiling sbo={sbo} at {H}x{W}")
    return bad


def check(dim, groups, channels, mults, hw):
    c = cfg(dim=dim, channels=channels, mults=mults, groups=groups, hw=hw)
    try:
        _lib.param_manifest(c)
        texts = [_lib.describe_plan(c, b) for b in BATCHES]
    except (ValueError, NotImplementedError):
        return None, False
    bad = sorted({v for t in texts for v in plan_violations(t, "bf16", LW, channels) + conv_violations(t)})
    return (f"dim={dim} groups={groups} ch={channels} mults={list(mults)} {hw[0]}x{hw[1]}: {'; '.join(bad[:3])}" if bad else
            None), True


def sweep():
    cfgs = [(d, g, 4, (1, 2, 4), (16, 16)) for d, g in itertools.product(DIMS, GROUPS)]
    cfgs += [(16, 4, 4, m, hw) for m, hw in itertools.product(MULTS, LATENTS)]
    cfgs += [(d, 4, c, (1, 2, 4), (16, 16)) for d, c in itertools.product((16, 64), CHANNELS)]
    cfgs += [(d, 4, 4, (1, 2, 4), hw) for d, hw in itertools.product(DIMS, ((8, 8), (16, 8), (4, 64), (12, 12)))]
    every = [c for c in itertools.product(DIMS, GROUPS, CHANNELS, MULTS, LATENTS) if c[0] * max(c[3]) <= 256]
    cfgs += random.Random(7).sample(every, 120)
    return list(dict.fromkeys(cfgs))


def test_every_accepted_mask_shape_plans_only_kernels_that_index_it():
    results = [check(*c) for c in sweep()]
    failures = [f for f, _ in results if f]
    accepted = sum(a for _, a in results)
    assert accepted >= 50, accepted
    assert not failures, f"{len(failures)} configs plan kernels outside their preconditions:\n" + "\n".join(failures[:40])


@pytest.mark.parametrize("hw", [(8, 8), (16, 8), (4, 64), (12, 12)])
def test_5x5_fusion_off_the_16x16_strip_mode(hw):
    """The 5x5 conv plans at these latents, or the whole config is refused for a reason other than the conv."""
    c = cfg(dim=16, mults=(1, 2, 4), hw=hw)
    try:
        text = _lib.describe_plan(c, 300)
    except NotImplementedError as e:
        assert "mask_fusion_conv" not in str(e) and "k_conv_umma" not in str(e), str(e)
        return
    line = conv_lines(text)["mask_fusion_conv.0"]
    assert " k=5 " in line and not conv_violations(text)
