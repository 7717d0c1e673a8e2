"""The shape space the planner accepts, against what its kernels can run (host only, no GPU).

Every U-Net configuration either is refused with ValueError / NotImplementedError before anything runs, or plans only
kernels whose indexing holds for its shapes.  The preconditions below are each kernel's own, taken from what it indexes
(kernels_simt.cu, fused.cu): k_gn_tma, k_gn_warp and k_gn find pixels, channel blocks and samples with shifts and masks,
so a plan that sends them a 6-group or 12x12 GroupNorm would read and write past its tensors."""
import ctypes
import itertools
import random
import re

import pytest

from flocoder_b200 import _lib

DIMS = (8, 16, 24, 32, 48, 64)
GROUPS = (1, 2, 3, 4, 6, 8)
CHANNELS = (1, 2, 3, 4, 8, 16)
MULTS = ((1,), (1, 2), (1, 3), (1, 2, 4), (1, 2, 3), (1, 2, 4, 8), (1, 1, 2, 2, 4))      # depth 1 to 5
LATENTS = ((16, 16), (8, 8), (4, 4), (32, 32), (64, 64), (16, 8), (8, 32), (4, 64), (12, 12), (20, 12), (48, 48), (48, 64))
# (compute dtype, flags, mask_cond)
PATHS = (("fp32", 0, False), ("fp32", 0, True), ("bf16", 0, False), ("fp16", 0, False), ("bf16", _lib.FLO_FLAG_LAYERWISE, False))
BATCHES = (8, 300)
SMEM_MAX = 227 * 1024           # shared memory a CTA may use on sm_100a


def pow2(x):
    return x > 0 and x & (x - 1) == 0


def gn_kernel_holds(variant, C, H, W, groups, bf16):
    """Whether the GroupNorm kernel `variant` indexes a C x H x W tensor with `groups` groups correctly."""
    cpg, hw = C // groups, H * W
    pair = cpg == 4                         # two 4-channel groups share one 8-channel block
    if variant == "any":                    # k_gn_any: scalar loads, integer divisions; fp32 outputs only
        return not bf16
    if not (pair or cpg % 8 == 0):          # the other three read whole channel quads of the blocked layout
        return False
    if not (pow2(W) and pow2(hw)):          # pixel -> (h, w) and float4 index -> channel block are shifts and masks
        return False
    if variant == "tma":                    # unit = channel-block pair or one group; 2-deep ring of units in 72 KB
        units, unit_bytes = (C // 8, hw * 32) if pair else (groups, cpg * hw * 4)
        return pow2(units) and hw >= 16 and pow2(unit_bytes) and 2048 <= unit_bytes <= 16384
    if variant == "warp":                   # unit held in one warp's registers: T <= 32 lanes x V <= 32 float4, both powers of two
        units, nvec = (C // 8, hw * 2) if pair else (groups, cpg * hw // 4)
        return pow2(units) and pow2(nvec) and 2 <= nvec <= 1024
    if variant == "cta":                    # one (sample, group) per CTA, blockIdx -> (sample, group) by shift: <= 256 x 8 float4
        return pow2(groups) and cpg * hw <= 256 * 8 * 4
    return False


def attn_kernel_holds(kind, n, bf16):
    if kind == "midattn":                   # k_midattn: the n x n scores of one head in shared memory
        return 1 <= n <= 64
    return n <= 256 or (not bf16 and n % 256 == 0)      # k_linattn: one CTA per head; k_linattn_big: fp32, 256-pixel tiles


def plan_violations(text, compute_dtype, flags, channels):
    """Every reason the described plan would run a kernel outside its preconditions."""
    bad = []
    bf16 = compute_dtype != "fp32"
    fused = "\nfused:" in text
    if fused != (bf16 and not flags & _lib.FLO_FLAG_LAYERWISE and channels <= 4):
        bad.append(f"fused={fused} is not the path this config selects")
    for line in text.splitlines():
        f = line.split()
        if not fused and len(f) > 1 and f[1] == "gn":
            C, (H, W), G = int(re.search(r" C=(\d+)", line).group(1)), map(int, f[4].split("x")), int(re.search(r"groups=(\d+)", line).group(1))
            v = re.search(r" gn=(\w+)", line)
            if v is None or not gn_kernel_holds(v.group(1), C, H, W, G, bf16):
                bad.append(f"{f[2]}: C={C} {H}x{W} groups={G} runs gn={v.group(1) if v else '?'}")
        elif not fused and len(f) > 1 and f[1] in ("linattn", "midattn"):
            n = int(re.search(r" n=(\d+)", line).group(1))
            if not attn_kernel_holds(f[1], n, bf16):
                bad.append(f"{f[2]}: {f[1]} at n={n}")
        elif fused and f and f[0] == "stage":
            H, W = map(int, f[4].split("x"))
            smem, tmem = int(re.search(r"smem=(\d+)", line).group(1)), int(re.search(r"tmem=(\d+)", line).group(1))
            if not (pow2(H) and pow2(W)) or smem > SMEM_MAX or not (pow2(tmem) and 32 <= tmem <= 512):
                bad.append(f"stage {f[3]}: {H}x{W} smem={smem} tmem={tmem}")
        elif fused and f and f[0] == "step":
            C, G = int(re.search(r" C=(\d+)", line).group(1)), int(re.search(r" G=(\d+)", line).group(1))
            if G and not (pow2(C) and pow2(G)):
                bad.append(f"step with C={C} G={G}")
    return bad


def config_id(dim, groups, channels, mults, hw, path):
    cd, flags, mask = path
    return (f"{cd}{'-layerwise' if flags else ''}{'-mask' if mask else ''} dim={dim} groups={groups} ch={channels} "
            f"mults={list(mults)} {hw[0]}x{hw[1]}")


def check_config(dim, groups, channels, mults, hw, path):
    """None when the config is refused or plans only valid kernels at every batch size, else what is wrong."""
    cd, flags, mask = path
    cfg = _lib.make_cfg(dim, channels, mults, groups, 0, hw[0], hw[1], cd, 0, flags, mask_cond=mask)
    L = _lib.lib()
    try:
        _lib.check(L.flo_param_count(ctypes.byref(cfg)))
        texts = [_lib.describe_plan(cfg, BATCHES[0])]
        if "\nfused:" in texts[0]:          # the layer-by-layer op program does not depend on the batch size; fused stages do
            texts += [_lib.describe_plan(cfg, b) for b in BATCHES[1:]]
    except (ValueError, NotImplementedError):
        return None
    bad = sorted({v for t in texts for v in plan_violations(t, cd, flags, channels)})
    return f"{config_id(dim, groups, channels, mults, hw, path)}: {'; '.join(bad[:3])}" if bad else None


def sweep_configs():
    """Four grids over the axes the kernels index by, plus a seeded sample of the whole product."""
    cfgs = []
    for path in PATHS:
        cfgs += [(d, g, 4, (1, 2, 4), (16, 16), path) for d, g in itertools.product(DIMS, GROUPS)]
        cfgs += [(16, 4, 4, m, hw, path) for m, hw in itertools.product(MULTS, LATENTS)]
        cfgs += [(d, 4, c, (1, 2, 4), (16, 16), path) for d, c in itertools.product((16, 32), CHANNELS)]
        cfgs += [(48, g, c, (1, 2, 4), hw, path) for g, c, hw in itertools.product((3, 6), (4, 8), ((16, 16), (12, 12)))]
    # host-side weight packing grows with the square of the widest level: keep it at 256 channels to bound the run time
    every = [c for c in itertools.product(DIMS, GROUPS, CHANNELS, MULTS, LATENTS, PATHS) if c[0] * max(c[3]) <= 256]
    cfgs += random.Random(2024).sample(every, 300)
    return list(dict.fromkeys(cfgs))


def test_every_accepted_shape_plans_only_kernels_that_index_it():
    cfgs = sweep_configs()
    failures = [f for f in (check_config(*c) for c in cfgs) if f]
    assert not failures, f"{len(failures)} of {len(cfgs)} configs plan kernels outside their preconditions:\n" + "\n".join(failures[:40])


# The shapes that used to plan and then index out of bounds (GroupNorm) or fail at the first forward (attention, and a
# GroupNorm unit too large for any 16-bit kernel).  Each is now either refused at plan time or planned onto k_gn_any.
LAYERWISE = ("bf16", _lib.FLO_FLAG_LAYERWISE, False)
FP32 = ("fp32", 0, False)
NAMED = {
    # name: (dim, groups, channels, mults, (H, W), path, refused)
    "fp32_dim48_groups6": (48, 6, 4, (1, 2, 4, 8), (16, 16), FP32, False),
    "fp32_dim24_groups3": (24, 3, 4, (1, 2, 4, 8), (16, 16), FP32, False),
    "fp32_dim24_groups6": (24, 6, 4, (1, 2, 4, 8), (16, 16), FP32, False),
    "fp32_12x12": (16, 4, 4, (1, 2, 4), (12, 12), FP32, False),
    "fp32_48x48": (16, 4, 4, (1, 2, 4, 8), (48, 48), FP32, True),          # linear attention at 24x24 = 576 pixels
    "fp32_one_level_16x16": (16, 4, 4, (1,), (16, 16), FP32, True),        # mid attention at n = 256
    "layerwise_dim48_groups6": (48, 6, 8, (1, 2, 4, 8), (16, 16), LAYERWISE, True),
    "layerwise_12x12": (16, 4, 8, (1, 2, 4), (12, 12), LAYERWISE, True),
    "layerwise_dim64_16x16": (64, 4, 4, (1, 2), (16, 16), LAYERWISE, True),   # GroupNorm(1, 64) over 16384 elements
}


@pytest.mark.parametrize("name", list(NAMED))
def test_shapes_that_indexed_out_of_bounds(name):
    dim, groups, ch, mults, hw, path, refused = NAMED[name]
    cd, flags, mask = path
    cfg = _lib.make_cfg(dim, ch, mults, groups, 0, hw[0], hw[1], cd, 0, flags)
    if refused:
        with pytest.raises(NotImplementedError, match="has no kernel"):
            _lib.describe_plan(cfg, 8)
        return
    text = _lib.describe_plan(cfg, 8)
    assert not plan_violations(text, cd, flags, ch)
    assert " gn=any" in text


def test_baseline_layerwise_plans_run_the_fast_groupnorm_kernels():
    """The BASELINE U-Net (dim 16, groups 4, 16x16) keeps k_gn_tma / k_gn_warp for every GroupNorm on the layer-wise paths."""
    for cd, flags in (("fp32", 0), ("bf16", _lib.FLO_FLAG_LAYERWISE)):
        cfg = _lib.make_cfg(16, 4, (1, 2, 4, 8), 4, 102, 16, 16, cd, 0, flags)
        text = _lib.describe_plan(cfg, 256)
        variants = re.findall(r" gn=(\w+)", text)
        assert len(variants) == len(re.findall(r"^ *\d+ gn ", text, re.M)) == 55
        assert set(variants) <= {"tma", "warp"}, variants
