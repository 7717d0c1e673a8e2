"""The C-ABI library: loads without a GPU, exports every symbol include/flocoder_b200.h declares,
and its host-side logic (manifest, validation, error mapping) behaves.  No compute calls here."""
import ctypes
import os
import re

import pytest
import torch

from conftest import CONFIGS, ROOT
from flocoder_b200 import _lib
from flocoder_b200.unet import Unet

HEADER = os.path.join(ROOT, "include", "flocoder_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"FLO_API\s+[\w\s\*]+?\b(flo_\w+)\s*\(", text)))


def test_library_is_built_and_loads():
    assert os.path.isfile(_lib.LIB_PATH), "run `python -m flocoder_b200.build`"
    L = _lib.lib()
    assert L.flo_version() == 100


def test_every_declared_symbol_is_exported():
    L = _lib.lib()
    names = declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(L, n), f"{n} declared in the header but not exported"
    assert sorted(_lib.EXPORTS) == names


@pytest.mark.parametrize("name", list(CONFIGS))
def test_manifest_matches_module_state_dict(name):
    n_classes = CONFIGS[name]
    m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes)
    cfg = _lib.make_cfg(16, 4, (1, 2, 4, 8), 4, n_classes, 16, 16, "fp32", 0)
    manifest = _lib.param_manifest(cfg)
    sd = m.state_dict()
    assert [n for n, _ in manifest] == list(sd.keys())
    for n, shape in manifest:
        assert tuple(sd[n].shape) == shape, n


def test_manifest_generic_dims():
    m = Unet(dim=32, channels=3, dim_mults=[1, 2, 2], resnet_block_groups=8, n_classes=5)
    cfg = _lib.make_cfg(32, 3, (1, 2, 2), 8, 5, 8, 8, "bf16", 0)
    manifest = _lib.param_manifest(cfg)
    assert [n for n, _ in manifest] == list(m.state_dict().keys())


def test_unsupported_configs_are_explicit_errors():
    L = _lib.lib()
    cfg = _lib.make_cfg(16, 4, (1, 2, 4, 8), 4, 0, 16, 16, "bf16", 0, mask_cond=True)   # inpainting U-Net: fp32 path only
    with pytest.raises(NotImplementedError):
        _lib.check(L.flo_param_count(ctypes.byref(cfg)))
    assert b"mask_cond" in L.flo_last_error()
    cfg = _lib.make_cfg(12, 4, (1, 2), 4, 0, 16, 16, "fp32", 0)       # dim not a multiple of 8
    with pytest.raises(NotImplementedError):
        _lib.check(L.flo_param_count(ctypes.byref(cfg)))
    cfg = _lib.make_cfg(16, 4, (1, 2, 4, 8), 4, 0, 12, 12, "fp32", 0)  # 12 not divisible by 8
    with pytest.raises(ValueError):
        _lib.check(L.flo_param_count(ctypes.byref(cfg)))
    cfg = _lib.make_cfg(24, 4, (1, 2), 4, 0, 16, 16, "bf16", 0)       # bf16 path needs dim % 16 == 0
    with pytest.raises(NotImplementedError):
        _lib.check(L.flo_param_count(ctypes.byref(cfg)))
    # the layer-wise 16-bit GroupNorm kernels index by shifts: 6 groups per sample and 12x12 planes have no kernel there.  The
    # manifest exists (the module can hold such weights); planning the forward refuses, naming the GroupNorm.
    for dim, groups, mults, hw in ((48, 6, (1, 2, 4, 8), 16), (16, 4, (1, 2, 4), 12)):
        cfg = _lib.make_cfg(dim, 8, mults, groups, 0, hw, hw, "bf16", 0, _lib.FLO_FLAG_LAYERWISE)
        _lib.check(L.flo_param_count(ctypes.byref(cfg)))
        with pytest.raises(NotImplementedError, match=r"GroupNorm 'downs\.0\.0\.block1' .* has no kernel"):
            _lib.describe_plan(cfg, 8)


def test_inpainting_manifest_matches_the_module():
    """mask_cond=1: the mask-fusion parameters in the reference's registration order (unet.py:214-235), for the
    midi_inpainting shape (dim = 8: two channels per GroupNorm group) as well."""
    for dim, hw in ((16, 16), (8, 8)):
        m = Unet(dim=dim, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True)
        cfg = _lib.make_cfg(dim, 4, (1, 2, 4, 8), 4, 0, hw, hw, "fp32", 0, mask_cond=True)
        manifest = _lib.param_manifest(cfg)
        sd = m.state_dict()
        assert [n for n, _ in manifest] == list(sd.keys())
        assert all(tuple(sd[n].shape) == shp for n, shp in manifest)
        text = _lib.describe_plan(cfg, 8)
        for op in ("mask_fusion_conv.0", "mask_fusion_conv.2", "mask_fusion_conv ", "down_mask_fusions.0.0", "down_mask_fusions.1.0",
                   "up_mask_fusions.0.0", "up_mask_fusions.1.0"):
            assert op in text, op


def test_nfe_counts():
    L = _lib.lib()
    assert L.flo_integrate_nfe(_lib.FLO_RK4, 50) == 196          # 49 intervals x 4 (SURVEY TL;DR)
    assert L.flo_integrate_nfe(_lib.FLO_EULER_LEGACY, 10) == 10
    assert L.flo_integrate_nfe(_lib.FLO_EULER_GRID, 10) == 9
    assert L.flo_integrate_nfe(99, 10) == -1


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_create_without_gpu_fails_loudly():
    m = Unet(dim=16, channels=4, n_classes=0)
    with pytest.raises(RuntimeError):
        _lib.Engine(dim=16, channels=4, dim_mults=(1, 2, 4, 8), groups=4, n_classes=0, height=16, width=16,
                    compute_dtype="fp32", device="cpu", state_dict=m.state_dict())


def test_fused_plan_decisions_round2():
    """Host-only planner checks (no GPU): (1) a stage that allocates all 512 tensor-memory columns must not fit twice on an SM
    (a second co-resident CTA would sit in tcgen05.alloc until the first exits: downs.1.2 ran as two waves before the planner
    asked for more than half an SM); (2) the small-batch plan gives the 4x4 / 2x2 attention blocks quarter-filled tiles."""
    import re
    cfg = _lib.make_cfg(dim=16, channels=4, dim_mults=[1, 2, 4, 8], groups=4, n_classes=0, height=16, width=16,
                        compute_dtype="bf16", device_index=0)
    lines = [l for l in _lib.describe_plan(cfg, 256).splitlines() if l.startswith("stage")]
    attn = [l for l in lines if " attn " in l]
    assert len(attn) == 9 and len(lines) == 19
    sm_bytes = 233472                                     # shared memory per SM; every CTA also reserves 1 KB
    for l in attn:
        smem, tmem = int(re.search(r"smem=(\d+)", l).group(1)), int(re.search(r"tmem=(\d+)", l).group(1))
        if tmem > 256:
            assert 2 * (smem + 1024) > sm_bytes, l
    by_name = {l.split()[3]: l for l in attn}
    assert "nb=2 " in by_name["downs.2.2"] and "ctas=128" in by_name["downs.2.2"]      # 4x4: 32 live rows per CTA
    assert "nb=8 " in by_name["downs.3.2"] and "ctas=32" in by_name["downs.3.2"]       # 2x2
    assert "nb=8 " in by_name["mid_attn"] and "full=1" in by_name["mid_attn"]


def test_environment_switches_are_the_ones_the_tests_use():
    """The library reads a FLO_* environment variable only to force a path that the planner also selects from the input, so that
    a test can compare the two on one input (FLO_TIMELINE: the clock64 instrumentation behind tools/gpu_timeline.py).  A losing
    A/B alternative goes together with its switch; a new switch comes with a test that uses it."""
    csrc = os.path.join(ROOT, "flocoder_b200", "csrc")
    read = set()
    for name in os.listdir(csrc):
        with open(os.path.join(csrc, name)) as f:
            read |= set(re.findall(r'getenv\("(FLO_\w+)"\)', f.read()))
    kept = {"FLO_SMALL_DIV", "FLO_ATTN_NO_KTRANS", "FLO_CFG_TWO_PASS", "FLO_GN_NO_TMA", "FLO_GN_CTA", "FLO_TIMELINE"}
    assert read == kept
    tests = os.path.join(ROOT, "tests")
    text = ""
    for name in os.listdir(tests):
        if name.endswith(".py") and name != os.path.basename(__file__):
            with open(os.path.join(tests, name)) as f:
                text += f.read()
    for switch in sorted(kept - {"FLO_TIMELINE"}):
        assert switch in text, f"{switch} is read by the library, but no test uses it"
