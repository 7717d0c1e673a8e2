"""Parity of the CUDA path (through the C ABI) with the oracle / the frozen reference outputs.

Bars (BASELINE.json north_star):
  fp32 : per-step velocity and final latent rel-L2 <= 1e-5 vs the reference (fp32 CPU)
  16-bit tensor-core paths: per-step velocity rel-L2 <= 2e-3, final latent rel-L2 <= 1e-2.
    * fp16 operands (same tcgen05 rate as bf16, 3 more mantissa bits) meet both bars directly against the fp32
      reference.
    * bf16 operands cannot meet 2e-3 per step against ANY reference: 8-bit mantissas put the format floor of this
      38-conv network at ~4.8e-3 per forward (SURVEY.md 8c), and a "precision-matched" oracle does not help because
      a 1e-7 input perturbation already moves the matched oracle itself by ~3e-3 (rounding decisions flip and the
      flips cascade; test_bf16_rounding_noise_floor measures it).  The bf16 tests therefore bound the CUDA error
      by the format floor (<= 1.35x the error of the bf16-emulating oracle vs fp32) and check the first blocks,
      before the cascade, tightly; the final-latent bar (1e-2) is met with a wide margin (~1.2e-3).
"""
import pytest
import torch

import oracle
from oracle.unet_oracle import BF16_MATCHED, FP32, FUSED_BF16, FUSED_FP16, OracleModel, UnetSpec, unet_forward
from conftest import CONFIGS, rel_l2, seeded_state_dict

pytestmark = pytest.mark.gpu

SHAPE = (8, 4, 16, 16)
FP32_STEP_TOL = 1e-5
FP32_FINAL_TOL = 1e-5
BF16_STEP_TOL = 2e-3
BF16_FINAL_TOL = 1e-2


def spec_for(n_classes):
    return UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=n_classes)


_models = {}


def gpu_model(n_classes, compute_dtype, layerwise=False):
    key = (n_classes, compute_dtype, layerwise)
    if key not in _models:
        from flocoder_b200 import _lib
        from flocoder_b200.unet import Unet
        torch.manual_seed(1234)
        m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes, compute_dtype=compute_dtype)
        if layerwise:
            m.engine_flags = _lib.FLO_FLAG_LAYERWISE
        _models[key] = m.cuda().eval()
    return _models[key]


def test_selftest_tcgen05_building_blocks():
    from flocoder_b200 import _lib
    rc, report = _lib.selftest_umma()
    print(report)
    assert rc == 0, f"flo_selftest_umma reported {rc} failing case(s):\n{report}"


@pytest.mark.parametrize("name", list(CONFIGS))
def test_fp32_forward_matches_reference_golden(goldens, name):
    g = goldens[name]
    m = gpu_model(g["n_classes"], "fp32")
    v = m(g["x0"].cuda(), g["fwd_t"].cuda())
    assert rel_l2(v, g["fwd_v"]) <= FP32_STEP_TOL
    v = m(g["x0"].cuda(), g["fwd_tvec"].cuda())                       # per-sample times
    assert rel_l2(v, g["fwd_v_tvec"]) <= FP32_STEP_TOL
    if g["n_classes"] > 0:
        v = m(g["x0"].cuda(), g["fwd_t"].cuda(), cond={"class_cond": g["cls"].cuda()})
        assert rel_l2(v, g["fwd_v_cls"]) <= FP32_STEP_TOL
        v = m(g["x0"].cuda(), g["fwd_t"].cuda(), cond={"class_cond": None})
        assert rel_l2(v, g["fwd_v"]) <= FP32_STEP_TOL


@pytest.mark.parametrize("name", list(CONFIGS))
def test_fp32_integrators_match_reference_golden(goldens, name):
    from flocoder_b200 import sampling
    g = goldens[name]
    m = gpu_model(g["n_classes"], "fp32")
    x0 = g["x0"].cuda()
    x1, nfe = sampling.generate_latents_rk4(m, SHAPE, n_steps=10, source=x0)
    assert nfe == g["rk4_10_nfe"]
    assert rel_l2(x1, g["rk4_10"]) <= FP32_FINAL_TOL
    assert torch.equal(x0.cpu(), g["x0"]), "the caller's source tensor must not be modified"
    x1, nfe = sampling.euler_sampler(m, SHAPE, 10, source=x0)
    assert nfe == 10 and x1.device.type == "cpu"
    assert rel_l2(x1, g["euler_10"]) <= FP32_FINAL_TOL
    x1, nfe = sampling.generate_latents_rk4(m, SHAPE, n_steps=10, source=x0, init_latents=g["init_latents"].cuda(),
                                            init_strength=0.3)
    assert nfe == g["rk4_10_init03_nfe"] and rel_l2(x1, g["rk4_10_init03"]) <= FP32_FINAL_TOL
    if g["n_classes"] > 0:
        cond = {"class_cond": g["cls"].cuda()}
        x1, _ = sampling.generate_latents_rk4(m, SHAPE, n_steps=10, cond=cond, cfg_strength=3.0, source=x0)
        assert rel_l2(x1, g["rk4_10_cfg3"]) <= FP32_FINAL_TOL
        x1, _ = sampling.generate_latents_rk4(m, SHAPE, n_steps=10, cond=cond, cfg_strength=0, source=x0)
        assert rel_l2(x1, g["rk4_10_cls_nocfg"]) <= FP32_FINAL_TOL


def test_fp32_rk4_50_final_latent(goldens):
    """BASELINE config shape (RK4, n_steps=50 -> 49 intervals, 196 evaluations) at B=8."""
    from flocoder_b200 import sampling
    g = goldens["flowers_sd"]
    m = gpu_model(102, "fp32")
    x1, nfe = sampling.generate_latents(m, SHAPE, method="rk4", n_steps=50, source=g["x0"].cuda())
    assert nfe == 200
    assert rel_l2(x1, g["rk4_50"]) <= FP32_FINAL_TOL


def _stage_activations(m, x, t, names, class_ids=None):
    """{name: fp32 CPU copy} of the activations of one CUDA forward that the engine keeps under these names (a fresh engine
    with FLO_FLAG_NO_BUFFER_REUSE, so every one of them survives the forward)."""
    from flocoder_b200 import _lib
    eng = _lib.Engine(dim=m.dim, channels=m.channels, dim_mults=m.dim_mults, groups=m.groups, n_classes=m.n_classes,
                      height=x.shape[2], width=x.shape[3], compute_dtype=m._resolved_compute_dtype(),
                      device=x.device, state_dict=m.state_dict(), flags=_lib.FLO_FLAG_NO_BUFFER_REUSE | m.engine_flags)
    eng.forward(x.float().contiguous(), t.float().contiguous(), class_ids)
    torch.cuda.synchronize()
    out = {}
    for name in names:
        try:
            out[name] = eng.read_activation(name, x.shape[0])
        except ValueError:
            continue
    eng.close()
    return out


def _layer_report(m, sd, spec, x, t, prec, names=None):
    """Per-op rel-L2 of the CUDA activations vs the oracle trace (needs FLO_FLAG_NO_BUFFER_REUSE)."""
    trace = {}
    with torch.no_grad():
        unet_forward(sd, spec, x.cpu(), t.cpu(), None, prec, trace)
    acts = _stage_activations(m, x, t, [name for name, ref in trace.items() if ref.dim() == 4])
    return [(name, rel_l2(acts[name], ref)) for name, ref in trace.items() if name in acts]


def test_fp32_per_layer_activations(goldens):
    g = goldens["midi_vqgan"]
    m = gpu_model(0, "fp32")
    _, sd = seeded_state_dict(0)
    rows = _layer_report(m, sd, spec_for(0), g["x0"].cuda(), g["fwd_t"].cuda(), FP32)
    assert len(rows) > 60
    worst = max(rows, key=lambda r: r[1])
    for name, e in rows:
        print(f"{name:40s} {e:.3e}")
    assert worst[1] <= 1e-5, worst


def _teacher_forced(m, trace):
    worst = 0.0
    for x_stage, t_stage, v_ref in trace:
        t_vec = torch.full((SHAPE[0],), float(t_stage)) * 999
        worst = max(worst, rel_l2(m(x_stage.cuda(), t_vec.cuda()), v_ref))
    return worst


@pytest.mark.parametrize("n_classes", [102, 0])
def test_fp16_teacher_forced_velocity_vs_fp32_reference(goldens, n_classes):
    """Per-step velocity bar (<= 2e-3) for the 16-bit tensor-core path, against the fp32 oracle itself: every stage
    input (y_stage, t_stage) of an fp32 RK4 trajectory is fed to the CUDA forward (isolates per-forward error
    from trajectory drift)."""
    g = goldens["flowers_sd" if n_classes else "midi_vqgan"]
    m = gpu_model(n_classes, "fp16")
    _, sd = seeded_state_dict(n_classes)
    trace = []
    oracle.generate_latents_rk4(OracleModel(sd, spec_for(n_classes), FP32), SHAPE, n_steps=6, source=g["x0"].clone(), trace=trace)
    assert len(trace) == 20
    worst = _teacher_forced(m, trace)
    print("fp16 worst per-step velocity rel-L2 vs fp32 oracle:", worst)
    assert worst <= BF16_STEP_TOL


def test_bf16_rounding_noise_floor():
    """Why bf16 has no meaningful per-step bar below ~3e-3: the bf16-emulating oracle is itself that sensitive."""
    _, sd = seeded_state_dict(0)
    x = torch.randn(8, 4, 16, 16, generator=torch.Generator().manual_seed(5678))
    t = torch.full((8,), 249.75)
    with torch.no_grad():
        a = unet_forward(sd, spec_for(0), x, t, prec=BF16_MATCHED)
        b = unet_forward(sd, spec_for(0), x * (1 + 1e-7 * torch.randn(x.shape, generator=torch.Generator().manual_seed(1))), t,
                         prec=BF16_MATCHED)
        f = unet_forward(sd, spec_for(0), x, t, prec=FP32)
    assert rel_l2(b, a) > 1e-3          # a 1e-7 perturbation moves the matched oracle by ~3e-3
    assert 3e-3 < rel_l2(a, f) < 8e-3   # format floor of bf16 GEMM operands (SURVEY.md 8c: 4.9e-3)


@pytest.mark.parametrize("layerwise", [False, True])
@pytest.mark.parametrize("n_classes", [102, 0])
def test_bf16_velocity_error_is_at_the_format_floor(goldens, n_classes, layerwise):
    """bf16: the CUDA path's per-step error vs fp32 must not exceed the error the bf16 *format* itself causes
    (the bf16-emulating oracle vs fp32) by more than 35 %."""
    g = goldens["flowers_sd" if n_classes else "midi_vqgan"]
    m = gpu_model(n_classes, "bf16", layerwise)
    _, sd = seeded_state_dict(n_classes)
    trace = []
    oracle.generate_latents_rk4(OracleModel(sd, spec_for(n_classes), FP32), SHAPE, n_steps=4, source=g["x0"].clone(), trace=trace)
    emul = OracleModel(sd, spec_for(n_classes), BF16_MATCHED if layerwise else FUSED_BF16)
    for x_stage, t_stage, v_ref in trace[::3]:
        t_vec = torch.full((SHAPE[0],), float(t_stage)) * 999
        e_cuda = rel_l2(m(x_stage.cuda(), t_vec.cuda()), v_ref)
        e_fmt = rel_l2(emul(x_stage, t_vec), v_ref)
        print(f"t={float(t_stage):.3f} cuda {e_cuda:.3e} format floor {e_fmt:.3e}")
        assert e_cuda <= 1.35 * e_fmt + 2e-4


@pytest.mark.parametrize("compute_dtype,layerwise", [("bf16", False), ("bf16", True), ("fp16", False)])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_16bit_final_latent_vs_fp32_reference(goldens, name, compute_dtype, layerwise):
    from flocoder_b200 import sampling
    g = goldens[name]
    m = gpu_model(g["n_classes"], compute_dtype, layerwise)
    x1, _ = sampling.generate_latents_rk4(m, SHAPE, n_steps=50, source=g["x0"].cuda())
    e = rel_l2(x1, g["rk4_50"])
    print(name, compute_dtype, "RK4-50 final latent rel-L2 vs fp32 reference:", e)
    assert e <= BF16_FINAL_TOL
    x1, _ = sampling.euler_sampler(m, SHAPE, 10, source=g["x0"].cuda())
    assert rel_l2(x1, g["euler_10"]) <= BF16_FINAL_TOL
    if g["n_classes"] > 0:
        x1, _ = sampling.generate_latents_rk4(m, SHAPE, n_steps=10, cond={"class_cond": g["cls"].cuda()}, cfg_strength=3.0,
                                              source=g["x0"].cuda())
        assert rel_l2(x1, g["rk4_10_cfg3"]) <= BF16_FINAL_TOL


@pytest.mark.parametrize("compute_dtype,prec,tol", [("bf16", FUSED_BF16, 3e-2), ("fp16", FUSED_FP16, 4e-3)])
def test_fused_per_stage_tensors_vs_emulating_oracle(goldens, compute_dtype, prec, tol):
    """Every stage-boundary tensor of the fused path (and, in debug mode, every ResnetBlock output) against the
    oracle that rounds at the same points; the first block must agree to accumulation-order / MUFU-approximation
    noise (a handful of flipped 16-bit roundings: ex2.approx + rcp.approx in the kernel's SiLU vs exact in the oracle)."""
    g = goldens["midi_vqgan"]
    m = gpu_model(0, compute_dtype)
    _, sd = seeded_state_dict(0)
    rows = dict(_layer_report(m, sd, spec_for(0), g["x0"].cuda(), g["fwd_t"].cuda(), prec))
    assert len(rows) > 40
    for name, e in rows.items():
        print(f"{name:40s} {e:.3e}")
    assert rows["init_conv"] <= 1e-6 and rows["downs.0.0"] <= (5e-4 if compute_dtype == "bf16" else 1e-4)
    worst = max(rows.items(), key=lambda r: r[1])
    assert worst[1] <= tol, worst


def test_layerwise_bf16_per_layer_activations_vs_matched_oracle(goldens):
    g = goldens["midi_vqgan"]
    m = gpu_model(0, "bf16", layerwise=True)
    _, sd = seeded_state_dict(0)
    rows = _layer_report(m, sd, spec_for(0), g["x0"].cuda(), g["fwd_t"].cuda(), BF16_MATCHED)
    worst = max(rows, key=lambda r: r[1])
    assert worst[1] <= 1e-2, worst       # bf16 storage of the compared tensor itself is ~2e-3


@pytest.mark.parametrize("compute_dtype", ["fp32", "bf16", "fp16"])
def test_batch_slices_are_independent_and_deterministic(compute_dtype):
    """Size-independent properties at a BASELINE-sized batch: a B=256 trajectory equals the trajectories of
    its slices (what batch sharding across GPUs relies on) and repeats bit-for-bit."""
    from flocoder_b200 import sampling
    m = gpu_model(0, compute_dtype)
    B = 256
    x0 = torch.randn(B, 4, 16, 16, generator=torch.Generator().manual_seed(5678)).cuda()
    full, _ = sampling.generate_latents_rk4(m, (B, 4, 16, 16), n_steps=5, source=x0)
    again, _ = sampling.generate_latents_rk4(m, (B, 4, 16, 16), n_steps=5, source=x0)
    assert torch.equal(full, again)
    assert torch.isfinite(full).all()
    # Slices that start on a multiple of every stage's samples-per-CTA (lcm = 96) see the same tiling -> bit-identical.
    # Other slices group samples differently inside a CTA, which only changes fp32 summation order (1e-7); on the
    # 16-bit paths that can flip roundings, so the bound there is the format's noise, not 1e-6.
    part, _ = sampling.generate_latents_rk4(m, (96, 4, 16, 16), n_steps=5, source=x0[96:192])
    assert torch.equal(part, full[96:192])
    tol = {"fp32": 1e-6, "fp16": 5e-4, "bf16": 4e-3}[compute_dtype]
    for lo, hi in ((0, 8), (100, 131), (248, 256)):
        part, _ = sampling.generate_latents_rk4(m, (hi - lo, 4, 16, 16), n_steps=5, source=x0[lo:hi])
        assert rel_l2(part, full[lo:hi]) <= tol


def test_generic_rk4_step_composes_with_our_forward(goldens):
    """rk4_step / v_func_cfg keep the reference semantics for an arbitrary f: composing them over
    Unet.forward must agree with the fused flo_integrate trajectory."""
    from flocoder_b200 import sampling
    g = goldens["stl_sd"]
    m = gpu_model(10, "fp32")
    x0 = g["x0"].cuda()
    ts = sampling.time_grid(6, device="cuda")
    t_vec = torch.zeros(8, device="cuda")
    cond = {"class_cond": g["cls"].cuda()}
    y = x0.clone()
    for i in range(len(ts) - 1):
        y = sampling.rk4_step(lambda x, t: sampling.v_func_cfg(m, cond, 2.0, t_vec, x, t), y, ts[i], ts[i + 1] - ts[i])
    fused, _ = sampling.generate_latents_rk4(m, SHAPE, n_steps=6, cond=cond, cfg_strength=2.0, source=x0)
    assert rel_l2(fused, y) <= 2e-6


def test_host_buffer_entry_point(goldens):
    from flocoder_b200 import _lib, sampling
    g = goldens["midi_vqgan"]
    m = gpu_model(0, "fp32")
    eng = m.engine(16, 16)
    x0 = g["x0"].clone().pin_memory()
    x1 = torch.empty_like(x0).pin_memory()
    ts = sampling.time_grid(10).tolist()
    eng.integrate_host(x0, x1, ts, _lib.FLO_RK4)
    assert rel_l2(x1, g["rk4_10"]) <= FP32_FINAL_TOL


def test_bf16_param_dtype_follows_module(goldens):
    """model.to(bfloat16): bf16 parameters -> bf16 compute path, bf16 in / bf16 out at the boundary."""
    from flocoder_b200.unet import Unet
    g = goldens["midi_vqgan"]
    torch.manual_seed(1234)
    m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0).cuda().to(torch.bfloat16)
    v = m(g["x0"].cuda().to(torch.bfloat16), g["fwd_t"].cuda())
    assert v.dtype == torch.bfloat16
    assert rel_l2(v.float(), g["fwd_v"]) <= 3e-2          # weights themselves are bf16-rounded here


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 7, 13, 100, 300, 600])
def test_ragged_and_large_batches_fused_vs_fp32_path(B):
    """Batch sizes that leave the last CTA / cluster group partly empty (1, 7, 13, 100) and sizes that select the other
    N-split variants of the low-resolution stages (up to the 32-36 clusters of 4 the GPCs hold, i.e. B <= 256..288: clusters of 4; 300: clusters of 2; 600: no split).  The
    fp16 fused path must stay within the per-step bar of the fp32 CUDA path (itself pinned to the reference above),
    per sample, and a class-conditional CFG trajectory must stay within the final-latent bar."""
    from flocoder_b200 import sampling
    m16 = gpu_model(102, "fp16")
    m32 = gpu_model(102, "fp32")
    gen = torch.Generator().manual_seed(4242 + B)
    x = torch.randn(B, 4, 16, 16, generator=gen).cuda()
    t = (torch.rand(B, generator=gen) * 999).cuda()                      # per-sample times: per-sample FiLM rows
    cls = torch.randint(0, 102, (B,), generator=gen).cuda()
    for cond in (None, {"class_cond": cls}):
        v16 = m16(x, t, cond).float()
        v32 = m32(x, t, cond).float()
        per_sample = (v16 - v32).flatten(1).norm(dim=1) / v32.flatten(1).norm(dim=1)
        assert torch.isfinite(v16).all()
        assert float(per_sample.max()) <= 3e-3, (B, float(per_sample.max()))     # worst single sample
        assert rel_l2(v16, v32) <= 2e-3
    if B <= 100:
        x16, _ = sampling.generate_latents_rk4(m16, (B, 4, 16, 16), n_steps=6, cond={"class_cond": cls}, cfg_strength=3.0, source=x)
        x32, _ = sampling.generate_latents_rk4(m32, (B, 4, 16, 16), n_steps=6, cond={"class_cond": cls}, cfg_strength=3.0, source=x)
        assert rel_l2(x16, x32) <= BF16_FINAL_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("dim,mults,hw,ncls", [(16, [1, 2, 4], 16, 10), (32, [1, 2, 4], 16, 0), (16, [1, 2, 4], 8, 0),
                                               (16, [1, 1, 2, 2], 16, 0)])
def test_other_unet_shapes_fused_vs_fp32_path(dim, mults, hw, ncls):
    """U-Nets other than the three BASELINE configurations (other widths, depths, latent sizes) go through the same
    planner: the fp16 fused path must agree with the fp32 CUDA path within the per-step bar."""
    from flocoder_b200.unet import Unet
    torch.manual_seed(7)
    m32 = Unet(dim=dim, channels=4, dim_mults=mults, n_classes=ncls, compute_dtype="fp32").cuda().eval()
    m16 = Unet(dim=dim, channels=4, dim_mults=mults, n_classes=ncls, compute_dtype="fp16").cuda().eval()
    m16.load_state_dict(m32.state_dict())
    x = torch.randn(5, 4, hw, hw).cuda()
    t = torch.rand(5).cuda() * 999
    assert rel_l2(m16(x, t), m32(x, t).cpu()) <= 2e-3


@pytest.mark.gpu
@pytest.mark.parametrize("dim,mults,hw,dtype", [(16, [1, 2, 4, 8], 32, "fp16"), (32, [1, 2, 4, 8], 16, "fp16"), (72, [1, 2], 16, "fp32")])
def test_unsupported_shapes_fail_loudly(dim, mults, hw, dtype):
    """Outside the supported envelope (DESIGN.md section 10) the library refuses at plan time; it never falls back."""
    from flocoder_b200.unet import Unet
    m = Unet(dim=dim, channels=4, dim_mults=mults, n_classes=0, compute_dtype=dtype).cuda().eval()
    with pytest.raises(NotImplementedError):
        m(torch.randn(2, 4, hw, hw).cuda(), torch.rand(2).cuda() * 999)


@pytest.mark.gpu
@pytest.mark.parametrize("dim,channels,mults,hw", [(32, 3, [1, 2, 4, 8], 32), (64, 4, [1, 2], 16)])
def test_fp32_path_large_latents_and_groupnorm_units_vs_oracle(dim, channels, mults, hw):
    """The fp32 path beyond the 16-bit envelope: configs/flowers_resize.yaml (3 x 32 x 32 "latents", Unet(dim=32): 1024 pixels ->
    tiled linear attention, GroupNorm(1, 32) over 32768 elements -> the generic GroupNorm kernel) and dim = 64 at 16 x 16."""
    from flocoder_b200.unet import Unet
    torch.manual_seed(11)
    m = Unet(dim=dim, channels=channels, dim_mults=mults, n_classes=0, compute_dtype="fp32")
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.cuda().eval()
    spec = UnetSpec(dim=dim, dim_mults=tuple(mults), channels=channels, groups=4, n_classes=0)
    gen = torch.Generator().manual_seed(12)
    x = torch.randn(3, channels, hw, hw, generator=gen)
    t = torch.rand(3, generator=gen) * 999
    with torch.no_grad():
        want = unet_forward(sd, spec, x, t)
    assert rel_l2(m(x.cuda(), t.cuda()), want) <= FP32_STEP_TOL


@pytest.mark.gpu
def test_sampler_with_our_unet_and_a_codec(goldens):
    """sampler() (sampling.py:187-229) end to end on the GPU: class-conditional CFG trajectory through flo_integrate, then
    the chunked decode through a caller-supplied codec."""
    from torch import nn
    from flocoder_b200 import sampling

    class Codec(nn.Module):
        def __init__(self):
            super().__init__()
            self.dec = nn.Conv2d(4, 3, 1)

        def decode(self, z):
            return torch.sigmoid(self.dec(z))

    g = goldens["flowers_sd"]
    m = gpu_model(102, "fp32")
    codec = Codec().cuda().eval()
    lat, img, nfe = sampling.sampler(m, codec, method="rk4", batch_size=8, n_steps=10, cond={"class_cond": g["cls"].cuda()},
                                     n_classes=102, cfg_strength=3.0, source=g["x0"].cuda())
    assert nfe == 40 and img.shape == (8, 3, 16, 16) and img.device.type == "cuda"
    assert rel_l2(lat, g["rk4_10_cfg3"]) <= 1e-5
    with torch.no_grad():
        assert torch.allclose(img, codec.decode(lat), atol=1e-6)


@pytest.mark.gpu
def test_stl_sd_euler_100_steps_batch_512():
    """BASELINE configs[4] per-GPU shape: stl_sd U-Net (n_classes=10), legacy Euler with 100 steps, 512 samples per GPU.
    The fp16 fused trajectory (100 graph-chained evaluations) stays within the final-latent bar of the fp32 CUDA path, and
    repeats bit-for-bit."""
    from flocoder_b200 import sampling
    m16, m32 = gpu_model(10, "fp16"), gpu_model(10, "fp32")
    x0 = torch.randn(512, 4, 16, 16, generator=torch.Generator().manual_seed(99)).cuda()
    a, nfe = sampling.euler_sampler(m16, (512, 4, 16, 16), 100, source=x0)
    b, _ = sampling.euler_sampler(m16, (512, 4, 16, 16), 100, source=x0)
    assert nfe == 100 and torch.equal(a, b)
    ref, _ = sampling.euler_sampler(m32, (512, 4, 16, 16), 100, source=x0[:64])
    assert rel_l2(a[:64], ref.cpu()) <= BF16_FINAL_TOL


@pytest.mark.gpu
def test_midi_vqgan_rk4_50_steps_batch_1024():
    """BASELINE configs[2] at full size: midi_vqgan-shaped U-Net (n_classes=0, inpainting off), RK4 n_steps=50, 1024
    samples on one GPU (the unsplit variant of the low-resolution stages).  Size-independent properties: the run repeats
    bit-for-bit, every sample is finite, and the first 32 samples stay within the final-latent bar of the fp32 CUDA path
    (itself pinned to the reference) integrating only that slice - samples never see each other (SURVEY 8e)."""
    from flocoder_b200 import sampling
    m16, m32 = gpu_model(0, "fp16"), gpu_model(0, "fp32")
    shape = (1024, 4, 16, 16)
    x0 = torch.randn(*shape, generator=torch.Generator().manual_seed(1024)).cuda()
    a, nfe = sampling.generate_latents_rk4(m16, shape, n_steps=50, source=x0)
    b, _ = sampling.generate_latents_rk4(m16, shape, n_steps=50, source=x0)
    assert nfe == 200 and a.shape == shape and torch.isfinite(a).all() and torch.equal(a, b)
    ref, _ = sampling.generate_latents_rk4(m32, (32, 4, 16, 16), n_steps=50, source=x0[:32])
    assert rel_l2(a[:32], ref.cpu()) <= BF16_FINAL_TOL


@pytest.mark.gpu
def test_groupnorm_pass_kernel_variants_agree(monkeypatch):
    """The standalone GroupNorm+FiLM+SiLU pass of the layer-wise path has three kernels chosen by unit size (k_gn_tma: bulk-copy
    staged warp teams; k_gn_warp: register-resident warp teams; k_gn: one CTA per unit).  Forced through each of them (the
    developer switches of DESIGN.md 5.2, read when a plan is captured), one forward of a ragged batch must agree: to fp32
    rounding in the fp32 mode (same formula, different summation order), and to the bf16 format floor in the bf16 mode
    (whose 16-bit variant also uses a one-pass variance and a MUFU SiLU in the staged / warp kernels).
    Default-init GroupNorms have gamma = 1, beta = 0, so the same forwards run again with oracle.trained_like weights, and each
    variant is also held against the fp64 oracle: <= 1e-5 in fp32, within 1.35x the bf16-emulating oracle's error + 2e-4 in bf16
    (the layer-wise rule of test_bf16_velocity_error_is_at_the_format_floor)."""
    from flocoder_b200 import _lib
    from flocoder_b200.unet import Unet
    from oracle.unet_oracle import trained_like
    gen = torch.Generator().manual_seed(77)
    x = torch.randn(37, 4, 16, 16, generator=gen).cuda()
    t = (torch.rand(37, generator=gen) * 999).cuda()
    torch.manual_seed(1234)
    sd0 = {k: v.detach().clone() for k, v in Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0).state_dict().items()}
    for weights, sd in (("default", sd0), ("trained_like", trained_like(sd0))):
        outs = {}
        for tag, env in (("tma", {}), ("warp", {"FLO_GN_NO_TMA": "1"}), ("cta", {"FLO_GN_CTA": "1"})):
            for k in ("FLO_GN_NO_TMA", "FLO_GN_CTA"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            for cd in ("fp32", "bf16"):
                m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, compute_dtype=cd)
                m.load_state_dict(sd)
                m.engine_flags = _lib.FLO_FLAG_LAYERWISE
                outs[tag, cd] = m.cuda().eval()(x, t).float().cpu()
                assert torch.isfinite(outs[tag, cd]).all()
        for tag in ("warp", "cta"):
            assert rel_l2(outs[tag, "fp32"], outs["tma", "fp32"]) <= 1e-5, (weights, tag)
            assert rel_l2(outs[tag, "bf16"], outs["tma", "bf16"]) <= 1.5e-2, (weights, tag)
        assert rel_l2(outs["tma", "bf16"], outs["tma", "fp32"]) <= 1.5e-2, weights
        with torch.no_grad():
            want = unet_forward({k: v.double() for k, v in sd.items()}, spec_for(0), x.cpu().double(), t.cpu().double())
            e_fmt = rel_l2(unet_forward(sd, spec_for(0), x.cpu(), t.cpu(), prec=BF16_MATCHED), want)
        for tag in ("tma", "warp", "cta"):
            e32, e16 = rel_l2(outs[tag, "fp32"], want), rel_l2(outs[tag, "bf16"], want)
            print(f"{weights:12s} {tag:4s} fp32 {e32:.3e} bf16 {e16:.3e} (format {e_fmt:.3e})")
            assert e32 <= 1e-5, (weights, tag, e32)
            assert e16 <= 1.35 * e_fmt + 2e-4, (weights, tag, e16, e_fmt)
