"""Per-sample RK45 on the device (``flo_integrate_rk45_per_sample``) against scipy's RK45 driving the fp64 oracle on each
sample alone, the B = 1 identity with the batched mode, the 16-bit and layer-wise paths against the fp32 path, batch
invariance, handle state, and the sharded sampler over NCCL.

* fp32 path: each sample's final latent within 1e-5 + 4 e32_i of the fp64 oracle's, e32_i being that sample's distance of
  the same oracle run with fp32 weights and velocities; at the loose tolerance 1e-3, within the tolerance itself.  There a
  lone sample takes 5 or 6 steps, its step sizes follow error norms that are differences of seven velocities, and the fp32
  path's velocity error (up to 1e-5 per forward, against 1e-7 for the CPU fp32 oracle) moves them enough to put a
  midi_vqgan sample 3.9e-4 from fp64 with the oracle's exact counts, where e32 is 5.8e-6.  Its (nfev, attempts) equal the oracle's where every fp64 error norm
  of that sample is clear of 1 by max(1e-3, 10 |n64 - n32|) and both oracles agree on the counts (the rule of
  test_gpu_rk45.py, per sample).
* fp16 / bf16 fused paths (both CFG routes) and the layer-wise flag: the batch within rel-L2 1e-2 of the fp32 path's
  per-sample run (the bar of the batched mode's test), every sample within 5e-2, and repeat runs bit-identical.  Measured
  on a B200, the worst single samples are 1.4e-2 in bf16 and 2.8e-2 with guidance 3 (CFG scales velocity errors by 1 + cfg),
  while most samples sit near 1e-3."""
import os
import socket
import sys

import pytest
import torch

from oracle.unet_oracle import OracleModel, UnetSpec, trained_like
from conftest import CONFIGS, GOLDEN_DIR, rel_l2, seeded_state_dict
from rk45_oracle import rk45_solve

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_FINAL_TOL = 1e-2          # final-latent bar of the 16-bit operand paths over the batch
BF16_SAMPLE_TOL = 5e-2         # ... and for the worst single sample
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
    """Seeded noise with a per-sample scale from 0.5 to 1.5, so samples differ in how hard they are to integrate."""
    x = torch.randn(b, 4, 16, 16, generator=torch.Generator().manual_seed(seed))
    return x * torch.linspace(0.5, 1.5, b)[:, None, None, None] if b > 1 else x


def sample_cond(cond, i):
    if cond is None:
        return None
    return {k: (v[i:i + 1] if torch.is_tensor(v) else v) for k, v in cond.items()}


def oracle_per_sample(sd, spec, y0, t0, tol, cond=None, cfg=0.0):
    """For every sample alone: (fp64 latent, fp32-oracle distance e32, nfev, attempts, counts robust)."""
    m64 = OracleModel({k: v.double() for k, v in sd.items()}, spec)
    m32 = OracleModel({k: v.float() for k, v in sd.items()}, spec)
    out = []
    for i in range(y0.shape[0]):
        c = sample_cond(cond, i)
        want, nfev, _, norms = rk45_solve(m64, y0[i:i + 1].double(), t0, 1.0, cond=c, cfg_strength=cfg, rtol=tol, atol=tol)
        y32, nfev32, _, norms32 = rk45_solve(m32, y0[i:i + 1].float(), t0, 1.0, cond=c, cfg_strength=cfg, rtol=tol, atol=tol)
        robust = nfev32 == nfev and len(norms32) == len(norms) and all(
            abs(a - 1.0) >= max(NORM_MARGIN, 10 * abs(a - b)) for a, b in zip(norms, norms32))
        out.append((want[0], rel_l2(y32, want), nfev, len(norms), robust))
    return out


def run_per_sample(m, x0, cond=None, cfg=0.0, init=None, init_strength=0.0, tol=1e-5):
    """(latents on the CPU, per-sample nfe [B]) of the public sampler with ``per_sample=True``."""
    from flocoder_b200 import sampling
    cond_d = None if cond is None else {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in cond.items()}
    got, nfe = sampling.generate_latents_rk45(m, tuple(x0.shape), cond=cond_d, cfg_strength=cfg, source=x0.cuda(),
                                              init_latents=None if init is None else init.cuda(),
                                              init_strength=init_strength, rtol=tol, atol=tol, per_sample=True)
    assert nfe.dtype == torch.int64 and nfe.device.type == "cpu" and nfe.shape == (x0.shape[0],)
    return got.cpu(), nfe


def check_vs_oracle(m, sd, spec, x0, t0, tol, cond=None, cfg=0.0, init=None, init_strength=0.0):
    """Returns the oracle's per-sample nfev and how many samples had their counts claimed."""
    y0 = x0.double() if init is None else (1 - init_strength) * x0.double() + init_strength * init.double()
    ref = oracle_per_sample(sd, spec, y0, t0, tol, cond, cfg)
    got, nfe = run_per_sample(m, x0, cond, cfg, init, init_strength, tol)
    claimed = 0
    for i, (want, e32, nfev, attempts, robust) in enumerate(ref):
        e = rel_l2(got[i], want)
        print(f"sample {i}: nfe {int(nfe[i])} (oracle {nfev} / {attempts} attempts), counts claimed: {robust}, "
              f"final rel-L2 {e:.2e} (fp32 oracle {e32:.2e})")
        if robust:
            assert int(nfe[i]) == nfev, f"sample {i}: device nfe {int(nfe[i])}, oracle {nfev}"
            assert (nfev - 2) // 6 == attempts
            claimed += 1
        bar = FP32_TOL + 4 * e32 if tol <= 1e-5 else max(FP32_TOL + 4 * e32, tol)
        assert e <= bar, f"sample {i}: final latents rel-L2 {e:.2e}, fp32 floor {e32:.2e}"
    if claimed == len(ref):                           # the batch runs until its slowest sample is done
        assert m.engine(16, 16).rk45_timing()[0] == max(r[3] for r in ref)
    return [r[2] for r in ref], claimed


# ---------------------------------------------------------------------------------------------------------------------
# fp32 path against scipy + the fp64 oracle, sample by sample
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tol", [1e-5, 1e-3])
@pytest.mark.parametrize("trained", [False, True])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_fp32_per_sample_matches_scipy_on_each_sample(name, trained, tol):
    n_classes = CONFIGS[name]
    b = 3 if name == "flowers_sd" else 2          # the oracle runs every sample alone, twice, on the CPU
    m = cuda_model(n_classes, "fp32", trained)
    nfevs, claimed = check_vs_oracle(m, state_dict(n_classes, trained), spec_for(n_classes), noise(b, 30 + n_classes),
                                     0.0, tol)
    if name == "flowers_sd" and trained and tol == 1e-5:
        assert len(set(nfevs)) > 1, f"the samples of this case need different nfev (oracle: {nfevs})"
        assert claimed > 0


def test_fp32_per_sample_class_conditioning_with_cfg():
    m = cuda_model(10, "fp32")
    cls = torch.tensor([3, 9])
    check_vs_oracle(m, state_dict(10, True), spec_for(10), noise(2, 11), 0.0, 1e-5, cond={"class_cond": cls}, cfg=3.0)


def test_fp32_per_sample_from_init_latents():
    from flocoder_b200 import sampling
    m = cuda_model(0, "fp32")
    t0 = float(sampling.warp_time(torch.tensor(0.3)))
    check_vs_oracle(m, state_dict(0, True), spec_for(0), noise(2, 12), t0, 1e-5, init=noise(2, 13), init_strength=0.3)


def test_fp32_per_sample_inpainting_with_a_soft_mask():
    from flocoder_b200.unet import Unet
    g = torch.load(os.path.join(GOLDEN_DIR, "inpaint_16.pt"), weights_only=False)
    torch.manual_seed(g["model_seed"])
    m = Unet(dim=g["dim"], channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True, compute_dtype="fp32")
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    m = m.cuda().eval()
    b = 2
    ramp = torch.linspace(-3, 3, 16)
    mask = torch.sigmoid(ramp[None, None, :, None] + ramp[None, None, None, :] * 0.5).expand(b, 4, 16, 16).contiguous()
    mask = mask * torch.tensor([1.0, 0.4])[:, None, None, None]             # a different mask per sample
    check_vs_oracle(m, sd, spec_for(0, g["dim"]), noise(b, 14), 0.0, 1e-5, cond={"mask_cond": mask})


# ---------------------------------------------------------------------------------------------------------------------
# B = 1: the per-sample mode is the batched mode
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("compute_dtype", ["fp32", "fp16"])
def test_b1_per_sample_equals_batched(compute_dtype):
    from flocoder_b200 import sampling
    m = cuda_model(102, compute_dtype)
    x0 = noise(1, 40).cuda()
    want, nfe = sampling.generate_latents_rk45(m, (1, 4, 16, 16), source=x0)
    attempts = m.engine(16, 16).rk45_timing()[0]
    got, nfe_ps = sampling.generate_latents_rk45(m, (1, 4, 16, 16), source=x0, per_sample=True)
    assert torch.equal(got, want)
    assert int(nfe_ps[0]) == nfe and m.engine(16, 16).rk45_timing()[0] == attempts
    counts = m.engine(16, 16).integrate_rk45_per_sample(x0.clone(), 0.0)
    assert int(counts[0, 0]) == nfe and int(counts[0, 1] + counts[0, 2]) == attempts


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit paths against the fp32 path, sample by sample
# ---------------------------------------------------------------------------------------------------------------------
_fp32_cache = {}


def fp32_per_sample(b, seed, cls=None, cfg=0.0):
    key = (b, seed, cls is not None, cfg)
    if key not in _fp32_cache:
        m = cuda_model(102, "fp32")
        _fp32_cache[key] = run_per_sample(m, noise(b, seed), None if cls is None else {"class_cond": cls}, cfg)
    return _fp32_cache[key]


def check16(m, b, seed, cls=None, cfg=0.0, what=""):
    got, nfe = run_per_sample(m, noise(b, seed), None if cls is None else {"class_cond": cls}, cfg)
    want, nfe32 = fp32_per_sample(b, seed, cls, cfg)
    errs = torch.tensor([rel_l2(got[i], want[i]) for i in range(b)])
    print(f"{what}: nfe min/median/max {int(nfe.min())}/{int(nfe.median())}/{int(nfe.max())} (fp32 path "
          f"{int(nfe32.min())}/{int(nfe32.median())}/{int(nfe32.max())}), batch rel-L2 {rel_l2(got, want):.2e}, "
          f"worst sample {float(errs.max()):.2e}, median sample {float(errs.median()):.2e}")
    assert rel_l2(got, want) <= BF16_FINAL_TOL
    assert float(errs.max()) <= BF16_SAMPLE_TOL, f"sample {int(errs.argmax())}: rel-L2 {float(errs.max()):.2e}"
    again, nfe2 = run_per_sample(m, noise(b, seed), None if cls is None else {"class_cond": cls}, cfg)
    assert torch.equal(nfe2, nfe) and torch.equal(again, got)


@pytest.mark.parametrize("B", [37, 300])
@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_per_sample_vs_fp32_path(compute_dtype, B):
    check16(cuda_model(102, compute_dtype), B, B, what=f"{compute_dtype} B={B}")


@pytest.mark.parametrize("two_pass", [False, True])
@pytest.mark.parametrize("compute_dtype", ["fp16", "bf16"])
def test_fused_per_sample_cfg_routes(compute_dtype, two_pass, monkeypatch):
    """B=150: guidance as one 300-sample forward (SF_CFG_2B), or the conditional + combining two-pass route (forced with
    FLO_CFG_TWO_PASS)."""
    if two_pass:
        monkeypatch.setenv("FLO_CFG_TWO_PASS", "1")
    B = 150
    check16(cuda_model(102, compute_dtype), B, 21, torch.arange(B) % 102, 3.0, what=f"{compute_dtype} cfg two_pass={two_pass}")


def test_layerwise_per_sample_vs_fp32_path():
    from flocoder_b200 import _lib
    check16(cuda_model(102, "bf16", flags=_lib.FLO_FLAG_LAYERWISE), 37, 37, what="bf16 layer-wise B=37")


# ---------------------------------------------------------------------------------------------------------------------
# batch invariance and handle state
# ---------------------------------------------------------------------------------------------------------------------
def test_permuted_batch_gives_the_permuted_result():
    sd, spec = state_dict(102, True), spec_for(102)
    x0 = noise(4, 50)
    ref = oracle_per_sample(sd, spec, x0.double(), 0.0, 1e-3)
    m = cuda_model(102, "fp32")
    got, nfe = run_per_sample(m, x0, tol=1e-3)
    perm = torch.tensor([2, 0, 3, 1])
    pgot, pnfe = run_per_sample(m, x0[perm], tol=1e-3)
    d = float((pgot - got[perm]).abs().max())
    print(f"max |permuted - unpermuted| {d:.2e}, nfe {nfe.tolist()}, oracle {[r[2] for r in ref]}")
    assert d <= 2e-6
    for j, i in enumerate(perm.tolist()):
        if ref[i][4]:
            assert int(pnfe[j]) == int(nfe[i]) == ref[i][2]


@pytest.mark.parametrize("compute_dtype, cfg", [("bf16", 0.0), ("fp16", 3.0), ("fp32", 3.0)])
def test_per_sample_run_leaves_the_handle_unchanged(compute_dtype, cfg):
    """batched RK45 -> per-sample RK45 -> batched RK45 -> RK4 on one handle: every run equals the same run on a fresh handle."""
    from flocoder_b200 import sampling
    B = 37
    cond = {"class_cond": (torch.arange(B) % 102).cuda()} if cfg else None
    x0 = noise(B, 5).cuda()
    kw = dict(cond=cond, cfg_strength=cfg, source=x0, rtol=1e-3, atol=1e-3)
    fresh = {}
    for what in ("batched", "per_sample", "rk4"):
        m = cuda_model(102, compute_dtype)
        if what == "rk4":
            fresh[what] = sampling.generate_latents_rk4(m, (B, 4, 16, 16), n_steps=6, cond=cond, cfg_strength=cfg, source=x0)
        else:
            fresh[what] = sampling.generate_latents_rk45(m, (B, 4, 16, 16), per_sample=what == "per_sample", **kw)
    m = cuda_model(102, compute_dtype)
    sampling.generate_latents_rk45(m, (B, 4, 16, 16), **kw)
    ps = sampling.generate_latents_rk45(m, (B, 4, 16, 16), per_sample=True, **kw)
    batched = sampling.generate_latents_rk45(m, (B, 4, 16, 16), **kw)
    rk4 = sampling.generate_latents_rk4(m, (B, 4, 16, 16), n_steps=6, cond=cond, cfg_strength=cfg, source=x0)
    assert torch.equal(ps[0], fresh["per_sample"][0]) and torch.equal(ps[1], fresh["per_sample"][1])
    assert torch.equal(batched[0], fresh["batched"][0]) and batched[1] == fresh["batched"][1]
    assert torch.equal(rk4[0], fresh["rk4"][0])


# ---------------------------------------------------------------------------------------------------------------------
# the sharded per-sample sampler over NCCL (two GPUs; skipped on a one-GPU box)
# ---------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, batch, out):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import torch.distributed as dist
    from flocoder_b200 import sampling
    from flocoder_b200.dist import generate_latents_sharded
    from flocoder_b200.unet import Unet
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(1234)
    m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=10, compute_dtype="fp32").to(dev).eval()
    x0 = noise(batch, 77)
    cond = {"class_cond": (torch.arange(batch) % 10).to(dev)}
    kw = dict(cond=cond, cfg_strength=2.0, sampler=sampling.generate_latents_rk45, per_sample=True, rtol=1e-4, atol=1e-4)
    full, nfe = generate_latents_sharded(m, (batch, 4, 16, 16), source=x0.to(dev), **kw)
    if rank == 0:
        ref, ref_nfe = sampling.generate_latents_rk45(m, (batch, 4, 16, 16), cond=cond, cfg_strength=2.0,
                                                      source=x0.to(dev), per_sample=True, rtol=1e-4, atol=1e-4)
        torch.save({"full": full.cpu(), "nfe": nfe, "ref": ref.cpu(), "ref_nfe": ref_nfe}, out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_per_sample_over_nccl_uneven_shards(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "nccl.pt")
    mp.spawn(_nccl_worker, args=(2, _free_port(), 9, out), nprocs=2, join=True)
    got = torch.load(out)
    assert float((got["full"] - got["ref"]).abs().max()) <= 2e-6
    assert torch.equal(got["nfe"], got["ref_nfe"])
