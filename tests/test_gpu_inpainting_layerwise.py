"""The inpainting U-Net (``Unet(mask_cond=True)``) on the layer-wise bf16 tcgen05 path (``compute_dtype="bf16"``,
``engine_flags = FLO_FLAG_LAYERWISE``): the 5x5 / 3x3 mask-fusion convolutions on k_conv_umma with their SiLU, residual,
unshuffled / upsampled copies and run-time bypass, and the 16-channel bf16 mask pyramid.

* forward: the final velocity and every mask op's activation within rel-L2 1e-2 of the bf16-matched oracle
  (``BF16_MATCHED``; 2e-2 with trained-like weights, see TRAINED_MATCHED_TOL), and against fp64 within 1.5x the matched
  oracle's own error + 1e-4;
* one handle switching between mask modes, 5x5 geometry off the 16x16 strip tiling, integrators and sharding."""
import os
import socket
import sys

import pytest
import torch

from oracle.unet_oracle import BF16_MATCHED, FP32, UnetSpec, trained_like, unet_forward
from conftest import GOLDEN_DIR, rel_l2

pytestmark = pytest.mark.gpu
BF16_FINAL_TOL = 1e-2      # final latent / velocity vs the reference on a 16-bit path
MATCHED_TOL = 1e-2         # per tensor vs the bf16-matched oracle (bf16 storage of the tensor itself is ~2e-3)
# With trained-like weights (sharp attention softmaxes) rounding flips grow through the bottleneck: without any mask the
# layer-wise path is already 1.1e-2 from the matched oracle at mid_attn (B200), and the mask ops after it inherit that.  The
# fp64 bound below (1.5x the matched oracle's own error) is what separates an implementation error from the format there.
TRAINED_MATCHED_TOL = 2e-2
MASK_OPS = ("mask_fusion_conv", "down_mask_fusions.0.0", "down_mask_fusions.1.0", "up_mask_fusions.0.0", "up_mask_fusions.1.0")
_cache = {}


def golden():
    if "g" not in _cache:
        _cache["g"] = torch.load(os.path.join(GOLDEN_DIR, "inpaint_16.pt"), weights_only=False)
    return _cache["g"]


def make_model(dim_mults=(1, 2, 4, 8), trained=True, compute_dtype="bf16", layerwise=True):
    """The inpaint_16 net (dim 16, seeded as the golden) with trained-like or default weights."""
    from flocoder_b200 import _lib
    from flocoder_b200.unet import Unet
    g = golden()
    torch.manual_seed(g["model_seed"])
    m = Unet(dim=g["dim"], channels=4, dim_mults=list(dim_mults), n_classes=0, mask_cond=True, compute_dtype=compute_dtype)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    if trained:
        sd = trained_like(sd)
        m.load_state_dict(sd)
    if layerwise:
        m.engine_flags = _lib.FLO_FLAG_LAYERWISE
    return m.cuda().eval(), sd, UnetSpec(dim=g["dim"], dim_mults=tuple(dim_mults), channels=4, groups=4, n_classes=0)


def make_mask(kind, b, h=16, w=16, seed=0):
    gen = torch.Generator().manual_seed(1000 + seed)
    soft = torch.sigmoid(4 * torch.randn(b, 4, h, w, generator=gen))
    if kind == "soft":
        return soft
    if kind == "ones":
        return torch.ones(b, 4, h, w)
    if kind == "half":                                  # half the samples all ones: the batch-wide bypass test fails
        soft[: b // 2] = 1.0
        return soft
    return None


def inputs(b, seed, h=16, w=16):
    gen = torch.Generator().manual_seed(seed)
    return torch.randn(b, 4, h, w, generator=gen), torch.rand(b, generator=gen) * 999


def cuda_activations(m, x, t, mask, names):
    """Final velocity and {name: activation} of one forward on a fresh handle that keeps every buffer."""
    from flocoder_b200 import _lib
    eng = _lib.Engine(dim=m.dim, channels=m.channels, dim_mults=m.dim_mults, groups=m.groups, n_classes=0,
                      height=x.shape[2], width=x.shape[3], compute_dtype="bf16", device=torch.device("cuda"),
                      state_dict=m.state_dict(), flags=_lib.FLO_FLAG_NO_BUFFER_REUSE | m.engine_flags, mask_cond=True)
    b = x.shape[0]
    eng.set_mask(None if mask is None else mask.cuda(), b)
    v = eng.forward(x.cuda().contiguous(), t.cuda().contiguous(), None)
    torch.cuda.synchronize()
    acts = {n: eng.read_activation(n, b) for n in names}
    eng.close()
    return v.cpu(), acts


def check_forward(m, sd, spec, x, t, mask, tol=TRAINED_MATCHED_TOL):
    cond = None if mask is None else {"mask_cond": mask}
    tr_bf, tr_64 = {}, {}
    with torch.no_grad():
        v_bf = unet_forward(sd, spec, x, t, cond, BF16_MATCHED, tr_bf)
        sd64 = {k: v.double() for k, v in sd.items()}
        cond64 = None if mask is None else {"mask_cond": mask.double()}
        v_64 = unet_forward(sd64, spec, x.double(), t.double(), cond64, FP32, tr_64)
    names = [n for n in MASK_OPS if n in tr_bf]
    v, acts = cuda_activations(m, x, t, mask, names)
    bad = []
    for name, got, want_bf, want_64 in [("velocity", v, v_bf, v_64)] + [(n, acts[n], tr_bf[n], tr_64[n]) for n in names]:
        e_bf, e_64, e_fmt = rel_l2(got, want_bf), rel_l2(got, want_64), rel_l2(want_bf, want_64)
        if not e_bf <= tol:
            bad.append(f"{name}: {e_bf:.3e} vs the matched oracle")
        if not e_64 <= 1.5 * e_fmt + 1e-4:
            bad.append(f"{name}: {e_64:.3e} vs fp64 > 1.5 x matched oracle {e_fmt:.3e} + 1e-4")
    return names, bad


@pytest.mark.parametrize("b", [5, 37, 300])
@pytest.mark.parametrize("kind", ["soft", "ones", "half", "none"])
def test_forward_vs_matched_oracle(kind, b):
    m, sd, spec = make_model()
    x, t = inputs(b, seed=b)
    names, bad = check_forward(m, sd, spec, x, t, make_mask(kind, b, seed=b))
    assert not bad, bad
    want = {"soft": 5, "half": 5, "ones": 4, "none": 0}[kind]       # all ones: only the first fusion is bypassed
    assert len(names) == want, names


@pytest.mark.parametrize("kind", ["soft", "half"])
def test_forward_default_weights_vs_matched_oracle(kind):
    m, sd, spec = make_model(trained=False)
    x, t = inputs(37, seed=21)
    names, bad = check_forward(m, sd, spec, x, t, make_mask(kind, 37, seed=21), tol=MATCHED_TOL)
    assert not bad, bad
    assert len(names) == 5


@pytest.mark.parametrize("hw", [(8, 8), (16, 8)])
def test_5x5_fusion_off_the_16x16_strip_tiling(hw):
    m, sd, spec = make_model(dim_mults=(1, 2, 4))
    x, t = inputs(37, seed=11, h=hw[0], w=hw[1])
    names, bad = check_forward(m, sd, spec, x, t, make_mask("soft", 37, hw[0], hw[1], seed=11))
    assert not bad, bad
    assert len(names) == 5


def test_mode_switching_on_one_handle():
    """One handle and one captured graph: mask -> ones -> none -> half -> mask, each against its oracle."""
    m, sd, spec = make_model()
    b = 37
    x, t = inputs(b, seed=3)
    out = []
    for kind in ("soft", "ones", "none", "half", "soft"):
        mask = make_mask(kind, b, seed=3)
        cond = None if mask is None else {"mask_cond": mask.cuda()}
        v = m(x.cuda(), t.cuda(), cond=cond).cpu()
        with torch.no_grad():
            want = unet_forward(sd, spec, x, t, None if mask is None else {"mask_cond": mask}, BF16_MATCHED)
        assert rel_l2(v, want) <= TRAINED_MATCHED_TOL, kind
        out.append(v)
    assert torch.equal(out[0], out[-1])
    assert rel_l2(out[0], out[2]) > 1e-2, "the mask must change the velocity"


# ---------------------------------------------------------------------------------------------------------------------
# integrators (default weights: the goldens were frozen with them)
# ---------------------------------------------------------------------------------------------------------------------
def test_rk4_and_euler_vs_reference_golden():
    from flocoder_b200 import sampling
    g = golden()
    m, _, _ = make_model(trained=False)
    x0 = g["x0"].cuda()
    shape = tuple(x0.shape)
    cond = {"mask_cond": g["mask_latents"].cuda()}
    x1, nfe = sampling.generate_latents_rk4(m, shape, n_steps=10, cond=cond, source=x0)
    assert nfe == 40 and rel_l2(x1, g["rk4_10_mask"]) <= BF16_FINAL_TOL
    again, _ = sampling.generate_latents_rk4(m, shape, n_steps=10, cond=cond, source=x0)
    assert torch.equal(x1, again)
    x1, nfe = sampling.euler_sampler(m, shape, 10, cond=cond, source=x0)
    assert nfe == 10 and rel_l2(x1, g["euler_10_mask"]) <= BF16_FINAL_TOL
    again, _ = sampling.euler_sampler(m, shape, 10, cond=cond, source=x0)
    assert torch.equal(x1, again)


@pytest.mark.parametrize("per_sample", [False, True])
def test_rk45_with_mask_vs_fp32_path(per_sample):
    from flocoder_b200 import sampling
    g = golden()
    m, _, _ = make_model(trained=False)
    ref, _, _ = make_model(trained=False, compute_dtype="fp32", layerwise=False)
    x0 = g["x0"].cuda()
    shape = tuple(x0.shape)
    cond = {"mask_cond": g["mask_latents"].cuda()}
    kw = dict(cond=cond, source=x0, rtol=1e-4, atol=1e-4, per_sample=per_sample)
    got, _ = sampling.generate_latents_rk45(m, shape, **kw)
    want, _ = sampling.generate_latents_rk45(ref, shape, **kw)
    assert rel_l2(got, want) <= BF16_FINAL_TOL
    again, _ = sampling.generate_latents_rk45(m, shape, **kw)
    assert torch.equal(got, again)


# ---------------------------------------------------------------------------------------------------------------------
# sharding over NCCL (two GPUs; skipped on a one-GPU box)
# ---------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, out):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import torch.distributed as dist
    from flocoder_b200 import _lib, sampling
    from flocoder_b200.dist import generate_latents_sharded
    from flocoder_b200.unet import Unet
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    g = torch.load(os.path.join(root, "tests", "golden", "inpaint_16.pt"), weights_only=False)
    torch.manual_seed(g["model_seed"])
    m = Unet(dim=g["dim"], channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True, compute_dtype="bf16")
    m.engine_flags = _lib.FLO_FLAG_LAYERWISE
    m = m.to(dev).eval()
    x0 = g["x0"][:7].to(dev)                                  # 4 + 3 samples
    cond = {"mask_cond": g["mask_latents"][:7].to(dev)}
    full, _ = generate_latents_sharded(m, tuple(x0.shape), n_steps=5, cond=cond, source=x0)
    if rank == 0:
        ref, _ = sampling.generate_latents_rk4(m, tuple(x0.shape), n_steps=5, cond=cond, source=x0)
        torch.save({"full": full.cpu(), "ref": ref.cpu()}, out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_sampling_with_mask(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "nccl.pt")
    mp.spawn(_nccl_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = torch.load(out)
    # a shard tiles its samples differently inside a CTA, which only reorders fp32 sums; on bf16 that can flip roundings
    assert rel_l2(got["full"], got["ref"]) <= 4e-3
