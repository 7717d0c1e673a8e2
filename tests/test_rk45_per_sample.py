"""Per-sample RK45 without a GPU: the foreign-model composition (``solve_ivp`` on each sample alone) against ``solve_ivp``
called directly, independence of a sample's result from its batch, argument errors before anything runs, the C ABI's
argument checks, a failing sample named in the error, and the sharded sampler over a world-size-2 gloo group."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy.integrate import solve_ivp

from flocoder_b200 import sampling

SHAPE = (3, 4, 5, 6)


class Toy(torch.nn.Module):
    """A foreign velocity model whose velocity depends on the sample's own state, time and class only."""

    def __init__(self, n_classes=5):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self.w = torch.nn.Parameter(torch.randn(4, 4, generator=g) * 0.5)
        self.emb = torch.nn.Parameter(torch.randn(max(n_classes, 1), 4, generator=g))
        self.calls = 0

    def forward(self, x, time, cond=None):
        self.calls += 1
        s = time[:, None, None, None] / 999
        v = torch.einsum("oc,bchw->bohw", self.w, torch.tanh(3 * x)) * (1 + 4 * s) + torch.sin(3 * s)
        if cond and cond.get("class_cond") is not None:
            v = v + self.emb[cond["class_cond"]][:, :, None, None]
        return v


def direct_one(model, y0, t0, cls=None, cfg=0.0, rtol=1e-5, atol=1e-5):
    """solve_ivp on one sample ([1,C,H,W]) called directly."""
    shape = tuple(y0.shape)
    cond = None if cls is None else {"class_cond": cls}

    def fun(t, yf):
        x = torch.from_numpy(yf).float().reshape(shape)
        tv = torch.ones(1) * t * 999
        v = model(x, tv, cond=cond)
        if cfg and cond is not None:
            v_nc = model(x, tv, cond={"class_cond": None})
            v = v_nc + cfg * (v - v_nc)
        return v.detach().double().numpy().ravel()
    return solve_ivp(fun, (t0, 1.0), y0.double().numpy().ravel(), method="RK45", rtol=rtol, atol=atol)


def noise(seed, shape=SHAPE):
    x = torch.randn(shape, generator=torch.Generator().manual_seed(seed))
    return x * torch.linspace(0.2, 3.0, shape[0])[:, None, None, None]      # samples of different difficulty


@pytest.mark.parametrize("case", ["plain", "cfg", "init"])
def test_foreign_model_is_solve_ivp_per_sample(case):
    m = Toy()
    y0 = noise(1)
    cls, cfg, init, t0 = None, 3.0, None, 0.0
    if case == "cfg":
        cls = torch.tensor([0, 3, 4])
    if case == "init":
        init = torch.randn(SHAPE, generator=torch.Generator().manual_seed(2))
        t0 = float(sampling.warp_time(torch.tensor(0.3)))
    with torch.no_grad():
        got, nfe = sampling.generate_latents_rk45(m, SHAPE, cond=None if cls is None else {"class_cond": cls},
                                                  cfg_strength=cfg, source=y0, init_latents=init, init_strength=0.3,
                                                  per_sample=True)
        start = y0 if init is None else (1 - 0.3) * y0 + 0.3 * init
        sols = [direct_one(m, start[i:i + 1], t0, None if cls is None else cls[i:i + 1], cfg) for i in range(SHAPE[0])]
    assert nfe.dtype == torch.int64 and nfe.device.type == "cpu" and nfe.shape == (SHAPE[0],)
    for i, sol in enumerate(sols):
        assert sol.success and int(nfe[i]) == sol.nfev and (sol.nfev - 2) % 6 == 0
        assert np.array_equal(got[i].double().numpy().ravel(), sol.y[:, -1].astype(np.float32).astype(np.float64)), i
    assert len(set(nfe.tolist())) > 1, "the samples should need different step counts"


def test_a_sample_does_not_depend_on_its_batch():
    m = Toy()
    y0 = noise(4, (5,) + SHAPE[1:])
    cls = torch.tensor([1, 0, 4, 2, 3])
    kw = dict(cfg_strength=2.0, rtol=1e-4, atol=1e-4, per_sample=True)
    with torch.no_grad():
        full, nfe = sampling.generate_latents_rk45(m, y0.shape, cond={"class_cond": cls}, source=y0, **kw)
        perm = torch.tensor([3, 0, 4, 1, 2])
        pf, pn = sampling.generate_latents_rk45(m, y0.shape, cond={"class_cond": cls[perm]}, source=y0[perm], **kw)
        one, n1 = sampling.generate_latents_rk45(m, (1,) + SHAPE[1:], cond={"class_cond": cls[2:3]}, source=y0[2:3], **kw)
    assert torch.equal(pf, full[perm]) and torch.equal(pn, nfe[perm])
    assert torch.equal(one[0], full[2]) and int(n1[0]) == int(nfe[2])


@pytest.mark.parametrize("kwargs", [dict(rtol=0.0), dict(rtol=-1e-5), dict(atol=-1e-9), dict(max_steps=0), dict(max_steps=2.5),
                                    dict(init_latents=torch.zeros(SHAPE), init_strength=1.0)])
def test_argument_errors_raise_before_anything_runs(kwargs):
    m = Toy()
    with pytest.raises(ValueError):
        sampling.generate_latents_rk45(m, SHAPE, per_sample=True, **kwargs)
    assert m.calls == 0


def test_max_steps_failure_names_the_sample():
    m = Toy()
    y0 = noise(5)
    with torch.no_grad():
        nfe = sampling.generate_latents_rk45(m, SHAPE, source=y0, per_sample=True)[1]
        y0 = y0[torch.argsort(nfe, stable=True)]          # sample 0 needs the fewest attempts
        nfe = nfe.sort().values
        assert nfe[1] > nfe[0]
        max_steps = (int(nfe[0]) - 2) // 6             # enough for sample 0 only
        with pytest.raises(RuntimeError, match=rf"sample 1 used max_steps={max_steps} "):
            sampling.generate_latents_rk45(m, SHAPE, source=y0, max_steps=max_steps, per_sample=True)


@pytest.mark.parametrize("args, what", [
    ((0.0, 1.0, 0.0, 1e-5), "rtol"), ((0.0, 1.0, 1e-5, -1.0), "atol"), ((1.0, 1.0, 1e-5, 1e-5), "t0"),
    ((0.5, 0.2, 1e-5, 1e-5), "t0"), ((0.0, float("nan"), 1e-5, 1e-5), "t0")])
def test_c_abi_argument_checks_need_no_device(args, what):
    from flocoder_b200 import _lib
    L = _lib.lib()
    counts = (ctypes.c_int32 * 6)()
    t0, t1, rtol, atol = args
    rc = L.flo_integrate_rk45_per_sample(None, None, t0, t1, rtol, atol, 999.0, None, 0.0, 100, counts, 2, None)
    assert rc == _lib.FLO_ERR_INVALID and what in L.flo_last_error().decode()
    rc = L.flo_integrate_rk45_per_sample(None, None, 0.0, 1.0, 1e-5, 1e-5, 999.0, None, 0.0, 0, counts, 2, None)
    assert rc == _lib.FLO_ERR_INVALID and "max_steps" in L.flo_last_error().decode()
    rc = L.flo_integrate_rk45_per_sample(None, None, 0.0, 1.0, 1e-5, 1e-5, 999.0, None, 0.0, 100, counts, 2, None)
    assert rc == _lib.FLO_ERR_INVALID and "NULL" in L.flo_last_error().decode()


def test_sharded_batched_rk45_is_still_refused():
    from flocoder_b200 import dist as fdist
    with pytest.raises(ValueError, match="per_sample"):
        fdist.generate_latents_sharded(Toy(), SHAPE, sampler=sampling.generate_latents_rk45, source=torch.randn(SHAPE),
                                       per_sample=False)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, batch, out):
    from flocoder_b200.dist import generate_latents_sharded
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shape = (batch,) + SHAPE[1:]
    x0 = noise(7, shape)
    init = torch.randn(shape, generator=torch.Generator().manual_seed(8))
    cond = {"class_cond": torch.arange(batch) % 5}
    kw = dict(cond=cond, cfg_strength=2.0, source=x0, sampler=sampling.generate_latents_rk45, per_sample=True,
              init_latents=init, init_strength=0.2, rtol=1e-4, atol=1e-4)
    with torch.no_grad():
        full, nfe = generate_latents_sharded(Toy(), shape, **kw)
        local, local_nfe = generate_latents_sharded(Toy(), shape, gather=False, **kw)
    if rank == 0:
        torch.save({"full": full, "nfe": nfe, "local": local, "local_nfe": local_nfe}, out)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("batch", [4, 5, 1])
def test_sharded_per_sample_rk45_equals_unsharded_gloo(tmp_path, batch):
    """Even (4 = 2 + 2), uneven (5 = 3 + 2) and one empty shard (1 = 1 + 0): latents and per-sample nfe equal the
    unsharded run."""
    from flocoder_b200.dist import shard_bounds
    out = str(tmp_path / "r0.pt")
    mp.spawn(_worker, args=(2, _free_port(), batch, out), nprocs=2, join=True)
    got = torch.load(out)
    shape = (batch,) + SHAPE[1:]
    with torch.no_grad():
        ref, ref_nfe = sampling.generate_latents_rk45(
            Toy(), shape, cond={"class_cond": torch.arange(batch) % 5}, cfg_strength=2.0, source=noise(7, shape),
            init_latents=torch.randn(shape, generator=torch.Generator().manual_seed(8)), init_strength=0.2,
            rtol=1e-4, atol=1e-4, per_sample=True)
    assert torch.equal(got["full"], ref)
    assert got["nfe"].dtype == torch.int64 and torch.equal(got["nfe"], ref_nfe)
    lo, hi = shard_bounds(batch, 2, 0)
    assert torch.equal(got["local"], ref[lo:hi]) and torch.equal(got["local_nfe"], ref_nfe[lo:hi])
