"""Benchmark of the hot path: fixed-step latent flow-matching sampling (SURVEY.md 8d).

    python bench.py --gpus N --steps K --warmup W                  # our sm_100a path (one rank per GPU)
    python bench.py --config {c2,c3,c4,c5} ...                     # another BASELINE configuration as the main line
    python bench.py --impl reference --steps K --warmup W          # the reference algorithm on the host cores
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's latents to DIR/*.npy

A "step" is one whole trajectory over one batch of synthetic latents.  BASELINE.json configs:

  c2 (default) flowers_sd U-Net (n_classes=102), RK4 n_steps=50 (49 intervals, 196 evaluations), 256 samples PER GPU
               (weak scaling: the line the driver's N = 1/2/4/8 runs report);
  c3           midi_vqgan shape (n_classes=0, inpainting off), RK4-50, 1024 samples on one GPU;
  c4           flowers_sd RK4-50, 8192 samples IN TOTAL sharded over the N GPUs (strong scaling) through
               flocoder_b200.dist.generate_latents_sharded, one final NCCL all-gather;
  c5           stl_sd U-Net (n_classes=10), legacy Euler 100 steps, 4096 samples in total over the N GPUs.

The default line also carries the other configurations the run can afford as sub-records (`other_configs`): c3 at N=1,
the strong-scaling point `strong_c4` at every N>1, and c5 at N=8 -- so the driver's own runs see them.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "samples/sec, 50-step RK4 latent sampling"
UNIT = "samples/s"
CONV_FLOP_PER_SAMPLE_FORWARD = 66_846_720      # SURVEY.md 8d: 2*M*N*K over the 75 convolutions
LATENT = (4, 16, 16)
CONFIGS = {
    "c2": dict(label="flowers_sd", n_classes=102, method="rk4", n_steps=50, per_gpu_batch=256, scaling="weak"),
    "c3": dict(label="midi_vqgan (inpainting off)", n_classes=0, method="rk4", n_steps=50, global_batch=1024, scaling="strong"),
    "c4": dict(label="flowers_sd", n_classes=102, method="rk4", n_steps=50, global_batch=8192, scaling="strong"),
    "c5": dict(label="stl_sd", n_classes=10, method="euler", n_steps=100, global_batch=4096, scaling="strong"),
}


def nfe_of(cfg):
    return 4 * (cfg["n_steps"] - 1) if cfg["method"] == "rk4" else cfg["n_steps"]


def metric_of(cfg):
    return METRIC if cfg["method"] == "rk4" else f"samples/sec, {cfg['n_steps']}-step Euler latent sampling"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def traffic_per_launch(kernel, args, batch):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/r02_traffic.json, else the
    round-1 file); only quoted when the run matches the captured configuration (fused path, 16-bit, batch 256), else null."""
    if args.layerwise or args.dtype == "fp32" or batch != 256:
        return None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)["kernels"][kernel]["dram_bytes_per_launch"]
        except Exception:
            continue
    return None


def workload_config(cfg, n_gpus, global_batch, dtype):
    steps = (f"RK4 n_steps={cfg['n_steps']} ({cfg['n_steps'] - 1} intervals, {nfe_of(cfg)} evaluations)" if cfg["method"] == "rk4"
             else f"legacy Euler {cfg['n_steps']} steps ({nfe_of(cfg)} evaluations)")
    return {
        "workload": f"{cfg['label']} latent U-Net (dim=16, mults 1-2-4-8, n_classes={cfg['n_classes']}, random init seed 1234), "
                    f"{steps}, cond=None",
        "global_batch": global_batch, "per_gpu_batch": -(-global_batch // n_gpus), "latent": list(LATENT),
        "nfe": nfe_of(cfg), "compute_dtype": dtype, "parallelism": f"batch-shard x{n_gpus} + final all-gather",
        "l2": "256 MiB memset between steps (inside the timed region)",
    }


DUMP_MAX_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` to out_dir/<name>.npy in float32, within DUMP_MAX_BYTES in all (headers included), so
    that two builds can be compared output for output.  A tensor over its share of the budget keeps a fixed, seeded sample
    of its rows (dim 0), in ascending order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_MAX_BYTES // len(arrays) - 4096                  # room for the .npy header
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        if 4 * t.numel() > share:
            n_rows = share // (4 * t[0].numel())
            if n_rows == 0:
                raise ValueError(f"{name}: one row of {tuple(t.shape)} exceeds the {share}-byte dump share")
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:n_rows]
            t = t[rows.sort().values]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.contiguous().numpy())


def seeded_state_dict(n_classes):
    from flocoder_b200.unet import Unet
    torch.manual_seed(1234)
    return {k: v.detach().clone() for k, v in
            Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes).state_dict().items()}


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm on the host cores
# --------------------------------------------------------------------------------------------------
def cpu_sample(cfg, batch, intervals, threads):
    """Times `intervals` RK4 intervals (4 evaluations each; Euler: `intervals` steps) of the CPU oracle at `batch` and scales
    to the full trajectory.  Returns (samples/s for the whole trajectory, seconds measured)."""
    import oracle
    from oracle.unet_oracle import OracleModel, UnetSpec
    torch.set_num_threads(threads)
    sd = seeded_state_dict(cfg["n_classes"])
    model = OracleModel(sd, UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=cfg["n_classes"]))
    x0 = torch.randn(batch, *LATENT, generator=torch.Generator().manual_seed(5678))
    t_vec = torch.zeros(batch)

    def f(x, t):
        return oracle.v_func_cfg(model, None, 0.0, t_vec, x, t)

    t0 = time.perf_counter()
    y = x0
    with torch.no_grad():
        if cfg["method"] == "rk4":
            ts = oracle.sampling_oracle.time_grid(cfg["n_steps"])
            total = cfg["n_steps"] - 1
            for i in range(intervals):
                y = oracle.rk4_step(f, y, ts[i], ts[i + 1] - ts[i])
        else:
            total = cfg["n_steps"]
            dt = 1.0 / total
            for i in range(intervals):
                y = y + f(y, torch.tensor(i / total * (1 - 1e-3) + 1e-3)) * dt
    dt_s = time.perf_counter() - t0
    return batch / (dt_s * total / intervals), dt_s


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    world = max(1, args.gpus)
    gb = cfg.get("global_batch") or cfg["per_gpu_batch"] * world
    total = cfg["n_steps"] - 1 if cfg["method"] == "rk4" else cfg["n_steps"]
    # ONE full trajectory (every interval, nothing extrapolated) at a small batch first: it anchors the bounded samples below.
    t0 = time.perf_counter()
    full_v, full_s = cpu_sample(cfg, 8, total, threads)
    full = {"batch": 8, "intervals": total, "seconds": round(full_s, 2), "samples_per_s": full_v}
    # Bounded sample: one RK4 interval of a shard-sized batch per step; if (warmup + steps) of those would not finish in
    # about 2.5 minutes on this host, the later steps use a proportionally smaller batch (throughput is per sample).
    batch, intervals = 256, 1
    budget_s, t_used, n_left = 150.0 - (time.perf_counter() - t0), 0.0, args.warmup + args.steps
    vals, secs, batches = [], 0.0, []
    for k in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        v, s = cpu_sample(cfg, batch, intervals, threads)
        t_used += time.perf_counter() - t0
        n_left -= 1
        if k >= args.warmup:
            vals.append(v); secs += s; batches.append(batch)
        if n_left > 0:
            per_sample = (time.perf_counter() - t0) / batch
            fit = int((budget_s - t_used) / n_left / per_sample) if per_sample > 0 else batch
            batch = max(8, min(256, (fit // 8) * 8))
    value = sum(vals) / len(vals)
    unit_name = "RK4 intervals" if cfg["method"] == "rk4" else "Euler steps"
    sample = (f"per step: B={batches if len(set(batches)) > 1 else batches[0]}, {intervals} of {total} {unit_name} of the CPU oracle "
              f"(PyTorch fp32, test-proven equal to the reference), scaled by {total}/{intervals}; every interval costs the same "
              f"(one full {total}-interval trajectory at B=8 in this run: {full_v:.2f} samples/s)")
    line = {
        "impl": "reference", "metric": metric_of(cfg), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * gb / value, "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # ms_per_step is the time the host would need for one whole-job step at this throughput: it is EXTRAPOLATED from
        # the bounded sample (the measured seconds are in cpu_baseline.seconds_measured)
        "extrapolated": True,
        # the same workload label as the GPU arm at this N; the host's cores process it sample by sample, so the
        # throughput of the bounded sample (one shard-sized batch) is the throughput of the whole job
        "config": workload_config(cfg, world, gb, "fp32"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "seconds_measured": round(secs, 2), "full_trajectory": full},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region through NVML in a background thread (spawning
    nvidia-smi every 100 ms was measured to halve the throughput of a launch-bound step by contending for the driver)."""

    def __init__(self, index, period=0.1):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.thread, self.stop_flag = None, False

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            self.h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.nv = nv
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self.thread is None:
            return out
        self.stop_flag = True
        self.thread.join(timeout=2)
        if self.samples:
            sm = sorted(self.samples)
            out.update(sm_mhz=sm[len(sm) // 2], reasons=sorted(self.reasons), samples=len(sm))
        return out


class Runner:
    """One BASELINE configuration on this rank's GPU: model, synthetic noise, the resident and the host-buffer step."""

    def __init__(self, cfg, args, world, rank, dev, batch_override=None):
        import torch.distributed as dist
        from flocoder_b200 import _lib, sampling
        from flocoder_b200.dist import generate_latents_sharded
        from flocoder_b200.unet import Unet
        self.cfg, self.world, self.rank, self.dev, self.dist = cfg, world, rank, dev, dist
        torch.manual_seed(1234)
        self.model = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=cfg["n_classes"], compute_dtype=args.dtype).to(dev).eval()
        if args.layerwise:
            self.model.engine_flags = _lib.FLO_FLAG_LAYERWISE
        self.eng = self.model.engine(LATENT[1], LATENT[2])
        n = cfg["n_steps"]
        self.cfg_strength = float(getattr(args, "cfg", 0.0) or 0.0)
        if self.cfg_strength and cfg["method"] == "rk4" and cfg["n_classes"] > 0 and cfg["scaling"] == "weak":
            # class-conditional sampling with classifier-free guidance (sampling.py:69-74): class_cond = arange(B) % n_classes,
            # two U-Net evaluations per stage (SURVEY 8d's optional variant)
            cg = self.cfg_strength
            ncls = cfg["n_classes"]
            one = lambda shape, src: sampling.generate_latents_rk4(                                                    # noqa: E731
                self.model, shape, n_steps=n, cond={"class_cond": (torch.arange(shape[0], device=dev) % ncls)}, cfg_strength=cg, source=src)
            shard_fn = sampling.generate_latents_rk4
        elif cfg["method"] == "rk4":
            one = lambda shape, src: sampling.generate_latents_rk4(self.model, shape, n_steps=n, source=src)          # noqa: E731
            shard_fn = sampling.generate_latents_rk4
        else:
            one = lambda shape, src: sampling.euler_latents(self.model, shape, n, source=src)                          # noqa: E731
            shard_fn = lambda m, shape, n_steps, cond, cfg_s, source=None: sampling.euler_latents(m, shape, n_steps, cond=cond, source=source)  # noqa: E731
        if cfg["scaling"] == "weak":
            # every rank integrates its own slice of per_gpu_batch samples; one all-gather assembles the global batch
            B = batch_override or cfg["per_gpu_batch"]
            self.global_batch, self.local_batch = B * world, B
            gen = torch.Generator().manual_seed(5678 + rank)
            self.x_host = torch.randn(B, *LATENT, generator=gen).pin_memory()
            self.x_dev = self.x_host.to(dev)
            gathered = torch.empty((world * B, *LATENT), device=dev) if world > 1 else None

            def run(src):
                x1, _ = one((B, *LATENT), src)
                if world > 1:
                    dist.all_gather_into_tensor(gathered, x1)
                    return gathered
                return x1
        else:
            # the global batch is cut into contiguous slices by flocoder_b200.dist (the product's own sharded entry point)
            G = batch_override or cfg["global_batch"]
            self.global_batch, self.local_batch = G, -(-G // world)
            gen = torch.Generator().manual_seed(5678)                 # the same global noise on every rank
            self.x_host = torch.randn(G, *LATENT, generator=gen).pin_memory()
            self.x_dev = self.x_host.to(dev)

            def run(src):
                x1, _ = generate_latents_sharded(self.model, (G, *LATENT), n, source=src, sampler=shard_fn)
                return x1
        self.run = run
        self.h2d = self.local_batch * 4 * LATENT[0] * LATENT[1] * LATENT[2]
        self.d2h = self.global_batch * 4 * LATENT[0] * LATENT[1] * LATENT[2]

    def step_resident(self):
        return self.run(self.x_dev)

    def step_e2e(self):
        # the call a user makes, with HOST buffers: H2D of this rank's noise, trajectory, D2H of the assembled latents
        out = self.run(self.x_host)
        return out.cpu()


def run_gpu_arm(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)

    cfg = CONFIGS[args.config]
    main = Runner(cfg, args, world, rank, dev, batch_override=args.batch)
    eng, B = main.eng, main.local_batch
    NFE = nfe_of(cfg) * (2 if main.cfg_strength else 1)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    step_ms = {}
    kept = {}                            # keep=True: what the region's last timed step returned (--dump-outputs)

    def timed(fn, steps, tag, keep=False):
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            if not os.environ.get("FLO_BENCH_NOFLUSH"):
                flush.zero_()
            out = fn()
            ev[i + 1].record()
        if keep:
            kept[tag] = out
        barrier()
        step_ms[tag] = [round(ev[i].elapsed_time(ev[i + 1]), 3) for i in range(steps)]
        ms = torch.tensor([ev[0].elapsed_time(ev[steps])], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # the sampler starts before the warm-up (NVML initialisation and its first query are slow and would otherwise
    # land inside the timed region); only the samples taken during the timed region are kept
    clocks = ClockSampler(local)
    if rank == 0 and not os.environ.get("FLO_BENCH_NOCLOCK"):
        clocks.start()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        flush.zero_()                    # also warms torch's fill kernel (its lazy first load cost 10-230 ms inside step 1)
        main.step_resident()
    torch.cuda.synchronize()
    clocks.samples.clear(); clocks.reasons.clear()
    l0 = eng.launch_count()
    ms = timed(main.step_resident, args.steps, "resident", keep=bool(args.dump_outputs))
    launches = eng.launch_count() - l0
    clk = clocks.stop() if rank == 0 else {}
    value = main.global_batch * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"latents": kept["resident"]})
    kept.clear()

    for _ in range(2):
        flush.zero_()
        main.step_e2e()
    ms_e2e = timed(main.step_e2e, args.steps, "e2e")
    e2e_value = main.global_batch * args.steps / (ms_e2e * 1e-3)

    # ---- the other BASELINE configurations this run can afford (every rank takes part: they are collective)
    others = {}
    if args.config == "c2" and not args.no_other and not args.cfg:
        extra = []
        if world == 1:
            extra.append(("c3", "c3"))
        else:
            extra.append(("strong_c4", "c4"))
            if world == 8:
                extra.append(("c5", "c5"))
        for tag, key in extra:
            try:
                r = Runner(CONFIGS[key], args, world, rank, dev)
                for _ in range(2):
                    flush.zero_()
                    r.step_resident()
                k = 2
                t_res = timed(r.step_resident, k, tag)
                r.step_e2e()
                t_e2e = timed(r.step_e2e, k, tag + "_e2e")
                others[tag] = {
                    "metric": metric_of(CONFIGS[key]), "value": r.global_batch * k / (t_res * 1e-3), "unit": UNIT,
                    "e2e": r.global_batch * k / (t_e2e * 1e-3), "ms_per_step": t_res / k, "steps": k, "warmup": 2,
                    "scaling": CONFIGS[key]["scaling"], "config": workload_config(CONFIGS[key], world, r.global_batch, args.dtype),
                    "tensor_frac_of_sustained": r.global_batch * k / (t_res * 1e-3) / world * nfe_of(CONFIGS[key]) *
                    CONV_FLOP_PER_SAMPLE_FORWARD / 1e12 / load_peaks()["bf16_tflops_sustained"],
                    "api": "flocoder_b200.dist.generate_latents_sharded" if CONFIGS[key]["scaling"] == "strong" else "generate_latents_rk4",
                }
                del r
            except Exception as exc:
                others[tag] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    # Per-launch durations measured live with CUDA events on the launching stream (one forward, launch by launch,
    # best of 5); achieved = ALGORITHMIC conv FLOPs of the dominant kernel's launches / their summed duration.
    KIND = {0: "k_init_conv", 1: "k_conv_umma (tcgen05 implicit-GEMM conv)", 2: "k_gn (GroupNorm+FiLM+SiLU+residual pass)",
            3: "k_linattn", 4: "k_midattn", 5: "k_final",
            6: "k_chain (fused ResnetBlock-chain stage: tcgen05 implicit-GEMM convs + GroupNorm/FiLM/SiLU/residual epilogues)",
            7: "k_attn (fused attention block: tcgen05 q/k/v/out convs + context/output contractions)"}
    info = eng.op_info()
    ms_ops = eng.profile_ops(B, reps=5)
    groups = {}
    for (name, kind, fl, by), t in zip(info, ms_ops):
        g = groups.setdefault(kind, {"n": 0, "ms": 0.0, "flop": 0.0, "bytes": 0.0})
        g["n"] += 1; g["ms"] += t; g["flop"] += fl * B; g["bytes"] += by * B
    fwd_ms = sum(ms_ops)
    conv_flop_sum = sum(fl for (_, _, fl, _) in info)
    dom = max((k for k in groups if k in (1, 6, 7)), key=lambda k: groups[k]["ms"])
    gd = groups[dom]
    # Event records between launches add ~6 us per launch that the graph replay of the timed region does not have, so the
    # kernel's duration inside the step is taken as (its share of the event-timed forward) x (the forward time of the
    # timed region); the raw event-timed figure is reported next to it.
    fwd_ms_in_step = ms / args.steps / NFE
    share = gd["ms"] / fwd_ms if fwd_ms > 0 else 0.0
    ms_in_step = share * fwd_ms_in_step
    achieved = gd["flop"] / (ms_in_step * 1e-3) / 1e12 if ms_in_step > 0 else 0.0
    achieved_event = gd["flop"] / (gd["ms"] * 1e-3) / 1e12 if gd["ms"] > 0 else 0.0
    peak = peaks["bf16_tflops_sustained"] if args.dtype in ("bf16", "fp16") else None      # kernel timed inside a long step
    roofline = {
        "bound": "tensor", "kernel": f"{KIND[dom]}, {gd['n']} launches/forward",
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
        "frac": (achieved / peak) if peak else None, "traffic": traffic_per_launch(KIND[dom].split(" ")[0], args, B),
        "peak_source": f"{peaks['source']} sustained bf16 cuBLAS (kernel duration taken inside the timed step)",
        "share_of_forward": share, "kernel_ms_per_forward_in_step": ms_in_step, "forward_ms_in_step": fwd_ms_in_step,
        "achieved_event_timed_alone": achieved_event,
        "end_to_end_tensor_frac_of_sustained": value / world * NFE * CONV_FLOP_PER_SAMPLE_FORWARD / 1e12 / peaks["bf16_tflops_sustained"],
        "forward_ms_sum_of_kernels": fwd_ms,
        "conv_flop_per_sample_forward": {"sum_over_launches": conv_flop_sum, "survey_8d": CONV_FLOP_PER_SAMPLE_FORWARD},
        "kernels": {KIND[k].split(" ")[0]: {"launches": g["n"], "ms": g["ms"], "conv_tflops": g["flop"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] else 0.0,
                                            "gbs": g["bytes"] / (g["ms"] * 1e-3) / 1e9 if g["ms"] else 0.0,
                                            "hbm_frac": g["bytes"] / (g["ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"] if g["ms"] else 0.0}
                    for k, g in groups.items()},
    }
    # The north star also asks for the GroupNorm+SiLU+FiLM pass to be judged by achieved HBM GB/s.  The fused path has no
    # such pass (GroupNorm runs on TMEM/SMEM-resident tiles inside k_chain), so the standalone kernels of the layer-wise
    # path (k_gn_tma / k_gn_warp) are timed here on tensors larger than L2 (B=4096, 100-235 MB per op), per launch with
    # CUDA events, best of 5.  Two byte counts: the bytes the kernel really moves (the layer-wise convs hand it fp32
    # accumulators and it writes fp32 masters next to the 16-bit operands), and SURVEY 8d's algorithmic figure for a pass
    # over 16-bit tensors (each normalised tensor read once and written once in bf16: 4 B per element).
    if world == 1 and args.dtype != "fp32" and not os.environ.get("FLO_BENCH_NO_GN"):
        try:
            from flocoder_b200 import _lib
            from flocoder_b200.unet import Unet
            lw = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=cfg["n_classes"], compute_dtype="bf16").to(dev).eval()
            lw.engine_flags = _lib.FLO_FLAG_LAYERWISE
            le = lw.engine(LATENT[1], LATENT[2])
            Bg = 4096
            li, lms = le.op_info(), le.profile_ops(Bg, reps=5)
            gn = [(n, by * Bg, t, fl * Bg / 10.0) for (n, k, fl, by), t in zip(li, lms) if k == 2 and by * Bg >= 64e6]   # flops = 10/element
            tot_b, tot_ms, tot_el = sum(r[1] for r in gn), sum(r[2] for r in gn), sum(r[3] for r in gn)
            best = max(gn, key=lambda r: r[1] / r[2])
            roofline["gn_pass"] = {
                "bound": "hbm", "kernel": "k_gn_tma (standalone GroupNorm+FiLM+SiLU+residual pass of the layer-wise path)",
                "batch": Bg, "launches": len(gn), "achieved": tot_b / (tot_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": tot_b / (tot_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "bytes_counted": "moved by the kernel (fp32 accumulator in, fp32 master + 16-bit operand copies out)",
                "survey_8d_bytes": {"achieved": tot_el * 4.0 / (tot_ms * 1e-3) / 1e9, "frac": tot_el * 4.0 / (tot_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                    "bytes_counted": "4 B per normalised element (bf16 read + bf16 write), SURVEY.md 8d"},
                "best_launch": {"op": best[0], "bytes": best[1], "us": best[2] * 1e3, "gbs": best[1] / (best[2] * 1e-3) / 1e9},
                "note": "all GN launches of one forward whose tensors exceed 64 MB; not on the default (fused) path"}
            del le, lw
        except Exception as exc:  # the headline numbers do not depend on this leg
            roofline["gn_pass"] = {"error": f"{type(exc).__name__}: {exc}"}
    cpu, parity, eager = None, None, None
    if world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        v_cpu, s_cpu = cpu_sample(cfg, 256, 2, threads)
        total = cfg["n_steps"] - 1 if cfg["method"] == "rk4" else cfg["n_steps"]
        cpu = {"value": v_cpu, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"B=256, 2 of {total} {'RK4 intervals' if cfg['method'] == 'rk4' else 'Euler steps'} of the CPU oracle "
                         f"(PyTorch fp32), {s_cpu:.1f} s measured, scaled by {total}/2"}
        parity = parity_record(main.model, cfg, args.dtype, dev)
        eager = torch_eager_cuda(cfg, dev, 256)
    line = {
        "metric": metric_of(cfg), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
        "dtype": {"bf16": "bf16", "fp16": "f16", "fp32": "f32"}[args.dtype], "data": "synthetic",
        "config": dict(workload_config(cfg, world, main.global_batch, args.dtype), name=args.config, cfg_strength=main.cfg_strength,
                       evaluations_per_stage=2 if main.cfg_strength else 1,
                       kernels="layerwise" if args.layerwise else "fused-stage", step_ms=step_ms),
        "clocks": {"sm_mhz": clk.get("sm_mhz"), "sm_max_mhz": clk.get("sm_max_mhz"), "reasons": clk.get("reasons", []),
                   "samples": clk.get("samples", 0)},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": main.h2d, "d2h_bytes_per_step": main.d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    if cpu:
        line["cpu_baseline"] = cpu
    if parity:
        line["parity"] = parity
    if eager:
        line["torch_eager_cuda"] = eager
    if others:
        line["other_configs"] = others
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def parity_record(model, cfg, dtype, dev):
    """The headline carries its own parity caveat: one forward and one short trajectory of THIS run's model and dtype against
    the fp32 CPU oracle (B=8, the golden inputs' seed), next to the north-star bars."""
    try:
        import oracle
        from oracle.unet_oracle import OracleModel, UnetSpec, unet_forward
        from flocoder_b200 import sampling
        sd = {k: v.detach().float().cpu().clone() for k, v in model.state_dict().items()}
        spec = UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=cfg["n_classes"])
        x0 = torch.randn(8, *LATENT, generator=torch.Generator().manual_seed(5678))
        t = torch.full((8,), 0.25 * 999)

        def rel(a, b):
            return float((a.double().cpu() - b.double()).norm() / b.double().norm())
        with torch.no_grad():
            v_ref = unet_forward(sd, spec, x0, t, None)
        e_step = rel(model(x0.to(dev), t.to(dev)), v_ref)
        ref, _ = oracle.generate_latents_rk4(OracleModel(sd, spec), (8, *LATENT), n_steps=10, source=x0.clone())
        x1, _ = sampling.generate_latents_rk4(model, (8, *LATENT), n_steps=10, source=x0.to(dev))
        return {"dtype": dtype, "step_velocity_rel_l2": e_step, "final_latent_rel_l2_rk4_10": rel(x1, ref),
                "vs": "fp32 CPU oracle (test-proven equal to the reference), B=8, t=0.25",
                "bars": {"step": 1e-5 if dtype == "fp32" else 2e-3, "final": 1e-5 if dtype == "fp32" else 1e-2},
                "note": ("bf16 operands: the per-step figure is the format floor of 8-bit mantissas (~4.8e-3, DESIGN.md 3), above the "
                         "2e-3 bar; --dtype fp16 runs the same kernels at the same speed and meets it") if dtype == "bf16" else ""}
    except Exception as exc:
        return {"error": f"{type(exc).__name__}: {exc}"}


def torch_eager_cuda(cfg, dev, batch):
    """Diagnostic: what a flocoder user gets on this B200 today -- the reference algorithm (the oracle restatement, PyTorch
    eager) on the GPU with the reference's host syncs per evaluation (sampling.py:60,64-67: .item(), empty_cache(),
    synchronize()).  fp32 with TF32 off for convs (the parity-grade setting) and the model cast to bfloat16."""
    out = {"batch": batch, "what": "oracle restatement of the reference, PyTorch eager on cuda, reference's per-evaluation host syncs"}
    try:
        import oracle
        from oracle.unet_oracle import OracleModel, UnetSpec
        spec = UnetSpec(dim=16, dim_mults=(1, 2, 4, 8), channels=4, groups=4, n_classes=cfg["n_classes"])
        sd32 = seeded_state_dict(cfg["n_classes"])
        x0 = torch.randn(batch, *LATENT, generator=torch.Generator().manual_seed(5678))
        old_tf32 = torch.backends.cudnn.allow_tf32
        # the *_no_host_syncs rows drop the reference's per-evaluation .item() / empty_cache() / synchronize(): eager PyTorch at its best
        for tag, dt, synced in (("fp32_tf32_off", torch.float32, True), ("bf16", torch.bfloat16, True),
                                ("fp32_tf32_off_no_host_syncs", torch.float32, False), ("bf16_no_host_syncs", torch.bfloat16, False)):
            torch.backends.cudnn.allow_tf32 = False
            sd = {k: (v.to(dev).to(dt) if v.is_floating_point() else v.to(dev)) for k, v in sd32.items()}
            inner = OracleModel(sd, spec)

            class Synced:
                def __call__(self, x, tt, cond=None):
                    v = inner(x, tt, cond=cond)
                    if synced:
                        _ = v.sum().item()
                        torch.cuda.empty_cache()
                        torch.cuda.synchronize()
                    return v

                def parameters(self):
                    return iter([next(iter(sd.values()))])
            m = Synced()
            src = x0.to(dev).to(dt)
            n = cfg["n_steps"]
            if cfg["method"] != "rk4":
                continue
            oracle.generate_latents_rk4(m, (batch, *LATENT), n_steps=3, source=src.clone())        # warm-up (cuDNN autotune etc.)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            oracle.generate_latents_rk4(m, (batch, *LATENT), n_steps=n, source=src.clone())
            torch.cuda.synchronize()
            out[tag] = {"samples_per_s": batch / (time.perf_counter() - t0)}
        torch.backends.cudnn.allow_tf32 = old_tf32
    except Exception as exc:
        out["error"] = f"{type(exc).__name__}: {exc}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE configuration of the main line")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--layerwise", action="store_true", help="one kernel per layer instead of the fused stage kernels")
    ap.add_argument("--batch", type=int, default=None, help="override: per-GPU batch (weak configs) / global batch (strong configs)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity / torch_eager_cuda legs")
    ap.add_argument("--no-other", action="store_true", help="skip the other_configs sub-records")
    ap.add_argument("--cfg", type=float, default=0.0,
                    help="class-conditional sampling with this classifier-free-guidance strength (weak RK4 configs: 2 evaluations per stage)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latents the last timed step returned to DIR/latents.npy (float32; a seeded row sample "
                         "above 64 MB); the inputs are seeded, so runs with the same arguments see the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU arm's latents; the reference arm times partial trajectories")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
