"""log_likelihood throughput on one GPU next to invert_latents: flowers_sd U-Net (dim 16, mults 1-2-4-8, 4x16x16, 102
classes) with trained-like weights (oracle.trained_like), fp32 path, B = 256, RK4-50 (196 evaluations), class-conditioned.

Prints one JSON line with the card name and power limit (read in the same run) and
* samples/s of log_likelihood with P = 1 and P = 4 Rademacher probes and of invert_latents(method="rk4", cfg_strength=0)
  on the same latents, timed alternately (best of --reps after one warm-up of each);
* ms per flo_unet_forward and per flo_unet_jvp with P = 1 and 4 at the same batch, from CUDA events over --calls calls each
  (each inside one window, alternated, best of --reps), and their ratio.

    python tools/bench_likelihood.py [--batch 256] [--reps 3] [--calls 20] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from bench_rk45 import card
    from conftest import seeded_state_dict
    from flocoder_b200 import sampling
    from flocoder_b200.unet import Unet
    from oracle.unet_oracle import trained_like

    assert torch.cuda.is_available(), "bench_likelihood measures the GPU; there is no CPU number to report"
    name, power = card()
    b, n_steps = args.batch, 50
    m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=102, compute_dtype="fp32")
    m.load_state_dict(trained_like(seeded_state_dict(102)[1]))
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(b, 4, 16, 16, generator=g).cuda()
    cond = {"class_cond": (torch.arange(b) % 102).cuda()}
    probes = {p: (torch.randint(0, 2, (p, b, 4, 16, 16), generator=g).float() * 2 - 1).cuda() for p in (1, 4)}

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    arms = {
        "log_likelihood_p1": lambda: sampling.log_likelihood(m, x, n_steps=n_steps, cond=cond, probes=probes[1]),
        "log_likelihood_p4": lambda: sampling.log_likelihood(m, x, n_steps=n_steps, cond=cond, probes=probes[4]),
        "invert_latents_rk4": lambda: sampling.invert_latents(m, x, n_steps=n_steps, cond=cond, cfg_strength=0.0,
                                                              method="rk4"),
    }
    best = {k: float("inf") for k in arms}
    for k, fn in arms.items():
        timed(fn)                                   # warm-up: plans, graphs, modules
    for _ in range(args.reps):
        for k, fn in arms.items():
            best[k] = min(best[k], timed(fn))

    eng = m.engine(16, 16)
    t = torch.full((b,), 500.0, device="cuda")
    cls = cond["class_cond"]
    calls = {
        "forward": lambda: eng.forward(x, t, cls),
        "jvp_p1": lambda: eng.jvp(x, t, cls, probes[1]),
        "jvp_p4": lambda: eng.jvp(x, t, cls, probes[4]),
    }
    ms = {k: float("inf") for k in calls}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for k, fn in calls.items():
        fn()
    for _ in range(args.reps):
        for k, fn in calls.items():
            ev0.record()
            for _ in range(args.calls):
                fn()
            ev1.record()
            ev1.synchronize()
            ms[k] = min(ms[k], ev0.elapsed_time(ev1) / args.calls)

    rec = {"card": name, "power_limit": power, "net": "flowers_sd trained_like", "compute_dtype": "fp32", "batch": b,
           "n_steps": n_steps, "nfe": 4 * (n_steps - 1),
           "samples_per_s": {k: round(b / v, 1) for k, v in best.items()},
           "ms_per_call": {k: round(v, 4) for k, v in ms.items()},
           "jvp_p1_over_forward": round(ms["jvp_p1"] / ms["forward"], 3),
           "jvp_p4_over_forward": round(ms["jvp_p4"] / ms["forward"], 3)}
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
