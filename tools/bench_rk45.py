"""RK45 sampling throughput next to RK4-50 on one GPU: flowers_sd U-Net with trained-like weights (oracle.trained_like),
fp16 and bf16, B = 256 and 1024.

Per configuration: samples/s of the adaptive solve (rtol = atol = 1e-5), its nfe and attempts, and the host gap per attempt
= host wall time of the attempt (graph launch to status record on the host) minus the attempt graph's device time from
CUDA events (flo_integrate_rk45_timing); and samples/s of RK4-50 (200 evaluations) from the same run.  Prints one JSON line
per configuration, with the card name and power limit, and writes them to --out when given.

Reverse rows: invert_latents of the RK4-50 result back to t = 0, with RK4-50 over the reversed grid (the same graphs as the
forward RK4, so the same rate is expected) and with the adaptive solve (rtol = atol = 1e-5), alternating with the forward
integrators.

With --per-sample the per-sample RK45 (every sample its own step-size control) runs as a third arm, alternating with the
other two on the same inputs.  Besides samples/s, attempts (the batch's, = the most any sample made) and the host gap it
reports each sample's nfe (min / median / max) and the share of evaluated sample-forwards spent on samples that had already
reached t = 1: 1 - sum_i nfe_i / (B * (2 + 6 * attempts)).

    python tools/bench_rk45.py [--batches 256 1024] [--dtypes fp16 bf16] [--reps 3] [--per-sample] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return name, power
    except Exception as e:                     # the numbers are still printed, with the card unknown
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--dtypes", nargs="+", default=["fp16", "bf16"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--per-sample", action="store_true", help="also time the per-sample RK45")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from flocoder_b200 import sampling
    from flocoder_b200.unet import Unet
    from conftest import seeded_state_dict
    from oracle.unet_oracle import trained_like

    assert torch.cuda.is_available(), "bench_rk45 measures the GPU; there is no CPU number to report"
    name, power = card()
    sd = trained_like(seeded_state_dict(102)[1])
    lines = []
    for dt in args.dtypes:
        m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=102, compute_dtype=dt)
        m.load_state_dict(sd)
        m = m.cuda().eval()
        for b in args.batches:
            x0 = torch.randn(b, 4, 16, 16, generator=torch.Generator().manual_seed(b)).cuda()
            eng = m.engine(16, 16)

            def rk45():
                return sampling.generate_latents_rk45(m, (b, 4, 16, 16), source=x0)

            def rk45ps():
                return sampling.generate_latents_rk45(m, (b, 4, 16, 16), source=x0, per_sample=True)

            def rk4():
                return sampling.generate_latents_rk4(m, (b, 4, 16, 16), n_steps=50, source=x0)   # the reference's RK4-50: 49 intervals

            rk45(); x1, _ = rk4(); torch.cuda.synchronize()          # warm-up: plans, graphs, modules

            def rk45_rev():
                return sampling.invert_latents(m, x1, method="rk45")

            def rk4_rev():
                return sampling.invert_latents(m, x1, n_steps=50)

            rk45_rev(); rk4_rev(); torch.cuda.synchronize()
            if args.per_sample:
                rk45ps(); torch.cuda.synchronize()
            best45, best4, timing, nfe = float("inf"), float("inf"), None, 0
            best45r, best4r, timing_r, nfe_r = float("inf"), float("inf"), None, 0
            best_ps, timing_ps, nfe_ps = float("inf"), None, None
            for _ in range(args.reps):                               # alternate the integrators
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _, nfe = rk45()
                torch.cuda.synchronize()
                dt45 = time.perf_counter() - t0
                if dt45 < best45:
                    best45, timing = dt45, eng.rk45_timing()
                t0 = time.perf_counter()
                rk4()
                torch.cuda.synchronize()
                best4 = min(best4, time.perf_counter() - t0)
                t0 = time.perf_counter()
                _, nfe_r = rk45_rev()
                torch.cuda.synchronize()
                dt45r = time.perf_counter() - t0
                if dt45r < best45r:
                    best45r, timing_r = dt45r, eng.rk45_timing()
                t0 = time.perf_counter()
                rk4_rev()
                torch.cuda.synchronize()
                best4r = min(best4r, time.perf_counter() - t0)
                if args.per_sample:
                    t0 = time.perf_counter()
                    _, nfe_ps = rk45ps()
                    torch.cuda.synchronize()
                    dtps = time.perf_counter() - t0
                    if dtps < best_ps:
                        best_ps, timing_ps = dtps, eng.rk45_timing()
            attempts, wall_ms, graph_ms = timing
            rec = {"card": name, "power_limit": power, "dtype": dt, "batch": b, "net": "flowers_sd trained_like",
                   "rk45": {"rtol": 1e-5, "atol": 1e-5, "samples_per_s": b / best45, "nfe": nfe, "attempts": attempts,
                            "ms_per_attempt_wall": wall_ms / attempts, "ms_per_attempt_graph": graph_ms / attempts,
                            "host_gap_ms_per_attempt": (wall_ms - graph_ms) / attempts,
                            "host_gap_share": (wall_ms - graph_ms) / wall_ms},
                   "rk4_50": {"samples_per_s": b / best4, "nfe": 200},
                   "rk45_reverse": {"rtol": 1e-5, "atol": 1e-5, "samples_per_s": b / best45r, "nfe": nfe_r,
                                    "attempts": timing_r[0], "ms_per_attempt_graph": timing_r[2] / timing_r[0],
                                    "host_gap_share": (timing_r[1] - timing_r[2]) / timing_r[1]},
                   "rk4_50_reverse": {"samples_per_s": b / best4r, "nfe": 196},
                   "reps": args.reps, "timing": "best of reps, wall clock"}
            if args.per_sample:
                a_ps, wall_ps, graph_ps = timing_ps
                evaluated = b * (2 + 6 * a_ps)                       # sample-forwards the batch ran, finished samples included
                rec["rk45_per_sample"] = {
                    "rtol": 1e-5, "atol": 1e-5, "samples_per_s": b / best_ps, "attempts": a_ps,
                    "nfe_min": int(nfe_ps.min()), "nfe_median": int(nfe_ps.median()), "nfe_max": int(nfe_ps.max()),
                    "nfe_mean": float(nfe_ps.double().mean()),
                    "finished_forward_share": 1.0 - int(nfe_ps.sum()) / evaluated,
                    "ms_per_attempt_wall": wall_ps / a_ps, "ms_per_attempt_graph": graph_ps / a_ps,
                    "host_gap_ms_per_attempt": (wall_ps - graph_ps) / a_ps, "host_gap_share": (wall_ps - graph_ps) / wall_ps}
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
