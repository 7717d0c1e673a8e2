"""Inpainting sampling throughput: the fp32 CUDA-core path against the layer-wise bf16 tcgen05 path on one GPU.

The inpaint_16 net shape (``Unet(dim=16, dim_mults=(1, 2, 4, 8), channels=4, mask_cond=True)``) with trained-like weights
(oracle.trained_like) and a soft seeded mask in use (every mask branch runs), RK4-50 (200 evaluations), B = 256 and 1024.
Per configuration: samples/s (best of --reps wall-clock runs that end in a device synchronise, the two paths alternating on
the same inputs), and the share of one forward spent in the seven mask-fusion convolutions (flo_unet_profile_ops: best-of-5
CUDA-event time per op, ops launched one by one).  Prints one JSON line per configuration, with the card name and power
limit, and writes them to --out when given.

    python tools/bench_inpainting.py [--batches 256 1024] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_rk45 import card  # noqa: E402

MASK_OPS = ("mask_fusion_conv.0", "mask_fusion_conv.2", "mask_fusion_conv", "down_mask_fusions.0.0", "down_mask_fusions.1.0",
            "up_mask_fusions.0.0", "up_mask_fusions.1.0")
ARMS = (("fp32", 0), ("bf16", "layerwise"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from flocoder_b200 import _lib, sampling
    from flocoder_b200.unet import Unet
    from oracle.unet_oracle import trained_like

    assert torch.cuda.is_available(), "bench_inpainting measures the GPU; there is no CPU number to report"
    name, power = card()
    torch.manual_seed(1234)
    sd = trained_like(Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True).state_dict())
    models = {}
    for dt, route in ARMS:
        m = Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True, compute_dtype=dt)
        m.load_state_dict(sd)
        if route == "layerwise":
            m.engine_flags = _lib.FLO_FLAG_LAYERWISE
        models[dt] = m.cuda().eval()
    lines = []
    for b in args.batches:
        gen = torch.Generator().manual_seed(b)
        x0 = torch.randn(b, 4, 16, 16, generator=gen).cuda()
        mask = torch.sigmoid(4 * torch.randn(b, 4, 16, 16, generator=gen)).cuda()
        cond = {"mask_cond": mask}
        shape = (b, 4, 16, 16)

        def rk4(m):
            return sampling.generate_latents_rk4(m, shape, n_steps=50, cond=cond, source=x0)

        out = {}
        for dt, m in models.items():                          # warm-up: plans, graphs, modules
            out[dt], _ = rk4(m)
        torch.cuda.synchronize()
        best = {dt: float("inf") for dt in models}
        for _ in range(args.reps):
            for dt, m in models.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rk4(m)
                torch.cuda.synchronize()
                best[dt] = min(best[dt], time.perf_counter() - t0)
        rec = {"card": name, "power_limit": power, "batch": b, "net": "inpaint_16 trained_like, soft mask",
               "integrator": "rk4_50 (200 evaluations)", "reps": args.reps, "timing": "best of reps, wall clock"}
        for dt, m in models.items():
            eng = m.engine(16, 16)
            eng.set_mask(mask, b)
            ms = eng.profile_ops(b)
            names = eng.op_names()
            mask_ms = sum(t for n, t in zip(names, ms) if n in MASK_OPS)
            rec[dt if dt == "fp32" else "bf16_layerwise"] = {
                "samples_per_s": b / best[dt], "forward_ms_sum_of_ops": sum(ms), "mask_ops_ms": mask_ms,
                "mask_ops_share": mask_ms / sum(ms), "n_mask_ops": sum(n in MASK_OPS for n in names)}
        rec["speedup_bf16_layerwise_over_fp32"] = best["fp32"] / best["bf16"]
        rec["final_latent_rel_l2_bf16_vs_fp32"] = float((out["bf16"] - out["fp32"]).double().norm() / out["fp32"].double().norm())
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
