"""Freeze outputs of the UNMODIFIED reference into ``tests/golden/*.pt``.

TEST INFRASTRUCTURE ONLY.  Needs a checkout of the unmodified reference:

    python -m oracle.make_golden      # the checkout at oracle/_ref, or FLOCODER_REFERENCE=/path/to/flocoder

For each of the three U-Nets the BASELINE configs name (n_classes = 102 flowers_sd,
0 midi_vqgan, 10 stl_sd; SURVEY.md section 8) it seeds torch with 1234, builds the
reference ``Unet(dim=16, channels=4, dim_mults=[1,2,4,8], n_classes=N)``, draws the
latents from ``torch.Generator().manual_seed(5678)`` and records what the reference
computes on CPU in fp32.  Weights are NOT stored (10 MB each): they are regenerated
from the seed by ``flocoder_b200.unet.Unet`` -- whose construction order mirrors the
reference's so the RNG stream lines up -- and checked against the fingerprints stored
here.
"""
from __future__ import annotations

import hashlib
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_shim  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MODEL_SEED, NOISE_SEED, B = 1234, 5678, 8
CONFIGS = {"flowers_sd": 102, "midi_vqgan": 0, "stl_sd": 10}


def fingerprint(sd):
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(v.detach().contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


def main():
    ref_unet, ref_sampling = ref_shim.load()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(os.cpu_count())
    for name, n_classes in CONFIGS.items():
        torch.manual_seed(MODEL_SEED)
        model = ref_unet.Unet(dim=16, channels=4, dim_mults=[1, 2, 4, 8], n_classes=n_classes).eval()
        sd = model.state_dict()
        x0 = torch.randn(B, 4, 16, 16, generator=torch.Generator().manual_seed(NOISE_SEED))
        g = {
            "config": name, "n_classes": n_classes, "model_seed": MODEL_SEED, "noise_seed": NOISE_SEED,
            "torch_version": torch.__version__,
            "sd_sha256": fingerprint(sd), "sd_names": list(sd.keys()),
            "sd_abs_sum": float(sum(v.double().abs().sum() for v in sd.values())),
            "n_params": sum(p.numel() for p in model.parameters()),
            "x0": x0.clone(),
        }
        with torch.no_grad():
            t = torch.full((B,), 0.25 * 999)
            g["fwd_t"] = t.clone()
            g["fwd_v"] = model(x0, t).clone()
            # per-sample distinct times (the forward() API takes a [B] vector)
            tv = torch.linspace(0.0, 1.0, B) * 999
            g["fwd_tvec"] = tv.clone()
            g["fwd_v_tvec"] = model(x0, tv).clone()
            if n_classes > 0:
                cls = torch.arange(B) % n_classes
                g["cls"] = cls.clone()
                g["fwd_v_cls"] = model(x0, t, cond={"class_cond": cls}).clone()
            # integrators
            x1, nfe = ref_sampling.generate_latents_rk4(model, (B, 4, 16, 16), n_steps=10, source=x0.clone())
            g["rk4_10"], g["rk4_10_nfe"] = x1.clone(), nfe
            x1, nfe = ref_sampling.generate_latents(model, (B, 4, 16, 16), method="rk4", n_steps=50,
                                                    source=x0.clone())
            g["rk4_50"], g["rk4_50_nfe"] = x1.clone(), nfe
            g["euler_10"] = ref_shim.reference_euler(model, x0, 10).clone()
            if n_classes > 0:
                x1, _ = ref_sampling.generate_latents_rk4(model, (B, 4, 16, 16), n_steps=10,
                                                          cond={"class_cond": cls}, cfg_strength=3.0,
                                                          source=x0.clone())
                g["rk4_10_cfg3"] = x1.clone()
                x1, _ = ref_sampling.generate_latents_rk4(model, (B, 4, 16, 16), n_steps=10,
                                                          cond={"class_cond": cls}, cfg_strength=0,
                                                          source=x0.clone())
                g["rk4_10_cls_nocfg"] = x1.clone()
            # init-latents ("img2img") branch, sampling.py:104-109
            init = torch.randn(B, 4, 16, 16, generator=torch.Generator().manual_seed(NOISE_SEED + 1))
            g["init_latents"] = init.clone()
            x1, nfe = ref_sampling.generate_latents_rk4(model, (B, 4, 16, 16), n_steps=10, source=x0.clone(),
                                                        init_latents=init, init_strength=0.3)
            g["rk4_10_init03"], g["rk4_10_init03_nfe"] = x1.clone(), nfe
            g["ts_50"] = ref_sampling.warp_time(torch.linspace(0, 1, 50)).clone()
        path = os.path.join(GOLDEN_DIR, f"{name}.pt")
        torch.save(g, path)
        print(f"{name}: |x0|={x0.norm():.6f} |v|={g['fwd_v'].norm():.6f} |rk4_10|={g['rk4_10'].norm():.6f} "
              f"|euler_10|={g['euler_10'].norm():.6f} |rk4_50|={g['rk4_50'].norm():.6f} -> {path} "
              f"({os.path.getsize(path)/1024:.0f} KiB)")


# ---- inpainting U-Net (SURVEY.md 8f N3): mask_cond=True, cond['mask_cond'] from the reference's MaskEncoder --------------
INPAINT_CONFIGS = {
    # name: (dim, latent H = W, pixel-mask size)    -- midi_inpainting.yaml: latent (4, 8, 8), Unet(dim=H) (train_flow.py:291)
    "inpaint_16": (16, 16, 256),
    "midi_inpainting": (8, 8, 128),
}


def main_inpaint():
    """``python -m oracle.make_golden inpaint`` -> tests/golden/{inpaint_16,midi_inpainting}.pt"""
    ref_unet, ref_sampling = ref_shim.load()
    import flocoder.inpainting as ref_inp
    torch.set_num_threads(os.cpu_count())
    for name, (dim, hw, mask_px) in INPAINT_CONFIGS.items():
        torch.manual_seed(MODEL_SEED)
        model = ref_unet.Unet(dim=dim, channels=4, dim_mults=[1, 2, 4, 8], n_classes=0, mask_cond=True).eval()
        sd = model.state_dict()
        torch.manual_seed(MODEL_SEED + 1)
        enc = ref_inp.MaskEncoder().eval()                                  # train_flow.py:239
        shape = (B, 4, hw, hw)
        x0 = torch.randn(shape, generator=torch.Generator().manual_seed(NOISE_SEED))
        # pixel-space masks: one rectangle per sample (1 = region to inpaint), seeded
        gen = torch.Generator().manual_seed(NOISE_SEED + 2)
        mask_pixels = torch.zeros(B, 1, mask_px, mask_px)
        for i in range(B):
            y0, x0_ = (torch.randint(0, mask_px // 2, (2,), generator=gen)).tolist()
            hh, ww = (torch.randint(mask_px // 8, mask_px // 2, (2,), generator=gen)).tolist()
            mask_pixels[i, 0, y0:y0 + hh, x0_:x0_ + ww] = 1.0
        with torch.no_grad():
            mask_latents = enc(mask_pixels)                                 # [B,4,hw,hw] (inpainting.py:234-245)
            assert tuple(mask_latents.shape) == shape, mask_latents.shape
            cond = {"mask_cond": mask_latents}
            g = {
                "config": name, "dim": dim, "hw": hw, "model_seed": MODEL_SEED, "noise_seed": NOISE_SEED,
                "torch_version": torch.__version__, "sd_sha256": fingerprint(sd), "sd_names": list(sd.keys()),
                "n_params": sum(p.numel() for p in model.parameters()),
                "x0": x0.clone(), "mask_pixels": mask_pixels.to(torch.uint8), "mask_latents": mask_latents.clone(),
                "enc_sd_sha256": fingerprint(enc.state_dict()), "enc_sd_names": list(enc.state_dict().keys()),
            }
            t = torch.full((B,), 0.25 * 999)
            g["fwd_t"] = t.clone()
            g["fwd_v_mask"] = model(x0, t, cond=cond).clone()
            g["fwd_v_nomask"] = model(x0, t).clone()                         # every mask branch skipped (key_usable false)
            g["fwd_v_ones"] = model(x0, t, cond={"mask_cond": torch.ones(shape)}).clone()   # unet.py:301 bypass, scale fusions stay
            half = mask_latents.clone(); half[: B // 2] = 1.0                # some samples all ones: no bypass (batch-wide test)
            g["mask_half"] = half.clone()
            g["fwd_v_half"] = model(x0, t, cond={"mask_cond": half}).clone()
            x1, _ = ref_sampling.generate_latents_rk4(model, shape, n_steps=10, cond=cond, source=x0.clone())
            g["rk4_10_mask"] = x1.clone()
            g["euler_10_mask"] = ref_shim.reference_euler(model, x0, 10, cond=cond).clone()
        path = os.path.join(GOLDEN_DIR, f"{name}.pt")
        torch.save(g, path)
        print(f"{name}: |v_mask|={g['fwd_v_mask'].norm():.6f} |v_nomask|={g['fwd_v_nomask'].norm():.6f} "
              f"|v_ones|={g['fwd_v_ones'].norm():.6f} |rk4_10|={g['rk4_10_mask'].norm():.6f} -> {path} "
              f"({os.path.getsize(path)/1024:.0f} KiB)")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "inpaint":
        main_inpaint()
    else:
        main()
