"""sampler() / decode_latents() / g2rgb() (SURVEY.md section 8(f) N1): host logic checked on CPU with a toy velocity
model and a toy codec; against the unmodified reference's sampler where a checkout exists (oracle/_ref or FLOCODER_REFERENCE)."""
import pytest
import torch
from torch import nn

from flocoder_b200 import sampling
from oracle import ref_shim


class ToyFlow(nn.Module):
    """A small class-conditional velocity field with the reference U-Net's call signature."""
    def __init__(self, n_classes=10):
        super().__init__()
        self.conv = nn.Conv2d(4, 4, 3, padding=1)
        self.emb = nn.Embedding(n_classes, 4)

    def forward(self, x, time, cond=None):
        v = self.conv(x) * torch.cos(time / 999.0).view(-1, 1, 1, 1)
        if cond is not None and cond.get("class_cond") is not None:
            v = v + self.emb(cond["class_cond"]).view(-1, 4, 1, 1)
        return v


class ToyCodec(nn.Module):
    def __init__(self, out_ch=3):
        super().__init__()
        self.dec = nn.Conv2d(4, out_ch, 1)
        self.enc = nn.Conv2d(3, 4, 1)

    def decode(self, z):
        return torch.sigmoid(self.dec(z))

    def encode(self, img):
        return self.enc(img)[:, :, ::4, ::4][:, :, :16, :16]


def test_g2rgb_quantisation():
    g = torch.tensor([0.0, 0.3, 0.5, 0.74, 0.75, 1.0]).view(1, 1, 1, 6)
    rgb = sampling.g2rgb(g)
    assert rgb.shape == (1, 3, 1, 6)
    assert rgb[0, 0, 0].tolist() == [0, 0, 0, 0, 1, 1]          # red: >= .75
    assert rgb[0, 1, 0].tolist() == [0, 1, 1, 1, 0, 0]          # green: |g - .5| < .25
    assert rgb[0, 2].abs().sum() == 0
    bw = sampling.g2rgb(g, keep_gray=True)
    assert bw[0, :, 0, :].tolist() == [[0, 0, 0, 1, 1, 1]] * 3
    three = torch.rand(2, 3, 4, 4)
    assert sampling.g2rgb(three) is three


def test_decode_latents_chunking_matches_one_shot():
    torch.manual_seed(0)
    codec = ToyCodec()
    z = torch.randn(300, 4, 16, 16)
    with torch.no_grad():
        full = codec.decode(z)
        assert torch.allclose(sampling.decode_latents(codec, z, chunk_size=128), full, atol=1e-6)
        midi = sampling.decode_latents(ToyCodec(out_ch=1), z[:5], is_midi=True)
    assert midi.shape == (5, 3, 16, 16) and set(midi.unique().tolist()) <= {0.0, 1.0}


def test_sampler_semantics():
    torch.manual_seed(1)
    model, codec = ToyFlow().eval(), ToyCodec().eval()
    src = torch.randn(40, 4, 16, 16)
    cond = {}
    torch.manual_seed(7)
    lat, img, nfe = sampling.sampler(model, codec, batch_size=20, n_steps=6, cond=cond, n_classes=10, cfg_strength=2.0, source=src)
    assert lat.shape == (20, 4, 16, 16) and img.shape == (20, 3, 16, 16) and nfe == 24
    assert cond["class_cond"].shape == (20,) and torch.equal(cond["class_cond"][:10], cond["class_cond"][10:])   # 10 classes tiled
    # equals generate_latents with the same conditioning, then a one-shot decode
    ref_lat, _ = sampling.generate_latents(model, (20, 4, 16, 16), "rk4", 6, {"class_cond": cond["class_cond"]}, 2.0, source=src[:20])
    assert torch.allclose(lat, ref_lat, atol=1e-6)
    with torch.no_grad():
        assert torch.allclose(img, codec.decode(ref_lat), atol=1e-6)
    # init image: encoded once, repeated over the batch, integration starts at t = init_strength
    init = torch.rand(3, 64, 64)
    lat2, _, nfe2 = sampling.sampler(model, codec, batch_size=4, n_steps=10, cond={"class_cond": torch.arange(8)}, source=src,
                                     init_image=init, init_strength=0.3)
    with torch.no_grad():
        z0 = codec.encode(init.unsqueeze(0)).repeat(4, 1, 1, 1)
    ref2, _ = sampling.generate_latents(model, (4, 4, 16, 16), "rk4", 10, {"class_cond": torch.arange(4)}, 3.0, source=src[:4],
                                        init_latents=z0, init_strength=0.3)
    assert torch.allclose(lat2, ref2, atol=1e-6) and nfe2 == 28        # n_steps -> int(10 * (1 - 0.3)) = 7 (sampling.py:106)


@pytest.mark.skipif(not ref_shim.available(), reason="needs a flocoder reference checkout (oracle/_ref or FLOCODER_REFERENCE)")
def test_sampler_matches_unmodified_reference():
    _, ref_sampling = ref_shim.load()
    torch.manual_seed(2)
    model, codec = ToyFlow().eval(), ToyCodec().eval()
    src = torch.randn(30, 4, 16, 16)
    torch.manual_seed(11)
    a = sampling.sampler(model, codec, batch_size=30, n_steps=5, cond={}, n_classes=10, cfg_strength=3.0, source=src)
    torch.manual_seed(11)
    b = ref_sampling.sampler(model, codec, batch_size=30, n_steps=5, cond={}, n_classes=10, cfg_strength=3.0, source=src)
    assert torch.allclose(a[0], b[0], atol=1e-6) and torch.allclose(a[1], b[1], atol=1e-6) and a[2] == b[2]
    z = torch.rand(6, 1, 8, 8)
    assert torch.equal(sampling.g2rgb(z), ref_sampling.g2rgb(z)) and torch.equal(sampling.g2rgb(z, True), ref_sampling.g2rgb(z, True))


def test_generate_samples_config_helpers():
    """generate_samples.py:120-138 / general.py:50-75 without Hydra: section precedence and the latent shapes of the
    BASELINE configs (sd: image_size // 8; vqgan: image_size // 2^num_downsamples)."""
    from flocoder_b200.generate import infer_latent_shape, ldcfg
    cfg = {"image_size": 128, "codec": {"choice": "sd", "num_downsamples": 3}, "flow": {"dim_mults": [1, 2, 4, 8], "unet": {"n_classes": 102}}}
    assert infer_latent_shape(cfg) == (4, 16, 16)
    assert ldcfg(cfg, "dim_mults") == [1, 2, 4, 8] and ldcfg(cfg, "num_downsamples") == 3 and ldcfg(cfg, "nope", 5) == 5
    cfg = {"image_size": 128, "codec": {"choice": "vqgan", "num_downsamples": 4, "vq_embedding_dim": 4}}
    assert infer_latent_shape(cfg) == (4, 8, 8)                  # configs/midi_inpainting.yaml
    assert infer_latent_shape({"image_size": 32, "codec": {"choice": "resize"}}) == (3, 32, 32)
    with pytest.raises(ValueError):
        infer_latent_shape({"codec": {"choice": "other"}})
