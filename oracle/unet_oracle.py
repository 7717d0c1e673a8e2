"""Functional CPU restatement of the flocoder velocity-field U-Net (test oracle).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.

The network is restated as one pure function of ``(state_dict, x, time, cond)``
instead of the reference's ``nn.Module`` tree, so that every intermediate can be
named, traced and (for the bf16 parity bar) rounded at exactly the points where
the CUDA path stores bf16.  Each helper cites the reference lines it follows
(paths relative to ``/root/reference``).

Precision policies
------------------
``FP32``          plain fp32/fp64 arithmetic: must equal the imported reference
                  to rounding noise (tests/test_oracle.py).
``BF16_MATCHED``  the same arithmetic with the operands of every tensor-core
                  convolution (all 3x3/1x1 convs except ``init_conv`` and
                  ``final_conv``) rounded to bf16, fp32 accumulation, and q/k/v
                  rounded to bf16 where the CUDA path stores them; time
                  embedding, MLPs, GroupNorm, softmax and residual adds stay
                  fp32.  This is the "precision-matched oracle" of SURVEY.md
                  section 8c: it separates implementation error from the bf16
                  format error.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
HEADS = 4        # unet.py:100,126 (defaults, never overridden by Unet)
DIM_HEAD = 32    # unet.py:100,126


@dataclass(frozen=True)
class UnetSpec:
    """Constructor arguments of the reference ``Unet`` (unet.py:165-175)."""
    dim: int = 16
    dim_mults: Sequence[int] = (1, 2, 4, 8)
    channels: int = 4
    groups: int = 4
    n_classes: int = 0

    @property
    def dims(self) -> List[int]:            # unet.py:189
        return [self.dim] + [self.dim * m for m in self.dim_mults]

    @property
    def in_out(self):                       # unet.py:190
        d = self.dims
        return list(zip(d[:-1], d[1:]))

    @property
    def time_dim(self) -> int:              # unet.py:197
        return self.dim * 8


@dataclass(frozen=True)
class Precision:
    name: str = "fp32"
    gemm_operands_bf16: bool = False   # round conv inputs+weights (tensor-core convs) to the 16-bit type
    qkv_store_bf16: bool = False       # round to_qkv outputs where the layer-by-layer CUDA path stores 16-bit
    stream_16: bool = False            # fused path: the residual stream itself (block / attention / conv outputs)
                                       # is stored in the 16-bit type between ops
    dtype16: torch.dtype = torch.bfloat16

    def _r(self, t: Tensor) -> Tensor:
        return t.to(self.dtype16).to(t.dtype)

    def op(self, t: Tensor) -> Tensor:
        return self._r(t) if self.gemm_operands_bf16 else t

    def qkv(self, t: Tensor) -> Tensor:
        return self._r(t) if self.qkv_store_bf16 else t

    def act(self, t: Tensor) -> Tensor:
        return self._r(t) if self.stream_16 else t


FP32 = Precision("fp32")
BF16_MATCHED = Precision("bf16_matched", gemm_operands_bf16=True, qkv_store_bf16=True)
FUSED_BF16 = Precision("fused_bf16", gemm_operands_bf16=True, stream_16=True)
FUSED_FP16 = Precision("fused_fp16", gemm_operands_bf16=True, stream_16=True, dtype16=torch.float16)


def trained_like(sd: Dict[str, Tensor], seed: int = 3, qkv_scale: float = 4.0) -> Dict[str, Tensor]:
    """New weights with statistics a trained checkpoint has and default init lacks.  Not a model of any real checkpoint.

    Default init leaves every GroupNorm at gamma = 1, beta = 0, so a kernel that drops beta or reads gamma at the wrong
    channel computes the same numbers, and it gives q / k logits with a standard deviation of ~0.5, so the softmaxes are
    nearly uniform and pairing values with the wrong pixel barely moves the output.  Here:

    * every GroupNorm affine (``*.norm`` and the linear attention's ``*.to_out.1``) gets gamma = 1 + 0.3 N(0, 1) and
      beta = 0.3 N(0, 1), per channel;
    * every ``*.to_qkv.weight`` is multiplied by ``qkv_scale`` (x4 puts the logit std at ~2: sharp softmaxes);
    * every other tensor is returned unchanged (as a copy).

    Deterministic in ``seed``: values are drawn in fp32 in sorted key order and cast to each tensor's dtype, so an fp32
    state dict and its fp64 copy give the same weights."""
    gen = torch.Generator().manual_seed(seed)
    out = {}
    for k in sorted(sd):
        v = sd[k]
        affine = k.endswith((".norm.weight", ".norm.bias", ".to_out.1.weight", ".to_out.1.bias"))
        if affine:
            z = 0.3 * torch.randn(v.shape, generator=gen, dtype=torch.float32)
            v = (1 + z if k.endswith(".weight") else z).to(dtype=v.dtype, device=v.device)
        elif k.endswith(".to_qkv.weight"):
            v = v * qkv_scale
        out[k] = v.detach().clone()
    return {k: out[k] for k in sd}


def key_usable(d, key) -> bool:
    """general.py:18-20."""
    return (d is not None) and isinstance(d, dict) and (d.get(key) is not None)


# ----------------------------------------------------------------------------
# leaf ops
# ----------------------------------------------------------------------------

def sinusoidal_embedding(time: Tensor, dim: int) -> Tensor:
    """unet.py:23-30: [sin(t f_j), cos(t f_j)], f_j = exp(-j ln(1e4)/(half-1)), in time.dtype."""
    half = dim // 2
    c = math.log(10000) / (half - 1)
    freqs = torch.exp(torch.arange(half, device=time.device, dtype=time.dtype) * -c)
    arg = time[:, None] * freqs[None, :]
    return torch.cat((arg.sin(), arg.cos()), dim=-1)


def _conv(sd, name: str, x: Tensor, pad: int, prec: Precision, tensor_core: bool = True) -> Tensor:
    w = sd[name + ".weight"]
    b = sd.get(name + ".bias")
    if tensor_core:
        x, w = prec.op(x), prec.op(w)
    return F.conv2d(x, w, b, padding=pad)


def _linear(sd, name: str, x: Tensor) -> Tensor:
    return F.linear(x, sd[name + ".weight"], sd[name + ".bias"])


def _group_norm(sd, name: str, x: Tensor, groups: int) -> Tensor:
    """nn.GroupNorm(groups, C) with eps=1e-5 (unet.py:61,133,157)."""
    return F.group_norm(x, groups, sd[name + ".weight"], sd[name + ".bias"], eps=1e-5)


def block(sd, p: str, x: Tensor, groups: int, scale_shift, prec: Precision, tr=None) -> Tensor:
    """unet.py:64-73: conv3x3 -> GN -> [x*(scale+1)+shift] -> SiLU."""
    h = _conv(sd, p + ".proj", x, 1, prec)
    if tr is not None:
        tr[p + ".proj"] = h
    h = _group_norm(sd, p + ".norm", h, groups)
    if scale_shift is not None:
        scale, shift = scale_shift
        h = h * (scale + 1) + shift
    h = F.silu(h)
    if tr is not None:
        tr[p] = h
    return h


def resnet_block(sd, p: str, x: Tensor, t_emb: Tensor, groups: int, prec: Precision, tr=None) -> Tensor:
    """unet.py:88-96."""
    ss = _linear(sd, p + ".mlp.1", F.silu(t_emb))             # unet.py:79-82,90
    ss = ss[:, :, None, None]                                   # 'b c -> b c 1 1'
    scale, shift = ss.chunk(2, dim=1)                           # unet.py:92
    h = block(sd, p + ".block1", x, groups, (scale, shift), prec, tr)
    h = block(sd, p + ".block2", h, groups, None, prec, tr)
    if (p + ".res_conv.weight") in sd:                          # unet.py:86
        res = _conv(sd, p + ".res_conv", x, 0, prec)
    else:
        res = x
    out = prec.act(h + res)
    if tr is not None:
        tr[p] = out
    return out


def linear_attention(sd, p: str, x: Tensor, prec: Precision) -> Tensor:
    """unet.py:135-150 (p is the LinearAttention prefix, '...fn.fn')."""
    b, c, hh, ww = x.shape
    n = hh * ww
    qkv = prec.qkv(_conv(sd, p + ".to_qkv", x, 0, prec))       # [b, 3*128, h, w], no bias
    q, k, v = (t.reshape(b, HEADS, DIM_HEAD, n) for t in qkv.chunk(3, dim=1))
    q = q.softmax(dim=-2)                                       # over the 32 head channels
    k = k.softmax(dim=-1)                                       # over pixels
    q = q * (DIM_HEAD ** -0.5)
    context = torch.einsum("bhdn,bhen->bhde", k, v)
    out = torch.einsum("bhde,bhdn->bhen", context, q)
    out = out.reshape(b, HEADS * DIM_HEAD, hh, ww)
    out = _conv(sd, p + ".to_out.0", out, 0, prec)
    return _group_norm(sd, p + ".to_out.1", out, 1)


def attention(sd, p: str, x: Tensor, prec: Precision) -> Tensor:
    """unet.py:108-122 (p is the Attention prefix, 'mid_attn.fn.fn')."""
    b, c, hh, ww = x.shape
    n = hh * ww
    qkv = prec.qkv(_conv(sd, p + ".to_qkv", x, 0, prec))
    q, k, v = (t.reshape(b, HEADS, DIM_HEAD, n) for t in qkv.chunk(3, dim=1))
    q = q * (DIM_HEAD ** -0.5)
    sim = torch.einsum("bhdi,bhdj->bhij", q, k)
    sim = sim - sim.amax(dim=-1, keepdim=True)
    attn = sim.softmax(dim=-1)
    out = torch.einsum("bhij,bhdj->bhid", attn, v)
    out = out.permute(0, 1, 3, 2).reshape(b, HEADS * DIM_HEAD, hh, ww)   # 'b h (x y) d -> b (h d) x y'
    return _conv(sd, p + ".to_out", out, 0, prec)


def residual_prenorm(sd, p: str, x: Tensor, fn, prec: Precision, tr=None) -> Tensor:
    """Residual(PreNorm(dim, fn)): fn(GN1(x)) + x  (unet.py:38-39,159-161)."""
    xn = _group_norm(sd, p + ".fn.norm", x, 1)
    y = prec.act(fn(sd, p + ".fn.fn", xn, prec) + x)
    if tr is not None:
        tr[p + ".fn.norm"] = xn
        tr[p] = y
    return y


def downsample(sd, p: str, x: Tensor, prec: Precision) -> Tensor:
    """unet.py:51-54: 'b c (h p1) (w p2) -> b (c p1 p2) h w' then 1x1 conv."""
    return _conv(sd, p + ".1", F.pixel_unshuffle(x, 2), 0, prec)


def upsample(sd, p: str, x: Tensor, prec: Precision) -> Tensor:
    """unet.py:43-46: nearest x2 then 3x3 conv."""
    return _conv(sd, p + ".1", F.interpolate(x, scale_factor=2, mode="nearest"), 1, prec)


# ----------------------------------------------------------------------------
# the network
# ----------------------------------------------------------------------------

def time_conditioning(sd, spec: UnetSpec, time: Tensor, cond) -> Tensor:
    """unet.py:310-320: time_mlp(time) (+ class_cond_mlp(class ids))."""
    e = sinusoidal_embedding(time, spec.dim)
    t = _linear(sd, "time_mlp.3", F.gelu(_linear(sd, "time_mlp.1", e)))
    if cond is not None and isinstance(cond, dict):
        if cond.get("class_cond") is not None and "class_cond_mlp.0.weight" in sd:
            c = F.embedding(cond["class_cond"], sd["class_cond_mlp.0.weight"])
            c = _linear(sd, "class_cond_mlp.3", F.gelu(_linear(sd, "class_cond_mlp.1", c)))
            t = t + c
    return t


def unet_forward(sd: Dict[str, Tensor], spec: UnetSpec, x: Tensor, time: Tensor,
                 cond: Optional[dict] = None, prec: Precision = FP32,
                 trace: Optional[Dict[str, Tensor]] = None) -> Tensor:
    """unet.py:289-372.  ``time`` is already scaled by 999 (sampling.py:63)."""
    g = spec.groups
    tr = trace
    n_res = len(spec.in_out)

    x = prec.act(_conv(sd, "init_conv", x, 0, prec, tensor_core=False))   # unet.py:295
    if tr is not None:
        tr["init_conv"] = x
    # inpainting (SURVEY.md 8f N3): the mask branches exist iff the module was built with mask_cond=True, i.e. iff the
    # state dict holds their weights (unet.py:298 hasattr(self, 'mask_fusion_conv'))
    use_mask = key_usable(cond, "mask_cond") and "mask_fusion_conv.0.weight" in sd
    mask = cond["mask_cond"] if use_mask else None
    if use_mask and not torch.allclose(mask, torch.ones_like(mask)):    # unet.py:301: all-ones mask bypasses the fusion
        xf = torch.cat([x, mask], dim=1)                                # unet.py:302
        xf = F.silu(_conv(sd, "mask_fusion_conv.0", xf, 2, prec))       # unet.py:215-221 (5x5, 3x3, 3x3; SiLU between)
        xf = F.silu(_conv(sd, "mask_fusion_conv.2", xf, 1, prec))
        x = _conv(sd, "mask_fusion_conv.4", xf, 1, prec)                # unet.py:305: no residual
        if tr is not None:
            tr["mask_fusion_conv"] = x
    r = x                                                              # unet.py:308 (clone)
    t = time_conditioning(sd, spec, time, cond)
    if tr is not None:
        tr["t_emb"] = t

    skips: List[Tensor] = []
    for i in range(n_res):                                             # unet.py:326-343
        p = f"downs.{i}"
        x = resnet_block(sd, p + ".0", x, t, g, prec, tr)
        skips.append(x)
        x = resnet_block(sd, p + ".1", x, t, g, prec, tr)
        x = residual_prenorm(sd, p + ".2", x, linear_attention, prec, tr)
        skips.append(x)
        if use_mask and i < 2 and f"down_mask_fusions.{i}.0.weight" in sd:          # unet.py:336-340
            m = F.interpolate(mask, size=x.shape[-2:], mode="bilinear")
            x = x + F.silu(_conv(sd, f"down_mask_fusions.{i}.0", torch.cat([x, m], dim=1), 1, prec))
            if tr is not None:
                tr[f"down_mask_fusions.{i}.0"] = x
        if i < n_res - 1:
            x = prec.act(downsample(sd, p + ".3", x, prec))
        else:
            x = prec.act(_conv(sd, p + ".3", x, 1, prec))
        if tr is not None:
            tr[p + ".3"] = x

    x = resnet_block(sd, "mid_block1", x, t, g, prec, tr)              # unet.py:345-347
    x = residual_prenorm(sd, "mid_attn", x, attention, prec, tr)
    x = resnet_block(sd, "mid_block2", x, t, g, prec, tr)

    for i in range(n_res):                                             # unet.py:350-367
        p = f"ups.{i}"
        x = torch.cat((x, skips.pop()), dim=1)
        x = resnet_block(sd, p + ".0", x, t, g, prec, tr)
        x = torch.cat((x, skips.pop()), dim=1)
        x = resnet_block(sd, p + ".1", x, t, g, prec, tr)
        x = residual_prenorm(sd, p + ".2", x, linear_attention, prec, tr)
        if use_mask and i < 2 and f"up_mask_fusions.{i}.0.weight" in sd:            # unet.py:360-364
            m = F.interpolate(mask, size=x.shape[-2:], mode="bilinear")
            x = x + F.silu(_conv(sd, f"up_mask_fusions.{i}.0", torch.cat([x, m], dim=1), 1, prec))
            if tr is not None:
                tr[f"up_mask_fusions.{i}.0"] = x
        if i < n_res - 1:
            x = prec.act(upsample(sd, p + ".3", x, prec))
        else:
            x = prec.act(_conv(sd, p + ".3", x, 1, prec))
        if tr is not None:
            tr[p + ".3"] = x

    x = torch.cat((x, r), dim=1)                                       # unet.py:369
    x = resnet_block(sd, "final_res_block", x, t, g, prec, tr)
    out = _conv(sd, "final_conv", x, 0, prec, tensor_core=False)       # unet.py:372
    if tr is not None:
        tr["final_conv"] = out
    return out


class OracleModel:
    """Callable ``model(x, time, cond=None)`` over a state_dict, for the integrator oracle.

    Exposes ``parameters()`` because ``generate_latents_rk4`` derives device and
    dtype from ``next(model.parameters())`` (sampling.py:96).
    """

    def __init__(self, sd: Dict[str, Tensor], spec: UnetSpec, prec: Precision = FP32):
        self.sd, self.spec, self.prec = sd, spec, prec
        self.calls = 0

    def parameters(self):
        return iter(self.sd.values())

    def __call__(self, x, time, cond=None):
        self.calls += 1
        with torch.no_grad():
            return unet_forward(self.sd, self.spec, x, time, cond, self.prec)
