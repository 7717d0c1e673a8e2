"""``Unet`` -- drop-in for ``flocoder.unet.Unet`` on the sampling path (inference).

Same constructor arguments, same ``state_dict`` names/shapes/order and the same
``forward(x, time, cond=None)`` contract as the reference (``flocoder/unet.py:164-377``),
but the module tree only *holds parameters*: the forward pass is one call into the
sm_100a C-ABI library (``include/flocoder_b200.h``), never PyTorch ops.  There is no CPU
or eager fallback -- off-GPU, or without the built library, ``forward`` raises.

Construction order of the parameterised leaves (Conv2d / Linear / Embedding) follows the
reference's ``__init__`` (``unet.py:185-286``) so that the same ``torch.manual_seed`` yields
bit-identical random-init weights; ``tests/test_unet_module.py`` checks this against the
frozen fingerprints in ``tests/golden``.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence

import torch
from torch import nn

from . import _lib

HEADS, DIM_HEAD = 4, 32          # unet.py:100,126 defaults; Unet never overrides them


def key_usable(d, key) -> bool:
    """general.py:18-20."""
    return (d is not None) and isinstance(d, dict) and (d.get(key) is not None)


class _Holder(nn.Module):
    """A parameter container whose children are registered under explicit names
    (including numeric ones such as ``"1"``), so state_dict keys match the reference's
    ``nn.Sequential`` / wrapper nesting without reproducing those classes."""

    def put(self, name: str, module: nn.Module) -> nn.Module:
        self.add_module(str(name), module)
        return module


def _resnet_holder(dim_in: int, dim_out: int, time_dim: int, groups: int) -> _Holder:
    """Parameters of ResnetBlock (unet.py:76-86): mlp.1, block{1,2}.{proj,norm}, [res_conv]."""
    rb = _Holder()
    rb.put("mlp", _Holder()).put("1", nn.Linear(time_dim, dim_out * 2))
    for name, cin in (("block1", dim_in), ("block2", dim_out)):
        blk = rb.put(name, _Holder())
        blk.put("proj", nn.Conv2d(cin, dim_out, 3, padding=1))
        blk.put("norm", nn.GroupNorm(groups, dim_out))
    if dim_in != dim_out:
        rb.put("res_conv", nn.Conv2d(dim_in, dim_out, 1))
    return rb


def _attn_holder(dim: int, linear: bool) -> _Holder:
    """Residual(PreNorm(dim, [Linear]Attention(dim))) -> '<p>.fn.fn.*' then '<p>.fn.norm.*'
    (unet.py:33-39,99-106,125-133,153-157)."""
    hidden = HEADS * DIM_HEAD
    core = _Holder()
    core.put("to_qkv", nn.Conv2d(dim, hidden * 3, 1, bias=False))
    if linear:
        out = core.put("to_out", _Holder())
        out.put("0", nn.Conv2d(hidden, dim, 1))
        out.put("1", nn.GroupNorm(1, dim))
    else:
        core.put("to_out", nn.Conv2d(hidden, dim, 1))
    prenorm = _Holder()
    prenorm.put("fn", core)
    prenorm.put("norm", nn.GroupNorm(1, dim))
    res = _Holder()
    res.put("fn", prenorm)
    return res


class Unet(nn.Module):
    """Velocity-field U-Net whose forward runs on hand-written sm_100a kernels.

    Extra (non-reference) keyword: ``compute_dtype`` -- ``None`` (follow the parameter
    dtype: fp32 params -> fp32 kernels, bf16 params -> bf16 tensor-core kernels),
    ``"fp32"`` or ``"bf16"`` (e.g. fp32 master parameters with bf16 tcgen05 convolutions).
    Time embedding, MLPs, GroupNorm statistics, softmax and the integrator state are fp32
    in every mode.
    """

    def __init__(self, dim, dim_mults=(1, 2, 4, 8), channels=3, resnet_block_groups=4,
                 n_classes=10, mask_cond=False, use_checkpoint=False, compute_dtype: Optional[str] = None):
        super().__init__()
        self.mask_cond = bool(mask_cond)              # inpainting U-Net (unet.py:214-235): fp32 kernels, or bf16 with
                                                      # engine_flags = FLO_FLAG_LAYERWISE
        self.use_checkpoint = use_checkpoint          # accepted for signature parity; inference only
        self.dim = dim
        self.dim_mults = tuple(int(m) for m in dim_mults)
        self.channels = channels
        self.out_dim = channels
        self.groups = resnet_block_groups
        self.n_classes = int(n_classes)
        self.class_condition = n_classes > 0
        self.compute_dtype = compute_dtype

        dims = [dim] + [dim * m for m in self.dim_mults]
        in_out = list(zip(dims[:-1], dims[1:]))
        time_dim = dim * 8
        g = resnet_block_groups

        self.init_conv = nn.Conv2d(channels, dim, 1, padding=0)
        self.time_mlp = _Holder()
        self.time_mlp.put("1", nn.Linear(dim, time_dim))
        self.time_mlp.put("3", nn.Linear(time_dim, time_dim))
        if self.class_condition:
            self.class_cond_mlp = _Holder()
            self.class_cond_mlp.put("0", nn.Embedding(n_classes, time_dim))
            self.class_cond_mlp.put("1", nn.Linear(time_dim, time_dim))
            self.class_cond_mlp.put("3", nn.Linear(time_dim, time_dim))

        if self.mask_cond:                            # unet.py:214-235: nn.Sequential indices 0, 2, 4 / 0 hold the convs
            self.mask_fusion_conv = _Holder()
            self.mask_fusion_conv.put("0", nn.Conv2d(dim + channels, 2 * dim, 5, padding=2))
            self.mask_fusion_conv.put("2", nn.Conv2d(2 * dim, 2 * dim, 3, padding=1))
            self.mask_fusion_conv.put("4", nn.Conv2d(2 * dim, dim, 3, padding=1))
            self.down_mask_fusions = nn.ModuleList()
            for d_in, _ in in_out[:2]:
                fuse = _Holder()
                fuse.put("0", nn.Conv2d(d_in + channels, d_in, 3, padding=1))
                self.down_mask_fusions.append(fuse)
            self.up_mask_fusions = nn.ModuleList()
            for _, d_out in list(reversed(in_out))[:2]:
                fuse = _Holder()
                fuse.put("0", nn.Conv2d(d_out + channels, d_out, 3, padding=1))
                self.up_mask_fusions.append(fuse)

        # registration order (downs, ups, mid, final) fixes the state_dict order; construction
        # order (downs, mid, ups, final) fixes the RNG stream -- both as in unet.py:238-286
        self.downs = nn.ModuleList()
        self.ups = nn.ModuleList()
        n_res = len(in_out)
        for i, (d_in, d_out) in enumerate(in_out):
            last = i >= n_res - 1
            stage = nn.ModuleList([
                _resnet_holder(d_in, d_in, time_dim, g),
                _resnet_holder(d_in, d_in, time_dim, g),
                _attn_holder(d_in, linear=True),
            ])
            if last:
                stage.append(nn.Conv2d(d_in, d_out, 3, padding=1))
            else:
                down = _Holder()
                down.put("1", nn.Conv2d(d_in * 4, d_out, 1))
                stage.append(down)
            self.downs.append(stage)

        mid = dims[-1]
        self.mid_block1 = _resnet_holder(mid, mid, time_dim, g)
        self.mid_attn = _attn_holder(mid, linear=False)
        self.mid_block2 = _resnet_holder(mid, mid, time_dim, g)

        for i, (d_in, d_out) in enumerate(reversed(in_out)):
            last = i == n_res - 1
            stage = nn.ModuleList([
                _resnet_holder(d_out + d_in, d_out, time_dim, g),
                _resnet_holder(d_out + d_in, d_out, time_dim, g),
                _attn_holder(d_out, linear=True),
            ])
            if last:
                stage.append(nn.Conv2d(d_out, d_in, 3, padding=1))
            else:
                up = _Holder()
                up.put("1", nn.Conv2d(d_out, d_in, 3, padding=1))
                stage.append(up)
            self.ups.append(stage)

        self.final_res_block = _resnet_holder(dim * 2, dim, time_dim, g)
        self.final_conv = nn.Conv2d(dim, channels, 1)

        self._engine = None
        self._engine_key = None
        self.engine_flags = 0           # _lib.FLO_FLAG_* (e.g. FLO_FLAG_LAYERWISE: one kernel per layer)

    # ------------------------------------------------------------------ engine
    def _resolved_compute_dtype(self) -> str:
        if self.compute_dtype is not None:
            if self.compute_dtype not in ("fp32", "bf16", "fp16"):
                raise ValueError(f"compute_dtype must be None, 'fp32', 'bf16' or 'fp16', got {self.compute_dtype!r}")
            return self.compute_dtype
        p = next(self.parameters())
        if p.dtype == torch.float32:
            return "fp32"
        if p.dtype == torch.bfloat16:
            return "bf16"
        if p.dtype == torch.float16:
            return "fp16"
        raise TypeError(f"unsupported parameter dtype {p.dtype}: the B200 path computes in fp32 or bf16")

    def _params_key(self, height: int, width: int):
        ps = list(self.parameters())
        return (ps[0].device, self._resolved_compute_dtype(), height, width, self.engine_flags,
                tuple(p.data_ptr() for p in ps), tuple(p._version for p in ps))

    def engine(self, height: int, width: int) -> "_lib.Engine":
        """The native handle for this module's current parameters (re-packed when they change)."""
        key = self._params_key(height, width)
        if self._engine is None or key != self._engine_key:
            dev = key[0]
            if dev.type != "cuda":
                raise RuntimeError(
                    "flocoder_b200.Unet runs only on a CUDA (sm_100a) device; there is no CPU fallback. "
                    f"Parameters are on {dev}.")
            if self._engine is not None:
                self._engine.close()
            sd = self.state_dict()
            self._engine = _lib.Engine(
                dim=self.dim, channels=self.channels, dim_mults=self.dim_mults, groups=self.groups,
                n_classes=self.n_classes, height=height, width=width, compute_dtype=key[1],
                device=dev, state_dict=sd, flags=self.engine_flags, mask_cond=self.mask_cond)
            self._engine_key = key
        return self._engine

    def invalidate(self):
        if self._engine is not None:
            self._engine.close()
        self._engine, self._engine_key = None, None

    @staticmethod
    def split_cond(cond):
        """Returns the class-id tensor (or None) exactly as unet.py:298,313-320 would consume ``cond``."""
        if cond is None:
            return None
        if not isinstance(cond, dict):
            # the reference's non-dict branch dies on warnings.DeprecationWarning (unet.py:318)
            raise TypeError("non-dict cond is not supported; use cond={'class_cond': LongTensor[B]}")
        return cond.get("class_cond")

    def mask_of(self, cond):
        """cond['mask_cond'] if this module consumes it (unet.py:298: key_usable and hasattr(self, 'mask_fusion_conv'))."""
        return cond["mask_cond"] if (self.mask_cond and key_usable(cond, "mask_cond")) else None

    # ----------------------------------------------------------------- forward
    @torch.no_grad()
    def forward(self, x: torch.Tensor, time: torch.Tensor, cond=None) -> torch.Tensor:
        """x: [B,C,H,W]; time: [B] already scaled by 999 (sampling.py:63); returns v [B,C,H,W]."""
        if x.dim() != 4 or x.shape[1] != self.channels:
            raise ValueError(f"x must be [B,{self.channels},H,W], got {tuple(x.shape)}")
        cls = self.split_cond(cond)
        if cls is not None and not self.class_condition:
            cls = None                                   # unet.py:315 hasattr(self,'class_cond_mlp')
        b, _, h, w = x.shape
        eng = self.engine(h, w)
        if x.device != eng.device:
            raise RuntimeError(f"x is on {x.device} but the model is on {eng.device}")
        time = time.to(device=x.device, dtype=torch.float32).reshape(-1)
        if time.numel() != b:
            raise ValueError(f"time must have {b} elements, got {time.numel()}")
        eng.set_mask(self.mask_of(cond), b)
        v = eng.forward(x.to(torch.float32).contiguous(), time.contiguous(), cls)
        return v.to(x.dtype)

    def check_jvp_supported(self, height: int, width: int) -> None:
        """NotImplementedError unless :meth:`jvp` has kernels for this module at ``height x width``: the fp32 path only,
        no inpainting mask branches (their convolutions apply SiLU), at most 256 pixels (linear attention)."""
        if self._resolved_compute_dtype() != "fp32":
            raise NotImplementedError(f"JVPs run on the fp32 path only, this model computes in {self._resolved_compute_dtype()}")
        if self.mask_cond:
            raise NotImplementedError("JVPs of the inpainting U-Net (mask_cond=True) are not supported")
        if height * width > 256:
            raise NotImplementedError(f"JVPs need at most 256 latent pixels (linear attention), got {height}x{width}")

    @torch.no_grad()
    def jvp(self, x: torch.Tensor, time: torch.Tensor, tangents: torch.Tensor, cond=None):
        """``(v, dv)`` with ``v = forward(x, time, cond)`` and ``dv = J_x v . tangents``: exact forward-mode Jacobian-vector
        products, several tangents per sample in one pass.  ``tangents`` is ``[B,C,H,W]`` or ``[P,B,C,H,W]``; ``dv`` has its
        shape.  fp32 path only (NotImplementedError for 16-bit models, ``mask_cond`` and more than 256 pixels)."""
        if x.dim() != 4 or x.shape[1] != self.channels:
            raise ValueError(f"x must be [B,{self.channels},H,W], got {tuple(x.shape)}")
        single = tangents.dim() == 4
        dx = tangents.unsqueeze(0) if single else tangents
        if dx.dim() != 5 or tuple(dx.shape[1:]) != tuple(x.shape) or dx.shape[0] < 1:
            raise ValueError(f"tangents must be {tuple(x.shape)} or [P,{','.join(map(str, x.shape))}], got {tuple(tangents.shape)}")
        cls = self.split_cond(cond)
        if cls is not None and not self.class_condition:
            cls = None
        b, _, h, w = x.shape
        self.check_jvp_supported(h, w)
        eng = self.engine(h, w)
        if x.device != eng.device or dx.device != eng.device:
            raise RuntimeError(f"x / tangents are on {x.device} / {dx.device} but the model is on {eng.device}")
        time = time.to(device=x.device, dtype=torch.float32).reshape(-1)
        if time.numel() != b:
            raise ValueError(f"time must have {b} elements, got {time.numel()}")
        v, dv = eng.jvp(x.to(torch.float32).contiguous(), time.contiguous(), cls, dx.to(torch.float32).contiguous())
        return v.to(x.dtype), (dv[0] if single else dv).to(tangents.dtype)


def infer_unet_config(state_dict) -> dict:
    """U-Net constructor arguments recoverable from a reference ``state_dict`` (``generate_samples.py:91-101`` infers only
    ``dim`` and ``channels`` from ``init_conv.weight`` and takes the rest from a Hydra config):
    ``dim`` / ``channels`` from ``init_conv.weight [dim, channels, 1, 1]``; ``dim_mults`` from the output width of every
    level's down-sampling conv (``downs.{l}.3[.1].weight``, ``unet.py:251-255``); ``n_classes`` from the class embedding
    (``class_cond_mlp.0.weight [n_classes, time_dim]``, ``unet.py:206-212``; 0 if absent).  GroupNorm group counts are not
    stored in a state dict (reference default 4)."""
    w0 = state_dict["init_conv.weight"]
    dim, channels = int(w0.shape[0]), int(w0.shape[1])
    mults, level = [], 0
    while True:
        key = next((k for k in (f"downs.{level}.3.1.weight", f"downs.{level}.3.weight") if k in state_dict), None)
        if key is None:
            break
        dout = int(state_dict[key].shape[0])
        if dout % dim:
            raise ValueError(f"{key}: width {dout} is not a multiple of dim={dim}")
        mults.append(dout // dim)
        level += 1
    if not mults:
        raise ValueError("state_dict has no 'downs.*' levels: not a flocoder U-Net checkpoint")
    emb = state_dict.get("class_cond_mlp.0.weight")
    cfg = {"dim": dim, "channels": channels, "dim_mults": mults, "n_classes": int(emb.shape[0]) if emb is not None else 0}
    if "mask_fusion_conv.0.weight" in state_dict:          # inpainting checkpoint (train_flow.py:291 mask_cond=inpainting)
        cfg["mask_cond"] = True
    return cfg


def unet_from_checkpoint(checkpoint, device=None, compute_dtype=None, strict=False, **overrides) -> "Unet":
    """Build a :class:`Unet` from a flocoder flow checkpoint (a path to ``flow_*.pt`` / a dict with ``model_state_dict``,
    as written by ``train_flow.py``, or a bare ``state_dict``) the way ``generate_samples.py:78-108`` does — minus its
    invalid ``condition=`` keyword — and load the weights with the reference's ``strict=False``.  ``overrides`` replace
    inferred constructor arguments (e.g. ``resnet_block_groups``)."""
    if isinstance(checkpoint, (str, bytes)) or hasattr(checkpoint, "__fspath__"):
        checkpoint = torch.load(checkpoint, map_location="cpu", weights_only=False)
    sd = checkpoint["model_state_dict"] if "model_state_dict" in checkpoint else checkpoint
    cfg = infer_unet_config(sd)
    cfg.update(overrides)
    model = Unet(compute_dtype=compute_dtype, **cfg)
    missing, unexpected = model.load_state_dict(sd, strict=strict)
    model.load_report = {"missing": list(missing), "unexpected": list(unexpected), "config": cfg}
    if device is not None:
        model = model.to(device)
    return model.eval()
