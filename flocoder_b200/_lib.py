"""ctypes binding of ``include/flocoder_b200.h`` (the C-ABI shared library).

The library is built in-tree by ``python -m flocoder_b200.build`` (nvcc, sm_100a) into
``flocoder_b200/_C/libflocoder_b200.so``.  If it is missing this module raises -- the product
path never falls back to PyTorch or to the CPU oracle.
"""
from __future__ import annotations

import ctypes
import weakref
import math
import os
from ctypes import (POINTER, Structure, byref, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t,
                    c_void_p, create_string_buffer)
from typing import Dict, Optional, Sequence

import torch

LIB_PATH = os.environ.get("FLO_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_C", "libflocoder_b200.so")   # FLO_LIB: A/B-test another build of the same ABI

FLO_OK, FLO_ERR_INVALID, FLO_ERR_UNSUPPORTED, FLO_ERR_CUDA, FLO_ERR_NOMEM, FLO_ERR_STEP = 0, -1, -2, -3, -4, -5
FLO_F32, FLO_BF16, FLO_F16 = 0, 1, 2
FLO_RK4, FLO_EULER_LEGACY, FLO_EULER_GRID = 0, 1, 2
FLO_FLAG_NO_BUFFER_REUSE, FLO_FLAG_NO_GRAPH, FLO_FLAG_LAYERWISE = 1, 2, 4

# every symbol include/flocoder_b200.h declares (tests/test_cabi.py checks the .so exports them)
EXPORTS = (
    "flo_version", "flo_last_error", "flo_param_count", "flo_param_info", "flo_unet_create",
    "flo_unet_destroy", "flo_unet_set_time_freqs", "flo_workspace_bytes", "flo_unet_forward", "flo_integrate", "flo_integrate_host",
    "flo_integrate_nfe", "flo_unet_num_ops", "flo_unet_op_name", "flo_unet_launches_per_forward",
    "flo_unet_launch_count", "flo_unet_read_activation", "flo_selftest_umma", "flo_describe_plan",
    "flo_unet_op_info", "flo_unet_profile_ops", "flo_unet_read_timeline", "flo_unet_set_mask",
    "flo_integrate_rk45", "flo_integrate_rk45_timing", "flo_integrate_rk45_per_sample", "flo_integrate_rk45_reverse",
    "flo_integrate_rk45_per_sample_reverse", "flo_unet_jvp", "flo_integrate_divergence",
)


class FloUnetCfg(Structure):
    _fields_ = [
        ("dim", c_int32), ("channels", c_int32), ("n_mults", c_int32), ("mults", c_int32 * 8),
        ("groups", c_int32), ("n_classes", c_int32), ("height", c_int32), ("width", c_int32),
        ("compute_dtype", c_int32), ("mask_cond", c_int32), ("flags", c_int32), ("device", c_int32),
    ]


_lib_handle = None


def lib() -> ctypes.CDLL:
    """Load the C-ABI library (once).  Fails loudly when it has not been built."""
    global _lib_handle
    if _lib_handle is not None:
        return _lib_handle
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the flocoder_b200 CUDA extension is not built. "
            "Run `python -m flocoder_b200.build` (needs nvcc with sm_100a support). "
            "There is no PyTorch/CPU fallback for this path.")
    L = ctypes.CDLL(LIB_PATH)
    L.flo_version.restype = c_int
    L.flo_last_error.restype = c_char_p
    L.flo_param_count.argtypes = [POINTER(FloUnetCfg)]
    L.flo_param_info.argtypes = [POINTER(FloUnetCfg), c_int, c_char_p, c_int, POINTER(c_int64), POINTER(c_int)]
    L.flo_unet_create.argtypes = [POINTER(c_void_p), POINTER(FloUnetCfg), POINTER(c_void_p), c_int, c_void_p]
    L.flo_unet_destroy.argtypes = [c_void_p]
    L.flo_unet_set_time_freqs.argtypes = [c_void_p, POINTER(c_float), c_int]
    L.flo_workspace_bytes.argtypes = [c_void_p, c_int]
    L.flo_workspace_bytes.restype = c_size_t
    L.flo_unet_forward.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]
    L.flo_integrate.argtypes = [c_void_p, c_void_p, POINTER(c_float), c_int, c_int, c_float, c_float,
                                c_void_p, c_float, c_void_p, c_int, c_void_p]
    L.flo_integrate_host.argtypes = [c_void_p, c_void_p, c_void_p, POINTER(c_float), c_int, c_int, c_float,
                                     c_float, c_void_p, c_float, c_int, c_void_p]
    L.flo_unet_set_mask.argtypes = [c_void_p, c_void_p, c_int, c_void_p]
    L.flo_integrate_rk45.argtypes = [c_void_p, c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                     ctypes.c_double, c_float, c_void_p, c_float, c_int, POINTER(c_int), c_int, c_void_p]
    L.flo_integrate_rk45_reverse.argtypes = L.flo_integrate_rk45.argtypes
    L.flo_integrate_rk45_timing.argtypes = [c_void_p, POINTER(ctypes.c_double)]
    L.flo_integrate_rk45_per_sample.argtypes = [c_void_p, c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                                ctypes.c_double, c_float, c_void_p, c_float, c_int, POINTER(ctypes.c_int32),
                                                c_int, c_void_p]
    L.flo_integrate_rk45_per_sample_reverse.argtypes = L.flo_integrate_rk45_per_sample.argtypes
    L.flo_unet_jvp.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]
    L.flo_integrate_divergence.argtypes = [c_void_p, c_void_p, POINTER(c_float), c_int, c_float, c_void_p, c_void_p, c_int,
                                           c_void_p, c_int, c_void_p]
    L.flo_integrate_nfe.argtypes = [c_int, c_int]
    L.flo_unet_num_ops.argtypes = [c_void_p]
    L.flo_unet_op_name.argtypes = [c_void_p, c_int, c_char_p, c_int]
    L.flo_unet_launches_per_forward.argtypes = [c_void_p, c_int]
    L.flo_unet_launch_count.argtypes = [c_void_p]
    L.flo_unet_launch_count.restype = c_int64
    L.flo_unet_read_activation.argtypes = [c_void_p, c_char_p, c_int, c_void_p, c_int64, POINTER(c_int64),
                                           c_void_p]
    L.flo_selftest_umma.argtypes = [c_char_p, c_int, c_void_p]
    L.flo_describe_plan.argtypes = [POINTER(FloUnetCfg), c_int, c_char_p, c_int]
    L.flo_unet_op_info.argtypes = [c_void_p, c_int, POINTER(c_int), POINTER(ctypes.c_double), POINTER(ctypes.c_double)]
    L.flo_unet_profile_ops.argtypes = [c_void_p, c_int, c_int, POINTER(c_float), c_void_p]
    L.flo_unet_read_timeline.argtypes = [c_void_p, c_int, c_int, POINTER(ctypes.c_longlong)]
    _lib_handle = L
    return L


def check(status: int, what: str = "") -> None:
    """Map flo_status to the exception class the reference's Python surface would raise."""
    if status >= 0:
        return
    msg = lib().flo_last_error()
    msg = msg.decode() if msg else "unknown error"
    text = f"{what}: {msg}" if what else msg
    if status == FLO_ERR_INVALID:
        raise ValueError(text)
    if status == FLO_ERR_UNSUPPORTED:
        raise NotImplementedError(text)
    if status == FLO_ERR_NOMEM:
        raise MemoryError(text)
    raise RuntimeError(text)


def make_cfg(dim, channels, dim_mults, groups, n_classes, height, width, compute_dtype, device_index,
             flags=0, mask_cond=False) -> FloUnetCfg:
    if len(dim_mults) > 8:
        raise ValueError("at most 8 resolution levels are supported")
    cfg = FloUnetCfg()
    cfg.dim, cfg.channels, cfg.n_mults = dim, channels, len(dim_mults)
    for i, m in enumerate(dim_mults):
        cfg.mults[i] = int(m)
    cfg.groups, cfg.n_classes, cfg.height, cfg.width = groups, n_classes, height, width
    cfg.compute_dtype = {"fp32": FLO_F32, "bf16": FLO_BF16, "fp16": FLO_F16}[compute_dtype]
    cfg.mask_cond, cfg.flags, cfg.device = int(bool(mask_cond)), flags, device_index
    return cfg


def param_manifest(cfg: FloUnetCfg):
    """[(name, shape)] in reference state_dict order, as the C side expects them."""
    L = lib()
    n = L.flo_param_count(byref(cfg))
    check(n, "flo_param_count")
    out = []
    name = create_string_buffer(256)
    shape = (c_int64 * 4)()
    ndim = c_int()
    for i in range(n):
        check(L.flo_param_info(byref(cfg), i, name, 256, shape, byref(ndim)), "flo_param_info")
        out.append((name.value.decode(), tuple(shape[j] for j in range(ndim.value))))
    return out


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class Engine:
    """Owns one ``flo_unet_t`` (packed weights + workspaces) for one module state on one device."""

    def __init__(self, *, dim, channels, dim_mults, groups, n_classes, height, width, compute_dtype,
                 device, state_dict: Dict[str, torch.Tensor], flags: int = 0, mask_cond: bool = False):
        self.L = lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("flocoder_b200 runs only on CUDA devices (sm_100a); no CPU fallback")
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        self.channels, self.height, self.width = channels, height, width
        self.compute_dtype = compute_dtype
        self.mask_cond = bool(mask_cond)
        self.cfg = make_cfg(dim, channels, dim_mults, groups, n_classes, height, width, compute_dtype,
                            index, flags, mask_cond)
        manifest = param_manifest(self.cfg)
        tensors = []
        for name, shape in manifest:
            if name not in state_dict:
                raise KeyError(f"state_dict is missing '{name}'")
            t = state_dict[name]
            if tuple(t.shape) != shape:
                raise ValueError(f"'{name}' has shape {tuple(t.shape)}, expected {shape}")
            tensors.append(t.detach().to(device=self.device, dtype=torch.float32).contiguous())
        ptrs = (c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
        self.handle = c_void_p()
        with torch.cuda.device(self.device):
            check(self.L.flo_unet_create(byref(self.handle), byref(self.cfg), ptrs, len(tensors),
                                         _stream_ptr(self.device)), "flo_unet_create")
            torch.cuda.current_stream(self.device).synchronize()   # packing reads `tensors`
            # sinusoidal frequencies exactly as the reference forms them (unet.py:26-27): torch.exp in fp32
            half = dim // 2
            freqs = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1)))
            check(self.L.flo_unet_set_time_freqs(self.handle, (c_float * half)(*freqs.tolist()), half),
                  "flo_unet_set_time_freqs")
        del tensors

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.L.flo_unet_destroy(self.handle)
            self.handle = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- calls ---------------------------------------------------------------------------
    def _check_class_range(self, c: torch.Tensor):
        """nn.Embedding (class_cond_mlp.0, unet.py:207) raises IndexError for ids outside [0, n_classes); the kernel
        would clamp them silently.  One min/max per distinct tensor: a trajectory validates its ids once, and the
        per-evaluation calls of the generic rk4_step path see the cached verdict."""
        n = int(self.cfg.n_classes)
        if n <= 0 or c.numel() == 0:
            return
        ok = getattr(self, "_cls_ok", None)          # (weak reference to the validated tensor object, its version counter)
        if ok is not None and ok[0]() is c and ok[1] == c._version:
            return
        lo, hi = int(c.min()), int(c.max())
        if lo < 0 or hi >= n:
            raise IndexError(f"class_cond holds ids in [{lo}, {hi}] but the model has n_classes={n} "
                             "(index out of range in self, as nn.Embedding reports it)")
        self._cls_ok = (weakref.ref(c), c._version)

    def _cls_ptr(self, class_ids, b):
        if class_ids is None:
            return None, None
        self._check_class_range(class_ids)
        c = class_ids.to(device=self.device, dtype=torch.int64).contiguous().reshape(-1)
        if c.numel() != b:
            raise ValueError(f"class_cond must have {b} elements, got {c.numel()}")
        return c, c.data_ptr()

    def set_mask(self, mask: Optional[torch.Tensor], b: int) -> None:
        """cond['mask_cond'] for the following calls at batch size ``b`` (``flo_unet_set_mask``): resized to every level
        and tested against the reference's all-ones bypass on the device.  ``None`` switches every mask branch off.
        Sent before every forward / trajectory (two small launches): the library keeps the state per batch-size plan, and a
        plan can be evicted and rebuilt between calls, so nothing is cached on this side."""
        if not self.mask_cond:
            return                                   # unet.py:298: no mask_fusion_conv -> cond['mask_cond'] is ignored
        ptr = None
        if mask is not None:
            if tuple(mask.shape) != (b, self.channels, self.height, self.width):
                raise ValueError(f"mask_cond must be [{b},{self.channels},{self.height},{self.width}] (the latent shape, "
                                 f"unet.py:302), got {tuple(mask.shape)}")
            keep = mask.detach().to(device=self.device, dtype=torch.float32).contiguous()
            ptr = keep.data_ptr()
        with torch.cuda.device(self.device):
            check(self.L.flo_unet_set_mask(self.handle, ptr, b, _stream_ptr(self.device)), "flo_unet_set_mask")

    def forward(self, x: torch.Tensor, time: torch.Tensor, class_ids: Optional[torch.Tensor]) -> torch.Tensor:
        b = x.shape[0]
        v = torch.empty_like(x)
        keep, cptr = self._cls_ptr(class_ids, b)
        with torch.cuda.device(self.device):
            check(self.L.flo_unet_forward(self.handle, x.data_ptr(), time.data_ptr(), cptr, v.data_ptr(), b,
                                          _stream_ptr(self.device)), "flo_unet_forward")
        return v

    def jvp(self, x: torch.Tensor, time: torch.Tensor, class_ids: Optional[torch.Tensor], dx: torch.Tensor):
        """``(v, dv)``: the velocity at ``x`` and the Jacobian-vector products ``dv[p] = J_x v . dx[p]`` (``flo_unet_jvp``,
        exact forward mode on the fp32 path).  ``x`` [B,C,H,W], ``dx`` [P,B,C,H,W], fp32 contiguous on the engine's device."""
        assert x.dtype == torch.float32 and x.is_contiguous() and x.device == self.device
        assert dx.dtype == torch.float32 and dx.is_contiguous() and dx.device == self.device and dx.dim() == 5
        b, n_tan = x.shape[0], dx.shape[0]
        v, dv = torch.empty_like(x), torch.empty_like(dx)
        keep, cptr = self._cls_ptr(class_ids, b)
        with torch.cuda.device(self.device):
            check(self.L.flo_unet_jvp(self.handle, x.data_ptr(), time.data_ptr(), cptr, dx.data_ptr(), n_tan, v.data_ptr(),
                                      dv.data_ptr(), b, _stream_ptr(self.device)), "flo_unet_jvp")
        return v, dv

    def integrate_divergence(self, y: torch.Tensor, ts: Sequence[float], probes: torch.Tensor, t_scale: float = 999.0,
                             class_ids=None) -> torch.Tensor:
        """RK4 over ``ts`` in place on ``y`` with the Hutchinson divergence of the fixed ``probes`` [P,B,C,H,W] at every
        stage (``flo_integrate_divergence``).  Returns ``div`` [B] fp64 on the device: sum over the intervals of
        ``dt/6 (d1 + 2 d2 + 2 d3 + d4)``, ``d = mean_p probe_p . (J v probe_p)``."""
        assert y.dtype == torch.float32 and y.is_contiguous() and y.device == self.device
        assert probes.dtype == torch.float32 and probes.is_contiguous() and probes.device == self.device
        b = y.shape[0]
        ts_arr = (c_float * len(ts))(*[float(t) for t in ts])
        div = torch.empty(b, dtype=torch.float64, device=self.device)
        keep, cptr = self._cls_ptr(class_ids, b)
        with torch.cuda.device(self.device):
            check(self.L.flo_integrate_divergence(self.handle, y.data_ptr(), ts_arr, len(ts), float(t_scale), cptr,
                                                  probes.data_ptr(), probes.shape[0], div.data_ptr(), b,
                                                  _stream_ptr(self.device)), "flo_integrate_divergence")
        return div

    def integrate(self, y: torch.Tensor, ts: Sequence[float], method: int, dt: float = 0.0,
                  t_scale: float = 999.0, class_ids=None, cfg_strength: float = 0.0,
                  v_trace: Optional[torch.Tensor] = None) -> torch.Tensor:
        """In place on ``y`` ([B,C,H,W] fp32 contiguous, on the engine's device)."""
        assert y.dtype == torch.float32 and y.is_contiguous() and y.device == self.device
        b = y.shape[0]
        ts_arr = (c_float * len(ts))(*[float(t) for t in ts])
        keep, cptr = self._cls_ptr(class_ids, b)
        with torch.cuda.device(self.device):
            check(self.L.flo_integrate(self.handle, y.data_ptr(), ts_arr, len(ts), method, float(dt),
                                       float(t_scale), cptr, float(cfg_strength),
                                       None if v_trace is None else v_trace.data_ptr(), b,
                                       _stream_ptr(self.device)), "flo_integrate")
        return y

    def integrate_rk45(self, y: torch.Tensor, t0: float, t1: float = 1.0, rtol: float = 1e-5, atol: float = 1e-5,
                       t_scale: float = 999.0, class_ids=None, cfg_strength: float = 0.0, max_steps: int = 10000,
                       reverse: bool = False):
        """Adaptive Dormand-Prince 5(4) from ``t0`` to ``t1`` in place on ``y`` (``flo_integrate_rk45``: scipy's RK45 step
        control on the device, one host wait per attempt).  Returns ``(nfev, accepted, rejected)``; raises RuntimeError
        when the step size collapses or ``max_steps`` attempts do not reach ``t1``.  ``reverse=True`` integrates backwards
        from ``t0`` down to ``t1 < t0`` (``flo_integrate_rk45_reverse``)."""
        assert y.dtype == torch.float32 and y.is_contiguous() and y.device == self.device
        b = y.shape[0]
        keep, cptr = self._cls_ptr(class_ids, b)
        counts = (c_int * 3)()
        fn = "flo_integrate_rk45_reverse" if reverse else "flo_integrate_rk45"
        with torch.cuda.device(self.device):
            check(getattr(self.L, fn)(self.handle, y.data_ptr(), float(t0), float(t1), float(rtol), float(atol),
                                      float(t_scale), cptr, float(cfg_strength), int(max_steps), counts, b,
                                      _stream_ptr(self.device)), fn)
        return counts[0], counts[1], counts[2]

    def integrate_rk45_per_sample(self, y: torch.Tensor, t0: float, t1: float = 1.0, rtol: float = 1e-5,
                                  atol: float = 1e-5, t_scale: float = 999.0, class_ids=None, cfg_strength: float = 0.0,
                                  max_steps: int = 10000, reverse: bool = False) -> torch.Tensor:
        """As :meth:`integrate_rk45`, but every sample is its own RK45 problem with its own step-size control
        (``flo_integrate_rk45_per_sample``, or ``flo_integrate_rk45_per_sample_reverse`` with ``reverse=True``).
        Returns the CPU int64 tensor ``[B, 3]`` of per-sample ``(nfev, accepted, rejected)``; raises RuntimeError naming
        the sample when one fails."""
        assert y.dtype == torch.float32 and y.is_contiguous() and y.device == self.device
        b = y.shape[0]
        keep, cptr = self._cls_ptr(class_ids, b)
        counts = (ctypes.c_int32 * (3 * b))()
        fn = "flo_integrate_rk45_per_sample_reverse" if reverse else "flo_integrate_rk45_per_sample"
        with torch.cuda.device(self.device):
            check(getattr(self.L, fn)(self.handle, y.data_ptr(), float(t0), float(t1), float(rtol), float(atol),
                                      float(t_scale), cptr, float(cfg_strength), int(max_steps), counts, b,
                                      _stream_ptr(self.device)), fn)
        return torch.tensor(list(counts), dtype=torch.int64).reshape(b, 3)

    def rk45_timing(self):
        """(attempts, host wall ms, attempt-graph device ms) of the last :meth:`integrate_rk45` or
        :meth:`integrate_rk45_per_sample` call, either direction (per-sample: attempts of the whole batch, the most any
        sample made)."""
        out = (ctypes.c_double * 3)()
        check(self.L.flo_integrate_rk45_timing(self.handle, out), "flo_integrate_rk45_timing")
        return int(out[0]), out[1], out[2]

    def integrate_host(self, x0: torch.Tensor, x1: torch.Tensor, ts: Sequence[float], method: int,
                       dt: float = 0.0, t_scale: float = 999.0, class_ids=None, cfg_strength: float = 0.0):
        """Host-buffer entry: x0/x1 are CPU fp32 tensors (pinned for full PCIe speed)."""
        assert x0.device.type == "cpu" and x1.device.type == "cpu"
        assert x0.dtype == torch.float32 and x1.dtype == torch.float32
        assert x0.is_contiguous() and x1.is_contiguous()
        b = x0.shape[0]
        ts_arr = (c_float * len(ts))(*[float(t) for t in ts])
        cptr = None
        if class_ids is not None:
            self._check_class_range(class_ids)
            keep = class_ids.to(device="cpu", dtype=torch.int64).contiguous()
            cptr = keep.data_ptr()
        with torch.cuda.device(self.device):
            check(self.L.flo_integrate_host(self.handle, x0.data_ptr(), x1.data_ptr(), ts_arr, len(ts), method,
                                            float(dt), float(t_scale), cptr, float(cfg_strength), b,
                                            _stream_ptr(self.device)), "flo_integrate_host")
        return x1

    # -- introspection -------------------------------------------------------------------
    def op_names(self):
        n = self.L.flo_unet_num_ops(self.handle)
        buf = create_string_buffer(256)
        out = []
        for i in range(n):
            check(self.L.flo_unet_op_name(self.handle, i, buf, 256))
            out.append(buf.value.decode())
        return out

    def op_info(self):
        """[(name, kind, algorithmic flops per sample, algorithmic bytes per sample)] per op."""
        out = []
        kind, fl, by = c_int(), ctypes.c_double(), ctypes.c_double()
        for i, name in enumerate(self.op_names()):
            check(self.L.flo_unet_op_info(self.handle, i, byref(kind), byref(fl), byref(by)))
            out.append((name, kind.value, fl.value, by.value))
        return out

    def profile_ops(self, b: int, reps: int = 5):
        """Best-of-`reps` CUDA-event duration (ms) of every kernel of one forward at batch b."""
        n = self.L.flo_unet_num_ops(self.handle)
        ms = (c_float * n)()
        with torch.cuda.device(self.device):
            check(self.L.flo_unet_profile_ops(self.handle, b, reps, ms, _stream_ptr(self.device)),
                  "flo_unet_profile_ops")
        return list(ms)

    def read_timeline(self, b: int, stage: int):
        out = (ctypes.c_longlong * 128)()
        check(self.L.flo_unet_read_timeline(self.handle, b, stage, out), "flo_unet_read_timeline")
        return list(out)

    def launches_per_forward(self, b: int) -> int:
        n = self.L.flo_unet_launches_per_forward(self.handle, b)
        check(n, "flo_unet_launches_per_forward")
        return n

    def launch_count(self) -> int:
        return int(self.L.flo_unet_launch_count(self.handle))

    def workspace_bytes(self, b: int) -> int:
        return int(self.L.flo_workspace_bytes(self.handle, b))

    def read_activation(self, name: str, b: int) -> torch.Tensor:
        shape = (c_int64 * 4)()
        cap = 1 << 24
        out = torch.empty(cap, dtype=torch.float32)
        with torch.cuda.device(self.device):
            check(self.L.flo_unet_read_activation(self.handle, name.encode(), b, out.data_ptr(), cap, shape,
                                                  _stream_ptr(self.device)), f"read_activation({name})")
        shp = tuple(shape[i] for i in range(4))
        n = shp[0] * shp[1] * shp[2] * shp[3]
        return out[:n].reshape(shp).clone()


def describe_plan(cfg: FloUnetCfg, b: int) -> str:
    """Host-only description of the op program / buffers / tcgen05 tilings (no GPU needed)."""
    buf = create_string_buffer(1 << 20)
    check(lib().flo_describe_plan(byref(cfg), b, buf, len(buf)), "flo_describe_plan")
    return buf.value.decode()


def selftest_umma() -> tuple:
    L = lib()
    buf = create_string_buffer(1 << 16)
    rc = L.flo_selftest_umma(buf, len(buf), _stream_ptr(torch.device("cuda", torch.cuda.current_device())))
    return rc, buf.value.decode()
