"""CPU oracle for the flocoder latent flow-matching sampling path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``flocoder_b200/`` imports this
package; only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline``
/ ``--impl reference`` legs of ``bench.py`` may.  The product path is the CUDA
extension and fails loudly when it is missing.

Parity status: the reference ships no golden vectors or known-answer tests for
this path (its ``tests/test_flow.py`` is a 0-byte file), so the oracle is
pinned against *outputs of the unmodified reference itself*, imported in the
build container by ``oracle/ref_shim.py`` and frozen into ``tests/golden/`` by
``oracle/make_golden.py``.
"""
from .unet_oracle import (UnetSpec, Precision, unet_forward, FP32, BF16_MATCHED, FUSED_BF16,  # noqa: F401
                          FUSED_FP16, trained_like)
from .sampling_oracle import (  # noqa: F401
    warp_time, rk4_step, v_func_cfg, generate_latents_rk4, generate_latents, euler_sampler,
    rk4_stage_times,
)
