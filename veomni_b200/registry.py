"""The reference's operator surface, mirrored and (when VeOmni is importable) extended in place.

VeOmni dispatches kernels through two objects (SURVEY.md §8(b)):

* ``OpSlot(op_name, variant)`` placed in generated modeling files and bound by ``_bind_veomni_ops``
  (veomni/ops/dispatch.py:38-102, veomni/models/auto.py:63-103);
* ``KERNEL_REGISTRY`` holding ``KernelSpec``s with a ``HardwareRequirement`` gate
  (veomni/ops/kernel_registry.py:71-172).

This module provides the same three classes with the same names, argument meaning and error behaviour
(``KeyError`` for an unknown implementation, ``RuntimeError`` when the hardware gate fails, ``RuntimeError``
when an unbound slot is called) so code written against ``veomni.ops`` reads the same here, registers the
sm_100a kernels under the implementation name ``"b200"``, and :func:`register` adds the very same specs to
VeOmni's own registry / attention table / Ulysses choke point when the reference is installed:

    model.ops_implementation.rms_norm_implementation: b200
    model.ops_implementation.rotary_pos_emb_implementation: b200
    model.ops_implementation.swiglu_mlp_implementation: b200
    model.ops_implementation.moe_implementation: fused_b200
    model.ops_implementation.attn_implementation: veomni_b200_attention_with_sp
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Callable

import torch

IMPL_NAME = "b200"
ATTN_NAME = "veomni_b200_attention_with_sp"


@dataclass(frozen=True)
class HardwareRequirement:
    device_type: str = "gpu"
    min_compute_capability: int | None = None
    max_compute_capability: int | None = None

    def is_satisfied(self) -> bool:
        if self.device_type == "any":
            return True
        if self.device_type != "gpu":
            raise ValueError(f"Unknown device_type: {self.device_type!r} (expected 'gpu' | 'npu' | 'any')")
        if not torch.cuda.is_available():
            return False
        major, minor = torch.cuda.get_device_capability()
        cc = major * 10 + minor
        if self.min_compute_capability is not None and cc < self.min_compute_capability:
            return False
        if self.max_compute_capability is not None and cc > self.max_compute_capability:
            return False
        return True


@dataclass(frozen=True)
class KernelSpec:
    name: str
    op_name: str
    variant: str
    factory: Callable[[], Callable]
    hardware: HardwareRequirement
    description: str = ""


class KernelRegistry:
    """(op_name, variant) -> {impl_name: KernelSpec}; same contract as veomni.ops.kernel_registry.KernelRegistry."""

    def __init__(self):
        self._specs: dict[tuple[str, str], dict[str, KernelSpec]] = {}

    def register(self, spec: KernelSpec, force: bool = False) -> None:
        bucket = self._specs.setdefault((spec.op_name, spec.variant), {})
        if spec.name in bucket and not force:
            raise ValueError(
                f"Duplicate kernel registration: op='{spec.op_name}', variant='{spec.variant}', name='{spec.name}'"
            )
        bucket[spec.name] = spec

    def resolve(self, op_name: str, variant: str, impl_name: str) -> Callable | None:
        if impl_name == "eager":
            return None
        bucket = self._specs.get((op_name, variant), {})
        if impl_name not in bucket:
            raise KeyError(
                f"Unknown kernel '{impl_name}' for op='{op_name}', variant='{variant}'. Available: {list(bucket) + ['eager']}"
            )
        spec = bucket[impl_name]
        if not spec.hardware.is_satisfied():
            raise RuntimeError(
                f"Kernel '{impl_name}' for op='{op_name}' requires device_type='{spec.hardware.device_type}'"
                f", compute_capability>={spec.hardware.min_compute_capability}, but the current hardware does not satisfy this."
            )
        return spec.factory()

    def list_available(self, op_name: str, variant: str) -> list[str]:
        return list(self._specs.get((op_name, variant), {}).keys())


KERNEL_REGISTRY = KernelRegistry()


class OpSlot:
    """Named dispatch slot; see veomni/ops/dispatch.py:38-102."""

    def __init__(self, op_name: str, variant: str, registry: KernelRegistry | None = None):
        self.op_name, self.variant = op_name, variant
        self._registry = registry or KERNEL_REGISTRY
        self._kernel: Callable | None = None
        self._impl_name: str | None = None

    def bind(self, impl_name: str) -> None:
        self._kernel = self._registry.resolve(self.op_name, self.variant, impl_name)
        self._impl_name = impl_name

    @property
    def use_non_eager_impl(self) -> bool:
        return self._kernel is not None

    def bound_kernel(self) -> Callable | None:
        return self._kernel

    def __call__(self, *args: Any, **kwargs: Any) -> Any:
        if self._kernel is None:
            raise RuntimeError(
                f"OpSlot('{self.op_name}', '{self.variant}') has no kernel bound. "
                "Call .bind() first or check .use_non_eager_impl before calling."
            )
        return self._kernel(*args, **kwargs)


_B200 = HardwareRequirement("gpu", min_compute_capability=100)


def _specs() -> list[KernelSpec]:
    def f_rms():
        from .functional import rms_norm

        return rms_norm

    def f_rope():
        from .functional import apply_rotary_pos_emb

        return apply_rotary_pos_emb

    def f_swiglu():
        from .functional import swiglu_mlp

        return swiglu_mlp

    def f_moe():
        from .moe import moe_experts_forward

        return moe_experts_forward

    def f_ce_causal():
        # bound to the reference's own outer wrapper when VeOmni is installed (label shift + SP reduction live there),
        # else to the mirror in .cross_entropy
        from functools import partial

        from .cross_entropy import ForCausalLMLoss as own, b200_cross_entropy

        try:
            from veomni.ops.kernels.cross_entropy import ForCausalLMLoss as ref_wrapper
        except ImportError:
            ref_wrapper = own
        return partial(ref_wrapper, cross_entropy_fn=b200_cross_entropy)

    def f_ce_seq_cls():
        from functools import partial

        from .cross_entropy import b200_cross_entropy

        from veomni.ops.kernels.cross_entropy import ForSequenceClassificationLoss  # only exists inside VeOmni

        return partial(ForSequenceClassificationLoss, cross_entropy_fn=b200_cross_entropy)

    return [
        KernelSpec(IMPL_NAME, "cross_entropy_loss", "causal", f_ce_causal, _B200,
                   "sm_100a fused linear + cross-entropy (chunked lm_head on cuBLAS, in-place gradient kernel)"),
        KernelSpec(IMPL_NAME, "cross_entropy_loss", "seq_cls", f_ce_seq_cls, _B200,
                   "sm_100a cross-entropy for sequence-classification heads"),
        KernelSpec(IMPL_NAME, "rms_norm", "standard", f_rms, _B200, "sm_100a RMSNorm (bulk-async staged rows)"),
        KernelSpec(IMPL_NAME, "rotary_pos_emb", "full", f_rope, _B200, "sm_100a RoPE"),
        KernelSpec(IMPL_NAME, "swiglu_mlp", "standard", f_swiglu, _B200, "sm_100a SiLU*up between cuBLAS GEMMs"),
        KernelSpec(IMPL_NAME, "moe_experts", "standard", f_moe, _B200, "sm_100a fused MoE (tcgen05 GroupGEMM, EP over NVLink)"),
    ]


for _s in _specs():
    KERNEL_REGISTRY.register(_s, force=True)


def _token_fn_dispatcher(name: str, orig: Callable) -> Callable:
    """Stand-in for the reference's ``chunk_logprobs_function`` / ``chunk_topk_distill_function`` (``name``): when the
    installed ops config selects ``cross_entropy_loss_implementation == "b200"``, the call goes to the function of the
    same name in :mod:`veomni_b200.cross_entropy`, with ``sp_enabled`` read from the reference's parallel state;
    otherwise to ``orig``, unchanged. The selection is process-global, like ``LOSS_MAPPING`` and the shared OpSlots:
    the ops config in force at call time decides. ``orig`` stays reachable as ``_vb200_orig``."""

    def dispatch(*args, **kwargs):
        from veomni.ops.config.singleton import get_ops_config

        cfg = get_ops_config()
        if cfg is not None and getattr(cfg, "cross_entropy_loss_implementation", None) == IMPL_NAME:
            from veomni.distributed.parallel_state import get_parallel_state

            from . import cross_entropy as own

            return getattr(own, name)(*args, sp_enabled=get_parallel_state().sp_enabled, **kwargs)
        return dispatch._vb200_orig(*args, **kwargs)

    dispatch.__name__ = dispatch.__qualname__ = name
    dispatch.__doc__ = orig.__doc__
    dispatch._vb200 = True
    dispatch._vb200_orig = orig
    return dispatch


def register(force: bool = True) -> bool:
    """Plug the kernels into an installed VeOmni. Returns False (and does nothing) if it is not importable."""
    try:
        from veomni.ops import kernel_registry as ref_reg
    except ImportError:
        return False
    for s in _specs():
        ref_reg.KERNEL_REGISTRY.register(
            ref_reg.KernelSpec(name=s.name, op_name=s.op_name, variant=s.variant, factory=s.factory,
                               hardware=ref_reg.HardwareRequirement(device_type="gpu"), description=s.description),
            force=force,
        )
    # attention: a new entry in HF's table, next to veomni_flash_attention_{2,3,4}_with_sp
    from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS

    from .attention import flash_attention_forward

    ALL_ATTENTION_FUNCTIONS.register(ATTN_NAME, flash_attention_forward)
    # Ulysses: the single choke point (veomni/distributed/sequence_parallel/ulysses.py:125-135)
    from . import ulysses

    ulysses.install()
    # async Ulysses (Qwen3-VL / Wan attention front and back end, sequence_parallel/async_ulysses.py:469-503)
    from . import async_ulysses

    async_ulysses.install()
    # cross-entropy: besides the OpSlot, HF's LOSS_MAPPING is filled through a closed name list
    # (veomni/ops/kernels/cross_entropy/__init__.py:336-353,480-516) — add "b200" to it
    try:
        import veomni.ops.kernels.cross_entropy as ref_ce

        from .cross_entropy import b200_cross_entropy

        if not getattr(ref_ce._resolve_cross_entropy_fn, "_vb200", False):
            _orig_resolve = ref_ce._resolve_cross_entropy_fn

            def _resolve_cross_entropy_fn(impl: str):
                return b200_cross_entropy if impl == IMPL_NAME else _orig_resolve(impl)

            _resolve_cross_entropy_fn._vb200 = True
            ref_ce._resolve_cross_entropy_fn = _resolve_cross_entropy_fn
    except Exception:  # noqa: BLE001
        pass
    # per-token log-probs / top-k distillation: ForCausalLMLoss and _chunk_loss_dispatch call these module globals
    # when the caller passes return_log_probs=True (veomni/ops/kernels/cross_entropy/__init__.py:130-177,395-439)
    try:
        import veomni.ops.kernels.cross_entropy as ref_ce

        for name in ("chunk_logprobs_function", "chunk_topk_distill_function"):
            fn = getattr(ref_ce, name)
            if not getattr(fn, "_vb200", False):
                setattr(ref_ce, name, _token_fn_dispatcher(name, fn))
    except Exception:  # noqa: BLE001
        pass
    # fused MoE raw pointer (veomni/ops/kernels/moe/__init__.py:62-108)
    try:
        import veomni.ops.kernels.moe as ref_moe

        from .moe import fused_moe_forward

        _orig = getattr(ref_moe.apply_veomni_fused_moe_patch, "_vb200_orig", ref_moe.apply_veomni_fused_moe_patch)

        def apply_veomni_fused_moe_patch(fused_moe_kernel: str = "triton", *a, **k):
            # same keyword as the reference (ops/kernels/moe/__init__.py:60; called as fused_moe_kernel=... by auto.py:99)
            if fused_moe_kernel in (IMPL_NAME, f"fused_{IMPL_NAME}"):
                ref_moe._fused_moe_forward = fused_moe_forward
                return
            return _orig(fused_moe_kernel, *a, **k)

        apply_veomni_fused_moe_patch._vb200_orig = _orig
        ref_moe.apply_veomni_fused_moe_patch = apply_veomni_fused_moe_patch
    except Exception:  # noqa: BLE001  (reference without the MoE package on this platform)
        pass
    return True
