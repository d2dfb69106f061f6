"""The OpSlot / KERNEL_REGISTRY mirror keeps the reference's contract (veomni/ops/dispatch.py, kernel_registry.py)."""
import pytest

from veomni_b200 import registry as R


def test_eager_resolves_to_none_and_unknown_raises_keyerror():
    assert R.KERNEL_REGISTRY.resolve("rms_norm", "standard", "eager") is None
    with pytest.raises(KeyError):
        R.KERNEL_REGISTRY.resolve("rms_norm", "standard", "does_not_exist")
    assert "b200" in R.KERNEL_REGISTRY.list_available("rms_norm", "standard")
    for op, var in (("rotary_pos_emb", "full"), ("swiglu_mlp", "standard"), ("moe_experts", "standard"),
                    ("cross_entropy_loss", "causal"), ("cross_entropy_loss", "seq_cls")):
        assert "b200" in R.KERNEL_REGISTRY.list_available(op, var)


def test_unbound_slot_raises_and_eager_binding_is_falsy():
    slot = R.OpSlot("rms_norm", "standard")
    assert not slot.use_non_eager_impl
    with pytest.raises(RuntimeError):
        slot(1, 2, 3)
    slot.bind("eager")
    assert not slot.use_non_eager_impl and slot.bound_kernel() is None


def test_hardware_gate_fails_loudly_without_a_b200():
    import torch

    if torch.cuda.is_available() and torch.cuda.get_device_capability()[0] >= 10:
        pytest.skip("a Blackwell GPU is present")
    slot = R.OpSlot("rms_norm", "standard")
    with pytest.raises(RuntimeError):
        slot.bind("b200")  # no silent CPU fallback


def test_duplicate_registration_rejected():
    reg = R.KernelRegistry()
    spec = R.KernelSpec("x", "op", "v", lambda: (lambda: 1), R.HardwareRequirement("any"))
    reg.register(spec)
    with pytest.raises(ValueError):
        reg.register(spec)
    reg.register(spec, force=True)
    assert reg.resolve("op", "v", "x")() == 1


def test_register_into_the_real_reference_when_present():
    """With the reference package built into oracle/_ref (oracle/build_ref.py), the b200 kernels land in ITS registry."""
    import sys

    from oracle.build_ref import REF_DIR

    if not (REF_DIR / "veomni").is_dir():
        pytest.skip("oracle/_ref holds no reference package (build() found no reference source)")
    sys.path.insert(0, str(REF_DIR))
    try:
        assert R.register() is True
        from transformers.modeling_utils import ALL_ATTENTION_FUNCTIONS
        from veomni.ops.kernel_registry import KERNEL_REGISTRY as REF

        for op, var in (("rms_norm", "standard"), ("rotary_pos_emb", "full"), ("swiglu_mlp", "standard"), ("moe_experts", "standard"),
                        ("cross_entropy_loss", "causal"), ("cross_entropy_loss", "seq_cls")):
            assert "b200" in REF.list_available(op, var)
        # the causal-LM loss factory binds OUR kernel into THEIR wrapper (label shift + SP reduce stay theirs)
        import veomni.ops.kernels.cross_entropy as ref_ce
        from veomni_b200.cross_entropy import b200_cross_entropy

        spec = [s for s in R._specs() if s.op_name == "cross_entropy_loss" and s.variant == "causal"][0]
        bound = spec.factory()
        assert bound.func is ref_ce.ForCausalLMLoss and bound.keywords["cross_entropy_fn"] is b200_cross_entropy
        assert R.ATTN_NAME in ALL_ATTENTION_FUNCTIONS.valid_keys()
        import veomni.distributed.sequence_parallel.ulysses as u

        assert u.all_to_all_tensor.__module__ == "veomni_b200.ulysses"
    finally:
        sys.path.remove(str(REF_DIR))
