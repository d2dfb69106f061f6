"""The REAL reference, on the GPU, through the drop-in boundary — against what its stock ops compute.

tests/golden/reference_boundary.json (tests/golden/make_reference_boundary.py) holds the loss and global gradient norm
of the unmodified reference's toy Qwen3 and Qwen3-MoE (its ``build_foundation_model`` -> ``_bind_veomni_ops``, bf16 on a
B200, eager ops and flash-attn-2 varlen attention) for the weights and packed 3-sequence batch that module draws.

* ``test_reference_models_with_b200_ops_match_reference_stock_ops``: the reference package that ``build()`` places in
  ``oracle/_ref`` (oracle/build_ref.py) builds the same models again, with ``b200`` selected for every op
  ``veomni_b200.registry.register()`` installs (``rms_norm`` / ``rotary_pos_emb`` / ``swiglu_mlp`` /
  ``cross_entropy_loss`` / ``moe_experts`` OpSlots, the HF attention table entry and the fused-MoE pointer). Skips only
  when ``oracle/_ref`` holds no reference package.
* ``test_host_models_match_reference_stock_ops``: the host mirror of the same models on the veomni_b200 kernels.

Both apply the reference's own cross-backend bar: loss and grad-norm within 1e-2 relative
(tests/models/test_models_patch.py:327-329).
"""
import importlib.util
import json
import sys
from pathlib import Path

import pytest
import torch

from oracle.build_ref import REF_DIR

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"
_spec = importlib.util.spec_from_file_location("make_reference_boundary", GOLDEN / "make_reference_boundary.py")
MRB = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(MRB)
CASES = [("qwen3", MRB.QWEN3_TOY), ("qwen3_moe", MRB.QWEN3_MOE_TOY)]


def _check(name: str, loss: float, gn: float, launches: int) -> None:
    ref = json.loads((GOLDEN / "reference_boundary.json").read_text())[name]
    print(json.dumps({"model": name, "loss_ref": ref["loss"], "loss_b200": loss, "grad_norm_ref": ref["grad_norm"],
                      "grad_norm_b200": gn, "b200_kernel_launches": launches}))
    assert launches > 0, "not a single veomni_b200 kernel launched"
    assert abs(loss - ref["loss"]) / abs(ref["loss"]) < 1e-2, (loss, ref["loss"])
    assert abs(gn - ref["grad_norm"]) / ref["grad_norm"] < 1e-2, (gn, ref["grad_norm"])


@pytest.mark.parametrize("name,cfg", CASES)
def test_reference_models_with_b200_ops_match_reference_stock_ops(cuda_dev, name, cfg):
    if not (REF_DIR / "veomni").is_dir():
        pytest.skip("oracle/_ref holds no reference package (build() found no reference source)")
    from veomni_b200 import _lib, registry

    sys.path.insert(0, str(REF_DIR))
    try:
        assert registry.register(), "veomni_b200.registry.register() found no importable VeOmni"
        _lib.reset_launch_count()
        res = MRB.reference_run(cfg, cuda_dev, attn_implementation=registry.ATTN_NAME, rms_norm_implementation="b200",
                                rotary_pos_emb_implementation="b200", swiglu_mlp_implementation="b200",
                                cross_entropy_loss_implementation="b200",
                                moe_implementation="fused_b200" if name == "qwen3_moe" else "eager")
    finally:
        sys.path.remove(str(REF_DIR))
    _check(name, res["loss"], res["grad_norm"], _lib.launch_count())


@pytest.mark.parametrize("name,cfg", CASES)
def test_host_models_match_reference_stock_ops(cuda_dev, name, cfg):
    from veomni_b200 import _lib

    model = MRB.toy_model(cfg).to(cuda_dev).to(torch.bfloat16)
    model.train()
    ids, labels, lens = MRB.toy_batch(cfg["vocab_size"])
    pos = torch.cat([torch.arange(n) for n in lens])[None]
    cu = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), dtype=torch.int32, device=cuda_dev)
    _lib.reset_launch_count()
    loss = model(ids.to(cuda_dev), pos.to(cuda_dev), cu, max(lens), labels=labels.to(cuda_dev))
    loss.backward()
    gn = torch.sqrt(sum((p.grad.float() ** 2).sum() for p in model.parameters() if p.grad is not None))
    _check(name, float(loss.detach()), float(gn), _lib.launch_count())
