"""Generate tests/golden/reference_boundary.json: loss and gradient norm of the REFERENCE's own toy models on a B200.

Needs the unmodified reference (VeOmni) importable and a CUDA GPU with flash-attn:

    PYTHONPATH=<VeOmni source tree> python tests/golden/make_reference_boundary.py

For each toy config the reference's ``build_foundation_model`` -> ``_bind_veomni_ops`` (veomni/models/auto.py:63-103)
builds its patched model in bf16 on the GPU with its stock ops (eager, flash-attn-2 varlen attention), loads the weights
``toy_model`` draws, runs one forward + backward over ``toy_batch`` and records the loss and the global gradient norm.
tests/test_reference_boundary_gpu.py runs the same weights and batch through the same reference models with the b200
ops selected (``reference_run`` with overrides), and through the host models, on the sm_100a kernels.
"""
from __future__ import annotations

import json
import sys
import tempfile
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
REPO = HERE.parent.parent
OUT = HERE / "reference_boundary.json"

QWEN3_TOY = dict(hidden_size=1024, intermediate_size=2048, num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=2,
                 head_dim=128, vocab_size=2048, max_position_embeddings=4096, rms_norm_eps=1e-6, tie_word_embeddings=False,
                 rope_theta=1000000.0, architectures=["Qwen3ForCausalLM"], model_type="qwen3")
QWEN3_MOE_TOY = dict(hidden_size=1024, intermediate_size=2048, moe_intermediate_size=256, num_experts=8, num_experts_per_tok=2,
                     num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=2, head_dim=128, vocab_size=2048,
                     max_position_embeddings=4096, rms_norm_eps=1e-6, tie_word_embeddings=False, rope_theta=1000000.0,
                     decoder_sparse_step=1, mlp_only_layers=[], norm_topk_prob=True, output_router_logits=False,
                     router_aux_loss_coef=0.0, architectures=["Qwen3MoeForCausalLM"], model_type="qwen3_moe")
TOYS = {"qwen3": QWEN3_TOY, "qwen3_moe": QWEN3_MOE_TOY}


def toy_model(cfg_dict: dict):
    """The host model of ``cfg_dict`` on the CPU in fp32, weights drawn by its ``init_weights(seed=0)`` (CPU generator,
    so the same on every machine). Both arms run it in bf16."""
    if str(REPO) not in sys.path:
        sys.path.insert(0, str(REPO))
    from veomni_b200.host_qwen3 import Qwen3Config, Qwen3ForCausalLM
    from veomni_b200.host_qwen3_moe import Qwen3MoeConfig, Qwen3MoeForCausalLM

    base = Qwen3Config.from_hf_dict(cfg_dict)
    if cfg_dict["model_type"] == "qwen3_moe":
        cfg = Qwen3MoeConfig(**vars(base), num_experts=cfg_dict["num_experts"], num_experts_per_tok=cfg_dict["num_experts_per_tok"],
                             moe_intermediate_size=cfg_dict["moe_intermediate_size"], norm_topk_prob=cfg_dict["norm_topk_prob"])
        model = Qwen3MoeForCausalLM(cfg)
    else:
        model = Qwen3ForCausalLM(base)
    model.init_weights(seed=0)
    return model


def toy_batch(vocab: int):
    """One packed row of three sequences: input ids, labels (-100 on each sequence's first token), sequence lengths."""
    lens = [300, 212, 512]
    g = torch.Generator().manual_seed(11)
    ids = torch.randint(0, vocab, (1, sum(lens)), generator=g)
    labels = ids.clone()
    off = 0
    for n in lens:
        labels[0, off] = -100
        off += n
    return ids, labels, lens


STOCK_OPS = dict(attn_implementation="flash_attention_2", moe_implementation="eager", cross_entropy_loss_implementation="eager",
                 rms_norm_implementation="eager", swiglu_mlp_implementation="eager", rotary_pos_emb_implementation="eager",
                 load_balancing_loss_implementation="eager", rms_norm_gated_implementation="eager",
                 causal_conv1d_implementation="eager", chunk_gated_delta_rule_implementation="eager")


def reference_run(cfg_dict: dict, dev: torch.device, **ops_overrides) -> dict:
    """Loss and global gradient norm of the reference's own model of ``cfg_dict`` on ``toy_model``'s weights and
    ``toy_batch``, built with ``STOCK_OPS`` updated by ``ops_overrides``. Needs ``veomni`` importable."""
    from veomni.arguments.arguments_types import OpsImplementationConfig
    from veomni.models import build_foundation_model

    ops = OpsImplementationConfig(**{**STOCK_OPS, **ops_overrides})
    with tempfile.TemporaryDirectory() as d:
        (Path(d) / "config.json").write_text(json.dumps(cfg_dict))
        model = build_foundation_model(config_path=d, weights_path=None, torch_dtype="bfloat16", init_device="cuda",
                                       ops_implementation=ops)
    state = {k: v.to(torch.bfloat16) for k, v in toy_model(cfg_dict).state_dict().items()}
    model.load_state_dict(state)
    model.train()
    ids, labels, lens = toy_batch(cfg_dict["vocab_size"])
    pos = torch.cat([torch.arange(n) for n in lens])[None]
    cu = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), dtype=torch.int32, device=dev)
    out = model(input_ids=ids.to(dev), labels=labels.to(dev), position_ids=pos.to(dev), attention_mask=torch.ones_like(ids).to(dev),
                cu_seq_lens_q=cu, cu_seq_lens_k=cu, max_length_q=max(lens), max_length_k=max(lens), use_cache=False)
    out.loss.backward()
    gn = torch.sqrt(sum((p.grad.float() ** 2).sum() for p in model.parameters() if p.grad is not None))
    return {"loss": float(out.loss.detach()), "grad_norm": float(gn)}


def main() -> None:
    import flash_attn

    dev = torch.device("cuda", 0)
    res = {name: reference_run(cfg, dev) for name, cfg in TOYS.items()}
    res["provenance"] = {"device": torch.cuda.get_device_name(dev), "torch": torch.__version__, "flash_attn": flash_attn.__version__,
                         "ops": "reference stock: eager rms_norm / rope / swiglu / moe / cross-entropy, flash_attention_2"}
    OUT.write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
