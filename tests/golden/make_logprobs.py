"""Generate tests/golden/logprobs.pt from the reference's own per-token log-probs and top-k distillation functions.

Needs the reference source tree (``$VEOMNI_SRC``, else ``oracle.build_ref.DEFAULT_SRC``):

    VEOMNI_SRC=<VeOmni source tree> python tests/golden/make_logprobs.py

For every case it runs the reference's ``chunk_logprobs_function`` / ``chunk_topk_distill_function``
(veomni/ops/kernels/cross_entropy/chunk_logprobs.py, chunk_topk_distill.py) on CPU, takes the gradient of a seeded
weighted sum of the differentiable outputs w.r.t. hidden states and lm_head weight, checks that the oracle
(``oracle/logprobs.py``) agrees, and stores inputs, upstream weights and reference results.

Inputs: hidden [2, 40, 64], lm_head weight [517, 64] (a ragged vocabulary: bf16 rows start off the 16-byte grid, so
the kernels' scalar head and tail run), scattered ignored labels and a fully ignored second sequence, teacher top-k
K = 8 with one duplicated id per position. Hidden states and weights are bf16 values, stored once and used in both
dtypes; the clamp is a bf16 value, so clamping in either dtype agrees.
"""

from __future__ import annotations

import os
import sys
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
REPO = HERE.parent.parent
sys.path.insert(0, str(REPO))

from oracle import logprobs as O  # noqa: E402
from oracle.build_ref import DEFAULT_SRC  # noqa: E402

B, L, H, V, K = 2, 40, 64, 517, 8
CLAMP = -6.0
# (name, dtype, temperature, top-k, clamp)
CASES = [
    ("fp32_t1_logprobs", torch.float32, 1.0, False, None),
    ("fp32_t07_topk", torch.float32, 0.7, True, None),
    ("fp32_t1_topk_clamp", torch.float32, 1.0, True, CLAMP),
    ("bf16_t07_logprobs", torch.bfloat16, 0.7, False, None),
    ("bf16_t1_topk", torch.bfloat16, 1.0, True, None),
    ("bf16_t07_topk_clamp", torch.bfloat16, 0.7, True, CLAMP),
]
NAMES = ("log_probs", "entropy", "distillation_losses", "student_mass", "teacher_mass")


def inputs():
    g = torch.Generator().manual_seed(17)
    hidden = torch.randn(B, L, H, generator=g).to(torch.bfloat16)
    weight = (0.2 * torch.randn(V, H, generator=g)).to(torch.bfloat16)
    labels = torch.randint(0, V, (B, L), generator=g)
    labels[0, torch.tensor([3, 4, 11, 25, 39])] = -100
    labels[1] = -100
    ids = torch.randint(0, V, (B, L, K), generator=g)
    ids[..., 7] = ids[..., 2]  # a duplicated id: its teacher probability counts twice
    tlp = torch.log_softmax(2.0 * torch.randn(B, L, K, generator=g), dim=-1) - 1.0
    ups = [torch.randn(B, L, generator=g) for _ in range(3)]  # upstream weights of log_probs, entropy, distill
    return {"hidden": hidden, "weight": weight, "labels": labels, "ids": ids, "tlp": tlp, "upstream": ups}


def reference_case(inp, dtype, temperature, topk, clamp):
    import veomni.ops.kernels.cross_entropy.chunk_logprobs as ref_lp
    from veomni.ops.kernels.cross_entropy import chunk_logprobs_function, chunk_topk_distill_function

    # flash-attn's Triton cross-entropy needs a GPU: on CPU use the reference's own log_softmax + gather path
    # (chunk_logprobs.py:107-110)
    ref_lp._FA_CE_AVAILABLE = False

    h = inp["hidden"].to(dtype).requires_grad_(True)
    w = inp["weight"].to(dtype).requires_grad_(True)
    if topk:
        outs = chunk_topk_distill_function(h, w, inp["labels"], inp["ids"], inp["tlp"].to(dtype), chunk_size=32,
                                           temperature=temperature, log_prob_min_clamp=clamp)
    else:
        outs = chunk_logprobs_function(h, w, inp["labels"], chunk_size=32, temperature=temperature)
    total = sum((o.float() * u).sum() for o, u in zip(outs[:3], inp["upstream"]))
    dh, dw = torch.autograd.grad(total, (h, w))
    return {n: o.detach() for n, o in zip(NAMES, outs)}, dh, dw


def oracle_case(inp, dtype, temperature, topk, clamp):
    h, lab, teacher = O.shift_for_logprobs(inp["hidden"].to(dtype), inp["labels"],
                                           (inp["ids"], inp["tlp"].to(dtype)) if topk else ())
    ups = [u[:, :-1].reshape(-1) for u in inp["upstream"]]
    kw = dict(ids=teacher[0].reshape(-1, K), tlp=teacher[1].reshape(-1, K), clamp=clamp) if topk else {}
    stats, dh, dw = O.fused_linear_token_logprobs(h.reshape(-1, H), inp["weight"].to(dtype), lab.reshape(-1),
                                                  temperature=temperature, chunk_size=32,
                                                  upstream=ups if topk else ups[:2] + [None], **kw)
    outs = {n: O.pad_last(stats[n].view(B, L - 1)) for n in NAMES if n in stats}
    dh = torch.nn.functional.pad(dh.view(B, L - 1, H), (0, 0, 0, 1))
    return outs, dh, dw


def main():
    sys.path.insert(0, os.environ.get("VEOMNI_SRC") or DEFAULT_SRC)  # the reference package, imported by reference_case
    inp = inputs()
    out = {"inputs": inp, "clamp": CLAMP, "cases": {}}
    for name, dtype, temperature, topk, clamp in CASES:
        ref, rdh, rdw = reference_case(inp, dtype, temperature, topk, clamp)
        orc, odh, odw = oracle_case(inp, dtype, temperature, topk, clamp)
        fp32 = dtype == torch.float32
        for n, v in ref.items():
            tol = dict(atol=1e-5, rtol=1e-5) if fp32 or n != "teacher_mass" else dict(atol=1e-2, rtol=1e-2)
            torch.testing.assert_close(orc[n], v.float(), **tol, msg=lambda m, n=n: f"{name} {n}: {m}")
        gtol = dict(atol=1e-6, rtol=1e-4) if fp32 else dict(atol=2e-3, rtol=2e-2)
        torch.testing.assert_close(odh.float(), rdh.float(), **gtol, msg=lambda m: f"{name} d hidden: {m}")
        torch.testing.assert_close(odw.float(), rdw.float(), **gtol, msg=lambda m: f"{name} d weight: {m}")
        assert all(float(v[1].abs().max()) == 0.0 for v in ref.values()), "fully ignored sequence must give 0"
        if clamp is not None:  # the clamp is active on some student top-k log-probs
            x = O.temper(inp["hidden"].to(dtype)[0, :-1] @ inp["weight"].to(dtype).t(), temperature)
            slp = x.log_softmax(-1).gather(-1, inp["ids"][0, 1:])
            assert 0 < int((slp < clamp).sum()) < slp.numel()
        print(f"  pinned: {name}")
        out["cases"][name] = {"dtype": dtype, "temperature": temperature, "topk": topk, "clamp": clamp,
                              "outputs": ref, "grad_hidden": rdh, "grad_weight": rdw}
    torch.save(out, HERE / "logprobs.pt")
    print("wrote", HERE / "logprobs.pt", (HERE / "logprobs.pt").stat().st_size, "bytes")


if __name__ == "__main__":
    main()
