"""GPU parity of the per-token log-probs / entropy / top-k distillation path (token_stats_kernel, token_grad_kernel).

* Fixture parity: ``chunk_logprobs_function``, ``chunk_topk_distill_function`` and ``ForCausalLMLoss(
  return_log_probs=True)`` against the reference's own outputs and gradients (tests/golden/make_logprobs.py).
  fp32: outputs atol/rtol 1e-5, gradients atol 1e-6 / rtol 1e-4. bf16: per-token outputs atol 2e-2 (cuBLAS and the CPU
  may round a logit one bf16 ulp apart), gradients atol 2e-3 / rtol 2e-2 (the fused-linear bar of test_loss_gpu.py).
* Kernel vs oracle on identical logits: statistics rtol 1e-5 against the oracle in fp64; gradients within 1 bf16 ulp
  of the oracle's value rounded once, 2 ulp with a temperature (the reference rounds twice), plus 8 fp32 ulp of the
  largest summed term where the terms cancel; ignored rows exactly 0;
  every combination of absent upstream gradients; two runs bit-identical.
* Through the real reference: the toy Qwen3 of tests/golden/make_reference_boundary.py built from ``oracle/_ref`` with
  ``cross_entropy_loss_implementation="b200"`` and called with ``return_log_probs=True``.
"""
import importlib.util
import itertools
import json
import sys
from pathlib import Path

import pytest
import torch

from oracle import logprobs as O
from oracle.build_ref import REF_DIR

pytestmark = pytest.mark.gpu
GOLDEN = Path(__file__).resolve().parent / "golden"
NAMES = ("log_probs", "entropy", "distillation_losses", "student_mass", "teacher_mass")


def _cpu(t):
    return t.detach().float().cpu()


def _report(what, got, want):
    d = (_cpu(got) - _cpu(want)).abs().max().item() if got.numel() else 0.0
    print(json.dumps({"check": what, "max_abs_dev": d}))


@pytest.fixture(scope="module")
def case_inputs(golden):
    f = golden("logprobs.pt")
    return f["inputs"], f["cases"]


def _run_public(fn_kind, inp, c, dev):
    from veomni_b200.cross_entropy import ForCausalLMLoss, chunk_logprobs_function, chunk_topk_distill_function

    dtype = c["dtype"]
    h = inp["hidden"].to(dtype).to(dev).requires_grad_(True)
    w = inp["weight"].to(dtype).to(dev).requires_grad_(True)
    labels = inp["labels"].to(dev)
    ids, tlp = inp["ids"].to(dev), inp["tlp"].to(dtype).to(dev)
    kw = dict(chunk_size=32, temperature=c["temperature"])
    if fn_kind == "function":
        if c["topk"]:
            outs = chunk_topk_distill_function(h, w, labels, ids, tlp, log_prob_min_clamp=c["clamp"], **kw)
        else:
            outs = chunk_logprobs_function(h, w, labels, **kw)
    else:
        extra = dict(teacher_topk_ids=ids, teacher_topk_log_probs=tlp, log_prob_min_clamp=c["clamp"]) if c["topk"] else {}
        loss, logits, aux = ForCausalLMLoss(labels=labels, vocab_size=w.shape[0], hidden_states=h, weights=w,
                                            return_log_probs=True, **kw, **extra)
        assert loss is None and logits is None
        outs = tuple(getattr(aux, n) for n in NAMES if getattr(aux, n) is not None)
    total = sum((o.float() * u.to(dev)).sum() for o, u in zip(outs[:3], inp["upstream"]))
    dh, dw = torch.autograd.grad(total, (h, w))
    return outs, dh, dw


@pytest.mark.parametrize("kind", ["function", "ForCausalLMLoss"])
@pytest.mark.parametrize("case", ["fp32_t1_logprobs", "fp32_t07_topk", "fp32_t1_topk_clamp", "bf16_t07_logprobs",
                                  "bf16_t1_topk", "bf16_t07_topk_clamp"])
def test_fixture_parity(cuda_dev, case_inputs, case, kind):
    inp, cases = case_inputs
    c = cases[case]
    outs, dh, dw = _run_public(kind, inp, c, cuda_dev)
    fp32 = c["dtype"] == torch.float32
    assert len(outs) == len(c["outputs"])
    for n, o in zip(NAMES, outs):
        want = c["outputs"][n]
        assert o.shape == want.shape and o.dtype == torch.float32
        assert torch.all(_cpu(o)[:, -1] == 0) and torch.all(_cpu(o)[1] == 0)  # padded slot, ignored sequence
        _report(f"{case}/{kind}/{n}", o, want)
        torch.testing.assert_close(_cpu(o), want.float(), **(dict(atol=1e-5, rtol=1e-5) if fp32 else dict(atol=2e-2, rtol=0)))
    if c["topk"]:
        assert not outs[3].requires_grad and not outs[4].requires_grad
    gtol = dict(atol=1e-6, rtol=1e-4) if fp32 else dict(atol=2e-3, rtol=2e-2)
    _report(f"{case}/{kind}/dh", dh, c["grad_hidden"])
    _report(f"{case}/{kind}/dw", dw, c["grad_weight"])
    torch.testing.assert_close(_cpu(dh), c["grad_hidden"].float(), **gtol)
    torch.testing.assert_close(_cpu(dw), c["grad_weight"].float(), **gtol)


def _bf16_ulp(v: torch.Tensor) -> torch.Tensor:
    _, e = torch.frexp(v)
    return torch.ldexp(torch.ones_like(v), e - 8)


def _term_scale(x, labels, ups, stats):
    """Per element, the magnitude of the largest term summed into the gradient (ignored rows are exactly 0 anyway)."""
    p = torch.softmax(x, dim=-1)
    s = torch.zeros_like(x)
    if ups[0] is not None:
        s = s + ups[0].abs().double()[:, None] * p
    if ups[1] is not None:
        s = s + ups[1].abs().double()[:, None] * p * ((x - stats["lse"][:, None]).abs() + stats["entropy"].abs()[:, None])
    if ups[2] is not None:
        s = s + ups[2].abs().double()[:, None] * p * stats["teacher_mass"][:, None]
    return s


def _launch_pair(logits, labels, temperature, ids, tlp, clamp, ups):
    """forward statistics, then the in-place gradient, on a copy of ``logits``; returns (stats dict, grad)."""
    from veomni_b200.cross_entropy import _token_launch

    rows, dev = logits.size(0), logits.device
    f = lambda: torch.empty(rows, dtype=torch.float32, device=dev)  # noqa: E731
    st = {n: f() for n in ("lse", "log_probs", "entropy")}
    if ids is not None:
        st.update({n: f() for n in NAMES[2:]})
    _token_launch(False, logits, labels, -100, temperature, st["lse"], st["entropy"], ids, tlp, clamp,
                  logp=st["log_probs"], dist=st.get("distillation_losses"), sm=st.get("student_mass"),
                  tm=st.get("teacher_mass"))
    g = logits.clone()
    _token_launch(True, g, labels, -100, temperature, st["lse"], st["entropy"], ids, tlp, clamp, ups=ups)
    return st, g


@pytest.mark.parametrize("rows,vocab,dtype", [(5, 17, torch.bfloat16), (33, 4096, torch.bfloat16),
                                              (64, 32003, torch.bfloat16), (16, 151936, torch.float32),
                                              (1024, 151936, torch.bfloat16)])
@pytest.mark.parametrize("temperature", [1.0, 0.7])
def test_kernel_vs_oracle(cuda_dev, rows, vocab, dtype, temperature):
    from veomni_b200 import _lib

    g = torch.Generator(device=cuda_dev).manual_seed(rows * 31 + vocab)
    x_in = (3 * torch.randn(rows, vocab, generator=g, device=cuda_dev)).to(dtype)
    labels = torch.randint(0, vocab, (rows,), generator=g, device=cuda_dev)
    labels[1::3] = -100
    K = min(64, vocab)
    ids = torch.randint(0, vocab, (rows, K), generator=g, device=cuda_dev)
    ids[:, -1] = ids[:, 0]  # duplicate
    ids[0, :3] = torch.tensor([0, vocab - 1, vocab // 2], device=cuda_dev)  # scalar head / tail entries
    tlp = torch.log_softmax(2 * torch.randn(rows, K, generator=g, device=cuda_dev), -1) - 1.0
    clamp = -float(torch.log(torch.tensor(float(vocab)))) - 1.0  # active on part of the student top-k
    ups = [torch.randn(rows, generator=g, device=cuda_dev) for _ in range(3)]
    x = O.temper(x_in, temperature).double()
    valid = labels != -100
    ref = O.token_stats(x, labels, ids=ids, tlp=tlp, clamp=clamp)
    _lib.reset_launch_count()
    st, _ = _launch_pair(x_in, labels, temperature, ids, tlp, clamp, ups)
    assert _lib.launch_count() == 2
    for n, v in st.items():
        assert torch.all(v[~valid] == 0) or n == "lse"
        torch.testing.assert_close(v.double(), ref[n], atol=1e-5, rtol=1e-5, msg=lambda m, n=n: f"{n}: {m}")
    n_ulp = 1 if temperature == 1.0 else 2
    combos = [c for r in range(1, 4) for c in itertools.combinations(range(3), r)]
    if rows * vocab > 1 << 24:
        combos = [(0, 1, 2)]  # the large shapes: everything at once
    for combo in combos:
        u = [ups[i] if i in combo else None for i in range(3)]
        _, gk = _launch_pair(x_in, labels, temperature, ids, tlp, clamp, u)
        go = O.token_grad(x, labels, *u, ids=ids, tlp=tlp, clamp=clamp)
        if dtype == torch.bfloat16:
            want = go.float().to(torch.bfloat16).double() / temperature  # the rounding before the division
            err = (gk.double() - want).abs()
            # where the dense terms cancel (log p + H near 0) a correct fp32 evaluation is off by a few fp32 ulp of the
            # terms, which can exceed a bf16 ulp of the small result: allow 8 fp32 ulp of the largest term on top
            bound = n_ulp * _bf16_ulp(want.float()).double() + 8 * 2.0**-24 * _term_scale(x, labels, u, ref) / temperature
            bad = err > bound
            assert not bad.any(), f"{combo}: {int(bad.sum())} entries beyond {n_ulp} ulp, worst {float((err / bound).max())}"
        else:
            torch.testing.assert_close(gk.double(), go / temperature, atol=1e-6, rtol=1e-4)
        assert torch.all(gk[~valid] == 0)
    # determinism
    st2, g2 = _launch_pair(x_in, labels, temperature, ids, tlp, clamp, ups)
    st3, g3 = _launch_pair(x_in, labels, temperature, ids, tlp, clamp, ups)
    assert torch.equal(g2, g3) and all(torch.equal(st2[n], st3[n]) for n in st2)


def test_rejects_cpu_tensors_and_wide_topk(cuda_dev):
    from veomni_b200._lib import VB200Error
    from veomni_b200.cross_entropy import chunk_logprobs_function, chunk_topk_distill_function

    with pytest.raises(VB200Error):
        chunk_logprobs_function(torch.randn(1, 4, 8), torch.randn(16, 8), torch.zeros(1, 4, dtype=torch.int64))
    h, w = torch.randn(1, 4, 8, device=cuda_dev), torch.randn(2048, 8, device=cuda_dev)
    lab = torch.zeros(1, 4, dtype=torch.int64, device=cuda_dev)
    ids = torch.zeros(1, 4, 1025, dtype=torch.int64, device=cuda_dev)
    with pytest.raises(VB200Error, match="1024"):
        chunk_topk_distill_function(h, w, lab, ids, torch.zeros(1, 4, 1025, device=cuda_dev))


def _load_mrb():
    spec = importlib.util.spec_from_file_location("make_reference_boundary", GOLDEN / "make_reference_boundary.py")
    mrb = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mrb)
    return mrb


def test_reference_model_return_log_probs_uses_b200(cuda_dev, monkeypatch):
    if not (REF_DIR / "veomni").is_dir():
        pytest.skip("oracle/_ref holds no reference package (build() found no reference source)")
    from veomni_b200 import _lib, registry

    mrb = _load_mrb()
    sys.path.insert(0, str(REF_DIR))
    try:
        assert registry.register()
        import veomni.ops.kernels.cross_entropy as ref_ce
        import veomni.ops.kernels.cross_entropy.chunk_logprobs as ref_lp
        from veomni.arguments.arguments_types import OpsImplementationConfig
        from veomni.models import build_foundation_model

        ops = OpsImplementationConfig(**{**mrb.STOCK_OPS, "attn_implementation": registry.ATTN_NAME,
                                         "cross_entropy_loss_implementation": "b200"})
        cfg = mrb.QWEN3_TOY
        import tempfile

        with tempfile.TemporaryDirectory() as d:
            (Path(d) / "config.json").write_text(json.dumps(cfg))
            model = build_foundation_model(config_path=d, weights_path=None, torch_dtype="bfloat16", init_device="cuda",
                                           ops_implementation=ops)
        model.load_state_dict({k: v.to(torch.bfloat16) for k, v in mrb.toy_model(cfg).state_dict().items()})
        ids, labels, lens = mrb.toy_batch(cfg["vocab_size"])
        pos = torch.cat([torch.arange(n) for n in lens])[None]
        cu = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), dtype=torch.int32, device=cuda_dev)
        fwd = dict(input_ids=ids.to(cuda_dev), labels=labels.to(cuda_dev), position_ids=pos.to(cuda_dev),
                   attention_mask=torch.ones_like(ids).to(cuda_dev), cu_seq_lens_q=cu, cu_seq_lens_k=cu,
                   max_length_q=max(lens), max_length_k=max(lens), use_cache=False)
        captured = {}  # the final norm's output is the hidden state the loss wrapper receives
        model.model.norm.register_forward_hook(lambda mod, inp, out: captured.__setitem__("h", out))
        from veomni_b200 import cross_entropy as own

        token_launches = []
        real_launch = own._token_launch
        monkeypatch.setattr(own, "_token_launch", lambda *a, **k: token_launches.append(a[0]) or real_launch(*a, **k))
        g = torch.Generator().manual_seed(23)
        T, Kt = ids.shape[1], 16
        t_ids = torch.randint(0, cfg["vocab_size"], (1, T, Kt), generator=g).to(cuda_dev)
        t_lp = (torch.log_softmax(torch.randn(1, T, Kt, generator=g), -1) - 1.0).to(cuda_dev)
        ups = [torch.randn(1, T, generator=g).to(cuda_dev) for _ in range(3)]
        monkeypatch.setattr(ref_lp, "_FA_CE_AVAILABLE", False)  # the reference side runs its log_softmax + gather path
        for teacher in (False, True):
            orig_name = "chunk_topk_distill_function" if teacher else "chunk_logprobs_function"
            orig = getattr(ref_ce, orig_name)._vb200_orig
            orig_calls = []
            monkeypatch.setattr(getattr(ref_ce, orig_name), "_vb200_orig",
                                lambda *a, **k: orig_calls.append(1) or orig(*a, **k))
            extra = dict(teacher_topk_ids=t_ids, teacher_topk_log_probs=t_lp, log_prob_min_clamp=-9.0) if teacher else {}
            model.zero_grad(set_to_none=True)
            _lib.reset_launch_count()
            token_launches.clear()
            out = model(**fwd, return_log_probs=True, temperature=0.9, **extra)
            aux = out.fused_linear_aux
            names = NAMES if teacher else NAMES[:2]
            ours = [getattr(aux, n) for n in names]
            total = sum((o * u).sum() for o, u in zip(ours[:3], ups))
            total.backward()
            launches = _lib.launch_count()
            assert launches > 0 and not orig_calls, "the b200 path must not call the reference's function"
            assert False in token_launches and True in token_launches  # token_stats_kernel and token_grad_kernel ran
            w = model.lm_head.weight
            gw_ours = w.grad.detach().clone()
            # the reference's own function on the same last hidden states and lm_head weight
            hs = captured["h"].detach().requires_grad_(True)
            wr = w.detach().clone().requires_grad_(True)
            lab = labels.to(cuda_dev)
            if teacher:
                ref = orig(hs, wr, lab, t_ids, t_lp, temperature=0.9, log_prob_min_clamp=-9.0)
            else:
                ref = orig(hs, wr, lab, temperature=0.9)
            (gw_ref,) = torch.autograd.grad(sum((o * u).sum() for o, u in zip(ref[:3], ups)), (wr,))
            for n, o, r in zip(names, ours, ref):
                _report(f"qwen3_toy/{n}", o, r)
                torch.testing.assert_close(_cpu(o), _cpu(r), atol=2e-2, rtol=0)
            _report("qwen3_toy/d lm_head", gw_ours, gw_ref)
            torch.testing.assert_close(_cpu(gw_ours), _cpu(gw_ref), atol=2e-3, rtol=2e-2)
    finally:
        sys.path.remove(str(REF_DIR))
