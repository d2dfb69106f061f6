"""Oracle for the per-token paths of the causal-LM loss wrapper: log-probs + entropy, and top-k forward-KL distillation.

TEST INFRASTRUCTURE ONLY — see ``oracle/__init__.py``.

Restates, in torch (any device, any float dtype for the statistics):
* ``_ChunkedLinearLogProbs`` (veomni/ops/kernels/cross_entropy/chunk_logprobs.py:126-268): logits = h @ W^T in the
  compute dtype, divided by the temperature in that dtype and upcast (173-176); log p(label) and the entropy
  lse - sum(softmax * x) (87-123), 0 at ignored rows; the closed-form dlogits (225-249) rounded to the compute dtype
  and then divided by the temperature in that dtype (251-258);
* ``_ChunkedLinearTopkDistill`` (chunk_topk_distill.py:79-326): student / teacher mass before the clamp, the forward
  KL on the clamped top-k log-probs (157-190) and its gradient through the clamp gate (266-306);
* the target choice and padding of ``chunk_logprobs_function`` / ``chunk_topk_distill_function``
  (chunk_logprobs.py:319-351, chunk_topk_distill.py:377-416).
One deliberate difference: the teacher log-probs are upcast before they are clamped and exponentiated (the reference
exponentiates bf16 teacher log-probs in bf16 for ``teacher_mass``). Pinned against the reference on CPU, with
tolerances, in tests/golden/make_logprobs.py.
"""

from __future__ import annotations

import torch


def temper(logits: torch.Tensor, temperature: float) -> torch.Tensor:
    """chunk_logprobs.py:173-176: divide in the logits dtype, then upcast to fp32."""
    if temperature != 1.0:
        logits = logits / temperature
    return logits.float()


def token_stats(x: torch.Tensor, labels: torch.Tensor, ignore_index: int = -100, ids: torch.Tensor | None = None,
                tlp: torch.Tensor | None = None, clamp: float | None = None) -> dict:
    """Per-row statistics of tempered logits ``x`` [rows, V] (fp32, or fp64 for a tighter truth): lse, log_probs,
    entropy and, with ``ids``/``tlp`` [rows, K], distillation_losses, student_mass, teacher_mass."""
    mask = labels != ignore_index
    zero = torch.zeros(x.size(0), dtype=x.dtype, device=x.device)
    lse = torch.logsumexp(x, dim=-1)
    logsm = x.log_softmax(dim=-1)
    lp = logsm.gather(-1, labels.clamp(min=0)[:, None]).squeeze(-1)
    ent = lse - (x.softmax(dim=-1) * x).sum(dim=-1)
    out = {"lse": lse, "log_probs": torch.where(mask, lp, zero), "entropy": torch.where(mask, ent, zero)}
    if ids is None:
        return out
    slp = logsm.gather(-1, ids)
    t = tlp.to(x.dtype)
    sm, tm = slp.exp().sum(dim=-1), t.exp().sum(dim=-1)
    if clamp is not None:
        slp, t = slp.clamp_min(clamp), t.clamp_min(clamp)
    kl = (t.exp() * (t - slp)).sum(dim=-1)
    out.update(distillation_losses=torch.where(mask, kl, zero), student_mass=torch.where(mask, sm, zero),
               teacher_mass=torch.where(mask, tm, zero))
    return out


def token_grad(x: torch.Tensor, labels: torch.Tensor, dlp=None, dent=None, ddist=None, ids=None, tlp=None,
               clamp: float | None = None, ignore_index: int = -100) -> torch.Tensor:
    """d(sum dlp*log_probs + dent*entropy + ddist*distillation_losses) / d x, in x's dtype, before any rounding."""
    probs = x.softmax(dim=-1)
    mask = (labels != ignore_index).to(x.dtype)
    g = torch.zeros_like(probs)
    if dlp is not None:
        onehot = torch.zeros_like(probs).scatter_(-1, labels.clamp(min=0)[:, None], 1.0)
        g = g + (dlp.to(x.dtype) * mask)[:, None] * (onehot - probs)
    if dent is not None:
        h = torch.logsumexp(x, dim=-1) - (probs * x).sum(dim=-1)
        g = g + probs * (x.log_softmax(dim=-1) + h[:, None]) * (-(dent.to(x.dtype) * mask))[:, None]
    if ddist is not None:
        t = tlp.to(x.dtype)
        pk = (t.clamp_min(clamp) if clamp is not None else t).exp()
        if clamp is not None:
            pk = pk * (x.log_softmax(dim=-1).gather(-1, ids) >= clamp).to(x.dtype)
        pt = torch.zeros_like(probs).scatter_add_(-1, ids, pk)
        g = g + (ddist.to(x.dtype) * mask)[:, None] * (pk.sum(dim=-1, keepdim=True) * probs - pt)
    return g


def finish_grad(g: torch.Tensor, dtype: torch.dtype, temperature: float) -> torch.Tensor:
    """chunk_logprobs.py:251-258: round to the compute dtype first, then divide by the temperature in that dtype."""
    g = g.to(dtype)
    return g / temperature if temperature != 1.0 else g


def fused_linear_token_logprobs(hidden, weight, labels, ids=None, tlp=None, temperature: float = 1.0, clamp=None,
                                ignore_index: int = -100, chunk_size: int = 1024, upstream=(None, None, None)):
    """Chunked lm_head + per-token statistics on already-shifted, flattened inputs (hidden [T, H], labels [T],
    ids / tlp [T, K]); returns (statistics dict, d hidden, d weight) for the upstream (dlp, dent, ddist) [T] each."""
    T = hidden.size(0)
    stats: dict[str, list] = {}
    dh, dw = torch.zeros_like(hidden), torch.zeros_like(weight)
    for r0 in range(0, T, chunk_size):
        r1 = min(T, r0 + chunk_size)
        x = temper(hidden[r0:r1] @ weight.t(), temperature)
        sl = slice(r0, r1)
        kw = dict(ids=ids[sl], tlp=tlp[sl], clamp=clamp) if ids is not None else {}
        for k, v in token_stats(x, labels[sl], ignore_index, **kw).items():
            stats.setdefault(k, []).append(v)
        ups = [u[sl] if u is not None else None for u in upstream]
        g = finish_grad(token_grad(x, labels[sl], *ups, ignore_index=ignore_index, **kw), hidden.dtype, temperature)
        dh[sl] = g @ weight
        dw += g.t() @ hidden[sl]
    return {k: torch.cat(v) for k, v in stats.items()}, dh, dw


def shift_for_logprobs(hidden, labels, teacher=()):
    """chunk_logprobs.py:337-338 / chunk_topk_distill.py:385-393 (no SP, no explicit shift_labels): hidden[..., :-1, :]
    predicts labels[..., 1:], and the teacher tensors are shifted with the labels."""
    return hidden[..., :-1, :], labels[..., 1:], tuple(t[..., 1:, :] for t in teacher)


def pad_last(t: torch.Tensor) -> torch.Tensor:
    """The zero slot the shifted outputs get at the end of the sequence (chunk_logprobs.py:344-350)."""
    return torch.nn.functional.pad(t, (0, 1), value=0.0)
