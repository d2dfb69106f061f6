"""Cross-entropy over the vocabulary: the inner kernel of VeOmni's loss wrappers.

Mirrors veomni/ops/kernels/cross_entropy/:
* :func:`b200_cross_entropy` has the ``cross_entropy_fn`` contract of ``eager_cross_entropy`` (eager.py:23-38) and
  ``fused_liger_kernel_cross_entropy`` (liger.py:24-57): ``(logits, labels, vocab_size, num_items_in_batch,
  ignore_index, shift_labels, hidden_states=, weights=) -> (loss, logits)``. With ``logits`` it is the eager
  arithmetic (``fixed_cross_entropy``: mean over non-ignored rows, or sum / num_items_in_batch); with
  ``hidden_states`` + ``weights`` it is the fused-linear form: the ``lm_head`` projection runs chunk by chunk on cuBLAS,
  the CUDA kernel turns each logits chunk into its gradient in place, and the full ``[T, V]`` logits (2.5 GB in
  fp32 at T=4096, V=151936) never exist.
* :func:`ForCausalLMLoss` is the outer policy (__init__.py:89-221): label shift unless SP, flatten, SP loss reduce.
* :func:`chunk_logprobs_function` / :func:`chunk_topk_distill_function` are the ``return_log_probs=True`` paths
  (chunk_logprobs.py, chunk_topk_distill.py): per-token log-probs and entropy, and top-k forward-KL distillation,
  through the same chunked lm_head; each logits chunk is turned into its gradient in place in backward.

No host synchronisation: the valid-token count stays on the device and scales loss and gradient there.
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import Any, Callable

import torch
import torch.nn.functional as F

from . import _lib
from ._lib import VB200Error, check, stream_ptr

_DT = {torch.bfloat16: 0, torch.float32: 1}


def _check(logits: torch.Tensor, labels: torch.Tensor) -> None:
    if not logits.is_cuda or not labels.is_cuda:
        raise VB200Error("cross_entropy runs on CUDA tensors only (no CPU fallback)")
    if logits.dtype not in _DT:
        raise VB200Error(f"cross_entropy: logits must be bf16 or fp32, got {logits.dtype}")
    if logits.dim() != 2 or logits.stride(1) != 1:
        raise VB200Error("cross_entropy: logits must be [rows, vocab] with contiguous rows")
    if labels.dtype != torch.int64 or labels.dim() != 1 or labels.numel() != logits.size(0):
        raise VB200Error("cross_entropy: labels must be int64 [rows]")


def _ptr(t: torch.Tensor | None) -> int | None:
    return t.data_ptr() if t is not None else None


def _launch(logits, labels, ignore_index, loss_rows, lse, lse_given, grad, scale, scale_dev, upstream) -> None:
    lib = _lib.load()
    with torch.cuda.device(logits.device):
        check(lib.vb200_cross_entropy(
            logits.data_ptr(), _DT[logits.dtype], logits.size(0), logits.size(1), logits.stride(0), labels.data_ptr(),
            int(ignore_index), _ptr(loss_rows), _ptr(lse), int(lse_given), _ptr(grad),
            grad.stride(0) if grad is not None else 0, float(scale), _ptr(scale_dev), _ptr(upstream), stream_ptr(),
        ), "vb200_cross_entropy")


def valid_label_recip(labels: torch.Tensor, ignore_index: int = -100) -> torch.Tensor:
    """Device tensor ``[1/count, count]`` of labels != ignore_index. With no valid label the factor is 0, so the loss and
    its gradient are exactly 0 for that batch (csrc/cross_entropy.cu ``ce_valid_recip_kernel``) — NOT the NaN that
    ``F.cross_entropy(reduction="mean")`` returns for an all-ignored batch: a fully masked micro-batch does not poison
    the step. Callers that want the eager NaN can test ``out[1] == 0`` themselves."""
    out = torch.empty(2, dtype=torch.float32, device=labels.device)
    lab = labels.reshape(-1).contiguous()
    if not lab.is_cuda or lab.dtype != torch.int64:
        raise VB200Error("valid_label_recip: labels must be a CUDA int64 tensor")
    with torch.cuda.device(lab.device):
        check(_lib.load().vb200_count_valid_labels(lab.data_ptr(), lab.numel(), int(ignore_index), out.data_ptr(),
                                                   stream_ptr()), "vb200_count_valid_labels")
    return out


def _scales(labels: torch.Tensor, num_items_in_batch, ignore_index: int) -> tuple[float, torch.Tensor | None]:
    """(host factor, device factor) of the reduction: mean over valid rows, or sum / num_items_in_batch
    (transformers fixed_cross_entropy)."""
    if num_items_in_batch is None:
        return 1.0, valid_label_recip(labels, ignore_index)[:1]
    if torch.is_tensor(num_items_in_batch):
        return 1.0, (1.0 / num_items_in_batch.to(device=labels.device, dtype=torch.float32)).reshape(1)
    return 1.0 / float(num_items_in_batch), None


class _CrossEntropy(torch.autograd.Function):
    """loss = reduce(logsumexp(x) - x[label]); backward re-reads the logits with the saved logsumexp."""

    @staticmethod
    def forward(ctx: Any, logits: torch.Tensor, labels: torch.Tensor, ignore_index: int, scale: float,
                scale_dev: torch.Tensor | None):
        _check(logits, labels)
        rows = logits.size(0)
        loss_rows = torch.empty(rows, dtype=torch.float32, device=logits.device)
        lse = torch.empty(rows, dtype=torch.float32, device=logits.device)
        _launch(logits, labels, ignore_index, loss_rows, lse, 0, None, 1.0, None, None)
        loss = loss_rows.sum() * scale
        if scale_dev is not None:
            loss = loss * scale_dev[0]
        ctx.save_for_backward(logits, labels, lse, scale_dev)
        ctx.ignore_index, ctx.scale = ignore_index, scale
        return loss

    @staticmethod
    def backward(ctx: Any, g: torch.Tensor):
        logits, labels, lse, scale_dev = ctx.saved_tensors
        grad = torch.empty_like(logits)
        up = g.detach().to(torch.float32).reshape(1).contiguous()
        _launch(logits, labels, ctx.ignore_index, None, lse, 1, grad, ctx.scale, scale_dev, up)
        return grad, None, None, None, None


class _FusedLinearCrossEntropy(torch.autograd.Function):
    """lm_head projection + cross-entropy, chunked over rows; the gradients w.r.t. hidden states and weights are
    produced during the forward pass (as the liger kernel the reference binds does) and scaled by the incoming
    gradient in backward."""

    @staticmethod
    def forward(ctx: Any, hidden: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor, ignore_index: int,
                scale: float, scale_dev: torch.Tensor | None, chunk_size: int):
        if hidden.dim() != 2 or weight.dim() != 2 or hidden.size(1) != weight.size(1):
            raise VB200Error("fused linear cross-entropy: hidden [T, H] and weight [V, H] expected")
        if hidden.dtype != weight.dtype:
            raise VB200Error("fused linear cross-entropy: hidden states and weights must share a dtype")
        T, V = hidden.size(0), weight.size(0)
        need_h, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        loss_rows = torch.empty(T, dtype=torch.float32, device=hidden.device)
        grad_h = torch.empty_like(hidden) if need_h else None
        grad_w = torch.zeros_like(weight) if need_w else None
        wt = weight.t()
        for r0 in range(0, T, chunk_size):
            r1 = min(T, r0 + chunk_size)
            h_c = hidden[r0:r1]
            logits = torch.mm(h_c, wt)  # [chunk, V] in the compute dtype (cuBLAS)
            lab = labels[r0:r1]
            _check(logits, lab)
            grad = logits if (need_h or need_w) else None  # in place: the chunk becomes dLoss/dlogits
            _launch(logits, lab, ignore_index, loss_rows[r0:r1], None, 0, grad, scale, scale_dev, None)
            if need_h:
                torch.mm(logits, weight, out=grad_h[r0:r1])
            if need_w:
                grad_w.addmm_(logits.t(), h_c)
        loss = loss_rows.sum() * scale
        if scale_dev is not None:
            loss = loss * scale_dev[0]
        ctx.save_for_backward(grad_h, grad_w)
        return loss

    @staticmethod
    def backward(ctx: Any, g: torch.Tensor):
        grad_h, grad_w = ctx.saved_tensors
        gh = grad_h * g.to(grad_h.dtype) if grad_h is not None else None
        gw = grad_w * g.to(grad_w.dtype) if grad_w is not None else None
        return gh, gw, None, None, None, None, None


class _FusedLinearTokenLogProbs(torch.autograd.Function):
    """lm_head projection + per-token log-probs and entropy, plus top-k forward-KL distillation when ``ids`` is given
    (K = ids.size(1) > 0): the arithmetic of _ChunkedLinearLogProbs / _ChunkedLinearTopkDistill
    (chunk_logprobs.py:126-268, chunk_topk_distill.py:79-326), chunked over rows.

    Forward: per chunk, logits on cuBLAS, then ``token_stats_kernel``; only the fp32 ``[T]`` statistics are kept.
    Backward: per chunk, the same GEMM recomputes the logits, ``token_grad_kernel`` turns them into dlogits in place,
    and two GEMMs give dh and dw. The weight saved here is the lm_head parameter, which FSDP2's pre-backward hook has
    unsharded again by the time backward runs (the reference's contract, chunk_logprobs.py:42-48).
    Outputs: ``(logp, entropy)``, or with K > 0 ``(logp, entropy, distill, student_mass, teacher_mass)``, the last
    two non-differentiable."""

    @staticmethod
    def forward(ctx: Any, hidden: torch.Tensor, weight: torch.Tensor, labels: torch.Tensor, ids: torch.Tensor | None,
                tlp: torch.Tensor | None, temperature: float, chunk_size: int, ignore_index: int, clamp: float | None):
        ctx.set_materialize_grads(False)
        _check_token_inputs(hidden, weight, labels, ids, tlp)
        T, dev = hidden.size(0), hidden.device
        K = ids.size(1) if ids is not None else 0
        f32 = dict(dtype=torch.float32, device=dev)
        lse, logp, ent = torch.empty(T, **f32), torch.empty(T, **f32), torch.empty(T, **f32)
        dist, sm, tm = (torch.empty(T, **f32) for _ in range(3)) if K else (None, None, None)
        wt = weight.t()
        for r0 in range(0, T, chunk_size):
            r1 = min(T, r0 + chunk_size)
            logits = torch.mm(hidden[r0:r1], wt)  # [chunk, V] in the compute dtype (cuBLAS)
            _token_launch(False, logits, labels[r0:r1], ignore_index, temperature, lse[r0:r1], ent[r0:r1],
                          ids[r0:r1] if K else None, tlp[r0:r1] if K else None, clamp,
                          logp=logp[r0:r1], dist=dist[r0:r1] if K else None, sm=sm[r0:r1] if K else None,
                          tm=tm[r0:r1] if K else None)
        ctx.save_for_backward(hidden, weight, labels, lse, ent, ids, tlp)
        ctx.temperature, ctx.chunk_size, ctx.ignore_index, ctx.clamp = temperature, chunk_size, ignore_index, clamp
        if not K:
            return logp, ent
        ctx.mark_non_differentiable(sm, tm)
        return logp, ent, dist, sm, tm

    @staticmethod
    def backward(ctx: Any, *grads):
        ups = list(grads[:3]) + [None] * (3 - len(grads[:3]))  # dlogp, dentropy, ddistill (absent for K = 0)
        nones = (None,) * 9
        if all(g is None for g in ups):
            return nones
        hidden, weight, labels, lse, ent, ids, tlp = ctx.saved_tensors
        need_h, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_h or need_w):
            return nones
        ups = [g.detach().reshape(-1).to(torch.float32).contiguous() if g is not None else None for g in ups]
        K = ids.size(1) if ids is not None else 0
        grad_h = torch.empty_like(hidden) if need_h else None
        grad_w = torch.zeros_like(weight) if need_w else None
        wt = weight.t()
        cs = ctx.chunk_size
        for r0 in range(0, hidden.size(0), cs):
            r1 = min(hidden.size(0), r0 + cs)
            h_c = hidden[r0:r1]
            logits = torch.mm(h_c, wt)
            _token_launch(True, logits, labels[r0:r1], ctx.ignore_index, ctx.temperature, lse[r0:r1], ent[r0:r1],
                          ids[r0:r1] if K else None, tlp[r0:r1] if K else None, ctx.clamp,
                          ups=[u[r0:r1] if u is not None else None for u in ups])  # logits now hold dlogits
            if need_h:
                torch.mm(logits, weight, out=grad_h[r0:r1])
            if need_w:
                grad_w.addmm_(logits.t(), h_c)
        return (grad_h, grad_w) + nones[2:]


def _check_token_inputs(hidden, weight, labels, ids, tlp) -> None:
    if not (hidden.is_cuda and weight.is_cuda and labels.is_cuda):
        raise VB200Error("token log-probs run on CUDA tensors only (no CPU fallback)")
    if hidden.dim() != 2 or weight.dim() != 2 or hidden.size(1) != weight.size(1):
        raise VB200Error("token log-probs: hidden [T, H] and weight [V, H] expected")
    if hidden.dtype != weight.dtype or hidden.dtype not in _DT:
        raise VB200Error("token log-probs: hidden states and weights must share a dtype, bf16 or fp32")
    if labels.dtype != torch.int64 or labels.shape != (hidden.size(0),):
        raise VB200Error("token log-probs: labels must be int64 [T]")
    if ids is None:
        return
    if not (ids.is_cuda and tlp.is_cuda):
        raise VB200Error("token log-probs: teacher top-k tensors must be CUDA tensors")
    if ids.dtype != torch.int64 or ids.dim() != 2 or ids.size(0) != hidden.size(0) or tlp.shape != ids.shape:
        raise VB200Error("token log-probs: teacher_topk_ids int64 [T, K] and teacher_topk_log_probs [T, K] expected")
    if tlp.dtype not in _DT:
        raise VB200Error(f"token log-probs: teacher log-probs must be bf16 or fp32, got {tlp.dtype}")
    if not (ids.is_contiguous() and tlp.is_contiguous()):
        raise VB200Error("token log-probs: teacher top-k tensors must be contiguous")


def _token_launch(backward: bool, logits, labels, ignore_index, temperature, lse, ent, ids, tlp, clamp,
                  logp=None, dist=None, sm=None, tm=None, ups=None) -> None:
    """One ``vb200_token_logprobs`` (forward) or ``vb200_token_logprobs_bwd`` (backward, in place) call on a chunk."""
    _check(logits, labels)
    lib = _lib.load()
    K = ids.size(1) if ids is not None else 0
    topk = (K, _ptr(ids), _ptr(tlp), _DT[tlp.dtype] if K else 0, int(clamp is not None),
            float(clamp) if clamp is not None else 0.0)
    head = (logits.data_ptr(), _DT[logits.dtype], logits.size(0), logits.size(1), logits.stride(0), labels.data_ptr(),
            int(ignore_index), float(temperature))
    with torch.cuda.device(logits.device):
        if backward:
            check(lib.vb200_token_logprobs_bwd(*head, lse.data_ptr(), ent.data_ptr(), *map(_ptr, ups), *topk,
                                               logits.data_ptr(), logits.stride(0), stream_ptr()),
                  "vb200_token_logprobs_bwd")
        else:
            check(lib.vb200_token_logprobs(*head, lse.data_ptr(), logp.data_ptr(), ent.data_ptr(), *topk, _ptr(dist),
                                           _ptr(sm), _ptr(tm), stream_ptr()), "vb200_token_logprobs")


def _shift_for_logprobs(hidden_states, labels, shift_labels, sp_enabled, teacher=()):
    """The target choice of chunk_logprobs.py:319-338 / chunk_topk_distill.py:379-393: explicit ``shift_labels`` as
    given; SP already shifted by the collator; otherwise ``labels[..., 1:]`` against ``hidden[..., :-1, :]`` (and the
    teacher tensors shifted with the labels). Returns (hidden, labels, teacher tensors, pad the outputs?)."""
    if shift_labels is not None:
        return hidden_states, shift_labels, teacher, False
    if sp_enabled:
        return hidden_states, labels, teacher, False
    return hidden_states[..., :-1, :], labels[..., 1:], tuple(t[..., 1:, :] for t in teacher), True


def _token_logprobs(hidden_states, weights, labels, teacher, chunk_size, ignore_index, temperature, clamp, pad):
    if not (hidden_states.is_cuda and weights.is_cuda and labels.is_cuda):
        raise VB200Error("token log-probs run on CUDA tensors only (no CPU fallback)")
    shape = labels.shape
    h = hidden_states.reshape(-1, hidden_states.size(-1))
    lab = labels.reshape(-1).to(torch.int64)
    ids = tlp = None
    if teacher:
        K = teacher[0].size(-1)
        ids = teacher[0].reshape(-1, K).to(torch.int64).contiguous()
        tlp = teacher[1].reshape(-1, K).contiguous()
    outs = _FusedLinearTokenLogProbs.apply(h, weights, lab, ids, tlp, float(temperature), int(chunk_size),
                                           int(ignore_index), None if clamp is None else float(clamp))
    outs = [o.view(shape) for o in outs]
    if pad:  # the final input token has no next-token target: one zero slot keeps the shape of ``labels``
        outs = [F.pad(o, (0, 1), value=0.0) for o in outs]
    if teacher:
        outs[3], outs[4] = outs[3].detach(), outs[4].detach()
    return tuple(outs)


def chunk_logprobs_function(
    hidden_states: torch.Tensor,
    weights: torch.Tensor,
    labels: torch.Tensor,
    chunk_size: int = 1024,
    ignore_index: int = -100,
    shift_labels: torch.Tensor | None = None,
    temperature: float = 1.0,
    *,
    sp_enabled: bool = False,
) -> tuple[torch.Tensor, torch.Tensor]:
    """Per-token ``log p(label)`` and softmax entropy through the chunked lm_head, without the ``[T, V]`` logits
    (the contract of chunk_logprobs.py:271-351). Both outputs have the shape of ``labels`` and are 0 at ignored
    positions; without ``shift_labels`` and SP the causal shift is applied here and the last slot is 0.
    ``sp_enabled`` stands for the reference's global parallel state: labels already shifted by the SP collator."""
    h, lab, _, pad = _shift_for_logprobs(hidden_states, labels, shift_labels, sp_enabled)
    return _token_logprobs(h, weights, lab, (), chunk_size, ignore_index, temperature, None, pad)


def chunk_topk_distill_function(
    hidden_states: torch.Tensor,
    weights: torch.Tensor,
    labels: torch.Tensor,
    teacher_topk_ids: torch.Tensor,
    teacher_topk_log_probs: torch.Tensor,
    chunk_size: int = 1024,
    ignore_index: int = -100,
    shift_labels: torch.Tensor | None = None,
    temperature: float = 1.0,
    log_prob_min_clamp: float | None = None,
    *,
    sp_enabled: bool = False,
) -> tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """``(log_probs, entropy, distillation_losses, student_mass, teacher_mass)`` of the top-k forward KL
    (chunk_topk_distill.py:329-416): ``teacher_topk_ids`` int64 ``[..., K]`` (K <= 1024) and
    ``teacher_topk_log_probs`` bf16 / fp32 ``[..., K]`` aligned with ``labels``. The two masses are detached."""
    h, lab, teacher, pad = _shift_for_logprobs(hidden_states, labels, shift_labels, sp_enabled,
                                               (teacher_topk_ids, teacher_topk_log_probs))
    return _token_logprobs(h, weights, lab, teacher, chunk_size, ignore_index, temperature, log_prob_min_clamp, pad)


@dataclass
class FusedLinearAuxOutput:
    """Per-token tensors of the log-probs paths; the field names of veomni.utils.model_outputs.FusedLinearAuxOutput."""

    log_probs: torch.Tensor | None = None
    entropy: torch.Tensor | None = None
    distillation_losses: torch.Tensor | None = None
    student_mass: torch.Tensor | None = None
    teacher_mass: torch.Tensor | None = None


class _ReduceLoss(torch.autograd.Function):
    """Token-weighted mean of the per-rank losses over the SP group (sequence_parallel/loss.py:27-60):
    forward sum_r(loss_r * n_r) / max(sum_r n_r, 1), a rank without valid tokens contributing 0;
    backward world * n_local / max(n_global, 1) * g."""

    @staticmethod
    def forward(ctx: Any, loss: torch.Tensor, num_valid: torch.Tensor, group):
        loss = torch.where(num_valid > 0, loss, torch.zeros_like(loss))
        local_n = num_valid.detach().clone()
        total = loss * num_valid
        global_n = num_valid.detach().clone()
        torch.distributed.all_reduce(total, group=group)
        torch.distributed.all_reduce(global_n, group=group)
        ctx.save_for_backward(local_n, global_n)
        ctx.world = torch.distributed.get_world_size(group)
        return total / global_n.clamp_min(1)

    @staticmethod
    def backward(ctx: Any, g: torch.Tensor):
        local_n, global_n = ctx.saved_tensors
        return ctx.world * local_n * g / global_n.clamp(min=1), None, None


def b200_cross_entropy(
    logits: torch.Tensor | None = None,
    labels: torch.Tensor | None = None,
    vocab_size: int | None = None,
    num_items_in_batch: int | torch.Tensor | None = None,
    ignore_index: int = -100,
    shift_labels: torch.Tensor | None = None,
    **kwargs,
) -> tuple[torch.Tensor, torch.Tensor | None]:
    """``cross_entropy_fn`` for ForCausalLMLoss / ForSequenceClassificationLoss. Prefers the fused-linear form when the
    caller passes ``hidden_states`` and ``weights`` (then no logits are returned, as with the liger kernel)."""
    hidden_states = kwargs.pop("hidden_states", None)
    weights = kwargs.pop("weights", None)
    chunk_size = int(kwargs.pop("chunk_size", 1024))
    labels = labels.reshape(-1)
    scale, scale_dev = _scales(labels, num_items_in_batch, ignore_index)
    if hidden_states is not None and weights is not None:
        hidden_states = hidden_states.reshape(-1, hidden_states.size(-1))
        loss = _FusedLinearCrossEntropy.apply(hidden_states, weights, labels, ignore_index, scale, scale_dev, chunk_size)
        return loss, logits
    if logits is None:
        raise VB200Error("b200_cross_entropy needs logits, or hidden_states and weights")
    logits = logits.reshape(-1, vocab_size if vocab_size is not None else logits.size(-1))
    return _CrossEntropy.apply(logits, labels, ignore_index, scale, scale_dev), logits


def ForCausalLMLoss(
    logits: torch.Tensor | None = None,
    labels: torch.Tensor | None = None,
    vocab_size: int | None = None,
    num_items_in_batch: int | None = None,
    ignore_index: int = -100,
    shift_labels: torch.Tensor | None = None,
    *,
    cross_entropy_fn: Callable = b200_cross_entropy,
    sp_group=None,
    **kwargs,
):
    """Outer policy of the causal-LM loss (reference __init__.py:89-221, loss path only): shift labels unless the
    sequence is SP-sharded (then the data pipeline already shifted them), flatten, call the kernel, and reduce the
    loss over the SP group weighted by each rank's valid-token count (sequence_parallel/loss.py).
    Returns ``(loss, logits, None)`` like the reference wrapper.

    With ``return_log_probs=True`` (reference __init__.py:107-177) the loss path is skipped: the per-token tensors of
    :func:`chunk_logprobs_function`, or of :func:`chunk_topk_distill_function` when ``teacher_topk_ids`` and
    ``teacher_topk_log_probs`` are passed, come back as ``(None, None, FusedLinearAuxOutput)``. ``temperature``,
    ``log_prob_min_clamp`` and ``chunk_size`` are forwarded to them."""
    hidden_states = kwargs.pop("hidden_states", None)
    weights = kwargs.pop("weights", None)
    if kwargs.pop("return_log_probs", False):
        sp_enabled = sp_group is not None and torch.distributed.get_world_size(sp_group) > 1
        return None, None, _log_probs_branch(hidden_states, weights, labels, ignore_index, shift_labels, sp_enabled,
                                             **kwargs)
    if hidden_states is None and logits is None:
        raise VB200Error("hidden_states or logits must be provided.")
    sp_enabled = sp_group is not None and torch.distributed.get_world_size(sp_group) > 1
    if not sp_enabled:
        if shift_labels is None:
            labels = F.pad(labels, (0, 1), value=ignore_index)
            shift_labels = labels[..., 1:].contiguous()
    else:
        shift_labels = labels
    shift_labels = shift_labels.reshape(-1)
    if hidden_states is not None:
        hidden_states = hidden_states.reshape(-1, hidden_states.size(-1))
    if logits is not None:
        logits = logits.reshape(-1, vocab_size)
    loss, logits = cross_entropy_fn(logits, shift_labels, vocab_size, num_items_in_batch, ignore_index,
                                    hidden_states=hidden_states, weights=weights, **kwargs)
    if sp_enabled:
        loss = _ReduceLoss.apply(loss, (shift_labels != ignore_index).sum(), sp_group)
    return loss, logits, None


def _log_probs_branch(hidden_states, weights, labels, ignore_index, shift_labels, sp_enabled, temperature=1.0,
                      teacher_topk_ids=None, teacher_topk_log_probs=None, log_prob_min_clamp=None, chunk_size=1024,
                      **_ignored) -> FusedLinearAuxOutput:
    """The ``return_log_probs=True`` branch of ForCausalLMLoss, with the reference's errors (__init__.py:135-143)."""
    if hidden_states is None:
        raise ValueError("return_log_probs=True requires hidden_states (fused-linear path).")
    if weights is None:
        raise ValueError("return_log_probs=True requires weights (lm_head weight).")
    if (teacher_topk_ids is None) != (teacher_topk_log_probs is None):
        raise ValueError("teacher_topk_ids and teacher_topk_log_probs must be provided together for "
                         "the top-k distillation path.")
    common = dict(chunk_size=chunk_size, ignore_index=ignore_index, shift_labels=shift_labels, temperature=temperature,
                  sp_enabled=sp_enabled)
    if teacher_topk_ids is not None:
        lp, ent, dist, sm, tm = chunk_topk_distill_function(hidden_states, weights, labels, teacher_topk_ids,
                                                            teacher_topk_log_probs, log_prob_min_clamp=log_prob_min_clamp,
                                                            **common)
        return FusedLinearAuxOutput(log_probs=lp, entropy=ent, distillation_losses=dist, student_mass=sm, teacher_mass=tm)
    lp, ent = chunk_logprobs_function(hidden_states, weights, labels, **common)
    return FusedLinearAuxOutput(log_probs=lp, entropy=ent)
