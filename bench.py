#!/usr/bin/env python
"""bench.py — tokens/sec of the Qwen3-8B FSDP2 bf16 training step (seq_len 4096, synthetic packed text).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W [--workload qwen3_8b|ulysses32k|moe30b]
    python bench.py --impl reference ...      # the reference's eager CPU path on this box's host cores

One "step" = forward + backward (per-layer gradient checkpointing, as VeOmni's default) + grad-norm clip + AdamW step +
zero_grad of the full model (random init), one packed micro-batch per data-parallel rank (weak scaling). Every op on the
hot path (RMSNorm, q/k-norm+RoPE, varlen attention, SwiGLU / MoE route + GroupGEMM, fused linear-cross-entropy, FSDP2
all-gather / reduce-scatter, Ulysses all-to-all, EP dispatch / combine, clip and AdamW) is a veomni_b200 sm_100a kernel;
dense projections are cuBLAS. Prints ONE JSON line (rank 0).

Workloads (BASELINE.json configs):
  qwen3_8b    configs[1]  Qwen3-8B FSDP2 bf16 seq 4096, DP only — the headline. At 1 GPU the model is NOT wrapped in FSDP
                          (as the reference: veomni/distributed/torch_parallelize.py:438-440,465).
  ulysses32k  configs[2]  Qwen3-8B FSDP2 + Ulysses SP degree 4 (degree = world if world < 4), one 32768-token sample per SP group
  moe30b      configs[3]  Qwen3-30B-A3B FSDP2 + EP degree = world (8 in the config), GroupGEMM path, seq 4096

At world > 1 the line carries "parity" (bit-exact checks of the NVLink collectives against NCCL-moved expected data and
FSDP2 gradients vs PyTorch's NCCL comm, run in this very process group before the timed region), "comm" (achieved NVLink
GB/s of the FSDP kernels inside the step) and "nccl_ab" (the same step on PyTorch's default NCCL FSDP2 collectives).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

SEQ_LEN = 4096
METRIC = "tokens/sec (Qwen3-8B FSDP2 bf16 seq4096)"
CPU_SAMPLE_TOKENS = 256  # the bounded CPU sample: one definition for `cpu_baseline` and `--impl reference`
DUMP_SAMPLE = 4096  # --dump-outputs: sampled elements per parameter (Qwen3-8B: 399 parameters, 5.4 MB in all)

# DRAM bytes per launch (read + write) of the three attention kernels at T=4096, 32/8 heads, D=128, from ncu --set full
# (profiles/r02_topkernels_ncu.txt: attn_bwd_dkdv_tc_kernel, attn_bwd_dq_n128_kernel, attn_fwd_tc_kernel<W8>)
NCU_TRAFFIC_BYTES = {"bwd_dkdv": 85890304 + 3582464, "bwd_dq": 84962560 + 9859072, "fwd": 50362368 + 2289920}


def _peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "how": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "how": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 8 for i in range(4) if r[4 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's eager path (restated in oracle/qwen3_cpu.py) on a bounded sample of the workload
# ------------------------------------------------------------------------------------------------
def _pick_threads() -> int:
    import torch

    ncpu = os.cpu_count() or 1
    # all host threads are available to the CPU arm, but bf16 GEMMs of this size stop scaling long before 128+ threads:
    # time a small matmul at a few thread counts and keep the fastest
    best, best_t = ncpu, float("inf")
    a, b = torch.randn(256, 4096).bfloat16(), torch.randn(12288, 4096).bfloat16()
    for c in sorted({c for c in (ncpu, ncpu // 2, ncpu // 4, 32, 16) if 1 <= c <= ncpu}):
        torch.set_num_threads(c)
        torch.nn.functional.linear(a, b)
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.linear(a, b)
        t = time.perf_counter() - t0
        if t < best_t:
            best, best_t = c, t
    return best


def cpu_sample(steps: int, warmup: int, budget_s: float) -> dict:
    """Time `steps` sample steps (after `warmup`) of oracle.qwen3_cpu.SampleStep; stops early past `budget_s` seconds."""
    import torch

    from oracle.qwen3_cpu import SampleStep

    cores = _pick_threads()
    torch.set_num_threads(cores)
    t_init = time.perf_counter()
    s = SampleStep(tokens=CPU_SAMPLE_TOKENS, layers=36, threads=cores, seq_len=SEQ_LEN)
    t_init = time.perf_counter() - t_init
    t_start = time.perf_counter()
    for _ in range(warmup):
        s.run()
        if time.perf_counter() - t_start > budget_s / 3:
            break
    times = []
    for _ in range(max(1, steps)):
        times.append(s.run())
        if time.perf_counter() - t_start > budget_s:
            break
    sec = sum(times) / len(times)
    return {"value": round(CPU_SAMPLE_TOKENS / sec, 3), "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"one sample step = the full Qwen3-8B (36 layers + embedding + lm_head + causal-LM loss, bf16 eager ops as in "
                      f"oracle/qwen3_cpu.py) forward + per-layer recompute + backward on {CPU_SAMPLE_TOKENS} of the step's {SEQ_LEN} "
                      f"tokens, clip_grad_norm, and AdamW over {CPU_SAMPLE_TOKENS}/{SEQ_LEN} of the 8.19 B fp32 parameters; every step "
                      f"really executed (no extrapolation); {len(times)} timed steps, mean",
            "seconds_per_sample_step": round(sec, 3), "steps_timed": len(times), "init_s": round(t_init, 1), "loss": round(s.loss, 4)}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    base = cpu_sample(steps=args.steps, warmup=min(args.warmup, 1), budget_s=150.0)
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "tokens/s", "n_gpus": args.gpus,
           "steps": base["steps_timed"], "warmup": min(args.warmup, 1), "ms_per_step": round(base["seconds_per_sample_step"] * 1e3, 1),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": f"Qwen3-8B bf16 seq_len 4096 training step (BASELINE configs[1]) on host CPU cores, reference eager ops; "
                                  f"each timed step is a bounded {CPU_SAMPLE_TOKENS}-token sample of the {SEQ_LEN}-token step (see cpu_baseline.sample)",
                      "global_batch": 1, "seq_len": SEQ_LEN, "sample_tokens": CPU_SAMPLE_TOKENS},
           "cpu_baseline": base,
           "e2e": {"value": base["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": round(time.time() - t0, 1)}
    print(json.dumps(out), flush=True)


def dump_outputs(out_dir: Path, model, opt, loss: float, grad_norm) -> None:
    """Write what the last timed step handed back as float arrays, for output-for-output comparison of two builds:
    ``loss.npy`` and ``grad_norm.npy`` (float64, shape [1]) and ``params_sample.npy`` (float32), the updated parameters
    (the optimizer's fp32 masters where it keeps them) at DUMP_SAMPLE seeded positions each, in ``named_parameters``
    order. Under FSDP the sample is this rank's shard."""
    import numpy as np
    import torch
    from torch.distributed.tensor import DTensor

    g = torch.Generator().manual_seed(0)
    parts = []
    with torch.no_grad():
        for _, p in model.named_parameters():
            t = opt.state[p].get("master", p) if p in opt.state else p
            t = (t.to_local() if isinstance(t, DTensor) else t).reshape(-1)
            if t.numel():
                idx = torch.randint(0, t.numel(), (min(DUMP_SAMPLE, t.numel()),), generator=g)
                parts.append(t[idx.to(t.device)].float().cpu())
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "loss.npy", np.array([loss], dtype=np.float64))
    np.save(out_dir / "grad_norm.npy", np.array([float(grad_norm)], dtype=np.float64))
    np.save(out_dir / "params_sample.npy", torch.cat(parts).numpy())


# ------------------------------------------------------------------------------------------------
def run_b200(args) -> None:
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (see module docstring)")
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29517")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)

    from veomni_b200 import _lib, prof
    from veomni_b200 import attention as vattn
    from veomni_b200.clip_grad_norm import clip_grad_norm
    from veomni_b200.host_qwen3 import Qwen3Config, Qwen3ForCausalLM, flops_per_token
    from veomni_b200.optim import B200AdamW
    from veomni_b200.parallel_state import init_parallel_state
    from veomni_b200.parallelize import build_parallelize_model

    _lib.load()  # fail loudly if the CUDA library is missing
    wl = args.workload
    sp = 1
    seq_len = SEQ_LEN
    if wl == "ulysses32k":
        sp = 4 if world % 4 == 0 else world
        seq_len = 32768
        if world < 2:
            raise SystemExit("--workload ulysses32k needs at least 2 GPUs")
    dp = world // sp
    ep = world if wl == "moe30b" else 1
    if wl == "moe30b" and world < 2:
        raise SystemExit("--workload moe30b needs at least 2 GPUs (expert parallelism)")
    if world > 1:
        init_parallel_state(dp_size=dp, dp_shard_size=dp, ulysses_size=sp, ep_size=ep)
    if wl == "moe30b":
        from veomni_b200.host_qwen3_moe import Qwen3MoeConfig, Qwen3MoeForCausalLM

        cfg = Qwen3MoeConfig.qwen3_30b_a3b()
    else:
        cfg = Qwen3Config.qwen3_8b()
    if args.layers:
        cfg.num_hidden_layers = args.layers  # debugging only; reported in config and marks the run invalid
    with torch.device("meta"):
        model = Qwen3MoeForCausalLM(cfg) if wl == "moe30b" else Qwen3ForCausalLM(cfg)
    reshard = bool(args.reshard)
    comm_kw = dict(b200_comm=not args.nccl_comm, comm_ctas=args.comm_ctas, rs_mode=args.rs_mode, fuse_copy_out=not args.no_fuse_copy_out,
                   enable_reshard_after_forward=reshard,
                   # Ulysses stages q/k/v (+ their gradients) of the local 32768/SP tokens in the symmetric region
                   misc_bytes=(1536 << 20) if wl == "ulysses32k" else (256 << 20))
    if wl == "moe30b":
        # 30.5 B parameters never exist unsharded: slice / shard on the meta device, then materialise and initialise the shards
        model = build_parallelize_model(model, init_device="meta", **comm_kw)
    else:
        model.to_empty(device=dev)
        model.init_weights(seed=0)
        model = build_parallelize_model(model, **comm_kw)
    inner = model
    inner.inv_freq = (1.0 / (cfg.rope_theta ** (torch.arange(0, cfg.head_dim, 2, device=dev).float() / cfg.head_dim)))
    model.train()
    if sp > 1:
        from veomni_b200.parallel_state import get_parallel_state

        model.sp_group = get_parallel_state().ulysses_group
    if ep > 1:
        from veomni_b200 import moe as vmoe
        from veomni_b200.ep import EPContext
        from veomni_b200.parallel_state import get_parallel_state

        from veomni_b200.symm import get_symmetric_memory

        ep_group = get_parallel_state().ep_group
        # dispatch / combine staging: 4 buffers of T*K*H*2 = 134 MB each (grown 1.5x on demand) + the counts exchange
        vmoe.set_ep_group(EPContext(ep_group, get_symmetric_memory(ep_group, 3 << 30, tag="ep")))
    fsdp = world > 1
    if args.torch_adamw:
        opt = torch.optim.AdamW(model.parameters(), lr=1e-4, betas=(0.9, 0.95), weight_decay=0.0, fused=True)
    else:
        # one multi-tensor kernel; at 1 GPU it owns the fp32 masters and the model computes on the bf16 copy it maintains
        opt = B200AdamW(model.parameters(), lr=1e-4, betas=(0.9, 0.95), weight_decay=0.0, master_weights=not fsdp)
    if not fsdp and args.torch_adamw:
        model.to(torch.bfloat16)  # debugging: pure-bf16 parameters with torch's optimizer
    fold_clip = (not args.torch_adamw) and ep == 1

    # synthetic packed micro-batches in pinned host memory (DummyTextDataset: ids ~ U{0..1023}, first label ignored);
    # under Ulysses every rank of an SP group holds its contiguous slice of the same sample (SequenceParallelCollator)
    t_local = seq_len // sp
    sp_rank, dp_rank = rank % sp, rank // sp
    g = torch.Generator().manual_seed(1234 + dp_rank)
    nbuf = 4
    host = []
    for _ in range(nbuf):
        ids = torch.randint(0, 1024, (1, seq_len), generator=g, dtype=torch.int64)
        labels = ids.clone()
        labels[0, 0] = -100
        shift = torch.nn.functional.pad(labels, (0, 1), value=-100)[..., 1:]
        pos = torch.arange(seq_len, dtype=torch.int64)[None]
        sl = slice(sp_rank * t_local, (sp_rank + 1) * t_local)
        host.append(tuple(t[:, sl].contiguous().pin_memory() for t in (ids, shift, pos)))
    cu = torch.tensor([0, seq_len], dtype=torch.int32, device=dev)
    resident = [tuple(t.to(dev) for t in h) for h in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host[0])
    n_valid_local = [int((h[1] != -100).sum()) for h in host]
    sp_group = getattr(model, "sp_group", None)
    last_grad_norm = [None]  # device scalar of the latest step, kept for --dump-outputs

    def step(batch, i=0):
        ids, shift, pos = batch
        loss = model(ids, pos, cu, seq_len, shift_labels=shift)
        if sp > 1:  # mean over the SP group's valid tokens (sequence_parallel/loss.py): local mean * n_local / n_group
            loss = loss * (n_valid_local[i % nbuf] * sp / float(seq_len - 1))
        loss.backward()
        if fold_clip:
            last_grad_norm[0], coef = clip_grad_norm(model, 1.0, return_coef=True)  # veomni_clip_grad_norm semantics; the
            opt.step(grad_scale=coef)                                                # scaling pass is folded into AdamW
        else:
            last_grad_norm[0] = clip_grad_norm(model, 1.0)
            opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def timed(nsteps, e2e: bool):
        dist.barrier()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        last = None
        for i in range(nsteps):
            if e2e:
                batch = tuple(t.to(dev, non_blocking=True) for t in host[i % nbuf])
                last = step(batch, i).item()  # device->host read of the step's loss
            else:
                last = step(resident[i % nbuf], i)
        e.record()
        torch.cuda.synchronize()
        dist.barrier()
        t = torch.tensor([s.elapsed_time(e)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / nsteps, (last if isinstance(last, float) else float(last.item()))

    # ---- multi-GPU parity, in this process group, before anything is timed ------------------------------------------
    parity = None
    if fsdp and not args.skip_parity and not args.nccl_comm:
        from veomni_b200 import selfcheck

        t0 = time.time()
        symm = getattr(model, "_vb200_symm", None)
        if symm is not None and symm.world == world:
            parity = selfcheck.run_all(symm, dev, fsdp=True, ep=True)  # raises VB200Error on any mismatch
        elif symm is not None:
            parity = selfcheck.run_all(symm, dev, fsdp=False, ep=False)
            parity["note"] = f"collectives checked on the {symm.world}-rank FSDP shard group"
        if parity is not None:
            parity["seconds"] = round(time.time() - t0, 1)
        torch.cuda.synchronize()
        dist.barrier()

    for i in range(args.warmup):
        wl_ = step(resident[i % nbuf], i)
        if os.environ.get("VB200_BENCH_DEBUG"):  # untimed: one sync per warm-up step to see the loss of every rank
            print(f"[rank {rank}] warm-up step {i}: loss {float(wl_.item()):.5f}", file=sys.stderr, flush=True)
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _lib.reset_launch_count()
    # CUDA-event pairs around every launch of the attention kernels (the heaviest kernels of ours) and the collectives
    vattn.PROFILE = {"fwd": [], "bwd_dq": [], "bwd_dkdv": []}
    prof.ACTIVE = {"fsdp_all_gather": [], "fsdp_reduce_scatter": [], "ulysses_a2a": [], "ep_pull": [], "group_gemm": []}
    ms_dev, loss_dev = timed(args.steps, e2e=False)
    launches = _lib.launch_count()
    aprof, vattn.PROFILE = vattn.PROFILE, None
    cprof, prof.ACTIVE = prof.ACTIVE, None
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:  # before the e2e pass below moves the weights on
        dump_outputs(Path(args.dump_outputs), model, opt, loss_dev, last_grad_norm[0])
    prof_ms = {k: [a.elapsed_time(b) for a, b in v] for k, v in aprof.items()}
    comm_stats = prof.summarize(cprof)
    ms_e2e, loss_e2e = timed(args.steps, e2e=True)
    mem_gb = torch.cuda.max_memory_allocated() / 2**30
    clocks = sampler.stop() if rank == 0 else {}

    # ---- side measurements (outside the timed regions; none of them can take the headline line down) ---------------
    no_rc = None
    if not args.skip_no_recompute and wl == "qwen3_8b":
        prev = inner.gradient_checkpointing
        inner.gradient_checkpointing = False
        try:
            torch.cuda.reset_peak_memory_stats()
            for i in range(2):
                step(resident[i % nbuf], i)
            ms_nr, _ = timed(args.steps, e2e=False)
            no_rc = {"value": round(seq_len * dp / (ms_nr / 1e3), 1), "unit": "tokens/s", "ms_per_step": round(ms_nr, 2),
                     "max_mem_gb": round(torch.cuda.max_memory_allocated() / 2**30, 1)}
        except torch.OutOfMemoryError:
            no_rc = {"value": None, "note": "out of memory without recomputation"}
        except Exception as ex:  # noqa: BLE001
            no_rc = {"value": None, "note": f"{type(ex).__name__}: {str(ex)[:160]}"}
        inner.gradient_checkpointing = prev
    nccl_ab = None
    if fsdp and not args.skip_ab and not args.nccl_comm and ep == 1:
        try:  # the same step on PyTorch's default NCCL all-gather / reduce-scatter (same process, same weights)
            from veomni_b200.fsdp_comm import reinstall_fsdp_comm, uninstall_fsdp_comm

            saved = uninstall_fsdp_comm(model)
            for i in range(2):
                step(resident[i % nbuf], i)
            ms_nccl, _ = timed(args.steps, e2e=False)
            reinstall_fsdp_comm(model, saved)
            for i in range(1):
                step(resident[i % nbuf], i)
            ms_again, _ = timed(args.steps, e2e=False)
            nccl_ab = {"ms_per_step_nccl_comm": round(ms_nccl, 2), "ms_per_step_b200_comm": round(ms_again, 2),
                       "speedup": round(ms_nccl / ms_again, 4), "note": "same process, same weights; B200 comm re-timed right after the NCCL leg"}
        except Exception as ex:  # noqa: BLE001
            nccl_ab = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
    if args.torch_profile:  # debugging aid: per-kernel device time of one step on rank 0
        from torch.profiler import ProfilerActivity, profile

        dist.barrier()
        with profile(activities=[ProfilerActivity.CUDA]) as tp:
            step(resident[0])
            torch.cuda.synchronize()
        if rank == 0:
            with open(args.torch_profile, "w") as fh:
                fh.write(tp.key_averages().table(sort_by="cuda_time_total", row_limit=70, max_name_column_width=90))
                try:  # where the step idles: per-stream busy time and the compute stream's gaps (tools/stream_gaps.py)
                    from tools import stream_gaps

                    fh.write("\n" + stream_gaps.report(tp))
                except Exception as ex:  # noqa: BLE001
                    fh.write(f"\nstream_gaps failed: {type(ex).__name__}: {ex}\n")
        dist.barrier()

    if rank == 0:
        peaks = _peaks()
        tokens = seq_len * dp
        value = tokens / (ms_dev / 1e3)
        heads_local = cfg.num_attention_heads // sp
        fwd_flops = 4 * seq_len * seq_len * cfg.head_dim * heads_local / 2  # causal fwd per launch
        # algorithmic FLOPs per launch (SURVEY.md §8(d)): fwd = 2 matmuls, dQ = 1, dK+dV = 2 of the 5 backward matmuls
        kinfo = {"fwd": ("attn_fwd_tc_kernel (varlen causal attention forward, tcgen05)", fwd_flops),
                 "bwd_dkdv": ("attn_bwd_dkdv_tc_kernel (attention backward dK/dV, tcgen05)", fwd_flops * 2.5 * 0.6),
                 "bwd_dq": ("attn_bwd_dq_tc_kernel (attention backward dQ, tcgen05)", fwd_flops * 2.5 * 0.4)}
        totals = {k: sum(v) for k, v in prof_ms.items() if v}
        dom = max(totals, key=totals.get) if totals else "fwd"
        attn_ms = prof_ms.get(dom, [])
        attn_flops = kinfo[dom][1]
        attn_avg_ms = sum(attn_ms) / max(1, len(attn_ms))
        achieved = attn_flops / (attn_avg_ms * 1e-3) / 1e12 if attn_ms else None
        names = {"qwen3_8b": "Qwen3-8B FSDP2 bf16 seq_len 4096 training step (BASELINE configs[1])",
                 "ulysses32k": f"Qwen3-8B FSDP2 + Ulysses SP{sp} bf16, one 32768-token sample per SP group (BASELINE configs[2])",
                 "moe30b": f"Qwen3-30B-A3B FSDP2 + EP{ep} bf16 seq_len 4096, GroupGEMM path (BASELINE configs[3])"}
        par = ("single GPU, no FSDP wrap (as the reference at world_size 1)" if not fsdp else
               f"fsdp{dp * sp}" + (f" x ulysses{sp}" if sp > 1 else "") + (f" + ep{ep}" if ep > 1 else ""))
        out = {
            "metric": METRIC if wl == "qwen3_8b" else f"tokens/sec ({wl})", "value": round(value, 1), "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_dev, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": names[wl] + ": fwd+bwd with per-layer gradient checkpointing (attention o/lse are kept across the "
                                   "recompute instead of re-running the attention kernel — the reference recomputes it), clip_grad_norm, "
                                   f"AdamW; one {seq_len}-token packed sample per data-parallel rank",
                       "global_batch": dp, "seq_len": seq_len, "parallelism": par, "layers": cfg.num_hidden_layers,
                       "params_b": round(cfg.num_params() / 1e9, 3) if wl != "moe30b" else 30.5,
                       "l2": "inputs (>= 16 GB of bf16 weights per step) larger than L2",
                       "fsdp_comm": ("none (1 GPU)" if not fsdp else "nccl" if args.nccl_comm else
                                     f"veomni_b200 NVLink kernels: all-gather pull{' with fused copy-out' if not args.no_fuse_copy_out else ''}, "
                                     f"reduce-scatter {args.rs_mode or 'push'} ({args.comm_ctas} CTAs)"),
                       "reshard_after_forward": reshard if fsdp else None,
                       "optimizer": "torch.optim.AdamW(fused=True)" if args.torch_adamw else
                                    ("veomni_b200 multi-tensor AdamW" + (" on fp32 masters + bf16 model copy" if not fsdp else " on the fp32 shards")
                                     + (", clip coefficient folded in" if fold_clip else "")),
                       "valid": args.layers == 0},
            "tokens_per_sec_per_gpu": round(value / world, 1),
            "e2e": {"value": round(tokens / (ms_e2e / 1e3), 1), "unit": "tokens/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e, 2)},
            "gpu_launches": int(launches),
            "roofline": {"kernel": kinfo[dom][0] + f", {len(attn_ms) // max(1, args.steps)} launches/step",
                         "attention_ms_per_step": {k: round(v / max(1, args.steps), 2) for k, v in totals.items()},
                         "bound": "tensor", "achieved": round(achieved, 1) if achieved else None,
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": round(achieved / peaks["bf16_tflops_sustained"], 4) if achieved else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of
                         # the same kernel at the same shape (profiles/r02_topkernels_ncu.txt)
                         "traffic": NCU_TRAFFIC_BYTES.get(dom) if (wl == "qwen3_8b") else None,
                         "traffic_source": "profiles/r02_topkernels_ncu.txt (ncu --set full, one launch at the same shape)",
                         "peak_source": f"{peaks['how']} (sustained cuBLAS bf16, kernel timed inside a long step)",
                         "avg_launch_ms": round(attn_avg_ms, 4), "launches_timed": len(attn_ms),
                         "algorithmic_flops_per_launch": attn_flops},
            "clocks": clocks, "loss": round(loss_dev, 4), "loss_e2e": round(loss_e2e, 4), "max_mem_gb": round(mem_gb, 1),
        }
        if wl != "moe30b":
            fpt = flops_per_token(cfg, [seq_len])
            out["mfu_measured_peak"] = round(fpt * value / world / (peaks["bf16_tflops_sustained"] * 1e12), 4)
            out["mfu_2250"] = round(fpt * value / world / 2250e12, 4)
        if comm_stats:
            comm = {}
            for tag, st in comm_stats.items():
                per_step_ms = st["ms"] / max(1, args.steps)
                ent = {"launches_per_step": st["launches"] // max(1, args.steps), "busy_ms_per_step": round(per_step_ms, 2)}
                if tag == "group_gemm":
                    ent["achieved_tflops"] = round(st["rate"] / 1e12, 1)
                    ent["frac_of_peak"] = round(st["rate"] / 1e12 / peaks["bf16_tflops_sustained"], 3)
                else:
                    ent["nvlink_in_GBps"] = round(st["rate"] / 1e9, 1)
                    ent["frac_of_900"] = round(st["rate"] / 1e9 / 900.0, 3)
                comm[tag] = ent
            out["comm"] = comm
        if ep > 1:
            from veomni_b200 import moe as vmoe_

            st = dict(vmoe_._ep_state().stats)
            rows_sent = seq_len * cfg.num_experts_per_tok
            out["ep_routing"] = {"exchanges": st["calls"], "rows_sent_per_exchange": rows_sent, "rows_received_min": st["min_recv"],
                                 "rows_received_max": st["max_recv"],
                                 "rows_received_mean": round(st["sum_recv"] / max(1, st["calls"]), 1), "rank": rank}
        if parity is not None:
            out["parity"] = parity
        if nccl_ab is not None:
            out["nccl_ab"] = nccl_ab
        if no_rc is not None:
            out["no_recompute"] = no_rc
        if not args.no_cpu_baseline and world == 1:
            try:
                out["cpu_baseline"] = cpu_sample(steps=2, warmup=1, budget_s=40.0)
            except Exception as ex:  # noqa: BLE001
                out["cpu_baseline"] = {"value": None, "error": f"{type(ex).__name__}: {str(ex)[:160]}"}
        print(json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="qwen3_8b", choices=["qwen3_8b", "ulysses32k", "moe30b"])
    ap.add_argument("--layers", type=int, default=0, help="debug only: fewer layers (marks the line invalid)")
    ap.add_argument("--nccl-comm", action="store_true", help="debug: PyTorch's default NCCL FSDP2 collectives")
    ap.add_argument("--comm-ctas", type=int, default=32)
    ap.add_argument("--rs-mode", default=None, choices=["push", "pull", "f32"], help="reduce-scatter variant (default push: copy-in fused)")
    ap.add_argument("--no-fuse-copy-out", action="store_true", help="debug: all-gather into the buffer + torch split_with_sizes_copy")
    ap.add_argument("--reshard", type=int, default=0, help="FSDP2 reshard_after_forward (default 0: the bf16 parameters stay "
                                                            "gathered between forward and backward — 16 GB of the 180 GB)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--torch-adamw", action="store_true", help="debug: torch.optim.AdamW(fused=True) instead of the veomni_b200 kernel")
    ap.add_argument("--skip-no-recompute", action="store_true", help="skip the extra no-recomputation measurement")
    ap.add_argument("--skip-parity", action="store_true", help="skip the multi-GPU parity stage")
    ap.add_argument("--skip-ab", action="store_true", help="skip the NCCL-comm A/B side measurement")
    ap.add_argument("--torch-profile", default="", help="debug: write a torch.profiler kernel table of one extra step")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 training step")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
