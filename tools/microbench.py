"""Per-kernel timing of the veomni_b200 kernels at the BASELINE sizes (CUDA events, inputs > L2 or rotated).

Usage: python tools/microbench.py [--only rmsnorm,rope,...] [--iters N] — prints one JSON line per kernel:
algorithmic bytes (SURVEY.md §8(d)), microseconds, achieved GB/s and fraction of the measured HBM peak.
"""
import argparse
import json
import os
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

from veomni_b200 import _lib  # noqa: E402
from veomni_b200 import functional as F  # noqa: E402

BF = torch.bfloat16


def peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d["hbm_gbs"], d["bf16_tflops"], "measured"
    return 6650.0, 1590.0, "fallback"


def _profile_once():  # VB200_PROFILE_ONCE=1 (or --profile-once): under `ncu --profile-from-start off`, capture ONE call of every benchmarked callable
    return os.environ.get("VB200_PROFILE_ONCE", "0") == "1"


def time_fn(fn, sets, iters=20, warmup=5):
    """sets: list of argument tuples rotated so consecutive launches touch different memory (> L2 in total)."""
    n = len(sets)
    if _profile_once():  # two warm-up calls outside the capture range, one call inside it
        fn(*sets[0])
        fn(*sets[1 % n])
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.profiler.start()
        s.record()
        fn(*sets[2 % n])
        e.record()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return s.elapsed_time(e) * 1e3
    for i in range(warmup):
        fn(*sets[i % n])
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(iters):
        fn(*sets[i % n])
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) * 1e3 / iters  # us


def report(name, us, nbytes=None, flops=None):
    hbm, tf, how = peaks()
    r = {"kernel": name, "us": round(us, 2)}
    if nbytes:
        r["algo_MB"] = round(nbytes / 1e6, 2)
        r["GBps"] = round(nbytes / us / 1e3, 1)
        r["frac_hbm"] = round(nbytes / us / 1e3 / hbm, 3)
    if flops:
        r["TFLOPs"] = round(flops / us / 1e6, 1)
        r["frac_tensor"] = round(flops / us / 1e6 / tf, 3)
    r["peak"] = how
    print(json.dumps(r), flush=True)


def bench_rmsnorm(dev, iters):
    T, H = 4096, 4096
    lib = _lib.load()
    nset = 6  # 6 x (32+32 MB) > 126 MB L2
    sets = []
    for _ in range(nset):
        x = torch.randn(T, H, device=dev, dtype=BF)
        sets.append((x, torch.empty_like(x), torch.empty(T, device=dev, dtype=torch.float32)))
    w = torch.ones(H, device=dev, dtype=BF)
    st = torch.cuda.current_stream().cuda_stream

    def fwd(x, y, r):
        lib.vb200_rmsnorm_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), r.data_ptr(), T, H, 1e-6, st)

    report("rmsnorm_fwd[4096x4096]", time_fn(fwd, sets, iters), nbytes=2 * T * H * 2)
    nparts = lib.vb200_rmsnorm_bwd_partials(T, H)
    part = torch.empty(nparts, H, device=dev, dtype=torch.float32)
    dw = torch.empty(H, device=dev, dtype=torch.float32)
    bsets = [(x, y, r, torch.empty_like(x)) for (x, y, r) in sets]
    for x, y, r in sets:
        fwd(x, y, r)

    def bwd(x, dy, r, dx):
        lib.vb200_rmsnorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), r.data_ptr(), dx.data_ptr(), part.data_ptr(),
                              dw.data_ptr(), T, H, st)

    report("rmsnorm_bwd[4096x4096]", time_fn(bwd, bsets, iters), nbytes=3 * T * H * 2)
    # fused residual-add + norm (the decoder layer's two norms): x, residual -> h, y ; dy, h, dh -> dx
    asets = [(x, y, r, torch.empty_like(x), torch.empty_like(x)) for (x, y, r) in sets]

    def afwd(x, res, r, h, y):
        lib.vb200_add_rmsnorm_fwd(x.data_ptr(), res.data_ptr(), w.data_ptr(), h.data_ptr(), y.data_ptr(), r.data_ptr(), T, H, 1e-6, st)

    report("add_rmsnorm_fwd[4096x4096]", time_fn(afwd, asets, iters), nbytes=4 * T * H * 2)

    def abwd(dy, x, r, dres, dx):
        lib.vb200_rmsnorm_bwd_add(dy.data_ptr(), x.data_ptr(), w.data_ptr(), r.data_ptr(), dres.data_ptr(), dx.data_ptr(),
                                  part.data_ptr(), dw.data_ptr(), T, H, st)

    report("rmsnorm_bwd_add[4096x4096]", time_fn(abwd, asets, iters), nbytes=4 * T * H * 2)
    # the same kernels on 4x the rows (the Ulysses-32k per-rank shape x2): the 4096-row launches are 10 us of streaming plus
    # ~6 us of launch ramp and drain, so the fraction at this size says how much of the gap is fixed cost
    T4 = 4 * T
    big = [(torch.randn(T4, H, device=dev, dtype=BF), torch.empty(T4, H, device=dev, dtype=BF),
            torch.empty(T4, device=dev, dtype=torch.float32), torch.empty(T4, H, device=dev, dtype=BF)) for _ in range(2)]

    def fwd4(x, y, r, _d):
        lib.vb200_rmsnorm_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), r.data_ptr(), T4, H, 1e-6, st)

    report("rmsnorm_fwd[16384x4096]", time_fn(fwd4, big, iters), nbytes=2 * T4 * H * 2)
    part4 = torch.empty(lib.vb200_rmsnorm_bwd_partials(T4, H), H, device=dev, dtype=torch.float32)

    def bwd4(x, dy, r, dx):
        lib.vb200_rmsnorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), r.data_ptr(), dx.data_ptr(), part4.data_ptr(),
                              dw.data_ptr(), T4, H, st)

    report("rmsnorm_bwd[16384x4096]", time_fn(bwd4, big, iters), nbytes=3 * T4 * H * 2)
    del big
    # per-head norm shape (q heads)
    R, C = 4096 * 40, 128
    hs = [(torch.randn(R, C, device=dev, dtype=BF), torch.empty(R, C, device=dev, dtype=BF),
           torch.empty(R, device=dev, dtype=torch.float32)) for _ in range(4)]
    wh = torch.ones(C, device=dev, dtype=BF)

    def fwdh(x, y, r):
        lib.vb200_rmsnorm_fwd(x.data_ptr(), wh.data_ptr(), y.data_ptr(), r.data_ptr(), R, C, 1e-6, st)

    report("rmsnorm_fwd[163840x128]", time_fn(fwdh, hs, iters), nbytes=2 * R * C * 2)


def bench_rope(dev, iters):
    """Direct C-ABI calls with preallocated buffers (the Python autograd wrappers cost more CPU time than these kernels)."""
    T, Hq, Hk, D = 4096, 32, 8, 128
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    cos = torch.randn(T, D, device=dev, dtype=BF)
    sin = torch.randn(T, D, device=dev, dtype=BF)
    wq = torch.ones(D, device=dev, dtype=BF)
    sets = []
    for _ in range(6):
        q, k = torch.randn(T, Hq, D, device=dev, dtype=BF), torch.randn(T, Hk, D, device=dev, dtype=BF)
        sets.append((q, k, torch.empty_like(q), torch.empty_like(k), torch.empty(T, Hq, device=dev), torch.empty(T, Hk, device=dev)))
    nbytes = 2 * T * (Hq + Hk) * D * 2

    def rope(q, k, qo, ko, rq, rk):
        lib.vb200_rope(q.data_ptr(), qo.data_ptr(), k.data_ptr(), ko.data_ptr(), cos.data_ptr(), sin.data_ptr(), T, Hq, Hk, D,
                       Hq * D, D, Hk * D, D, Hq * D, D, Hk * D, D, 0, st)

    report("rope_qk[4096x(32+8)x128]", time_fn(rope, sets, iters), nbytes=nbytes)

    def fused(q, k, qo, ko, rq, rk):
        lib.vb200_qknorm_rope_fwd(q.data_ptr(), k.data_ptr(), wq.data_ptr(), wq.data_ptr(), cos.data_ptr(), sin.data_ptr(),
                                  qo.data_ptr(), ko.data_ptr(), rq.data_ptr(), rk.data_ptr(), T, Hq, Hk, D, 1e-6, st)

    report("qknorm_rope_fwd[4096x(32+8)x128]", time_fn(fused, sets, iters), nbytes=nbytes)
    part = torch.empty(lib.vb200_qknorm_rope_bwd_partials(T), 2 * D, device=dev)
    dwq, dwk = torch.empty(D, device=dev), torch.empty(D, device=dev)

    def fused_bwd(q, k, qo, ko, rq, rk):
        lib.vb200_qknorm_rope_bwd(qo.data_ptr(), ko.data_ptr(), q.data_ptr(), k.data_ptr(), wq.data_ptr(), wq.data_ptr(),
                                  cos.data_ptr(), sin.data_ptr(), rq.data_ptr(), rk.data_ptr(), qo.data_ptr(), ko.data_ptr(),
                                  part.data_ptr(), dwq.data_ptr(), dwk.data_ptr(), T, Hq, Hk, D, st)

    report("qknorm_rope_bwd[4096x(32+8)x128]", time_fn(fused_bwd, sets, iters), nbytes=3 * T * (Hq + Hk) * D * 2)


def bench_swiglu(dev, iters):
    T, I = 4096, 12288
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    sets = [(torch.randn(T, I, device=dev, dtype=BF), torch.randn(T, I, device=dev, dtype=BF), torch.empty(T, I, device=dev, dtype=BF),
             torch.empty(T, I, device=dev, dtype=BF)) for _ in range(2)]

    def fwd(g, u, o, o2):
        lib.vb200_swiglu_fwd(g.data_ptr(), u.data_ptr(), o.data_ptr(), T, I, I, I, st)

    report("swiglu_fwd[4096x12288]", time_fn(fwd, sets, iters), nbytes=3 * T * I * 2)

    def bwd(g, u, o, o2):
        lib.vb200_swiglu_bwd(o.data_ptr(), g.data_ptr(), u.data_ptr(), o.data_ptr(), o2.data_ptr(), T, I, I, I, I, st)

    report("swiglu_bwd[4096x12288]", time_fn(bwd, sets, iters), nbytes=5 * T * I * 2)


def bench_loss(dev, iters):
    """One 1024-row chunk of the 151936-entry vocabulary, bf16, gradient written in place: read + write once."""
    rows, V = 1024, 151936
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    labels = torch.randint(0, V, (rows,), device=dev)
    sets = [(torch.randn(rows, V, device=dev, dtype=BF), torch.empty(rows, device=dev, dtype=torch.float32)) for _ in range(2)]

    def fused(x, lr):  # forward statistics + in-place gradient (the fused-linear path's kernel)
        lib.vb200_cross_entropy(x.data_ptr(), 0, rows, V, V, labels.data_ptr(), -100, lr.data_ptr(), None, 0, x.data_ptr(), V,
                                1.0 / rows, None, None, st)

    report("cross_entropy_fwd+grad_inplace[1024x151936 bf16]", time_fn(fused, sets, iters), nbytes=2 * rows * V * 2)

    def fwd(x, lr):  # loss only
        lib.vb200_cross_entropy(x.data_ptr(), 0, rows, V, V, labels.data_ptr(), -100, lr.data_ptr(), None, 0, None, 0,
                                1.0, None, None, st)

    report("cross_entropy_fwd[1024x151936 bf16]", time_fn(fwd, sets, iters), nbytes=rows * V * 2)
    x32 = torch.randn(rows, V, device=dev, dtype=torch.float32)
    g32 = torch.empty_like(x32)
    lr = torch.empty(rows, device=dev, dtype=torch.float32)

    def lib_ce():
        xx = x32.detach().requires_grad_(True)
        torch.nn.functional.cross_entropy(xx, labels).backward()

    report("(lib) torch cross_entropy fwd+bwd[1024x151936 fp32]", time_fn(lambda: lib_ce(), [()], iters))
    del g32, lr


def bench_logprobs(dev, iters):
    """Per-token log-probs / entropy / top-k distillation (token_stats_kernel, token_grad_kernel) on one 1024-row chunk of
    the 151936-entry vocabulary in bf16, without and with K = 64 teacher entries; then the fused-linear forward + backward
    at T = H = 4096 against the oracle's torch restatement of the reference arithmetic on the same CUDA tensors."""
    from oracle import logprobs as O
    from veomni_b200.cross_entropy import _token_launch, chunk_topk_distill_function

    rows, V, K = 1024, 151936, 64
    f32 = dict(dtype=torch.float32, device=dev)
    labels = torch.randint(0, V, (rows,), device=dev)
    ids = torch.randint(0, V, (rows, K), device=dev)
    tlp = torch.log_softmax(torch.randn(rows, K, device=dev), -1)
    st = [torch.empty(rows, **f32) for _ in range(6)]
    ups = [torch.randn(rows, **f32) for _ in range(3)]
    sets = [(torch.randn(rows, V, device=dev, dtype=BF),) for _ in range(2)]  # 2 x 311 MB > L2
    for k in (0, K):
        kid, ktl = (ids, tlp) if k else (None, None)

        def fwd(x):
            _token_launch(False, x, labels, -100, 1.0, st[0], st[1], kid, ktl, None, logp=st[2], dist=st[3], sm=st[4], tm=st[5])

        report(f"token_logprobs_fwd[1024x151936 bf16, K={k}]", time_fn(fwd, sets, iters), nbytes=rows * V * 2)
        fwd(sets[0][0])

        def bwd(x):  # in place; the values drift between calls, the traffic does not
            _token_launch(True, x, labels, -100, 1.0, st[0], st[1], kid, ktl, None, ups=ups if k else ups[:2] + [None])

        report(f"token_logprobs_grad_inplace[1024x151936 bf16, K={k}]", time_fn(bwd, sets, iters), nbytes=2 * rows * V * 2)
    del sets
    T, H = 4096, 4096
    h = (torch.randn(T, H, device=dev) * 0.5).to(BF).requires_grad_(True)
    w = (torch.randn(V, H, device=dev) * 0.02).to(BF).requires_grad_(True)
    lab = torch.randint(0, V, (T,), device=dev)
    tids = torch.randint(0, V, (T, K), device=dev)
    ttlp = torch.log_softmax(torch.randn(T, K, device=dev), -1)
    up = [torch.randn(T, **f32) for _ in range(3)]

    def ours():
        outs = chunk_topk_distill_function(h, w, lab, tids, ttlp, shift_labels=lab)
        torch.autograd.grad(sum((o * u).sum() for o, u in zip(outs[:3], up)), (h, w))

    def eager():  # the reference's per-chunk arithmetic: fp32 [1024, V] softmax / log_softmax / dense teacher temporaries
        with torch.no_grad():
            O.fused_linear_token_logprobs(h, w, lab, tids, ttlp, upstream=up)

    for name, fn in (("chunk_topk_distill fwd+bwd (veomni_b200)", ours), ("(oracle) eager restatement fwd+grads", eager)):
        fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        us = time_fn(lambda: fn(), [()], max(3, iters // 10), warmup=1)
        r = {"kernel": f"{name}[T=4096 H=4096 V=151936 K=64 bf16]", "ms": round(us / 1e3, 2),
             "peak_extra_GB": round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 2)}
        print(json.dumps(r), flush=True)


def bench_fsdp(dev, iters):
    """FSDP2 copy-in kernels and the gradient-clip kernels at Qwen3-8B layer-unit sizes (193 M parameters per unit)."""
    import ctypes

    from veomni_b200.clip_grad_norm import multi_scale_, multi_sumsq
    from veomni_b200.fsdp_comm import pack_plan

    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    H, I, Hq, Hk, D = 4096, 12288, 32, 8, 128
    shapes = [(Hq * D, H), (Hk * D, H), (Hk * D, H), (H, Hq * D), (D,), (D,), (I, H), (I, H), (H, I), (H,), (H,)]
    for world in (2, 8):
        plan, row = pack_plan(shapes, world)
        grads = [torch.randn(*s_, device=dev, dtype=BF) for s_ in shapes]
        out = torch.empty(world * row, device=dev, dtype=BF)
        flat = []
        for t, (numel, chunk, off) in zip(grads, plan):
            flat += [t.data_ptr(), numel, chunk, off]
        arr = (ctypes.c_int64 * len(flat))(*flat)
        n = sum(t.numel() for t in grads)

        def pack():
            lib.vb200_fsdp_pack_bf16(arr, len(plan), world, row, out.data_ptr(), 0, st)

        report(f"fsdp_pack_bf16 (reduce-scatter copy-in)[unit 193M, N={world}]", time_fn(lambda: pack(), [()], iters), nbytes=4 * n)

        def chunk_cat():
            torch._chunk_cat(grads, dim=0, num_chunks=world, out=out.view(world, -1))

        report(f"(lib) torch._chunk_cat bf16->bf16[unit 193M, N={world}]", time_fn(lambda: chunk_cat(), [()], iters), nbytes=4 * n)
    # all-gather copy-in: this rank's fp32 shards (1/8 of the unit) cast to bf16
    shards = [torch.randn((s_[0] + 7) // 8 * (s_[1] if len(s_) > 1 else 1), device=dev) for s_ in shapes]
    nsh = sum(t.numel() for t in shards)
    dst = torch.empty(nsh, device=dev, dtype=BF)
    flat, off = [], 0
    for t in shards:
        flat += [t.data_ptr(), t.numel(), t.numel(), off]
        off += t.numel()
    arr2 = (ctypes.c_int64 * len(flat))(*flat)
    report("fsdp_pack_bf16 (all-gather copy-in, fp32->bf16)[unit 193M / 8]",
           time_fn(lambda: lib.vb200_fsdp_pack_bf16(arr2, len(shards), 1, nsh, dst.data_ptr(), 1, st), [()], iters), nbytes=6 * nsh)
    big = [torch.randn(64 << 20, device=dev) for _ in range(4)] + [torch.randn(4096, device=dev) for _ in range(64)]
    tot = sum(t.numel() for t in big)
    multi_sumsq(big)
    report("multi_sumsq[256M fp32 + 64 small]", time_fn(lambda: multi_sumsq(big), [()], iters), nbytes=4 * tot)
    coef = torch.tensor(0.999, device=dev)
    report("multi_scale[256M fp32 + 64 small]", time_fn(lambda: multi_scale_(big, coef), [()], iters), nbytes=8 * tot)
    report("(lib) torch._foreach_norm", time_fn(lambda: torch._foreach_norm(big, 2.0), [()], iters), nbytes=4 * tot)
    report("(lib) torch._foreach_mul_", time_fn(lambda: torch._foreach_mul_(big, coef), [()], iters), nbytes=8 * tot)


BENCHES = {"rmsnorm": bench_rmsnorm, "rope": bench_rope, "swiglu": bench_swiglu, "loss": bench_loss, "logprobs": bench_logprobs,
           "fsdp": bench_fsdp}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--profile-once", action="store_true",
                    help="for `ncu --profile-from-start off --set full`: one captured launch per benchmarked callable")
    a = ap.parse_args()
    if a.profile_once:
        os.environ["VB200_PROFILE_ONCE"] = "1"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    names = [n for n in a.only.split(",") if n] or list(BENCHES)
    for n in names:
        mod = BENCHES.get(n)
        if mod is None:
            try:
                extra = __import__("tools.microbench_extra", fromlist=["BENCHES"]).BENCHES
                mod = extra[n]
            except Exception as ex:  # noqa: BLE001
                print(json.dumps({"kernel": n, "error": str(ex)}))
                continue
        mod(dev, a.iters)


if __name__ == "__main__":
    main()
