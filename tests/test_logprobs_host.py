"""Per-token log-probs / top-k distillation, host side: the oracle against the reference fixture, and the dispatcher
``veomni_b200.registry.register()`` installs over the reference's ``chunk_logprobs_function`` /
``chunk_topk_distill_function``."""
import importlib.util
import sys
from pathlib import Path

import pytest
import torch

from oracle.build_ref import REF_DIR

GOLDEN = Path(__file__).resolve().parent / "golden"
_spec = importlib.util.spec_from_file_location("make_logprobs", GOLDEN / "make_logprobs.py")
ML = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(ML)
NAMES = ("chunk_logprobs_function", "chunk_topk_distill_function")


@pytest.mark.parametrize("case", [c[0] for c in ML.CASES])
def test_oracle_reproduces_reference_fixture(golden, case):
    f = golden("logprobs.pt")
    c = f["cases"][case]
    outs, dh, dw = ML.oracle_case(f["inputs"], c["dtype"], c["temperature"], c["topk"], c["clamp"])
    fp32 = c["dtype"] == torch.float32
    assert set(outs) == set(c["outputs"])
    for n, v in c["outputs"].items():
        tol = dict(atol=1e-5, rtol=1e-5) if fp32 or n != "teacher_mass" else dict(atol=1e-2, rtol=1e-2)
        torch.testing.assert_close(outs[n], v.float(), **tol)
        assert torch.all(v[1] == 0) and torch.all(v[:, -1] == 0)  # ignored sequence, padded slot
    gtol = dict(atol=1e-6, rtol=1e-4) if fp32 else dict(atol=2e-3, rtol=2e-2)
    torch.testing.assert_close(dh.float(), c["grad_hidden"].float(), **gtol)
    torch.testing.assert_close(dw.float(), c["grad_weight"].float(), **gtol)


@pytest.fixture()
def ref_ce():
    if not (REF_DIR / "veomni").is_dir():
        pytest.skip("oracle/_ref holds no reference package (build() found no reference source)")
    sys.path.insert(0, str(REF_DIR))
    try:
        from veomni.ops.config import singleton

        import veomni.ops.kernels.cross_entropy as ce

        saved_cfg = singleton.get_ops_config()
        yield ce
        singleton.set_ops_config(saved_cfg)
    finally:
        sys.path.remove(str(REF_DIR))


class _Cfg:
    def __init__(self, impl):
        self.cross_entropy_loss_implementation = impl


def test_dispatcher_routes_b200_to_ours_and_everything_else_to_the_original(ref_ce, monkeypatch):
    from veomni.ops.config import singleton

    from veomni_b200 import cross_entropy as own
    from veomni_b200 import registry

    assert registry.register() is True
    calls = []

    def recorder(who, name):
        def fn(*args, **kwargs):
            calls.append((who, name, args, kwargs))
            return who
        return fn

    for name in NAMES:
        wrapped = getattr(ref_ce, name)
        assert wrapped._vb200 and wrapped.__name__ == name
        assert wrapped._vb200_orig.__module__.startswith("veomni.ops.kernels.cross_entropy.")
        monkeypatch.setattr(own, name, recorder("ours", name))
        monkeypatch.setattr(wrapped, "_vb200_orig", recorder("orig", name))
    for impl in ("b200", "eager", "liger_kernel", "chunk_loss", None):
        singleton.set_ops_config(_Cfg(impl) if impl else None)
        want = "ours" if impl == "b200" else "orig"
        calls.clear()
        assert ref_ce.chunk_logprobs_function("h", "w", "l", chunk_size=8) == want
        assert ref_ce.chunk_topk_distill_function("h", "w", "l", "i", "t", temperature=0.5) == want
        assert [(c[0], c[1]) for c in calls] == [(want, NAMES[0]), (want, NAMES[1])]
        assert calls[0][2] == ("h", "w", "l") and calls[1][2] == ("h", "w", "l", "i", "t")
        extra = {"sp_enabled": False} if want == "ours" else {}  # no SP group in this process
        assert calls[0][3] == {"chunk_size": 8, **extra} and calls[1][3] == {"temperature": 0.5, **extra}


def test_register_twice_wraps_once(ref_ce):
    from veomni_b200 import registry

    assert registry.register() is True
    first = {n: getattr(ref_ce, n) for n in NAMES}
    assert registry.register() is True
    for n in NAMES:
        fn = getattr(ref_ce, n)
        assert fn is first[n] and fn._vb200
        assert not getattr(fn._vb200_orig, "_vb200", False)
        assert fn._vb200_orig.__module__.startswith("veomni.ops.kernels.cross_entropy")
