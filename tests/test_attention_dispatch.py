"""The Python side of the attention kernels (ops/attention_sm100.py) exercised on the CPU with a stand-in extension
that honours the bindings' contract: ``attn_fwd`` / ``attn_bwd`` are computed in PyTorch from the documented semantics
(same outputs, log-sum-exp layout and dropout mask as the kernels), ``attn_decode`` runs the REAL decode kernel source on
CPU threads (tests/emu).  Covers what would otherwise first run on the GPU box: the first-use self-tests and their
fall-back decision, the autograd plumbing of dropout probability / seed, the zero-padding of ragged sequence lengths,
the decode dispatch."""
import ctypes
import math
import os
import sys
import warnings

import pytest
import torch

from megatron_llm_b200.ops import _ext, attention_sm100
from megatron_llm_b200.ops.attention import attention_reference, dropout_keep_mask, dropout_threshold

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
import host_build  # noqa: E402


def _scores(q, k, window, scale):
    """[b, n, sq, sk] masked scaled scores with the kv heads broadcast to the query heads."""
    b, sq, nq, hn = q.shape
    sk, nkv = k.size(1), k.size(2)
    kf = k.float().repeat_interleave(nq // nkv, dim=2)
    s = torch.einsum("bqnh,bknh->bnqk", q.float(), kf) * scale
    qi = torch.arange(sq).view(sq, 1) + (sk - sq)
    ki = torch.arange(sk).view(1, sk)
    allowed = ki <= qi
    if window is not None and window >= 0:
        allowed = allowed & (ki >= qi - window)
    return s.masked_fill(~allowed, float("-inf"))


class FakeExtension:
    """What csrc/attention_bind.cpp promises, in PyTorch (``broken`` scales the output like a faulty kernel would)."""

    def __init__(self, decode_lib, broken=False):
        self.lib, self.broken, self.calls = decode_lib, broken, []

    def _forward(self, q, k, v, window, scale, p, seed):
        b, s, nq, hn = q.shape
        sc = _scores(q, k, None if window < 0 else window, scale)
        lse = torch.logsumexp(sc, dim=-1)                                   # [b, n, s]
        prob = torch.softmax(sc, dim=-1)
        if p > 0:
            prob = prob * dropout_keep_mask(seed, p, b, nq, s, s) * dropout_threshold(p)[1]
        vf = v.float().repeat_interleave(nq // v.size(2), dim=2)
        out = torch.einsum("bnqk,bknh->bqnh", prob, vf)
        return out * (1.1 if self.broken else 1.0), lse

    def attn_fwd(self, q, k, v, causal, window, scale, dropout_p=0.0, seed=0):
        assert causal and q.size(1) % 128 == 0 and q.size(1) == k.size(1), "kernel contract: causal, tiles of 128"
        self.calls.append(("fwd", tuple(q.shape), str(q.dtype), dropout_p, seed))
        out, lse = self._forward(q, k, v, window, scale, dropout_p, seed)
        return out.to(q.dtype), lse

    def attn_bwd(self, dout, q, k, v, out, lse, causal, window, scale, dropout_p=0.0, seed=0):
        self.calls.append(("bwd", tuple(q.shape), str(q.dtype), dropout_p, seed))
        with torch.enable_grad():
            qf, kf, vf = (t.detach().float().requires_grad_() for t in (q, k, v))
            o, _ = self._forward(qf, kf, vf, window, scale, dropout_p, seed)
            o.backward(dout.float())
        return qf.grad.to(q.dtype), kf.grad.to(q.dtype), vf.grad.to(q.dtype)

    def attn_decode(self, q, k, v, window, scale, splits):
        b, sq, nq, hn = q.shape
        sk, nkv = k.size(1), k.size(2)
        assert attention_sm100._decode_aligned(q, k, v)
        n_splits = max(1, min((296 + b * nkv - 1) // (b * nkv), (sk + 255) // 256)) if splits <= 0 else splits
        kps = (((sk + n_splits - 1) // n_splits) + 31) // 32 * 32
        n_splits = (sk + kps - 1) // kps
        rows = b * nkv * n_splits * sq * (nq // nkv)
        part_o, part_ml = torch.empty(rows, hn), torch.empty(rows, 2)
        out = torch.empty(b, sq, nq, hn, dtype=q.dtype)
        st = lambda t: (ctypes.c_longlong * 3)(t.stride(0), t.stride(1), t.stride(2))
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        rc = self.lib.mlb_attn_decode(0 if q.dtype == torch.bfloat16 else 1, p(q), p(k), p(v), st(q), st(k), st(v), b, sq,
                                      sk, nq, nkv, hn, int(window), ctypes.c_float(scale), n_splits, kps, p(part_o),
                                      p(part_ml), p(out), None)
        assert rc == 0
        self.calls.append(("decode", tuple(q.shape), sk))
        return out * (1.1 if self.broken else 1.0)


@pytest.fixture(scope="module")
def decode_lib(tmp_path_factory):
    return ctypes.CDLL(host_build.build(["attention_decode.cu"], str(tmp_path_factory.mktemp("emu_dispatch"))))


@pytest.fixture
def fake(monkeypatch, decode_lib):
    ext = FakeExtension(decode_lib)
    monkeypatch.setattr(_ext, "load", lambda: ext)
    monkeypatch.setattr(attention_sm100, "_feature_state", {})
    for var in ("MLB200_ATTN", "MLB200_DISABLE_KERNELS", "MLB200_ATTN_FP16", "MLB200_ATTN_DROPOUT", "MLB200_ATTN_DECODE"):
        monkeypatch.delenv(var, raising=False)
    verdicts = lambda: [k for k in os.environ if k.startswith("MLB200_ATTN_SELFTEST_")]
    for var in verdicts():
        monkeypatch.delenv(var, raising=False)
    yield ext
    for var in verdicts():      # feature_ok publishes its verdicts to child processes through the environment
        os.environ.pop(var, None)


def test_selftests_admit_working_kernels_and_reject_broken_ones(fake, monkeypatch):
    dev = torch.device("cpu")
    for feature in ("fp16", "dropout", "decode"):
        assert attention_sm100.feature_ok(feature, 64, torch.bfloat16, dev), feature
    kinds = {c[0] for c in fake.calls}
    assert kinds == {"fwd", "bwd", "decode"}
    assert any(c[0] == "fwd" and c[2] == "torch.float16" for c in fake.calls)          # the fp16 self-test ran in fp16
    assert any(c[0] == "fwd" and c[3] > 0 and c[4] != 0 for c in fake.calls)           # dropout: with p and a seed
    n = len(fake.calls)
    assert attention_sm100.feature_ok("decode", 64, torch.bfloat16, dev) and len(fake.calls) == n   # decided once
    # a kernel that returns wrong numbers is switched off, loudly
    fake.broken = True
    monkeypatch.setattr(attention_sm100, "_feature_state", {})
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        for feature in ("fp16", "dropout", "decode"):
            assert not attention_sm100.feature_ok(feature, 128, torch.bfloat16, dev), feature
    assert len(w) == 3 and all("FAILED its self-test" in str(x.message) for x in w)
    # the verdicts are published to processes started from here (ranks, tools): they do not test again
    assert os.environ["MLB200_ATTN_SELFTEST_FP16_HD64"] == "1" and os.environ["MLB200_ATTN_SELFTEST_DECODE_HD128"] == "0"
    monkeypatch.setattr(attention_sm100, "_feature_state", {})
    n = len(fake.calls)
    assert not attention_sm100.feature_ok("decode", 128, torch.bfloat16, dev) and len(fake.calls) == n
    os.environ.pop("MLB200_ATTN_SELFTEST_DECODE_HD128")    # not monkeypatch.delenv: its undo would put the "0" back after the test
    # ... and so is one that raises; the environment switch overrides both ways
    monkeypatch.setattr(attention_sm100, "_feature_state", {})
    monkeypatch.setattr(fake, "attn_decode", lambda *a: (_ for _ in ()).throw(RuntimeError("launch failed")))
    with warnings.catch_warnings(record=True):
        warnings.simplefilter("always")
        assert not attention_sm100.feature_ok("decode", 128, torch.bfloat16, dev)
    monkeypatch.setattr(attention_sm100, "_feature_state", {})
    monkeypatch.setenv("MLB200_ATTN_DECODE", "1")
    assert attention_sm100.feature_ok("decode", 128, torch.bfloat16, dev)
    monkeypatch.setattr(attention_sm100, "_feature_state", {})
    monkeypatch.setenv("MLB200_ATTN_DECODE", "0")
    assert not attention_sm100.feature_ok("decode", 128, torch.bfloat16, dev)


def test_selftest_on_a_cuda_device_runs_in_a_throwaway_process(fake, monkeypatch):
    """On a GPU the first launch of a never-run kernel variant happens in a child process with a time limit: a sticky
    CUDA error or a dead-locked kernel costs that child, not the job.  Here the child sees no GPU (on a GPU machine too)
    and cannot pass -- what is checked is that a crashing child and one that overruns its limit both come back as a
    clean, loud 'no'."""
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")          # read by the child's CUDA start-up; this process uses no device
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    dev = torch.device("cuda", 0)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert not attention_sm100.feature_ok("fp16", 128, torch.float16, dev)
    assert len(w) == 1 and "self-test process exited with code" in str(w[0].message)
    assert not fake.calls                                       # nothing ran in this process
    assert os.environ["MLB200_ATTN_SELFTEST_FP16_HD128"] == "0"
    monkeypatch.setenv("MLB200_ATTN_SELFTEST_TIMEOUT", "0.05")
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert not attention_sm100.feature_ok("dropout", 64, torch.bfloat16, dev)
    assert len(w) == 1 and "did not finish within" in str(w[0].message)
    # a passing child: its last line carries the error
    import subprocess
    done = subprocess.CompletedProcess([], 0, stdout="noise\nMLB200_SELFTEST_ERR 2.5e-03\n", stderr="")
    monkeypatch.setattr(subprocess, "run", lambda *a, **k: done)
    assert attention_sm100.feature_ok("decode", 64, torch.bfloat16, dev)
    assert os.environ["MLB200_ATTN_SELFTEST_DECODE_HD64"] == "1"


@pytest.mark.parametrize("s,window,p", [(256, None, 0.0), (77, None, 0.1), (200, 64, 0.25)])
def test_attention_autograd_plumbing_padding_and_dropout(fake, monkeypatch, s, window, p):
    """ops.attention_sm100.attention: probability and seed reach forward AND backward, ragged lengths are padded to the
    tile and sliced back, gradients equal the fp32 oracle with the same mask."""
    seed = 0x0123_4567_89AB_CDEF
    monkeypatch.setattr(attention_sm100, "_draw_seed", lambda dp, n: seed if dp > 0 else 0)
    torch.manual_seed(s)
    b, nq, nkv, hn = 2, 4, 2, 64
    q, k, v = (torch.randn(b, s, n, hn).bfloat16().requires_grad_() for n in (nq, nkv, nkv))
    do = torch.randn(b, s, nq, hn).bfloat16()
    assert attention_sm100.supported(q, k, v, True, window, p)       # (p > 0: runs the dropout self-test first)
    fake.calls.clear()
    out = attention_sm100.attention(q, k, v, True, window, None, p)
    assert out.shape == (b, s, nq, hn)
    out.backward(do)
    sp = (s + 127) // 128 * 128
    assert [c[:2] for c in fake.calls if c[0] in ("fwd", "bwd")] == [("fwd", (b, sp, nq, hn)), ("bwd", (b, sp, nq, hn))]
    assert all(c[3] == p and c[4] == (seed if p > 0 else 0) for c in fake.calls if c[0] in ("fwd", "bwd"))
    qf, kf, vf = (t.detach().float().requires_grad_() for t in (q, k, v))
    keep = dropout_keep_mask(seed, p, b, nq, s, s) if p > 0 else None        # the mask of the un-padded positions
    ref = attention_reference(qf, kf, vf, True, window, None, p, keep)
    ref.backward(do.float())
    rel = lambda a, r: ((a.float() - r).norm() / r.norm()).item()
    assert rel(out, ref) < 1e-2                                              # (bf16 rounding of the outputs only)
    for mine, theirs in ((q, qf), (k, kf), (v, vf)):
        assert rel(mine.grad, theirs.grad) < 1e-2


def test_decode_dispatch_runs_the_split_kv_kernel(fake):
    """decode_supported / decode_attention on KV-cache views (CPU tensors, the real kernel source underneath)."""
    torch.manual_seed(0)
    b, nq, nkv, hn, s_max = 2, 8, 2, 64, 150
    kmem = torch.randn(s_max, b, nkv, hn).bfloat16()
    vmem = torch.randn(s_max, b, nkv, hn).bfloat16()
    with torch.no_grad():
        for t in (97, 98, 149):
            q = torch.randn(b, 1, nq, hn).bfloat16()
            k, v = kmem[:t + 1].transpose(0, 1), vmem[:t + 1].transpose(0, 1)
            assert attention_sm100.decode_supported(q, k, v, True, 0.0)
            out = attention_sm100.decode_attention(q, k, v, None, None)
            ref = attention_reference(q.float(), k.float(), v.float(), True)
            assert (out.float() - ref).abs().max().item() < 2e-2
    # not the decode shape / needs a gradient / misaligned rows -> not taken
    q = torch.randn(b, 1, nq, hn).bfloat16()
    k, v = kmem[:50].transpose(0, 1), vmem[:50].transpose(0, 1)
    assert not attention_sm100.decode_supported(q, k, v, False, 0.0)
    assert not attention_sm100.decode_supported(q, k, v, True, 0.1)
    assert not attention_sm100.decode_supported(torch.randn(b, 40, nq, hn).bfloat16(), k, v, True, 0.0)   # 160 rows / group
    qg = q.clone().requires_grad_()
    with torch.enable_grad():
        assert not attention_sm100.decode_supported(qg, k, v, True, 0.0)
    assert not attention_sm100.decode_supported(q, kmem[:50, :, :, 4:36].transpose(0, 1), v, True, 0.0)
