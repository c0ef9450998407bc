"""Kernel-level parity (GPU): each hand-written sm_100a kernel vs a plain fp32 torch / numpy
restatement of the same op, called through the C ABI (reverb_b200/_lib.py)."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _p(t):
    return C.c_void_p(t.data_ptr())


@pytest.fixture(scope="module")
def lib():
    from reverb_b200 import _lib
    return _lib.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(lib, rc):
    from reverb_b200 import _lib
    assert rc == 0, _lib.last_error()


def test_fbank_matches_oracle_and_torchaudio_golden(lib):
    from oracle import fbank_np
    from reverb_b200 import synth
    gold = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "fbank.npz")))
    for key, ref in gold.items():
        n = int(key.split("_")[0][1:])
        seed = int(key.split("seed")[1])
        pcm = synth.synth_audio(n / 16000.0 + 1e-9, seed=seed)[:n]
        for dtype in (torch.float32, torch.int16):
            w = torch.from_numpy(pcm.astype(np.float32 if dtype == torch.float32 else np.int16)).cuda()
            m = lib.rvb_fbank_num_frames(n)
            assert m == ref.shape[0]
            out = torch.empty(m, 80, device="cuda")
            fn = lib.rvb_fbank_f32 if dtype == torch.float32 else lib.rvb_fbank_i16
            _check(lib, fn(_p(w), n, _p(out), m, _stream()))
            got = out.cpu().numpy()
            # tolerance: fp32 FFT/mel vs torchaudio's fp32 pocketfft; log-mel values are O(10)
            np.testing.assert_allclose(got, ref, rtol=0, atol=2e-3)
            np.testing.assert_allclose(got, fbank_np.fbank(pcm.astype(np.float32)), rtol=0, atol=2e-3)


@pytest.mark.parametrize("d", [128, 256, 1024, 640])
def test_layernorm(lib, d):
    torch.manual_seed(d)
    M = 777
    x = torch.randn(M, d, device="cuda") * 3 + 1
    g = torch.randn(d, device="cuda")
    b = torch.randn(d, device="cuda")
    out_f = torch.empty(M, d, device="cuda")
    out_b = torch.empty(M, d, device="cuda", dtype=torch.bfloat16)
    _check(lib, lib.rvb_layernorm(_p(x), _p(g), _p(b), 1e-5, M, d, _p(out_b), _p(out_f), _stream()))
    ref = torch.nn.functional.layer_norm(x, (d,), g, b, 1e-5)
    torch.testing.assert_close(out_f, ref, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(out_b.float(), ref.bfloat16().float(), rtol=2e-2, atol=2e-2)


GEMM_SHAPES = [(128, 128, 64), (300, 256, 128), (257, 101, 128), (513, 1001, 192), (1000, 1024, 4096), (64, 384, 2432), (4096, 4096, 1024)]


@pytest.mark.parametrize("impl", [1, 0, 2], ids=["simt", "tcgen05", "tcgen05_2cta"])
@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_gemm_bias_act_modes(lib, impl, M, N, K):
    torch.manual_seed(M + N + K)
    lib.rvb_set_gemm_impl(impl)
    try:
        A = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
        W = (torch.randn(N, K, device="cuda") / math.sqrt(K)).bfloat16()
        bias = torch.randn(N, device="cuda")
        ref = A.float() @ W.float().t() + bias
        ldo = (N + 3) & ~3
        # fp32 out
        out = torch.zeros(M, ldo, device="cuda")
        _check(lib, lib.rvb_gemm_bf16(_p(A), _p(W), _p(bias), M, N, K, 0, 1, 1.0, _p(out), ldo, _stream()))
        torch.testing.assert_close(out[:, :N], ref, rtol=1e-3, atol=1e-3)
        assert bool((out[:, N:] == 0).all())              # row padding is never written
        # bf16 out + SiLU
        out_b = torch.zeros(M, ldo, device="cuda", dtype=torch.bfloat16)
        _check(lib, lib.rvb_gemm_bf16(_p(A), _p(W), _p(bias), M, N, K, 2, 0, 1.0, _p(out_b), ldo, _stream()))
        torch.testing.assert_close(out_b[:, :N].float(), torch.nn.functional.silu(ref), rtol=2e-2, atol=2e-2)
        # residual accumulate with alpha, ReLU
        res = torch.randn(M, ldo, device="cuda")
        res0 = res.clone()
        _check(lib, lib.rvb_gemm_bf16(_p(A), _p(W), _p(bias), M, N, K, 1, 2, 0.5, _p(res), ldo, _stream()))
        torch.testing.assert_close(res[:, :N], res0[:, :N] + 0.5 * torch.relu(ref), rtol=1e-3, atol=1e-3)
        assert torch.equal(res[:, N:], res0[:, N:])
        torch.cuda.synchronize()
    finally:
        lib.rvb_set_gemm_impl(-1)       # back to the default (env RVB_GEMM or the 2-CTA kernel)


@pytest.mark.parametrize("impl", [1, 0, 2], ids=["simt", "tcgen05", "tcgen05_2cta"])
@pytest.mark.parametrize("M,C,K", [(300, 64, 128), (1000, 256, 256), (4133, 1024, 1024)])
def test_gemm_glu_epilogue(lib, impl, M, C, K):
    """ACT_GLU: pointwise_conv1 + GLU in one GEMM (weight rows interleaved in groups of 32, include/rvb_b200.h)."""
    torch.manual_seed(M + C)
    lib.rvb_set_gemm_impl(impl)
    try:
        A = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
        W = (torch.randn(2 * C, K, device="cuda") / math.sqrt(K)).bfloat16()
        bias = torch.randn(2 * C, device="cuda")
        ref = torch.nn.functional.glu(A.float() @ W.float().t() + bias, dim=1)
        c = torch.arange(C, device="cuda")
        ra = 64 * (c // 32) + (c % 32)
        Wp = torch.empty_like(W)
        bp = torch.empty_like(bias)
        Wp[ra], Wp[ra + 32] = W[:C], W[C:]
        bp[ra], bp[ra + 32] = bias[:C], bias[C:]
        out = torch.zeros(M, C, device="cuda", dtype=torch.bfloat16)
        _check(lib, lib.rvb_gemm_bf16(_p(A), _p(Wp), _p(bp), M, 2 * C, K, 3, 0, 1.0, _p(out), C, _stream()))
        torch.testing.assert_close(out.float(), ref, rtol=2e-2, atol=2e-2)
    finally:
        lib.rvb_set_gemm_impl(-1)


@pytest.mark.parametrize("dk,H", [(64, 2), (32, 4), (128, 1)])
@pytest.mark.parametrize("pos", [True, False])
def test_attention(lib, dk, H, pos):
    torch.manual_seed(dk + H)
    B, T = 3, 150
    d = H * dk
    qkv = (torch.randn(B, T, 3 * d, device="cuda") * 0.7).bfloat16()
    p = (torch.randn(T, d, device="cuda") * 0.7).bfloat16()
    u = torch.randn(H, dk, device="cuda") * 0.3
    v = torch.randn(H, dk, device="cuda") * 0.3
    klens = torch.tensor([150, 97, 1], dtype=torch.int32, device="cuda")
    out = torch.zeros(B, T, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention(_p(qkv), C.c_void_p(qkv.data_ptr() + 2 * d), C.c_void_p(qkv.data_ptr() + 4 * d),
                                  _p(p) if pos else None, _p(u) if pos else None, _p(v) if pos else None, _p(out),
                                  3 * d, 3 * d, 3 * d, d, d, B, T, T, H, dk, 1, _p(klens), None, 0, scale, _stream()))
    q = qkv[..., :d].float().view(B, T, H, dk)
    k = qkv[..., d:2 * d].float().view(B, T, H, dk).transpose(1, 2)
    vv = qkv[..., 2 * d:].float().view(B, T, H, dk).transpose(1, 2)
    if pos:
        pp = p.float().view(1, T, H, dk).transpose(1, 2)
        qu = (q + u).bfloat16().float().transpose(1, 2)
        qv = (q + v).bfloat16().float().transpose(1, 2)
        s = (qu @ k.transpose(-1, -2) + qv @ pp.transpose(-1, -2)) * scale
    else:
        s = (q.transpose(1, 2) @ k.transpose(-1, -2)) * scale
    mask = torch.arange(T, device="cuda")[None, :] >= klens[:, None]
    s = s.masked_fill(mask[:, None, None, :], -float("inf"))
    a = torch.softmax(s, -1).masked_fill(mask[:, None, None, :], 0.0)
    ref = (a @ vv).transpose(1, 2).reshape(B, T, d)
    torch.testing.assert_close(out.float(), ref, rtol=3e-2, atol=3e-2)


def test_attention_causal_cross(lib):
    """decoder forms: causal self-attention with per-sequence lengths, and cross attention with q_per_kv."""
    torch.manual_seed(5)
    H, dk = 2, 64
    d = H * dk
    S, L, N, Tk = 6, 23, 3, 90
    qkv = (torch.randn(S, L, 3 * d, device="cuda") * 0.7).bfloat16()
    qlens = torch.tensor([23, 5, 1, 17, 23, 9], dtype=torch.int32, device="cuda")
    out = torch.zeros(S, L, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention(_p(qkv), C.c_void_p(qkv.data_ptr() + 2 * d), C.c_void_p(qkv.data_ptr() + 4 * d),
                                  None, None, None, _p(out), 3 * d, 3 * d, 3 * d, 0, d, S, L, L, H, dk, 1, None,
                                  _p(qlens), 1, scale, _stream()))
    q = qkv[..., :d].float().view(S, L, H, dk).transpose(1, 2)
    k = qkv[..., d:2 * d].float().view(S, L, H, dk).transpose(1, 2)
    v = qkv[..., 2 * d:].float().view(S, L, H, dk).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * scale
    j = torch.arange(L, device="cuda")
    ok = (j[None, None, :] <= j[None, :, None]) & (j[None, None, :] < qlens[:, None, None])
    s = s.masked_fill(~ok[:, None], -float("inf"))
    a = torch.softmax(s, -1).masked_fill(~ok[:, None], 0.0).nan_to_num(0.0)
    ref = (a @ v).transpose(1, 2).reshape(S, L, d)
    valid = (j[None, :] < qlens[:, None])
    torch.testing.assert_close(out.float()[valid], ref[valid], rtol=3e-2, atol=3e-2)
    # cross attention: S sequences share Tk memory rows of utterance s // N
    qx = (torch.randn(S, L, d, device="cuda") * 0.7).bfloat16()
    kv = (torch.randn(S // N, Tk, 2 * d, device="cuda") * 0.7).bfloat16()
    klens = torch.tensor([90, 41], dtype=torch.int32, device="cuda")
    _check(lib, lib.rvb_attention(_p(qx), _p(kv), C.c_void_p(kv.data_ptr() + 2 * d), None, None, None, _p(out),
                                  d, 2 * d, 2 * d, 0, d, S, L, Tk, H, dk, N, _p(klens), None, 0, scale, _stream()))
    q = qx.float().view(S, L, H, dk).transpose(1, 2)
    k = kv[..., :d].float().view(S // N, Tk, H, dk).transpose(1, 2).repeat_interleave(N, 0)
    v = kv[..., d:].float().view(S // N, Tk, H, dk).transpose(1, 2).repeat_interleave(N, 0)
    s = (q @ k.transpose(-1, -2)) * scale
    mask = (torch.arange(Tk, device="cuda")[None, :] >= klens.repeat_interleave(N)[:, None])
    s = s.masked_fill(mask[:, None, None, :], -float("inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(S, L, d)
    torch.testing.assert_close(out.float(), ref, rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("B,T,H", [(3, 150, 2), (2, 748, 4), (1, 128, 1), (2, 129, 2)])
def test_attention_tcgen05_relpos(lib, B, T, H):
    """tcgen05 attention with the folded rel-pos term (K'' = k + p, key bias c) vs the reference formula in fp32."""
    torch.manual_seed(B * 1000 + T)
    dk = 64
    d = H * dk
    qkv = (torch.randn(B, T, 3 * d, device="cuda") * 0.7).bfloat16()
    pos = (torch.randn(T, d, device="cuda") * 0.7).bfloat16()
    u = torch.randn(H, dk, device="cuda") * 0.3
    v = torch.randn(H, dk, device="cuda") * 0.3
    klens = torch.tensor([T, max(1, T * 2 // 3), 1][:B], dtype=torch.int32, device="cuda")
    kpp = torch.empty(B, T, d, device="cuda", dtype=torch.bfloat16)
    cb = torch.empty(B, H, T, device="cuda")
    _check(lib, lib.rvb_relpos_prep(C.c_void_p(qkv.data_ptr() + 2 * d), 3 * d, _p(pos), d, _p(u), _p(v), _p(kpp), _p(cb),
                                    B, T, H, dk, _stream()))
    out = torch.zeros(B, T, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention_tc(_p(qkv), _p(kpp), C.c_void_p(qkv.data_ptr() + 4 * d), _p(out), 3 * d, d, 3 * d, d,
                                     B, T, T, H, dk, _p(cb), _p(klens), 0, scale, _stream()))
    torch.cuda.synchronize()
    q = qkv[..., :d].float().view(B, T, H, dk)
    k = qkv[..., d:2 * d].float().view(B, T, H, dk).transpose(1, 2)
    vv = qkv[..., 2 * d:].float().view(B, T, H, dk).transpose(1, 2)
    pp = pos.float().view(1, T, H, dk).transpose(1, 2)
    # the pre-kernel itself: exact bf16 rounding of k + p, fp32 bias
    torch.testing.assert_close(kpp.float().view(B, T, H, dk).transpose(1, 2), (k + pp).bfloat16().float(), rtol=0, atol=0)
    want_cb = (u[None, :, None, :] * k).sum(-1) + (v[None, :, None, :] * pp).sum(-1)
    torch.testing.assert_close(cb, want_cb, rtol=1e-4, atol=1e-4)
    s = ((q + u).transpose(1, 2) @ k.transpose(-1, -2) + (q + v).transpose(1, 2) @ pp.transpose(-1, -2)) * scale
    mask = torch.arange(T, device="cuda")[None, :] >= klens[:, None]
    s = s.masked_fill(mask[:, None, None, :], -float("inf"))
    a = torch.softmax(s, -1).masked_fill(mask[:, None, None, :], 0.0)
    ref = (a @ vv).transpose(1, 2).reshape(B, T, d)
    torch.testing.assert_close(out.float(), ref, rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("persist", ["0", "1"])
def test_attention_tcgen05_persistent_many_items_mixed_lengths(lib, persist):
    """More (query tile, head, group) items than CTAs, so every CTA of the persistent kernel walks several items, with key
    lengths that give 0 (empty item -> zero rows), 1, 2 and 5 key tiles in mixed order: the rings (K'', V, S / P~, Q) and
    barrier phases must stay consistent across item boundaries — also when an item is a single tile long."""
    torch.manual_seed(77)
    H, dk = 4, 64
    d = H * dk
    G, T = 60, 300                                     # 3 query tiles x 4 heads x 60 groups = 720 items > 2 x 148 CTAs
    qkv = (torch.randn(G, T, 3 * d, device="cuda") * 0.7).bfloat16()
    bias = torch.randn(G, H, T, device="cuda") * 0.5
    lens = [300, 1, 64, 65, 0, 128, 17, 299, 63, 200]
    klens = torch.tensor([lens[i % len(lens)] for i in range(G)], dtype=torch.int32, device="cuda")
    out = torch.full((G, T, d), 7.0, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    import os
    os.environ["RVB_ATTN_PERSIST"] = persist            # "1": the persistent kernel (off by default: measured slower)
    try:
        _check(lib, lib.rvb_attention_tc(_p(qkv), C.c_void_p(qkv.data_ptr() + 2 * d), C.c_void_p(qkv.data_ptr() + 4 * d),
                                         _p(out), 3 * d, 3 * d, 3 * d, d, G, T, T, H, dk, _p(bias), _p(klens), 0, scale,
                                         _stream()))
        torch.cuda.synchronize()
        out2 = torch.empty_like(out)
        _check(lib, lib.rvb_attention_tc(_p(qkv), C.c_void_p(qkv.data_ptr() + 2 * d), C.c_void_p(qkv.data_ptr() + 4 * d),
                                         _p(out2), 3 * d, 3 * d, 3 * d, d, G, T, T, H, dk, _p(bias), _p(klens), 0, scale,
                                         _stream()))
        torch.cuda.synchronize()
    finally:
        del os.environ["RVB_ATTN_PERSIST"]
    q = qkv[..., :d].float().view(G, T, H, dk).transpose(1, 2)
    k = qkv[..., d:2 * d].float().view(G, T, H, dk).transpose(1, 2)
    v = qkv[..., 2 * d:].float().view(G, T, H, dk).transpose(1, 2)
    s = (q @ k.transpose(-1, -2) + bias[:, :, None, :]) * scale
    mask = torch.arange(T, device="cuda")[None, :] >= klens[:, None]
    s = s.masked_fill(mask[:, None, None, :], -float("inf"))
    a = torch.nan_to_num(torch.softmax(s, -1), nan=0.0).masked_fill(mask[:, None, None, :], 0.0)
    ref = (a @ v).transpose(1, 2).reshape(G, T, d)
    torch.testing.assert_close(out.float(), ref, rtol=3e-2, atol=3e-2)
    assert float(out[4].float().abs().max()) == 0.0      # klen 0: rows written as zeros
    # the same launch is deterministic run to run (no dependence on which CTA picked which items)
    assert torch.equal(out, out2)


def test_attention_tcgen05_grouped_cross(lib):
    """decoder source-attention form: groups of N*L query rows share one utterance's keys; no bias."""
    torch.manual_seed(11)
    H, dk = 2, 64
    d = H * dk
    G, Tq, Tk = 3, 230, 300
    qx = (torch.randn(G, Tq, d, device="cuda") * 0.7).bfloat16()
    kv = (torch.randn(G, Tk, 2 * d, device="cuda") * 0.7).bfloat16()
    klens = torch.tensor([300, 41, 128], dtype=torch.int32, device="cuda")
    out = torch.zeros(G, Tq, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention_tc(_p(qx), _p(kv), C.c_void_p(kv.data_ptr() + 2 * d), _p(out), d, 2 * d, 2 * d, d,
                                     G, Tq, Tk, H, dk, None, _p(klens), 0, scale, _stream()))
    q = qx.float().view(G, Tq, H, dk).transpose(1, 2)
    k = kv[..., :d].float().view(G, Tk, H, dk).transpose(1, 2)
    v = kv[..., d:].float().view(G, Tk, H, dk).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * scale
    mask = torch.arange(Tk, device="cuda")[None, :] >= klens[:, None]
    s = s.masked_fill(mask[:, None, None, :], -float("inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(G, Tq, d)
    torch.testing.assert_close(out.float(), ref, rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("ramp", [20.0, -20.0])
def test_attention_tcgen05_running_max_rescale(lib, ramp):
    """Scores whose magnitude grows (or shrinks) along the key axis: with ramp > 0 later key tiles exceed the running
    maximum by far more than 2^8, so the lazy rescale of the TMEM accumulator / row sum runs many times per row."""
    torch.manual_seed(5)
    H, dk = 2, 64
    d = H * dk
    G, Tq, Tk = 2, 200, 700
    qx = (torch.randn(G, Tq, d, device="cuda") * 0.7).bfloat16()
    kvf = torch.randn(G, Tk, 2 * d, device="cuda") * 0.7
    t = torch.arange(Tk, device="cuda", dtype=torch.float32) / Tk
    gain = 1.0 + abs(ramp) * (t if ramp > 0 else (1.0 - t))
    kvf[..., :d] *= gain[None, :, None]
    kv = kvf.bfloat16()
    klens = torch.tensor([700, 333], dtype=torch.int32, device="cuda")
    out = torch.zeros(G, Tq, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention_tc(_p(qx), _p(kv), C.c_void_p(kv.data_ptr() + 2 * d), _p(out), d, 2 * d, 2 * d, d,
                                     G, Tq, Tk, H, dk, None, _p(klens), 0, scale, _stream()))
    q = qx.float().view(G, Tq, H, dk).transpose(1, 2)
    k = kv[..., :d].float().view(G, Tk, H, dk).transpose(1, 2)
    v = kv[..., d:].float().view(G, Tk, H, dk).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * scale
    mask = torch.arange(Tk, device="cuda")[None, :] >= klens[:, None]
    s = s.masked_fill(mask[:, None, None, :], -float("inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(G, Tq, d)
    torch.testing.assert_close(out.float(), ref, rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("L", [164, 64, 300])
def test_attention_tcgen05_causal_self(lib, L):
    """decoder self-attention form: one group per hypothesis, causal mask + key-length mask (tgt_mask of
    decoder.py:139-146 = pad mask & subsequent_mask); rows at positions >= the hypothesis length are don't-care."""
    torch.manual_seed(L)
    H, dk = 2, 64
    d = H * dk
    S = 5
    qkv = (torch.randn(S, L, 3 * d, device="cuda") * 0.7).bfloat16()
    lens = torch.tensor([L, max(1, L * 2 // 3), 1, min(L, 130), min(L, 64)], dtype=torch.int32, device="cuda")
    out = torch.zeros(S, L, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention_tc(_p(qkv), C.c_void_p(qkv.data_ptr() + 2 * d), C.c_void_p(qkv.data_ptr() + 4 * d), _p(out),
                                     3 * d, 3 * d, 3 * d, d, S, L, L, H, dk, None, _p(lens), 1, scale, _stream()))
    q = qkv[..., :d].float().view(S, L, H, dk).transpose(1, 2)
    k = qkv[..., d:2 * d].float().view(S, L, H, dk).transpose(1, 2)
    v = qkv[..., 2 * d:].float().view(S, L, H, dk).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * scale
    pos = torch.arange(L, device="cuda")
    mask = (pos[None, :] > pos[:, None])[None] | (pos[None, None, :] >= lens[:, None, None])
    s = s.masked_fill(mask[:, None], -float("inf"))
    ref = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(S, L, d)
    for g in range(S):
        n = int(lens[g])
        torch.testing.assert_close(out[g, :n].float(), ref[g, :n], rtol=3e-2, atol=3e-2)


def test_resample_matches_torchaudio_golden(lib):
    """GPU resampler (csrc/resample.cu + the host filter table) vs torchaudio.transforms.Resample outputs
    (tests/golden/resample.npz): fp32 accumulation order differs from conv1d -> 2e-5 of the int16 full scale."""
    import reverb_b200
    from reverb_b200 import synth
    from reverb_b200.engine import Engine
    gold = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "resample.npz")))
    eng = Engine.__new__(Engine)             # the resampler needs no model: only the library handle and a device
    eng.lib, eng.device = lib, torch.device("cuda", 0)
    eng._stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for key, ref in gold.items():
        rate, n, seed = int(key.split("_")[0][1:]), int(key.split("_")[1][1:]), int(key.split("seed")[1])
        pcm = synth.synth_audio(n / 16000.0 + 1e-9, seed=seed)[:n]
        for dtype in (np.int16, np.float32):
            got = eng.resample(torch.from_numpy(pcm.astype(dtype)).cuda(), rate, 16000).cpu().numpy()
            assert got.shape == ref.shape
            np.testing.assert_allclose(got, ref, rtol=0, atol=32768 * 2e-5)


@pytest.mark.parametrize("chunk,left", [(16, -1), (8, 2), (50, 0), (1, 3), (200, 1)])
def test_attention_tcgen05_chunk_mask(lib, chunk, left):
    """bounded attention context (subsequent_chunk_mask, utils/mask.py:88-123) & key-length mask, with the rel-pos
    key bias: only the visible key tiles are visited, boundary tiles are masked per element."""
    torch.manual_seed(chunk * 7 + left)
    B, T, H, dk = 3, 300, 2, 64
    d = H * dk
    qkv = (torch.randn(B, T, 3 * d, device="cuda") * 0.7).bfloat16()
    cb = torch.randn(B, H, T, device="cuda") * 0.5
    klens = torch.tensor([T, 211, 37], dtype=torch.int32, device="cuda")
    out = torch.zeros(B, T, d, device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(dk)
    _check(lib, lib.rvb_attention_tc_chunked(_p(qkv), C.c_void_p(qkv.data_ptr() + 2 * d), C.c_void_p(qkv.data_ptr() + 4 * d),
                                             _p(out), 3 * d, 3 * d, 3 * d, d, B, T, T, H, dk, _p(cb), _p(klens), chunk,
                                             left, scale, _stream()))
    q = qkv[..., :d].float().view(B, T, H, dk).transpose(1, 2)
    k = qkv[..., d:2 * d].float().view(B, T, H, dk).transpose(1, 2)
    v = qkv[..., 2 * d:].float().view(B, T, H, dk).transpose(1, 2)
    s = (q @ k.transpose(-1, -2) + cb[:, :, None, :]) * scale
    i = torch.arange(T, device="cuda")
    lo = torch.zeros_like(i) if left < 0 else torch.clamp((i // chunk - left) * chunk, min=0)
    hi = torch.clamp((i // chunk + 1) * chunk, max=T)
    vis = (i[None, :] >= lo[:, None]) & (i[None, :] < hi[:, None])
    mask = ~vis[None] | (i[None, None, :] >= klens[:, None, None])
    s = s.masked_fill(mask[:, None], -float("inf"))
    ref = (torch.softmax(s, -1).nan_to_num(0.0) @ v).transpose(1, 2).reshape(B, T, d)
    for g in range(B):
        n = int(klens[g])
        torch.testing.assert_close(out[g, :n].float(), ref[g, :n], rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("impl", [0, 2], ids=["tcgen05", "tcgen05_2cta"])
@pytest.mark.parametrize("M,N,K", [(300, 1001, 128), (4133, 10001, 1024), (129, 257, 4096)])
def test_gemm_fused_logsoftmax_gather(lib, impl, M, N, K):
    """OUT_LSE epilogue + merge kernel: log_softmax(A W^T + b)[m, gather[m]] without writing the logits."""
    torch.manual_seed(M + N)
    lib.rvb_set_gemm_impl(impl)
    try:
        A = (torch.randn(M, K, device="cuda") * 0.5).bfloat16()
        W = (torch.randn(N, K, device="cuda") * (3.0 / math.sqrt(K))).bfloat16()
        bias = torch.randn(N, device="cuda")
        gather = torch.randint(0, N, (M,), device="cuda", dtype=torch.int32)
        gather[::7] = -1
        gather[1] = N - 1
        gather[2] = 0
        ws = torch.empty(int(lib.rvb_gemm_logsoftmax_gather_ws_bytes(M, N)), device="cuda", dtype=torch.uint8)
        out = torch.full((M,), 123.0, device="cuda")
        _check(lib, lib.rvb_gemm_logsoftmax_gather(_p(A), _p(W), _p(bias), M, N, K, _p(gather), _p(ws), _p(out), _stream()))
        logp = torch.log_softmax(A.float() @ W.float().t() + bias, dim=-1)
        g = gather.long().clamp(min=0)
        want = torch.where(gather >= 0, logp.gather(1, g[:, None])[:, 0], torch.zeros(M, device="cuda"))
        torch.testing.assert_close(out, want, rtol=1e-3, atol=2e-3)
    finally:
        lib.rvb_set_gemm_impl(-1)


# ------------------------------------------------------------------------------------------------------------------
# fp32-accurate "bf16x3" mode (rvb_model_config.precision = 1)
def _pair(lib, x):
    rows, width = x.shape
    out = torch.empty(rows, 2 * width, device="cuda", dtype=torch.bfloat16)
    _check(lib, lib.rvb_f32_to_bf16_pair(_p(x.contiguous()), _p(out), rows, width, _stream()))
    hi, lo = out[:, :width].float(), out[:, width:].float()
    assert torch.equal(hi, x.bfloat16().float()) and torch.equal(lo, (x - hi).bfloat16().float())
    return out


@pytest.mark.parametrize("impl", [0, 2], ids=["tcgen05", "tcgen05_2cta"])
@pytest.mark.parametrize("M,N,K", [(300, 256, 128), (1000, 1024, 4096), (4096, 4096, 1024), (513, 10001, 1024)])
def test_gemm_bf16x3_is_fp32_accurate(lib, impl, M, N, K):
    """Three tcgen05 passes over (hi, lo) operand pairs: |C - fp64 reference| must be ~2^-16 relative to the row scale —
    two orders of magnitude below the single-pass bf16 GEMM, at the level of an fp32 matmul."""
    torch.manual_seed(M + N + K)
    lib.rvb_set_gemm_impl(impl)
    try:
        A = torch.randn(M, K, device="cuda") * 0.5
        W = torch.randn(N, K, device="cuda") / math.sqrt(K)
        bias = torch.randn(N, device="cuda")
        ref = (A.double() @ W.double().t() + bias.double())
        Ap, Wp = _pair(lib, A), _pair(lib, W)
        ldo = (N + 3) & ~3
        out = torch.zeros(M, ldo, device="cuda")
        _check(lib, lib.rvb_gemm_bf16x3(_p(Ap), _p(Wp), _p(bias), M, N, K, 0, 1, 1.0, _p(out), ldo, _stream()))
        err3 = float((out[:, :N].double() - ref).abs().max())
        out1 = torch.zeros(M, ldo, device="cuda")
        Ab, Wb = A.bfloat16(), W.bfloat16()                       # keep the operands alive across the launch
        _check(lib, lib.rvb_gemm_bf16(_p(Ab), _p(Wb), _p(bias), M, N, K, 0, 1, 1.0, _p(out1), ldo, _stream()))
        err1 = float((out1[:, :N].double() - ref).abs().max())
        err32 = float(((A @ W.t() + bias).double() - ref).abs().max())      # torch's own fp32 matmul (may use tf32-free path)
        print(f"[x3 {M}x{N}x{K}] max abs err: bf16x3 {err3:.2e}, bf16 {err1:.2e}, torch fp32 {err32:.2e}")
        assert err3 < 2e-5 * math.sqrt(K / 128) and err3 < err1 / 50 and err3 < 30 * err32 + 1e-5
        if N % 128 == 0:
            # bf16 pair output + SiLU: hi + lo reproduces silu(ref) to ~2^-16
            outp = torch.zeros(M, 2 * N, device="cuda", dtype=torch.bfloat16)
            _check(lib, lib.rvb_gemm_bf16x3(_p(Ap), _p(Wp), _p(bias), M, N, K, 2, 0, 1.0, _p(outp), 0, _stream()))
            got = outp[:, :N].float() + outp[:, N:].float()
            want = torch.nn.functional.silu(ref).float()
            assert float((got - want).abs().max()) < 1e-4
            # residual accumulate
            res = torch.randn(M, N, device="cuda")
            res0 = res.clone()
            _check(lib, lib.rvb_gemm_bf16x3(_p(Ap), _p(Wp), _p(bias), M, N, K, 0, 2, 0.5, _p(res), N, _stream()))
            assert float((res.double() - (res0.double() + 0.5 * ref)).abs().max()) < 1e-4
    finally:
        lib.rvb_set_gemm_impl(-1)


def test_gemm_bf16x3_glu_pair_output(lib):
    torch.manual_seed(7)
    M, Cc, K = 1000, 256, 256
    A = torch.randn(M, K, device="cuda") * 0.5
    W = torch.randn(2 * Cc, K, device="cuda") / math.sqrt(K)
    bias = torch.randn(2 * Cc, device="cuda")
    ref = torch.nn.functional.glu(A.double() @ W.double().t() + bias.double(), dim=1).float()
    c = torch.arange(Cc, device="cuda")
    ra = 64 * (c // 32) + (c % 32)
    Wq, bq = torch.empty_like(W), torch.empty_like(bias)
    Wq[ra], Wq[ra + 32] = W[:Cc], W[Cc:]
    bq[ra], bq[ra + 32] = bias[:Cc], bias[Cc:]
    out = torch.zeros(M, 2 * Cc, device="cuda", dtype=torch.bfloat16)
    Ap, Wp = _pair(lib, A), _pair(lib, Wq)                       # keep the operands alive across the launch
    _check(lib, lib.rvb_gemm_bf16x3(_p(Ap), _p(Wp), _p(bq), M, 2 * Cc, K, 3, 0, 1.0, _p(out), 0, _stream()))
    torch.cuda.synchronize()
    got = out[:, :Cc].float() + out[:, Cc:].float()
    assert float((got - ref).abs().max()) < 1e-4
