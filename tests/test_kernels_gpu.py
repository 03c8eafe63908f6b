"""GPU: each sm_100a kernel, called through the C-ABI test hooks, against a plain torch fp32 reference of the
same op on the same (bf16-rounded) operands."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from avsep_b200.engine import Engine, EngineConfig
    e = Engine(EngineConfig(65, 64, 4, 1, 1, 2, "bf16"), 0)
    yield e
    e.close()


def _s():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(eng, rc):
    assert rc == 0, eng.lib.avsep_last_error(eng.h).decode()


@pytest.mark.parametrize("M,N,K,act,bn", [
    (128, 128, 64, 0, 0),          # single tile, single k-tile
    (256, 256, 256, 0, 0),
    (300, 192, 264, 1, 0),         # ragged M, N not a power of two, K tail (264 = 4*64 + 8), ReLU
    (1000, 768, 256, 0, 0),        # QKV shape
    (1000, 1024, 256, 2, 0),       # FFN1 + GELU
    (1000, 256, 1024, 0, 0),       # FFN2 (16 k-tiles: ring wraps several times)
    (77, 64, 64, 0, 0),            # tiny model (d=64)
    (500, 256, 128, 0, 128),       # frame_proj shape, forced 128-wide tiles
    (500, 512, 256, 2, 256),       # decoder hidden
    (4096, 768, 256, 0, 256),
])
def test_gemm_tcgen05(eng, M, N, K, act, bn):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    out = torch.full((M, N), float("nan"), device="cuda")
    _check(eng, eng.lib.avsep_test_gemm(eng.h, A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(),
                                        M, N, K, act, bn, _s()))
    torch.cuda.synchronize()
    ref = A.float() @ W.float().t() + bias
    if act == 1:
        ref = torch.relu(ref)
    elif act == 2:
        ref = torch.nn.functional.gelu(ref)
    err = (out - ref).abs().max().item()
    assert err < 2e-3, err


@pytest.mark.parametrize("M,act", [(128, 1), (1000, 1), (16128, 1), (12800, 2), (77, 2), (148 * 128 + 300, 1)])
def test_ffn_fused(eng, M, act):
    """linear1 -> ReLU / GELU -> linear2 -> +residual -> LayerNorm in one kernel (hidden stays on chip)."""
    g = torch.Generator(device="cuda").manual_seed(M + act)
    d, hid = 256, 1024
    a = torch.randn(M, d, device="cuda", generator=g).bfloat16()
    w1 = (torch.randn(hid, d, device="cuda", generator=g) / math.sqrt(d)).bfloat16()
    b1 = torch.randn(hid, device="cuda", generator=g) * 0.5
    w2 = (torch.randn(d, hid, device="cuda", generator=g) / math.sqrt(hid)).bfloat16()
    b2 = torch.randn(d, device="cuda", generator=g)
    x = torch.randn(M, d, device="cuda", generator=g) * 2 + 0.3
    gamma = torch.randn(d, device="cuda", generator=g)
    beta = torch.randn(d, device="cuda", generator=g)
    hdn = a.float() @ w1.float().t() + b1
    hdn = torch.relu(hdn) if act == 1 else torch.nn.functional.gelu(hdn)
    x_ref = x + hdn.bfloat16().float() @ w2.float().t() + b2        # the hidden is rounded to bf16 between the GEMMs
    ln_ref = torch.nn.functional.layer_norm(x_ref, (d,), gamma, beta, 1e-5)
    out = torch.zeros(M, d, device="cuda", dtype=torch.bfloat16)
    _check(eng, eng.lib.avsep_test_ffn_fused(eng.h, a.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                                             b2.data_ptr(), act, x.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                             out.data_ptr(), M, _s()))
    torch.cuda.synchronize()
    assert (x - x_ref).abs().max().item() < 2e-2          # bf16 rounding of the hidden at a different point of the tie
    assert (x - x_ref).abs().mean().item() < 2e-4
    assert (out.float() - ln_ref).abs().max().item() < 6e-2
    assert (out.float() - ln_ref).abs().mean().item() < 5e-3


@pytest.fixture(scope="module")
def eng32():
    from avsep_b200.engine import Engine, EngineConfig
    e = Engine(EngineConfig(65, 64, 4, 1, 1, 2, "tf32"), 0)
    yield e
    e.close()


@pytest.mark.parametrize("M,N,K,act", [(128, 128, 32, 0), (1000, 768, 256, 0), (300, 192, 264, 1), (1000, 256, 1024, 2),
                                       (77, 64, 64, 0)])
def test_gemm_tcgen05_tf32(eng32, M, N, K, act):
    def to_tf32(x):      # round to nearest (ties away), as cvt.rna.tf32.f32 and the library's weight packer do
        return ((x.view(torch.int32) + 0x1000) & -8192).view(torch.float32)
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = to_tf32(torch.randn(M, K, device="cuda", generator=g))
    W = to_tf32(torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K))
    bias = torch.randn(N, device="cuda", generator=g)
    out = torch.full((M, N), float("nan"), device="cuda")
    _check(eng32, eng32.lib.avsep_test_gemm(eng32.h, A.data_ptr(), W.data_ptr(), bias.data_ptr(), out.data_ptr(),
                                            M, N, K, act, 0, _s()))
    torch.cuda.synchronize()
    ref = A.double() @ W.double().t() + bias.double()
    if act == 1:
        ref = torch.relu(ref)
    elif act == 2:
        ref = torch.nn.functional.gelu(ref)
    err = (out.double() - ref).abs().max().item()
    assert err < 2e-4, err          # exact tf32 operands, fp32 accumulation


def test_attention_split_fp32_grade(eng32):
    B, H, hd, T, N = 2, 4, 64, 63, 50
    g = torch.Generator(device="cuda").manual_seed(5)
    d = H * hd
    q = torch.randn(B, T, d, device="cuda", generator=g)
    k = torch.randn(B, N, d, device="cuda", generator=g)
    v = torch.randn(B, N, d, device="cuda", generator=g)
    out = torch.zeros(B, T, d, device="cuda")
    _check(eng32, eng32.lib.avsep_test_attention(eng32.h, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                                 B, H, hd, T, T, N, _s()))
    torch.cuda.synchronize()
    up = lambda t: torch.nn.functional.interpolate(t.permute(0, 2, 1), size=T, mode="linear",
                                                   align_corners=False).permute(0, 2, 1)
    qh = q.view(B, T, H, hd).transpose(1, 2)
    kh = up(k).view(B, T, H, hd).transpose(1, 2)
    vh = up(v).view(B, T, H, hd).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) / math.sqrt(hd), -1) @ vh).transpose(1, 2).reshape(B, T, d)
    assert (out - ref).abs().max().item() < 1e-3     # fp32-grade contraction; the output is rounded to tf32 (2^-11)
    # self-attention (no interpolation), fp32 in / fp32 out
    out2 = torch.zeros(B, T, d, device="cuda")
    _check(eng32, eng32.lib.avsep_test_attention(eng32.h, q.data_ptr(), q.data_ptr(), q.data_ptr(), out2.data_ptr(),
                                                 B, H, hd, T, T, 0, _s()))
    torch.cuda.synchronize()
    ref2 = (torch.softmax(qh @ qh.transpose(-1, -2) / math.sqrt(hd), -1) @ qh).transpose(1, 2).reshape(B, T, d)
    assert (out2 - ref2).abs().max().item() < 2e-3


@pytest.mark.parametrize("M,N,K", [(1000, 256, 256), (16128, 256, 1024), (77, 64, 64), (300, 128, 512), (130, 32, 64),
                                   (148 * 128 + 700, 256, 256)])     # last: some CTAs run two tiles (both epilogue paths)
def test_gemm_fused_residual_layernorm(eng, M, N, K):
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    W = (torch.randn(N, K, device="cuda", generator=g) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, device="cuda", generator=g)
    x = torch.randn(M, N, device="cuda", generator=g) * 2 + 0.5
    gamma = torch.randn(N, device="cuda", generator=g)
    beta = torch.randn(N, device="cuda", generator=g)
    x_ref = x + A.float() @ W.float().t() + bias
    ln_ref = torch.nn.functional.layer_norm(x_ref, (N,), gamma, beta, 1e-5)
    out = torch.zeros(M, N, device="cuda", dtype=torch.bfloat16)
    _check(eng, eng.lib.avsep_test_gemm_ln(eng.h, A.data_ptr(), W.data_ptr(), bias.data_ptr(), x.data_ptr(),
                                           gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), M, N, K, _s()))
    torch.cuda.synchronize()
    assert (x - x_ref).abs().max().item() < 2e-3
    assert (out.float() - ln_ref).abs().max().item() < 5e-2
    assert (out.float() - ln_ref).abs().mean().item() < 4e-3
    # cast-only variant (gamma = None): out_op = bf16(x)
    x2 = x_ref.clone()
    _check(eng, eng.lib.avsep_test_gemm_ln(eng.h, A.data_ptr(), W.data_ptr(), bias.data_ptr(), x2.data_ptr(),
                                           None, None, out.data_ptr(), M, N, K, _s()))
    torch.cuda.synchronize()
    assert torch.equal(out, x2.bfloat16())


@pytest.mark.parametrize("B,L,N,K", [(2, 63, 256, 264), (3, 32, 64, 72), (1, 300, 256, 256), (5, 7, 64, 64)])
def test_conv1d_implicit_gemm(eng, B, L, N, K):
    g = torch.Generator(device="cuda").manual_seed(B + L + N + K)
    x = torch.randn(B, L, K, device="cuda", generator=g).bfloat16()
    xp = torch.zeros(B, L + 2, K, device="cuda", dtype=torch.bfloat16)
    xp[:, 1:L + 1] = x
    w = (torch.randn(N, K, 3, device="cuda", generator=g) / math.sqrt(3 * K)).bfloat16()   # (Cout, Cin, tap)
    w3 = w.permute(0, 2, 1).contiguous().reshape(N, 3 * K)                                   # k = tap*K + c
    bias = torch.randn(N, device="cuda", generator=g)
    out = torch.full((B * L, N), float("nan"), device="cuda")
    _check(eng, eng.lib.avsep_test_conv1d(eng.h, xp.data_ptr(), w3.data_ptr(), bias.data_ptr(), out.data_ptr(),
                                          B, L, N, K, _s()))
    torch.cuda.synchronize()
    ref = torch.nn.functional.conv1d(x.float().permute(0, 2, 1), w.float(), bias, padding=1).permute(0, 2, 1)
    err = (out.view(B, L, N) - ref).abs().max().item()
    assert err < 2e-3, err


@pytest.mark.parametrize("B,H,hd,Lq,Lk", [(2, 4, 64, 63, 63), (3, 4, 16, 32, 32), (1, 2, 64, 200, 200),
                                           (2, 8, 64, 50, 50), (1, 1, 32, 5, 5), (1, 2, 128, 70, 70),
                                           (1, 4, 64, 20, 60), (2, 4, 64, 64, 1), (2, 2, 64, 1, 64), (1, 4, 64, 64, 65)])
def test_attention_self(eng, B, H, hd, Lq, Lk):
    g = torch.Generator(device="cuda").manual_seed(B * 100 + Lq)
    d = H * hd
    q = torch.randn(B, Lq, d, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, Lk, d, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, Lk, d, device="cuda", generator=g).bfloat16()
    out = torch.zeros(B, Lq, d, device="cuda", dtype=torch.bfloat16)
    _check(eng, eng.lib.avsep_test_attention(eng.h, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                             B, H, hd, Lq, Lk, 0, _s()))
    torch.cuda.synchronize()
    qh, kh, vh = (t.float().view(B, -1, H, hd).transpose(1, 2) for t in (q, k, v))
    ref = torch.softmax(qh @ kh.transpose(-1, -2) / math.sqrt(hd), -1) @ vh
    ref = ref.transpose(1, 2).reshape(B, Lq, d)
    err = (out.float() - ref).abs().max().item()
    assert err < 3e-2, err       # bf16 P and bf16 output rounding on O(1) values


@pytest.mark.parametrize("B,H,hd,T,N", [(2, 4, 64, 63, 50), (2, 4, 16, 20, 30), (1, 4, 64, 300, 120), (2, 4, 16, 32, 10)])
def test_attention_cross_with_lerp_on_load(eng, B, H, hd, T, N):
    g = torch.Generator(device="cuda").manual_seed(T * 31 + N)
    d = H * hd
    q = torch.randn(B, T, d, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, N, d, device="cuda", generator=g)
    v = torch.randn(B, N, d, device="cuda", generator=g)
    out = torch.zeros(B, T, d, device="cuda", dtype=torch.bfloat16)
    _check(eng, eng.lib.avsep_test_attention(eng.h, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                             B, H, hd, T, T, N, _s()))
    torch.cuda.synchronize()
    up = lambda t: torch.nn.functional.interpolate(t.permute(0, 2, 1), size=T, mode="linear",
                                                   align_corners=False).permute(0, 2, 1)
    qh = q.float().view(B, T, H, hd).transpose(1, 2)
    kh = up(k).view(B, T, H, hd).transpose(1, 2)
    vh = up(v).view(B, T, H, hd).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) / math.sqrt(hd), -1) @ vh).transpose(1, 2).reshape(B, T, d)
    err = (out.float() - ref).abs().max().item()
    assert err < 3e-2, err


@pytest.mark.parametrize("M,d", [(1000, 256), (77, 64), (513, 512), (9, 1024)])
def test_add_layernorm(eng, M, d):
    g = torch.Generator(device="cuda").manual_seed(M + d)
    x = torch.randn(M, d, device="cuda", generator=g) * 3
    y = torch.randn(M, d, device="cuda", generator=g)
    gamma = torch.randn(d, device="cuda", generator=g)
    beta = torch.randn(d, device="cuda", generator=g)
    xo = torch.empty_like(x)
    out = torch.empty(M, d, device="cuda", dtype=torch.bfloat16)
    _check(eng, eng.lib.avsep_test_add_layernorm(eng.h, x.data_ptr(), y.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                                 xo.data_ptr(), out.data_ptr(), M, d, _s()))
    torch.cuda.synchronize()
    assert torch.equal(xo, x + y)
    ref = torch.nn.functional.layer_norm(x + y, (d,), gamma, beta, 1e-5)
    assert (out.float() - ref).abs().max().item() < 4e-2        # bf16 output rounding of O(5) values
    assert (out.float() - ref.bfloat16().float()).abs().max().item() < 4e-2
    # plain cast (gamma = None) and residual-only paths
    out2 = torch.empty(M, d, device="cuda", dtype=torch.bfloat16)
    _check(eng, eng.lib.avsep_test_add_layernorm(eng.h, x.data_ptr(), None, None, None, None, out2.data_ptr(), M, d, _s()))
    torch.cuda.synchronize()
    assert torch.equal(out2, x.bfloat16())


@pytest.mark.parametrize("Hh,Ww,M", [(32, 32, 1), (32, 32, 7), (32, 32, 8), (32, 32, 50), (32, 32, 601), (32, 32, 1203),
                                      (32, 32, 2501), (16, 16, 21), (15, 18, 7), (16, 16, 601), (31, 32, 50), (32, 31, 50),
                                      (64, 64, 50)])
def test_visual_cnn(Hh, Ww, M):
    """The frame size picks the kernel: 32x32 frames run the tcgen05 kernel (visual_cnn_tc.cu), every other size the
    generic mma.sync kernel (visual_cnn.cu)."""
    from oracle.weights import CONFIGS, make_state_dict
    from avsep_b200.engine import Engine, EngineConfig
    cfg = CONFIGS["tiny"]
    P = make_state_dict(cfg, seed=5, gain=2.0)
    e = Engine(EngineConfig(**cfg.as_dict()), 0)
    try:
        e.load_state({k: v for k, v in P.items() if v.ndim > 0})
        g = torch.Generator(device="cuda").manual_seed(M)
        frames = torch.rand(M, Hh, Ww, device="cuda", generator=g)
        pooled = torch.zeros(M, 128, device="cuda", dtype=torch.bfloat16)
        assert e.lib.avsep_test_visual_cnn(e.h, frames.data_ptr(), M, Hh, Ww, pooled.data_ptr(), _s()) == 0, \
            e.lib.avsep_last_error(e.h).decode()
        torch.cuda.synchronize()
        F = torch.nn.functional
        x = frames.view(M, 1, Hh, Ww)
        for idx in (0, 3, 6):
            t = lambda k: torch.from_numpy(P[k]).cuda()
            x = F.conv2d(x, t(f"visual_encoder.conv.{idx}.weight"), t(f"visual_encoder.conv.{idx}.bias"), stride=2, padding=1)
            bn = f"visual_encoder.conv.{idx + 1}"
            x = F.relu(F.batch_norm(x, t(bn + ".running_mean"), t(bn + ".running_var"), t(bn + ".weight"), t(bn + ".bias"),
                                    False, 0.1, 1e-5))
        ref = x.mean(dim=(2, 3))
        err = (pooled.float() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert err < 2e-2 * max(1.0, scale), (err, scale)
    finally:
        e.close()


@pytest.mark.parametrize("B,H,Lq,Lk", [(2, 4, 63, 63), (1, 4, 128, 128), (2, 2, 300, 300), (1, 4, 1251, 1251),
                                       (3, 4, 129, 257), (2, 4, 500, 500), (1, 1, 5, 5), (2, 4, 200, 77)])
def test_attention_tcgen05_self(eng, B, H, Lq, Lk):
    """tcgen05 flash-attention kernel (attention_tc.cu), forced on for every shape, against fp32 softmax attention."""
    hd = 64
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + Lq + Lk)
    d = H * hd
    q = torch.randn(B, Lq, d, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, Lk, d, device="cuda", generator=g).bfloat16()
    v = torch.randn(B, Lk, d, device="cuda", generator=g).bfloat16()
    out = torch.full((B, Lq, d), 7.0, device="cuda", dtype=torch.bfloat16)
    guard = out.clone()
    eng.set_option("attn_tc", 2)
    try:
        _check(eng, eng.lib.avsep_test_attention(eng.h, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                                 B, H, hd, Lq, Lk, 0, _s()))
        torch.cuda.synchronize()
    finally:
        eng.set_option("attn_tc", 1)
    qh, kh, vh = (t.float().view(B, -1, H, hd).transpose(1, 2) for t in (q, k, v))
    ref = torch.softmax(qh @ kh.transpose(-1, -2) / math.sqrt(hd), -1) @ vh
    ref = ref.transpose(1, 2).reshape(B, Lq, d)
    err = (out.float() - ref).abs().max().item()
    assert err < 3e-2, err
    assert not torch.equal(out, guard)


@pytest.mark.parametrize("B,H,T,N", [(2, 4, 63, 50), (1, 4, 300, 120), (2, 4, 1251, 500), (1, 2, 640, 64)])
def test_attention_tcgen05_cross_materialised_lerp(eng, B, H, T, N):
    hd = 64
    g = torch.Generator(device="cuda").manual_seed(T * 7 + N)
    d = H * hd
    q = torch.randn(B, T, d, device="cuda", generator=g).bfloat16()
    k = torch.randn(B, N, d, device="cuda", generator=g)
    v = torch.randn(B, N, d, device="cuda", generator=g)
    out = torch.zeros(B, T, d, device="cuda", dtype=torch.bfloat16)
    eng.set_option("attn_tc", 2)
    try:
        _check(eng, eng.lib.avsep_test_attention(eng.h, q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(),
                                                 B, H, hd, T, T, N, _s()))
        torch.cuda.synchronize()
    finally:
        eng.set_option("attn_tc", 1)
    up = lambda t: torch.nn.functional.interpolate(t.permute(0, 2, 1), size=T, mode="linear",
                                                   align_corners=False).permute(0, 2, 1)
    qh = q.float().view(B, T, H, hd).transpose(1, 2)
    kh = up(k).view(B, T, H, hd).transpose(1, 2)
    vh = up(v).view(B, T, H, hd).transpose(1, 2)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) / math.sqrt(hd), -1) @ vh).transpose(1, 2).reshape(B, T, d)
    err = (out.float() - ref).abs().max().item()
    assert err < 3e-2, err
