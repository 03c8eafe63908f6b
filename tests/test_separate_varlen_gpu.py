"""avsep_separate_varlen (Engine.separate(lengths=...)): the rebuild of `separated` from masks on a variable-length
batch.  Below each utterance's length the product is avsep_separate's single fp32 multiply, bit for bit; past it the
output is 0 and neither masks nor mixture is read, so NaN / Inf padding cannot leak in.  On the masks of a varlen
forward it reproduces that forward's `separated` exactly -- what the masks-only gather of a varlen batch relies on."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.weights import CONFIGS, make_inputs, make_state_dict
from tests.helpers import build_model

pytestmark = pytest.mark.gpu


def _engine(F, S):
    from avsep_b200.engine import Engine, EngineConfig
    return Engine(EngineConfig(F, 64, 1, 1, 1, S), 0)


def _lengths(B, T, seed):
    """1, T, T - 1, a few values around the 4-element group boundaries, then seeded ones."""
    rng = np.random.default_rng(seed)
    fixed = [1, T, max(1, T - 1), min(T, 2), min(T, 5), min(T, T // 2 + 1)]
    return np.asarray((fixed + list(rng.integers(1, T + 1, max(0, B - len(fixed)))))[:B], np.int32)


def _want(masks, mixed, lens):
    """CPU reference: the product below each length (model.py:220), 0 past it."""
    want = masks * mixed.unsqueeze(1)
    for b, tb in enumerate(lens):
        want[b, :, :, int(tb):] = 0.0
    return want


def _abi(eng, masks, mixed, lens_dev, out):
    B, S, F, T = masks.shape
    rc = eng.lib.avsep_separate_varlen(eng.h, masks.data_ptr(), mixed.data_ptr(),
                                       None if lens_dev is None else lens_dev.data_ptr(), B, T, out.data_ptr(),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream))
    eng._check(rc, "avsep_separate_varlen")
    return out


SHAPES = [(3, 2, 257, 63), (1, 3, 65, 32), (2, 1, 5, 7), (1, 2, 3, 1), (5, 3, 2, 1), (7, 2, 257, 63), (64, 2, 257, 63)]


@pytest.mark.parametrize("B,S,F,T", SHAPES)
def test_full_and_null_lengths_are_avsep_separate_bit_for_bit(B, S, F, T):
    g = torch.Generator().manual_seed(B * 100 + T)
    masks = torch.rand(B, S, F, T, generator=g).cuda()
    mixed = (torch.randn(B, F, T, generator=g) * 30.0).cuda()
    eng = _engine(F, S)
    want = eng.separate(masks, mixed)
    assert torch.equal(eng.separate(masks, mixed, lengths=[T] * B), want)
    assert torch.equal(_abi(eng, masks, mixed, None, torch.full_like(masks, float("nan"))), want)
    full = torch.full((B,), T, dtype=torch.int32, device="cuda")
    assert torch.equal(_abi(eng, masks, mixed, full, torch.full_like(masks, float("nan"))), want)
    eng.close()


@pytest.mark.parametrize("B,S,F,T", SHAPES)
def test_ragged_batch_is_the_product_below_each_length_and_zero_past_it(B, S, F, T):
    g = torch.Generator().manual_seed(B * 10 + T + 1)
    masks, mixed = torch.rand(B, S, F, T, generator=g), torch.randn(B, F, T, generator=g) * 30.0
    lens = _lengths(B, T, seed=B + T)
    eng = _engine(F, S)
    out = torch.full((B, S, F, T), float("nan"), device="cuda")
    assert eng.separate(masks.cuda(), mixed.cuda(), out=out, lengths=lens) is out
    assert torch.equal(out.cpu(), _want(masks, mixed, lens))
    eng.close()


@pytest.mark.parametrize("value", [float("nan"), float("inf"), -float("inf")])
def test_padding_is_never_read(value):
    B, S, F, T = 9, 2, 257, 63
    g = torch.Generator().manual_seed(3)
    masks, mixed = torch.rand(B, S, F, T, generator=g), torch.randn(B, F, T, generator=g)
    lens = _lengths(B, T, seed=3)
    eng = _engine(F, S)
    clean = eng.separate(masks.cuda(), mixed.cuda(), lengths=lens)
    masks_p, mixed_p = masks.clone(), mixed.clone()
    for b, tb in enumerate(lens):
        masks_p[b, :, :, tb:] = value
        mixed_p[b, :, tb:] = value
    got = eng.separate(masks_p.cuda(), mixed_p.cuda(), lengths=lens)
    assert torch.equal(got, clean) and torch.equal(got.cpu(), _want(masks, mixed, lens))
    eng.close()


@pytest.mark.parametrize("B", [1, 4, 5])
@pytest.mark.parametrize("off_masks,off_out", [(0, 0), (1, 1), (3, 3), (1, 2), (0, 2)])
def test_both_alignment_paths(B, off_masks, off_out):
    """Equal misalignment of masks and output keeps the 16-byte walk (head and tail elements one by one; groups that
    straddle a length or a plane load element-wise); different misalignment takes the element-wise kernel.  Nothing
    outside the output view is written."""
    S, F, T = 2, 257, 63
    n = B * S * F * T
    g = torch.Generator().manual_seed(B * 16 + off_masks * 4 + off_out)
    masks_h, mixed_h = torch.rand(B, S, F, T, generator=g), torch.randn(B, F, T, generator=g)
    lens = _lengths(B, T, seed=B + off_masks)
    eng = _engine(F, S)
    masks = torch.full((n + 4,), float("nan"), device="cuda")[off_masks:off_masks + n].view(B, S, F, T)
    masks.copy_(masks_h)
    block = torch.full((n + 8,), 7.0, device="cuda")
    out = block[off_out:off_out + n].view(B, S, F, T)
    eng.separate(masks, mixed_h.cuda(), out=out, lengths=lens)
    assert torch.equal(out.cpu(), _want(masks_h, mixed_h, lens))
    assert bool((block[:off_out] == 7.0).all()) and bool((block[off_out + n:] == 7.0).all())
    eng.close()


def test_device_lengths_are_clamped():
    B, S, F, T = 6, 2, 257, 63
    g = torch.Generator().manual_seed(6)
    masks, mixed = torch.rand(B, S, F, T, generator=g).cuda(), torch.randn(B, F, T, generator=g).cuda()
    raw = np.array([0, -5, T + 1, 1 << 30, 17, -(1 << 30)], np.int32)
    eng = _engine(F, S)
    got = eng.separate(masks, mixed, lengths=torch.from_numpy(raw).cuda())
    assert torch.equal(got, eng.separate(masks, mixed, lengths=np.clip(raw, 1, T)))
    eng.close()


def test_one_launch():
    from torch.profiler import ProfilerActivity, profile
    B, S, F, T = 64, 2, 257, 63
    eng = _engine(F, S)
    masks, mixed = torch.rand(B, S, F, T, device="cuda"), torch.randn(B, F, T, device="cuda")
    lens = torch.from_numpy(_lengths(B, T, seed=8)).cuda()
    out = torch.empty_like(masks)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.separate(masks, mixed, out=out, lengths=lens)
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert len(kernels) == 1 and "separate_kernel" in kernels[0], kernels
    eng.close()


def test_host_length_errors():
    eng = _engine(65, 2)
    masks, mixed = torch.rand(4, 2, 65, 8, device="cuda"), torch.rand(4, 65, 8, device="cuda")
    for bad in ([8] * 3, [0, 8, 8, 8], [9, 8, 8, 8], np.full(4, 8.0), torch.full((4,), 8, dtype=torch.int64, device="cuda")):
        with pytest.raises(ValueError, match="separate"):
            eng.separate(masks, mixed, lengths=bad)
    eng.close()


@pytest.mark.parametrize("cname,T,N", [("default", 63, 50), ("tiny", 40, 12)])
def test_varlen_forward_separated_is_separate_varlen_of_its_masks(cname, T, N):
    """The masks-only gather's rebuild: separate_varlen(masks, NaN-padded mixed, lengths) of a varlen forward's masks
    equals that forward's `separated` bit for bit, zeros past the lengths included."""
    cfg = CONFIGS[cname]
    side = 32 if cname == "default" else 16
    B = 7
    model = build_model(cfg, make_state_dict(cfg, seed=91, gain=2.0), "bf16")
    mixed, frames = make_inputs(cfg, B, T, N, side, side, seed=91, kind="dataset")
    lens = _lengths(B, T, seed=92)
    flens = np.maximum(1, np.round(lens * N / T)).astype(np.int32)
    m_d, f_d = torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda()
    for b in range(B):
        m_d[b, :, lens[b]:] = float("nan")
        f_d[b, flens[b]:] = float("nan")
    sep, masks = model(m_d, f_d, lengths=lens, frame_lengths=flens)
    eng = model.engine
    assert torch.isfinite(sep).all() and torch.isfinite(masks).all()
    assert torch.equal(eng.separate(masks, m_d, lengths=lens), sep)
    lens_d = torch.from_numpy(lens).cuda()
    assert torch.equal(eng.separate(masks, m_d, lengths=lens_d), sep)
