"""Variable-length batches (avsep_forward_varlen; ``lengths`` / ``frame_lengths`` of Engine.forward and
AVSeparationTransformer.forward): every utterance of a ragged batch gives what the model gives on that utterance
alone, its outputs past its length are 0, and the padding of the inputs is never read."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import avsep_oracle as onp
from oracle import avsep_oracle_torch as otorch
from oracle.weights import CONFIGS, make_inputs, make_state_dict
from tests.helpers import TOL, build_model

pytestmark = pytest.mark.gpu

# (config, precision, B, T, N, frame side, attn_tc): the fused stack path (two utterances per tile), one utterance per
# tile, fused stacks with the K|V interpolation as its own lerp_rows launch (the audio rows do not fit a visual tile
# slot), the unfused path with tcgen05 attention, head dim 16, d = 512 (add + LayerNorm kernel), and the TF32 path
CASES = {
    "default_63_50": ("default", "bf16", 6, 63, 50, 32, None),
    "default_100_80": ("default", "bf16", 4, 100, 80, 32, None),
    "default_100_50": ("default", "bf16", 4, 100, 50, 32, None),
    "default_300_120_tc": ("default", "bf16", 3, 300, 120, 32, 1),
    "tiny_40_12": ("tiny", "bf16", 5, 40, 12, 16, None),
    "scaled_63_50": ("scaled", "bf16", 3, 63, 50, 32, None),
    "default_tf32_63_50": ("default", "tf32", 3, 63, 50, 32, None),
}


def _setup(name, seed=61):
    cname, prec, B, T, N, side, attn_tc = CASES[name]
    cfg = CONFIGS[cname]
    P = make_state_dict(cfg, seed=seed, gain=2.0)
    mixed, frames = make_inputs(cfg, B, T, N, side, side, seed=seed, kind="dataset")
    model = build_model(cfg, P, prec)
    model.prepack()
    if attn_tc is not None:
        model.engine.set_option("attn_tc", attn_tc)
    return cfg, P, prec, model, mixed, frames


def _ragged(B, T, N, seed):
    """Seeded lengths that include 1 and the maximum on both sides."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, T + 1, B).astype(np.int32)
    flens = rng.integers(1, N + 1, B).astype(np.int32)
    lens[0], flens[0] = 1, N
    lens[1], flens[1] = T, 1
    return lens, flens


def _pad(mixed, frames, lens, flens, value):
    """Copies with everything past each utterance's lengths set to `value`."""
    m, f = mixed.copy(), frames.copy()
    for b in range(len(lens)):
        m[b, :, lens[b]:] = value
        f[b, flens[b]:] = value
    return m, f


def _run(model, mixed, frames, **kw):
    sep, masks = model(torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda(), **kw)
    torch.cuda.synchronize()
    return sep.cpu().numpy(), masks.cpu().numpy()


def _run_varlen_abi(model, mixed, frames, lens_dev=None, flens_dev=None):
    """avsep_forward_varlen through the C ABI (NULL length pointers when None)."""
    eng = model.engine
    m, f = torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda()
    B, F, T = m.shape
    N, Hh, Ww = f.shape[1:]
    sep = torch.empty(B, eng.cfg.num_speakers, F, T, device="cuda")
    masks = torch.empty_like(sep)
    rc = eng.lib.avsep_forward_varlen(eng.h, m.data_ptr(), f.data_ptr(),
                                      None if lens_dev is None else lens_dev.data_ptr(),
                                      None if flens_dev is None else flens_dev.data_ptr(), B, T, N, Hh, Ww,
                                      sep.data_ptr(), masks.data_ptr(), None, 0,
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream))
    eng._check(rc, "avsep_forward_varlen")
    torch.cuda.synchronize()
    return sep.cpu().numpy(), masks.cpu().numpy()


@pytest.mark.parametrize("name", list(CASES))
def test_full_lengths_are_a_no_op(name):
    cfg, P, prec, model, mixed, frames = _setup(name)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    sep, masks = _run(model, mixed, frames)
    full_t, full_n = np.full(B, T, np.int32), np.full(B, N, np.int32)
    for kw in (dict(lengths=full_t, frame_lengths=full_n), dict(lengths=list(full_t)), dict(frame_lengths=full_n)):
        sep_v, masks_v = _run(model, mixed, frames, **kw)
        assert np.array_equal(sep_v, sep) and np.array_equal(masks_v, masks), (name, list(kw))
    sep_n, masks_n = _run_varlen_abi(model, mixed, frames)       # both pointers NULL
    assert np.array_equal(sep_n, sep) and np.array_equal(masks_n, masks), name
    dev = torch.from_numpy(full_t).cuda(), torch.from_numpy(full_n).cuda()
    sep_d, masks_d = _run_varlen_abi(model, mixed, frames, *dev)
    assert np.array_equal(sep_d, sep) and np.array_equal(masks_d, masks), name


@pytest.mark.parametrize("name", list(CASES))
def test_ragged_batch_matches_reference_per_utterance(name):
    cfg, P, prec, model, mixed, frames = _setup(name)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    lens, flens = _ragged(B, T, N, seed=62)
    sep, masks = _run(model, mixed, frames, lengths=lens, frame_lengths=flens)
    Pt = otorch.to_torch(P) if cfg.d_model >= 256 else None
    tol = TOL[prec]
    for b in range(B):
        tb, nb = int(lens[b]), int(flens[b])
        assert not masks[b, :, :, tb:].any() and not sep[b, :, :, tb:].any(), (name, b)
        assert np.array_equal(sep[b, :, :, :tb], masks[b, :, :, :tb] * mixed[b, None, :, :tb]), (name, b)
        m1, f1 = mixed[b:b + 1, :, :tb], frames[b:b + 1, :nb]
        if Pt is None:
            sep_ref, masks_ref = onp.forward(P, cfg, m1, f1)
        else:
            sep_ref, masks_ref = (x.numpy() for x in otorch.forward(Pt, cfg, torch.from_numpy(m1), torch.from_numpy(f1)))
        em = float(np.abs(masks[b, :, :, :tb] - masks_ref[0]).max())
        es = float((np.abs(sep[b, :, :, :tb] - sep_ref[0]) / np.maximum(1.0, np.abs(m1[0]))[None]).max())
        assert em < tol and es < tol, (name, b, tb, nb, em, es)


def test_alone_equals_in_batch_bit_for_bit_on_the_fused_path():
    """T_b in 33..63 and N_b in 33..50 keep the two-utterance tile layout a stand-alone call at (T_b, N_b) uses, and
    masked key columns contribute exact zeros: each utterance's valid region is the stand-alone result, bit for bit."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=63, gain=2.0)
    B, T, N = 8, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=63, kind="dataset")
    model = build_model(cfg, P, "bf16")
    rng = np.random.default_rng(64)
    lens = rng.integers(33, T + 1, B).astype(np.int32)
    flens = rng.integers(33, N + 1, B).astype(np.int32)
    lens[0], flens[0] = 33, 50
    lens[1], flens[1] = 63, 33
    sep, masks = _run(model, mixed, frames, lengths=lens, frame_lengths=flens)
    for b in range(B):
        tb, nb = int(lens[b]), int(flens[b])
        sep_1, masks_1 = _run(model, np.ascontiguousarray(mixed[b:b + 1, :, :tb]), np.ascontiguousarray(frames[b:b + 1, :nb]))
        assert np.array_equal(masks[b, :, :, :tb], masks_1[0]), (b, tb, nb)
        assert np.array_equal(sep[b, :, :, :tb], sep_1[0]), (b, tb, nb)


@pytest.mark.parametrize("name", ["default_63_50", "tiny_40_12", "default_tf32_63_50"])
def test_padding_is_never_read(name):
    cfg, P, prec, model, mixed, frames = _setup(name, seed=65)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    lens, flens = _ragged(B, T, N, seed=66)
    m0, f0 = _pad(mixed, frames, lens, flens, 0.0)
    sep, masks = _run(model, m0, f0, lengths=lens, frame_lengths=flens)
    assert np.isfinite(sep).all() and np.isfinite(masks).all()
    for value in (np.nan, 1e30):
        mv, fv = _pad(mixed, frames, lens, flens, value)
        sep_v, masks_v = _run(model, mv, fv, lengths=lens, frame_lengths=flens)
        assert np.array_equal(sep_v, sep) and np.array_equal(masks_v, masks), (name, value)


def test_many_tiles_ragged_sub_batches_reproduce_their_rows():
    """B = 701 ragged utterances on the default model: every CTA of the stack kernels walks several tiles; three
    sub-batches run alone with their own lengths give their rows of the full call bit for bit."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=67, gain=2.0)
    B, T, N = 701, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=67, kind="dataset")
    lens, flens = _ragged(B, T, N, seed=68)
    model = build_model(cfg, P, "bf16")
    sep, masks = _run(model, mixed, frames, lengths=lens, frame_lengths=flens)
    assert np.isfinite(sep).all() and masks.min() >= 0.0 and masks.max() <= 1.0
    for b in range(B):
        assert not masks[b, :, :, lens[b]:].any() and not sep[b, :, :, lens[b]:].any(), b
    for sub in (slice(0, 4), slice(296, 303), slice(690, 701)):
        sep_s, masks_s = _run(model, mixed[sub], frames[sub], lengths=lens[sub], frame_lengths=flens[sub])
        assert np.array_equal(masks_s, masks[sub]) and np.array_equal(sep_s, sep[sub]), sub


def test_graph_replay_follows_the_device_lengths():
    """Fixed input, output and length buffers: the graph is captured once and every replay reads whatever the length
    tensors hold at that moment; each result equals an eager run with the same lengths."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=69, gain=2.0)
    B, T, N = 16, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=69, kind="dataset")
    model = build_model(cfg, P, "bf16")
    m, f = torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda()
    sep = torch.empty(B, cfg.num_speakers, cfg.freq_bins, T, device="cuda")
    masks = torch.empty_like(sep)
    lens_d = torch.empty(B, dtype=torch.int32, device="cuda")
    flens_d = torch.empty_like(lens_d)
    sets = [_ragged(B, T, N, seed=70 + k) for k in range(5)]
    got = []
    for lens, flens in sets:
        lens_d.copy_(torch.from_numpy(lens))
        flens_d.copy_(torch.from_numpy(flens))
        model(m, f, out=(sep, masks), lengths=lens_d, frame_lengths=flens_d)
        got.append((sep.cpu().numpy(), masks.cpu().numpy()))
    model.engine.set_option("use_graph", 0)
    for (lens, flens), (sep_g, masks_g) in zip(sets, got):
        sep_e, masks_e = _run(model, mixed, frames, lengths=lens, frame_lengths=flens)
        assert np.array_equal(sep_g, sep_e) and np.array_equal(masks_g, masks_e)
    assert not np.array_equal(got[0][1], got[1][1])


@pytest.mark.parametrize("name", ["default_63_50", "tiny_40_12"])
def test_varlen_launches_the_same_kernels(name):
    cfg, P, prec, model, mixed, frames = _setup(name, seed=71)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    _run(model, mixed, frames)
    uniform = model.engine.launch_count()
    lens, flens = _ragged(B, T, N, seed=72)
    _run(model, mixed, frames, lengths=lens, frame_lengths=flens)
    assert model.engine.launch_count() == uniform, (name, uniform, model.engine.launch_count())


def test_length_errors_and_device_clamping():
    cfg, P, prec, model, mixed, frames = _setup("default_63_50", seed=73)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    m, f = torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda()
    full = [T] * B
    for bad in ([T] * (B - 1), np.full((B, 1), T), np.full(B, 10.0), [0] + full[1:], [T + 1] + full[1:],
                torch.full((B,), T, dtype=torch.int64, device="cuda")):
        with pytest.raises(ValueError):
            model(m, f, lengths=bad)
    for bad in ([0] + [N] * (B - 1), [N + 1] + [N] * (B - 1)):
        with pytest.raises(ValueError):
            model(m, f, frame_lengths=bad)
    with pytest.raises(ValueError):
        model(torch.from_numpy(mixed), torch.from_numpy(frames), lengths=full)
    # device tensors are not read on the host: out-of-range values behave as the nearest bound
    lens, flens = _ragged(B, T, N, seed=74)
    raw_t, raw_n = lens.copy(), flens.copy()
    raw_t[2], raw_t[3] = 0, T + 5
    raw_n[2], raw_n[3] = 0, N + 5
    lens[2], lens[3] = 1, T
    flens[2], flens[3] = 1, N
    sep_c, masks_c = _run_varlen_abi(model, mixed, frames, torch.from_numpy(raw_t).cuda(), torch.from_numpy(raw_n).cuda())
    sep, masks = _run(model, mixed, frames, lengths=lens, frame_lengths=flens)
    assert np.array_equal(sep_c, sep) and np.array_equal(masks_c, masks)
