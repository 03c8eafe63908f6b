"""Variable-length waveform batches (avsep_stft_varlen / avsep_istft_varlen; ``lengths`` of Engine.stft, Engine.istft
and AVSeparationTransformer.separate_waveforms): every utterance of a ragged batch gives, bit for bit, what the same
call gives on that utterance alone, everything past its length is 0, and the padding is never read - including
through the partner frame the two-frames-per-FFT packing gives each frame."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import waveform_oracle as wo
from oracle.weights import CONFIGS, make_inputs, make_state_dict
from tests.helpers import TOL, build_model
from tests.test_waveform_gpu import TOL_WAVE, _wave_err

pytestmark = pytest.mark.gpu

# (n_fft, hop, L): radix-8 analysis and inverse (hop 128 and 100), radix-8 analysis with the radix-2 inverse (hop 32),
# radix-2 both ways (the tiny model's F = 65), a hop of a whole frame, and the smallest frame
GEOMS = [(512, 128, 8000), (512, 100, 2696), (512, 32, 900), (128, 32, 1000), (2048, 2048, 5000), (8, 3, 777)]
IDS = [f"{n}_{h}" for n, h, _ in GEOMS]


@pytest.fixture(scope="module")
def eng():
    from avsep_b200.engine import Engine, EngineConfig
    return Engine(EngineConfig(freq_bins=257, d_model=256, nhead=4, num_encoder_layers=2, num_fusion_layers=2,
                               num_speakers=2), 0)


def _ragged(L, hop, B=10, seed=0):
    """Sample lengths with 1, L, L - 1, a value below one hop and values that put the last frame T_b - 1 on both sides
    of a frame pair (odd and even), plus seeded ones."""
    T = 1 + L // hop
    k = T // 2
    rng = np.random.default_rng(seed)
    lens = [1, L, max(1, hop // 2), min(L, hop * k + 1), min(L, hop * (k + 1) + hop // 3), max(1, L - 1),
            min(L, hop * 1 + 1), min(L, hop * 2)]
    lens = lens[:B] + list(rng.integers(1, L + 1, max(0, B - len(lens))))
    return np.asarray(lens, np.int32)


def _frames(lens, hop, T):
    return np.minimum(T, 1 + lens // hop)


def _solid(L, n_fft, hop, T):
    """Samples whose overlap-add window sum exceeds 1e-3 (the split tests/test_waveform_gpu.py's _wave_err uses)."""
    wss = np.zeros((T - 1) * hop + n_fft)
    for i in range(T):
        wss[i * hop:i * hop + n_fft] += np.hanning(n_fft) ** 2
    return wss[:L] > 1e-3


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _stft_abi(eng, x, n_fft, hop, lens_dev=None, flens_dev=None):
    B, L = x.shape
    T = 1 + L // hop
    spec = torch.empty(B, n_fft // 2 + 1, T, dtype=torch.complex64, device="cuda")
    mag = torch.empty(B, n_fft // 2 + 1, T, device="cuda")
    rc = eng.lib.avsep_stft_varlen(eng.h, x.data_ptr(), None if lens_dev is None else lens_dev.data_ptr(), B, L,
                                   n_fft, hop, spec.data_ptr(), mag.data_ptr(),
                                   None if flens_dev is None else flens_dev.data_ptr(), _stream())
    eng._check(rc, "avsep_stft_varlen")
    assert eng.launch_count() == 1
    return spec, mag


def _istft_abi(eng, spec, masks, L, n_fft, hop, lens_dev=None):
    B, F, T = spec.shape
    S = 1 if masks is None else masks.shape[1]
    out = torch.empty(B, S, L, device="cuda")
    rc = eng.lib.avsep_istft_varlen(eng.h, spec.data_ptr(), None if masks is None else masks.data_ptr(),
                                    None if lens_dev is None else lens_dev.data_ptr(), B, S, T, n_fft, hop, L,
                                    out.data_ptr(), _stream())
    eng._check(rc, "avsep_istft_varlen")
    assert eng.launch_count() == 1
    return out


def _bits(t):
    t = t.detach()
    return torch.view_as_real(t).cpu() if t.is_complex() else t.cpu()


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _inputs(n_fft, hop, L, B, seed, S=2):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = 0.3 * torch.randn(B, L, device="cuda", generator=g)
    T = 1 + L // hop
    masks = torch.rand(B, S, n_fft // 2 + 1, T, device="cuda", generator=g)
    return x, masks


@pytest.mark.parametrize("n_fft,hop,L", GEOMS, ids=IDS)
def test_full_lengths_are_a_no_op(eng, n_fft, hop, L):
    B = 3
    x, masks = _inputs(n_fft, hop, L, B, seed=1)
    T = 1 + L // hop
    spec, mag = eng.stft(x, n_fft, hop)
    spec_v, mag_v, fl = eng.stft(x, n_fft, hop, lengths=[L] * B)
    assert _same(spec_v, spec) and _same(mag_v, mag)
    assert fl.dtype == torch.int32 and fl.tolist() == [T] * B
    spec_n, mag_n = _stft_abi(eng, x, n_fft, hop)                        # both pointers NULL
    assert _same(spec_n, spec) and _same(mag_n, mag)
    fl_d = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    spec_f, mag_f = _stft_abi(eng, x, n_fft, hop, None, fl_d)           # NULL lengths, frame counts requested
    assert _same(spec_f, spec) and _same(mag_f, mag) and fl_d.tolist() == [T] * B
    full = torch.full((B,), L, dtype=torch.int32, device="cuda")
    for m in (masks, None):
        y = eng.istft(spec, m, L, n_fft, hop)
        assert _same(eng.istft(spec, m, L, n_fft, hop, lengths=np.full(B, L)), y)
        assert _same(_istft_abi(eng, spec, m, L, n_fft, hop), y)
        assert _same(_istft_abi(eng, spec, m, L, n_fft, hop, full), y)


@pytest.mark.parametrize("n_fft,hop,L", GEOMS, ids=IDS)
def test_alone_equals_in_batch_bit_for_bit(eng, n_fft, hop, L):
    B = 10
    lens = _ragged(L, hop, B, seed=n_fft + hop)
    x, masks = _inputs(n_fft, hop, L, B, seed=2)
    T = 1 + L // hop
    spec, mag, fl = eng.stft(x, n_fft, hop, lengths=lens)
    tb_all = 1 + lens // hop
    assert fl.tolist() == tb_all.tolist()
    spec_full, _ = eng.stft(x, n_fft, hop)                               # an arbitrary full-length spectrum
    y = eng.istft(spec_full, masks, L, n_fft, hop, lengths=lens)
    y1 = eng.istft(spec_full, None, L, n_fft, hop, lengths=lens)
    for b in range(B):
        lb, tb = int(lens[b]), int(tb_all[b])
        s1, m1 = eng.stft(x[b:b + 1, :lb].contiguous(), n_fft, hop)
        assert s1.shape[2] == tb
        assert _same(spec[b, :, :tb], s1[0]) and _same(mag[b, :, :tb], m1[0]), (b, lb)
        assert not spec[b, :, tb:].abs().any() and not mag[b, :, tb:].any(), (b, lb)
        tf = min(T, 1 + lb // hop)
        sp = spec_full[b:b + 1, :, :tf].contiguous()
        want = eng.istft(sp, masks[b:b + 1, :, :, :tf].contiguous(), lb, n_fft, hop)
        assert _same(y[b, :, :lb], want[0]) and not y[b, :, lb:].any(), (b, lb)
        want1 = eng.istft(sp, None, lb, n_fft, hop)
        assert _same(y1[b, :, :lb], want1[0]) and not y1[b, :, lb:].any(), (b, lb)


@pytest.mark.parametrize("n_fft,hop,L", GEOMS, ids=IDS)
def test_padding_is_never_read(eng, n_fft, hop, L):
    B = 10
    lens = _ragged(L, hop, B, seed=3 * hop)
    T = 1 + L // hop
    tb = _frames(lens, hop, T)
    x, masks = _inputs(n_fft, hop, L, B, seed=3)
    spec_full, _ = eng.stft(x, n_fft, hop)

    def padded(value):
        xv, sv, mv = x.clone(), spec_full.clone(), masks.clone()
        for b in range(B):
            xv[b, lens[b]:] = value
            sv[b, :, tb[b]:] = complex(value, value)
            mv[b, :, :, tb[b]:] = value
        return xv, sv, mv

    x0, s0, m0 = padded(0.0)
    spec, mag, _ = eng.stft(x0, n_fft, hop, lengths=lens)
    y = eng.istft(s0, m0, L, n_fft, hop, lengths=lens)
    assert torch.isfinite(mag).all() and torch.isfinite(y).all()
    for value in (float("nan"), 1e30):
        xv, sv, mv = padded(value)
        spec_v, mag_v, _ = eng.stft(xv, n_fft, hop, lengths=lens)
        assert _same(spec_v, spec) and _same(mag_v, mag), value
        assert _same(eng.istft(sv, mv, L, n_fft, hop, lengths=lens), y), value


@pytest.mark.parametrize("n_fft,hop,L", [GEOMS[0], GEOMS[2], GEOMS[3]], ids=[IDS[0], IDS[2], IDS[3]])
def test_device_lengths_are_clamped(eng, n_fft, hop, L):
    B = 6
    lens = _ragged(L, hop, B, seed=4)
    raw = lens.copy()
    raw[2], raw[3] = 0, L + 5
    lens[2], lens[3] = 1, L
    x, masks = _inputs(n_fft, hop, L, B, seed=4)
    fl_d = torch.empty(B, dtype=torch.int32, device="cuda")
    spec_c, mag_c = _stft_abi(eng, x, n_fft, hop, torch.from_numpy(raw).cuda(), fl_d)
    spec, mag, fl = eng.stft(x, n_fft, hop, lengths=lens)
    assert _same(spec_c, spec) and _same(mag_c, mag) and torch.equal(fl_d, fl)
    y_c = _istft_abi(eng, spec, masks, L, n_fft, hop, torch.from_numpy(raw).cuda())
    assert _same(y_c, eng.istft(spec, masks, L, n_fft, hop, lengths=lens))


def _default_model(seed):
    cfg = CONFIGS["default"]
    return cfg, build_model(cfg, make_state_dict(cfg, seed=seed, gain=2.0), "bf16")


def _wave_inputs(cfg, B, L, N, side, seed):
    _, frames = make_inputs(cfg, B, 1, N, side, side, seed=seed, kind="dataset")
    g = torch.Generator(device="cuda").manual_seed(seed)
    return 0.3 * torch.randn(B, L, device="cuda", generator=g), torch.from_numpy(frames).cuda()


def test_separate_waveforms_alone_equals_in_batch_on_the_default_model():
    """L_b in [4096, 8000] gives T_b in [33, 63] and N_b in [33, 50]: the forward keeps the fused stack kernel's tile
    layout of a stand-alone call, so the whole waveform path is bit-identical per utterance."""
    cfg, model = _default_model(81)
    B, L, N = 8, 8000, 50
    wave, lips = _wave_inputs(cfg, B, L, N, 32, seed=81)
    rng = np.random.default_rng(82)
    lens = rng.integers(4096, L + 1, B).astype(np.int32)
    flens = rng.integers(33, N + 1, B).astype(np.int32)
    lens[0], flens[0] = 4096, N
    lens[1], flens[1] = L, 33
    waves, masks = model.separate_waveforms(wave, lips, lengths=lens, frame_lengths=flens)
    assert waves.shape == (B, 2, L) and masks.shape == (B, 2, 257, 63)
    for b in range(B):
        lb, nb = int(lens[b]), int(flens[b])
        tb = 1 + lb // 128
        w1, m1 = model.separate_waveforms(wave[b:b + 1, :lb].contiguous(), lips[b:b + 1, :nb].contiguous())
        assert _same(waves[b, :, :lb], w1[0]) and not waves[b, :, lb:].any(), (b, lb, nb)
        assert _same(masks[b, :, :, :tb], m1[0]) and not masks[b, :, :, tb:].any(), (b, lb, nb)


def test_separate_waveforms_short_utterances_on_the_tiny_model():
    cfg = CONFIGS["tiny"]
    model = build_model(cfg, make_state_dict(cfg, seed=83, gain=2.0), "bf16")
    B, L, N, n_fft, hop = 6, 1000, 12, 128, 32
    wave, lips = _wave_inputs(cfg, B, L, N, 16, seed=83)
    lens = np.array([1, L, 20, 33, 500, 777], np.int32)
    flens = np.array([N, 1, 3, 12, 7, 5], np.int32)
    waves, masks = model.separate_waveforms(wave, lips, n_fft, hop, lengths=lens, frame_lengths=flens)
    assert waves.shape == (B, 2, L) and masks.shape == (B, 2, 65, 1 + L // hop)
    spec, _, _ = model.engine.stft(wave, n_fft, hop, lengths=lens)
    for b in range(B):
        lb, nb = int(lens[b]), int(flens[b])
        tb = 1 + lb // hop
        _, m1 = model.separate_waveforms(wave[b:b + 1, :lb].contiguous(), lips[b:b + 1, :nb].contiguous(), n_fft, hop)
        assert (masks[b, :, :, :tb] - m1[0]).abs().max().item() < TOL["bf16"], (b, lb, nb)
        assert not masks[b, :, :, tb:].any() and not waves[b, :, lb:].any(), b
        sb, mb = spec[b:b + 1, :, :tb].contiguous(), masks[b:b + 1, :, :, :tb].contiguous()
        assert _same(waves[b, :, :lb], model.engine.istft(sb, mb, lb, n_fft, hop)[0]), (b, lb)
        want = wo.istft_masked(sb[0].cpu().numpy(), mb[0].cpu().numpy(), lb, n_fft, hop)
        got = waves[b, :, :lb].cpu().numpy()
        if _solid(lb, n_fft, hop, tb).any():
            assert _wave_err(got, want, n_fft, hop, tb) <= TOL_WAVE, (b, lb)
        else:                               # no sample with a solid window sum: _wave_err's loose bound only
            assert (np.abs(got - want) / np.maximum(1.0, np.abs(want))).max() <= 1e-3, (b, lb)


def test_graph_replay_follows_the_device_lengths():
    cfg, model = _default_model(85)
    B, L, N = 8, 8000, 50
    wave, lips = _wave_inputs(cfg, B, L, N, 32, seed=85)
    lens_d = torch.empty(B, dtype=torch.int32, device="cuda")
    flens_d = torch.empty_like(lens_d)
    rng = np.random.default_rng(86)
    sets = [(rng.integers(1, L + 1, B).astype(np.int32), rng.integers(1, N + 1, B).astype(np.int32)) for _ in range(4)]
    got = []
    for _ in range(2):                      # the second pass replays graphs captured in the first
        for lens, flens in sets:
            lens_d.copy_(torch.from_numpy(lens))
            flens_d.copy_(torch.from_numpy(flens))
            w, m = model.separate_waveforms(wave, lips, lengths=lens_d, frame_lengths=flens_d)
            got.append((w.clone(), m.clone()))
    model.engine.set_option("use_graph", 0)
    for k, (w_g, m_g) in enumerate(got):
        lens, flens = sets[k % len(sets)]
        w_e, m_e = model.separate_waveforms(wave, lips, lengths=lens, frame_lengths=flens)
        assert _same(w_g, w_e) and _same(m_g, m_e), k
    assert not _same(got[0][1], got[1][1])


def test_ragged_batch_at_size():
    """B = 256 one-second clips with L_b = 128 (T_b - 1) + 64, T_b in [16, 63]: three sub-batches run alone with their
    own lengths reproduce their rows bit for bit; the analysis and the inverse are one launch each and the forward
    launches what a uniform forward launches."""
    cfg, model = _default_model(87)
    B, L, N = 256, 8000, 50
    wave, lips = _wave_inputs(cfg, B, L, N, 32, seed=87)
    rng = np.random.default_rng(88)
    tb = rng.integers(16, 64, B)
    lens = (128 * (tb - 1) + 64).astype(np.int32)
    flens = np.maximum(1, np.round(50 * tb / 63)).astype(np.int32)
    waves, masks = model.separate_waveforms(wave, lips, lengths=lens, frame_lengths=flens)
    assert torch.isfinite(waves).all()
    for b in range(B):
        assert not waves[b, :, lens[b]:].any() and not masks[b, :, :, tb[b]:].any(), b
    for sub in (slice(0, 4), slice(100, 107), slice(245, 256)):
        w_s, m_s = model.separate_waveforms(wave[sub].contiguous(), lips[sub].contiguous(), lengths=lens[sub],
                                            frame_lengths=flens[sub])
        assert _same(w_s, waves[sub]) and _same(m_s, masks[sub]), sub
    eng = model.engine
    spec, mag = eng.stft(wave, 512, 128)
    eng.forward(mag, lips)
    uniform = eng.launch_count()
    spec, mag, fl = eng.stft(wave, 512, 128, lengths=lens)
    assert eng.launch_count() == 1 and fl.tolist() == tb.tolist()
    _, m = eng.forward(mag, lips, lengths=fl, frame_lengths=flens)
    assert eng.launch_count() == uniform
    eng.istft(spec, m, L, 512, 128, lengths=lens)
    assert eng.launch_count() == 1


def test_length_errors():
    cfg = CONFIGS["tiny"]
    model = build_model(cfg, make_state_dict(cfg, seed=89, gain=2.0), "bf16")
    B, L, N, n_fft, hop = 4, 1000, 12, 128, 32
    wave, lips = _wave_inputs(cfg, B, L, N, 16, seed=89)
    model.prepack()
    eng = model.engine
    spec, _ = eng.stft(wave, n_fft, hop)
    full = [L] * B
    bads = ([L] * (B - 1), np.full((B, 1), L), np.full(B, 10.0), [0] + full[1:], [L + 1] + full[1:],
            torch.full((B,), L, dtype=torch.int64, device="cuda"))
    for bad in bads:
        with pytest.raises(ValueError, match="stft"):
            eng.stft(wave, n_fft, hop, lengths=bad)
        with pytest.raises(ValueError, match="istft"):
            eng.istft(spec, None, L, n_fft, hop, lengths=bad)
        with pytest.raises(ValueError, match="separate_waveforms"):
            model.separate_waveforms(wave, lips, lengths=bad)
    for bad in ([0] + [N] * (B - 1), [N + 1] + [N] * (B - 1), [N] * (B + 1)):
        with pytest.raises(ValueError, match="separate_waveforms"):
            model.separate_waveforms(wave, lips, frame_lengths=bad)
    with pytest.raises(ValueError):
        model.separate_waveforms(wave.cpu(), lips.cpu(), lengths=full)
    with pytest.raises(ValueError):
        model.separate_waveforms(wave, lips.cpu(), lengths=full)
