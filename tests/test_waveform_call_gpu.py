"""Waveforms in, waveforms out in one call (avsep_separate_waveforms and its host-buffer forms): bit for bit what the
three-call composition Engine.stft -> Engine.forward -> Engine.istft gives, on every kernel path the forward can take,
with one launch fewer, and the host-buffer forms equal to the device call."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.weights import CONFIGS, make_inputs, make_state_dict
from tests.helpers import build_model

pytestmark = pytest.mark.gpu

# name -> (config, precision, B, L, N, frame side, n_fft, hop, debug)
CASES = {
    "default_bf16_b256": ("default", "bf16", 256, 8000, 50, 32, 512, 128, False),   # fused stack kernels
    "default_tf32": ("default", "tf32", 16, 8000, 50, 32, 512, 128, False),
    "default_long": ("default", "bf16", 8, 128 * 159, 50, 32, 512, 128, False),     # T = 160 > 128: per-layer kernels
    "default_debug": ("default", "bf16", 8, 8000, 50, 32, 512, 128, True),
    "tiny_nfft128": ("tiny", "bf16", 6, 1000, 12, 16, 128, 32, False),              # radix-2 analysis / inverse
}
_MODELS = {}


def _model(cfg_name, precision, seed=91):
    key = (cfg_name, precision)
    if key not in _MODELS:
        cfg = CONFIGS[cfg_name]
        _MODELS[key] = build_model(cfg, make_state_dict(cfg, seed=seed, gain=2.0), precision)
        _MODELS[key].prepack()
    return _MODELS[key]


def _inputs(cfg_name, B, L, N, side, seed):
    _, frames = make_inputs(CONFIGS[cfg_name], B, 1, N, side, side, seed=seed, kind="dataset")
    g = torch.Generator(device="cuda").manual_seed(seed)
    return 0.3 * torch.randn(B, L, device="cuda", generator=g), torch.from_numpy(frames).cuda()


def _ragged(B, L, N, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, L + 1, B).astype(np.int32)
    flens = rng.integers(1, N + 1, B).astype(np.int32)
    lens[0], flens[0] = L, N
    if B > 1:
        lens[1], flens[1] = 1, 1
    return lens, flens


def _same(a, b):
    return a.shape == b.shape and torch.equal(a.detach().cpu(), b.detach().cpu())


def _composed(eng, wave, lips, n_fft, hop, lens=None, flens=None):
    L = wave.shape[1]
    if lens is None:
        spec, mag = eng.stft(wave, n_fft, hop)
        _, masks = eng.forward(mag, lips, frame_lengths=flens)
    else:
        spec, mag, fl = eng.stft(wave, n_fft, hop, lengths=lens)
        _, masks = eng.forward(mag, lips, lengths=fl, frame_lengths=flens)
    return eng.istft(spec, masks, L, n_fft, hop, lengths=lens), masks


@pytest.mark.parametrize("name", list(CASES))
def test_device_call_equals_the_composition(name):
    cfg_name, prec, B, L, N, side, n_fft, hop, debug = CASES[name]
    model = _model(cfg_name, prec)
    eng = model.engine
    eng.set_debug(debug)
    try:
        wave, lips = _inputs(cfg_name, B, L, N, side, seed=92)
        w_ref, m_ref = _composed(eng, wave, lips, n_fft, hop)
        w, m = eng.separate_waveforms(wave, lips, n_fft, hop)
        assert _same(w, w_ref) and _same(m, m_ref)
        w2, m2 = eng.separate_waveforms(wave, lips, n_fft, hop, want_masks=False)
        assert m2 is None and _same(w2, w_ref)
        lens, flens = _ragged(B, L, N, seed=93)
        w_ref, m_ref = _composed(eng, wave, lips, n_fft, hop, lens, flens)
        w, m = eng.separate_waveforms(wave, lips, n_fft, hop, lengths=lens, frame_lengths=flens)
        assert _same(w, w_ref) and _same(m, m_ref)
        w2, _ = eng.separate_waveforms(wave, lips, n_fft, hop, lengths=lens, frame_lengths=flens, want_masks=False)
        assert _same(w2, w_ref)
        # lip-frame lengths alone (every sample present)
        w_ref, m_ref = _composed(eng, wave, lips, n_fft, hop, flens=flens)
        w, m = eng.separate_waveforms(wave, lips, n_fft, hop, frame_lengths=flens)
        assert _same(w, w_ref) and _same(m, m_ref)
    finally:
        eng.set_debug(False)


def _abi_call(eng, wave, lips, n_fft, hop, out, masks, lens_d=None, flens_d=None):
    B, L = wave.shape
    _, N, Hh, Ww = lips.shape
    rc = eng.lib.avsep_separate_waveforms(eng.h, wave.data_ptr(), lips.data_ptr(),
                                          None if lens_d is None else lens_d.data_ptr(),
                                          None if flens_d is None else flens_d.data_ptr(), B, L, N, Hh, Ww, n_fft, hop,
                                          out.data_ptr(), None if masks is None else masks.data_ptr(), None, 0,
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
    eng._check(rc, "avsep_separate_waveforms")
    return eng.launch_count()


def test_launches_profile_and_graph_replay():
    model = _model("default", "bf16")
    eng = model.engine
    B, L, N = 64, 8000, 50
    wave, lips = _inputs("default", B, L, N, 32, seed=94)
    spec, mag = eng.stft(wave, 512, 128)
    n_stft = eng.launch_count()
    _, masks = eng.forward(mag, lips)
    n_fwd = eng.launch_count()
    eng.istft(spec, masks, L, 512, 128)
    n_istft = eng.launch_count()
    want = n_stft + n_fwd + n_istft - 1
    assert want == 7
    out = torch.empty(B, 2, L, device="cuda")
    mk = torch.empty(B, 2, 257, 63, device="cuda")
    counts, results = [], []
    for _ in range(4):                      # eager, capture, replay, replay
        out.fill_(float("nan"))
        mk.fill_(float("nan"))
        counts.append(_abi_call(eng, wave, lips, 512, 128, out, mk))
        results.append((out.clone(), mk.clone()))
    assert counts == [want] * 4, counts
    for w, m in results[1:]:
        assert _same(w, results[0][0]) and _same(m, results[0][1])
    # device lengths: a new ragged batch in the same length buffers replays the cached graph
    lens_d = torch.empty(B, dtype=torch.int32, device="cuda")
    flens_d = torch.empty_like(lens_d)
    for seed in (95, 96, 97):
        lens, flens = _ragged(B, L, N, seed)
        lens_d.copy_(torch.from_numpy(lens))
        flens_d.copy_(torch.from_numpy(flens))
        assert _abi_call(eng, wave, lips, 512, 128, out, mk, lens_d, flens_d) == want
        w_ref, m_ref = _composed(eng, wave, lips, 512, 128, lens, flens)
        assert _same(out, w_ref) and _same(mk, m_ref), seed
    eng.set_profile(True)
    try:
        eng.profile_report(reset=True)
        _abi_call(eng, wave, lips, 512, 128, out, None)
        rep = eng.profile_report(reset=True)
    finally:
        eng.set_profile(False)
    assert "prep_audio" not in rep and "stft" in rep and "istft" in rep, rep
    assert sum(n for n, _ in rep.values()) == want


@pytest.fixture(scope="module")
def default_model():
    return _model("default", "bf16")


def _host_inputs(B, seed, L=8000, N=50):
    wave, lips = _inputs("default", B, L, N, 32, seed)
    return wave, lips, wave.cpu().pin_memory(), lips.cpu().pin_memory()


@pytest.mark.parametrize("B,chunk,lanes", [(1, 0, 0), (57, 0, 0), (256, 0, 0), (57, 16, 3)])
def test_host_call_equals_device_call(default_model, B, chunk, lanes):
    eng = default_model.engine
    wave, lips, wave_h, lips_h = _host_inputs(B, seed=100 + B)
    w_d, m_d = eng.separate_waveforms(wave, lips)
    eng.set_option("host_chunk", chunk)
    eng.set_option("host_lanes", lanes)
    try:
        w_h, m_h = eng.separate_waveforms_host(wave_h, lips_h)
        assert not w_h.is_cuda and _same(w_h, w_d) and _same(m_h, m_d)
        w_h, m_h = eng.separate_waveforms_host(wave_h, lips_h, want_masks=False)
        assert m_h is None and _same(w_h, w_d)
        # pageable buffers give the same results
        w_p, m_p = eng.separate_waveforms_host(wave.cpu(), lips.cpu(), out=(torch.empty(B, 2, 8000),
                                                                          torch.empty(B, 2, 257, 63)))
        assert _same(w_p, w_d) and _same(m_p, m_d)
    finally:
        eng.set_option("host_chunk", 0)
        eng.set_option("host_lanes", 0)


def test_async_slots_cycle_over_batches(default_model):
    eng = default_model.engine
    batches = []
    for k in range(8):
        B = (24, 57, 8, 40)[k % 4]
        wave, lips, wave_h, lips_h = _host_inputs(B, seed=110 + k)
        w_d, m_d = eng.separate_waveforms(wave, lips)
        out = torch.empty(B, 2, 8000).pin_memory()
        mk = torch.empty(B, 2, 257, 63).pin_memory() if k % 3 else None
        batches.append((wave_h, lips_h, out, mk, w_d, m_d))
    torch.cuda.synchronize()

    def check(k):
        _, _, out, mk, w_d, m_d = batches[k]
        assert _same(out, w_d), k
        assert mk is None or _same(mk, m_d), k

    for k, (wave_h, lips_h, out, mk, _, _) in enumerate(batches):
        slot = k % 4
        if k >= 4:
            eng.host_wait(slot)
            check(k - 4)
        eng.separate_waveforms_host_async(wave_h, lips_h, out, mk, slot)
    for k in range(4, 8):
        eng.host_wait(k % 4)
        check(k)


def test_async_waveform_and_spectrogram_forms_interleave(default_model):
    eng = default_model.engine
    B = 32
    wave, lips, wave_h, lips_h = _host_inputs(B, seed=120)
    w_d, m_d = eng.separate_waveforms(wave, lips)
    _, mag = eng.stft(wave, 512, 128)
    sep_d, masks_d = eng.forward(mag, lips)
    mag_h = mag.cpu().pin_memory()
    torch.cuda.synchronize()
    for _ in range(2):
        sep = torch.empty(B, 2, 257, 63).pin_memory()
        masks = torch.empty_like(sep).pin_memory()
        out = torch.empty(B, 2, 8000).pin_memory()
        mk = torch.empty(B, 2, 257, 63).pin_memory()
        eng.forward_host_async(mag_h, lips_h, sep, masks, 0)
        eng.separate_waveforms_host_async(wave_h, lips_h, out, mk, 1)
        eng.host_wait(0)
        eng.host_wait(1)
        assert _same(sep, sep_d) and _same(masks, masks_d)
        assert _same(out, w_d) and _same(mk, m_d)


def test_model_routes_cpu_inputs_through_the_host_call(default_model):
    wave, lips, wave_h, lips_h = _host_inputs(12, seed=130)
    w_d, m_d = default_model.separate_waveforms(wave, lips)
    w_h, m_h = default_model.separate_waveforms(wave_h, lips_h)
    assert not w_h.is_cuda and not m_h.is_cuda
    assert _same(w_h, w_d) and _same(m_h, m_d)


def test_errors_name_the_call(default_model):
    eng = default_model.engine
    wave, lips, wave_h, lips_h = _host_inputs(2, seed=140)
    with pytest.raises(RuntimeError, match="avsep_separate_waveforms: n_fft"):
        eng.separate_waveforms(wave, lips, 256, 128)
    with pytest.raises(RuntimeError, match="avsep_separate_waveforms_host: n_fft"):
        eng.separate_waveforms_host(wave_h, lips_h, 256, 128)
    with pytest.raises(RuntimeError, match="avsep_separate_waveforms: .*power of two"):
        eng.separate_waveforms(wave, lips, 512, 513)
    long_wave = torch.zeros(1, 128 * 5000, device="cuda")
    with pytest.raises(RuntimeError, match="avsep_separate_waveforms: .*positional table"):
        eng.separate_waveforms(long_wave, lips[:1].contiguous(), 512, 128)
    with pytest.raises(ValueError, match="separate_waveforms"):
        eng.separate_waveforms(wave, lips[:1].contiguous())
    with pytest.raises(ValueError, match="separate_waveforms"):
        default_model.separate_waveforms(wave_h, lips_h, lengths=[8000, 8000])
    B, L = wave.shape
    out = torch.empty(B, 2, L, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for w_ptr, l_ptr, o_ptr in ((None, lips.data_ptr(), out.data_ptr()), (wave.data_ptr(), None, out.data_ptr()),
                                (wave.data_ptr(), lips.data_ptr(), None)):
        rc = eng.lib.avsep_separate_waveforms(eng.h, w_ptr, l_ptr, None, None, B, L, 50, 32, 32, 512, 128, o_ptr, None,
                                              None, 0, stream)
        assert rc != 0 and b"null buffer" in eng.lib.avsep_last_error(eng.h)
    assert eng.lib.avsep_waveform_workspace_bytes(eng.h, B, L, 50, 32, 32, 256, 128) == 0
    ws = eng.lib.avsep_waveform_workspace_bytes(eng.h, B, L, 50, 32, 32, 512, 128)
    assert ws > eng.lib.avsep_workspace_bytes(eng.h, B, 63, 50, 32, 32)
    buf = torch.empty(ws + 1024, dtype=torch.uint8, device="cuda")
    base = (buf.data_ptr() + 1023) // 1024 * 1024          # the workspace must be 1024-byte aligned
    mk = torch.empty(B, 2, 257, 63, device="cuda")
    rc = eng.lib.avsep_separate_waveforms(eng.h, wave.data_ptr(), lips.data_ptr(), None, None, B, L, 50, 32, 32, 512,
                                          128, out.data_ptr(), mk.data_ptr(), base, ws - 1, stream)
    assert rc != 0 and b"avsep_waveform_workspace_bytes" in eng.lib.avsep_last_error(eng.h)
    rc = eng.lib.avsep_separate_waveforms(eng.h, wave.data_ptr(), lips.data_ptr(), None, None, B, L, 50, 32, 32, 512,
                                          128, out.data_ptr(), mk.data_ptr(), base, ws, stream)
    eng._check(rc, "avsep_separate_waveforms")
    w_d, m_d = eng.separate_waveforms(wave, lips)
    assert _same(out, w_d) and _same(mk, m_d)
