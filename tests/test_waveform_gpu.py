"""GPU parity of the waveform side (SURVEY 8f rank 4): avsep_stft / avsep_istft through the C ABI against the
reference's `_stft` magnitudes (tests/golden/waveform_stft.npz), the oracle (oracle/waveform_oracle.py) and the
round-trip / linearity identities at full size.  Floating point: the in-kernel transform is fp32 (like numpy's
single-precision path), so spectra are compared relative to the largest magnitude and waveforms absolutely."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "av-separation-transformer_b200"))
from oracle import waveform_oracle as wo   # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden", "waveform_stft.npz")
TOL_SPEC_REL = 2e-6        # of max|spec|
TOL_WAVE = 5e-6            # absolute, waveforms are O(1)


def _wave_err(got, want, n_fft, hop, T=None):
    """max |got - want| / max(1, |want|) over the samples whose overlap-add denominator is solid (> 1e-3).  The first
    (and, for signals the frames overrun, last) samples of a Hann analysis have a tiny window sum: arbitrary masked
    spectra come out there with magnitudes in the hundreds and the fp32 transform error is amplified by 1/wss, so
    those samples get a looser relative bound."""
    L = want.shape[-1]
    w2 = np.hanning(n_fft) ** 2
    T = 1 + L // hop if T is None else T
    wss = np.zeros((T - 1) * hop + n_fft)
    for i in range(T):
        wss[i * hop:i * hop + n_fft] += w2
    solid = wss[:L] > 1e-3
    rel = np.abs(got - want) / np.maximum(1.0, np.abs(want))
    assert rel[..., ~solid].max(initial=0.0) <= 1e-3
    return rel[..., solid].max()


@pytest.fixture(scope="module")
def eng():
    from avsep_b200.engine import Engine, EngineConfig
    return Engine(EngineConfig(freq_bins=257, d_model=256, nhead=4, num_encoder_layers=2, num_fusion_layers=2,
                               num_speakers=2), 0)


@pytest.mark.parametrize("name", ("default", "short", "ragged"))
def test_stft_matches_reference_magnitudes_and_oracle_phase(eng, name):
    z = np.load(GOLD)
    n_fft, hop = (int(v) for v in z[name + "_geom"])
    x = z[name + "_wave"]
    spec, mag = eng.stft(torch.from_numpy(x).cuda()[None].contiguous(), n_fft, hop)
    ref = wo.stft_complex(x, n_fft, hop)
    scale = np.abs(ref).max()
    got = spec[0].cpu().numpy()
    assert got.shape == ref.shape and mag.shape[1:] == ref.shape
    assert np.abs(got - ref).max() <= TOL_SPEC_REL * scale
    assert np.abs(mag[0].cpu().numpy() - z[name + "_mag"]).max() <= TOL_SPEC_REL * scale
    assert torch.equal(mag, spec.abs()) or (mag - spec.abs()).abs().max().item() <= 1e-6 * scale


def _stft_matches_synthesis(kw):
    from avsep_b200.dataset import SyntheticAVDataset
    from oracle import synth_oracle as so
    ds = SyntheticAVDataset(**kw)
    cfg = so.SynthConfig(**kw)
    idxs = (0, 1, 2, 3)
    waves = []
    for i in idxs:
        amps, freqs, phases = so.draw_item(cfg, i)[:3]
        waves.append(so.waveforms(cfg, amps, freqs, phases)[1])
    b = ds.batch(idxs, want_clean=False)
    x = torch.from_numpy(np.stack(waves).astype(np.float32)).cuda()
    _, mag = ds.engine.stft(x, cfg.n_fft, cfg.hop_length)
    scale = b["mixed_spec"].abs().max().item()
    assert (mag - b["mixed_spec"]).abs().max().item() <= TOL_SPEC_REL * scale


def test_stft_magnitude_agrees_with_the_synthesis_path():
    """avsep_stft on the mixture waveform of dataset items reproduces the mixed_spec avsep_synth_batch makes (same
    framing and transform; the waveform here comes from the synthesis oracle, so allow the fp32 transform tolerance)."""
    _stft_matches_synthesis({})


def test_stft_magnitude_agrees_with_the_synthesis_path_radix2():
    """The same at n_fft = 256, where both run the radix-2 analysis kernel."""
    _stft_matches_synthesis(dict(sample_rate=16000, duration=0.5, n_fft=256, hop_length=64, num_frames=10, frame_h=16,
                                 frame_w=24, speaker_freqs=(200.0, 330.0, 512.0)))


@pytest.mark.parametrize("name", ("default", "short", "ragged"))
def test_istft_matches_oracle_with_masks(eng, name):
    z = np.load(GOLD)
    n_fft, hop = (int(v) for v in z[name + "_geom"])
    x = z[name + "_wave"]
    rng = np.random.default_rng(11)
    ref_spec = wo.stft_complex(x, n_fft, hop).astype(np.complex64)
    masks = rng.uniform(0, 1, (3,) + ref_spec.shape).astype(np.float32)
    want = wo.istft_masked(ref_spec, masks, len(x), n_fft, hop)
    got = eng.istft(torch.from_numpy(ref_spec).cuda()[None].contiguous(), torch.from_numpy(masks).cuda()[None].contiguous(),
                    len(x), n_fft, hop)
    assert got.shape == (1, 3, len(x))
    assert _wave_err(got[0].cpu().numpy(), want, n_fft, hop) <= TOL_WAVE


def test_istft_ignores_imaginary_dc_and_nyquist_like_irfft(eng):
    rng = np.random.default_rng(12)
    n_fft, hop, T = 64, 16, 12
    spec = (rng.standard_normal((2, n_fft // 2 + 1, T)) + 1j * rng.standard_normal((2, n_fft // 2 + 1, T))).astype(np.complex64)
    L = (T - 1) * hop + n_fft
    got = eng.istft(torch.from_numpy(spec).cuda(), None, L, n_fft, hop).cpu().numpy()
    for b in range(2):
        want = wo.istft_masked(spec[b], None, L, n_fft, hop, direct=True)
        assert _wave_err(got[b], want, n_fft, hop, T) <= TOL_WAVE
    assert (got[:, :, 0] == 0).all() and (got[:, :, L - 1] == 0).all()


@pytest.mark.parametrize("hop,L", [(128, 1000), (100, 2696), (64, 1500), (512, 4000), (300, 1000), (32, 900), (129, 127)])
def test_n_fft_512_geometries_match_oracle(eng, hop, L):
    """n_fft = 512 takes the register radix-8 kernels for hop >= 64 (any hop for the analysis) and the radix-2 ones
    below; hops that do not divide n_fft, a hop of a whole frame, and a signal shorter than one hop."""
    rng = np.random.default_rng(hop)
    x = (0.3 * rng.standard_normal((2, L))).astype(np.float32)
    spec, mag = eng.stft(torch.from_numpy(x).cuda(), 512, hop)
    T = 1 + L // hop
    assert spec.shape == (2, 257, T)
    masks = rng.uniform(0, 1, (2, 2, 257, T)).astype(np.float32)
    got = eng.istft(spec, torch.from_numpy(masks).cuda(), L, 512, hop).cpu().numpy()
    for b in range(2):
        ref = wo.stft_complex(x[b], 512, hop)
        assert np.abs(spec[b].cpu().numpy() - ref).max() <= TOL_SPEC_REL * np.abs(ref).max()
        want = wo.istft_masked(spec[b].cpu().numpy(), masks[b], L, 512, hop)
        assert _wave_err(got[b], want, 512, hop) <= TOL_WAVE


@pytest.mark.parametrize("B,L,n_fft,hop", [(256, 8000, 512, 128), (4, 160000, 512, 128), (3, 5000, 2048, 2048), (5, 777, 8, 3)])
def test_round_trip_and_mask_linearity_at_size(eng, B, L, n_fft, hop):
    g = torch.Generator(device="cuda").manual_seed(3)
    x = 0.3 * torch.randn(B, L, device="cuda", generator=g)
    spec, mag = eng.stft(x, n_fft, hop)
    T = 1 + L // hop
    if (T - 1) * hop + n_fft < L:
        pytest.skip("frames do not cover the signal")
    y = eng.istft(spec, None, L, n_fft, hop)[:, 0]
    w = torch.from_numpy(np.hanning(n_fft)).cuda()
    # samples every covering frame weights with exactly 0 cannot come back (n = 0; with hop == n_fft also frame ends)
    wss = torch.zeros((T - 1) * hop + n_fft, dtype=torch.float64, device="cuda")
    for i in range(T):
        wss[i * hop:i * hop + n_fft] += w * w
    ok = wss[:L] > 1e-11
    small = wss[:L] < 1e-3      # near-zero window sums amplify fp32 rounding: compare those loosely
    err = (y - x).abs()
    assert err[:, ok & ~small].max().item() <= 2e-5
    assert (y[:, ~ok] == 0).all()
    m0 = torch.rand(B, 1, n_fft // 2 + 1, T, device="cuda", generator=g)
    parts = eng.istft(spec, torch.cat([m0, 1 - m0], 1).contiguous(), L, n_fft, hop)
    assert (parts.sum(1) - y).abs()[:, ~small].max().item() <= 2e-5


def test_istft_rejects_bad_geometry(eng):
    spec = torch.zeros(1, 257, 4, dtype=torch.complex64, device="cuda")
    with pytest.raises(RuntimeError, match="do not reach"):
        eng.istft(spec, None, 5000, 512, 128)
    with pytest.raises(RuntimeError, match="power of two"):
        eng.istft(torch.zeros(1, 151, 4, dtype=torch.complex64, device="cuda"), None, 100, 300, 100)
    with pytest.raises(ValueError):
        eng.istft(spec.cpu(), None, 100, 512, 128)


def _forward_and_wide_stft(dev):
    """A default-model forward and an n_fft = 2048 STFT on cuda:dev (both launch kernels that need more than 48 KB of
    shared memory)."""
    from avsep_b200 import AVSeparationTransformer
    torch.manual_seed(0)
    model = AVSeparationTransformer().eval()
    g = torch.Generator().manual_seed(6)
    mixed, lips = torch.rand(2, 257, 63, generator=g), torch.rand(2, 50, 32, 32, generator=g)
    x = torch.randn(3, 6000, generator=g)
    sep, masks = model(mixed.to(dev), lips.to(dev))
    spec, mag = model.engine.stft(x.to(dev), 2048, 512)
    torch.cuda.synchronize(dev)
    return [t.cpu() for t in (sep, masks, spec, mag)]


def test_second_device_after_the_first_matches_a_fresh_process(tmp_path):
    """The shared-memory opt-in is per device: a process that ran on cuda:0 must still opt in on cuda:1."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import subprocess
    here = [_forward_and_wide_stft(0), _forward_and_wide_stft(1)]
    for dev in (0, 1):
        out = tmp_path / f"fresh{dev}.pt"
        code = (f"import sys; sys.path[:0] = {[ROOT, os.path.join(ROOT, 'av-separation-transformer_b200')]!r}; "
                f"import torch; from tests.test_waveform_gpu import _forward_and_wide_stft as f; "
                f"torch.save(f({dev}), {str(out)!r})")
        subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)
        fresh = torch.load(out)
        assert all(torch.equal(a, b) for a, b in zip(here[dev], fresh)), dev


def test_separate_waveforms_end_to_end():
    from avsep_b200 import AVSeparationTransformer
    torch.manual_seed(0)
    model = AVSeparationTransformer().eval()
    g = torch.Generator(device="cuda").manual_seed(4)
    wave = 0.3 * torch.randn(4, 8000, device="cuda", generator=g)
    lips = torch.rand(4, 50, 32, 32, device="cuda", generator=g)
    waves, masks = model.separate_waveforms(wave, lips)
    assert waves.shape == (4, 2, 8000) and masks.shape == (4, 2, 257, 63)
    # the same result assembled by hand from the public pieces and the oracle inverse
    spec, mag = model.engine.stft(wave, 512, 128)
    _, masks2 = model(mag, lips)
    assert torch.equal(masks, masks2)
    want = wo.istft_masked(spec[1].cpu().numpy(), masks[1].cpu().numpy(), 8000, 512, 128)
    assert _wave_err(waves[1].cpu().numpy(), want, 512, 128) <= TOL_WAVE
