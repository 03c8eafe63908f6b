"""The checks of the reference project's own test file (AV-Separation-Transformer, tests/test_model.py) on the
inference path, restated against whatever ``av_separation`` resolves to.

tests/test_reference_conformance_gpu.py runs this file in a fresh interpreter with the B200 drop-in first on the
path; it is not collected by a plain ``pytest tests`` (it needs a GPU and that import setup).  Like the reference's
tests, it builds every module at the reference's tiny shapes (F=65, T=32, d=64, 4 heads, B=2, 10 lip frames of 16x16,
2 speakers), calls it with CPU tensors and checks shapes, value ranges and which input an output depends on; the
values themselves are pinned by the golden vectors under tests/golden.  The reference's gradient, loss and
training-step tests are not restated: this build implements the forward path only.
"""
import pytest
import torch

from av_separation import AVSeparationTransformer, SyntheticAVDataset
from av_separation.model import (AudioEncoder, CrossModalFusion, PositionalEncoding, SeparationDecoder,
                                 VisualEncoder)

FREQ_BINS, T, D_MODEL, NHEAD, BATCH, NUM_FRAMES, H, W, NUM_SPEAKERS = 65, 32, 64, 4, 2, 10, 16, 16, 2


@pytest.fixture(autouse=True)
def _seed():
    torch.manual_seed(0)


def _mixed(t=T):
    return torch.randn(BATCH, FREQ_BINS, t).abs()


def _frames(n=NUM_FRAMES):
    return torch.rand(BATCH, n, H, W)


class TestPositionalEncoding:
    def test_output_shape(self):
        x = torch.randn(BATCH, T, D_MODEL)
        assert PositionalEncoding(D_MODEL)(x).shape == x.shape

    def test_encoding_is_nonzero(self):
        assert PositionalEncoding(D_MODEL)(torch.zeros(1, T, D_MODEL)).abs().sum() > 0


class TestAudioEncoder:
    def test_output_shape(self):
        enc = AudioEncoder(FREQ_BINS, D_MODEL, NHEAD, num_layers=2)
        out = enc(_mixed())
        assert out.shape == (BATCH, T, D_MODEL) and torch.isfinite(out).all()

    @pytest.mark.parametrize("t", [16, 32, 64])
    def test_variable_lengths(self, t):
        assert AudioEncoder(FREQ_BINS, D_MODEL, NHEAD, num_layers=2)(_mixed(t)).shape == (BATCH, t, D_MODEL)


class TestVisualEncoder:
    def test_output_shape(self):
        out = VisualEncoder(D_MODEL, NHEAD, num_layers=2)(_frames(), target_len=T)
        assert out.shape == (BATCH, T, D_MODEL) and torch.isfinite(out).all()

    @pytest.mark.parametrize("target_len", [20, 32, 50])     # 10 lip frames: down- and up-sampled in time
    def test_target_lengths(self, target_len):
        out = VisualEncoder(D_MODEL, NHEAD, num_layers=2)(_frames(), target_len=target_len)
        assert out.shape == (BATCH, target_len, D_MODEL)


class TestCrossModalFusion:
    def test_output_shape(self):
        fusion = CrossModalFusion(D_MODEL, NHEAD, num_layers=2)
        out = fusion(torch.randn(BATCH, T, D_MODEL), torch.randn(BATCH, T, D_MODEL))
        assert out.shape == (BATCH, T, D_MODEL) and torch.isfinite(out).all()

    def test_output_depends_on_visual(self):
        fusion = CrossModalFusion(D_MODEL, NHEAD, num_layers=2)
        audio = torch.randn(BATCH, T, D_MODEL)
        a = fusion(audio, torch.randn(BATCH, T, D_MODEL))
        b = fusion(audio, torch.randn(BATCH, T, D_MODEL))
        assert not torch.allclose(a, b)


class TestSeparationDecoder:
    def test_mask_shape(self):
        dec = SeparationDecoder(D_MODEL, FREQ_BINS, NUM_SPEAKERS)
        assert dec(torch.randn(BATCH, T, D_MODEL)).shape == (BATCH, NUM_SPEAKERS, FREQ_BINS, T)

    def test_masks_in_unit_range(self):
        masks = SeparationDecoder(D_MODEL, FREQ_BINS, NUM_SPEAKERS)(10.0 * torch.randn(BATCH, T, D_MODEL))
        assert masks.min() >= 0.0 and masks.max() <= 1.0

    def test_separate(self):
        dec = SeparationDecoder(D_MODEL, FREQ_BINS, NUM_SPEAKERS)
        masks, mixed = torch.rand(BATCH, NUM_SPEAKERS, FREQ_BINS, T), _mixed()
        sep = dec.separate(masks, mixed)
        assert sep.shape == (BATCH, NUM_SPEAKERS, FREQ_BINS, T)
        assert torch.equal(sep, masks * mixed.unsqueeze(1))


class TestAVSeparationTransformer:
    def _model(self):
        return AVSeparationTransformer(freq_bins=FREQ_BINS, d_model=D_MODEL, nhead=NHEAD, num_encoder_layers=2,
                                       num_fusion_layers=2, num_speakers=NUM_SPEAKERS)

    def test_forward_shapes(self):
        sep, masks = self._model()(_mixed(), _frames())
        assert sep.shape == masks.shape == (BATCH, NUM_SPEAKERS, FREQ_BINS, T)
        assert torch.isfinite(sep).all() and torch.isfinite(masks).all()

    def test_masks_in_unit_range(self):
        _, masks = self._model()(_mixed(), _frames())
        assert masks.min() >= 0.0 and masks.max() <= 1.0

    def test_separated_is_masks_times_mixture(self):
        mixed = _mixed()
        sep, masks = self._model()(mixed, _frames())
        assert torch.allclose(sep, masks * mixed.unsqueeze(1), rtol=1e-5, atol=1e-5)

    @pytest.mark.parametrize("t", [16, 32, 64])
    def test_variable_lengths(self, t):
        sep, masks = self._model()(_mixed(t), _frames())
        assert sep.shape == masks.shape == (BATCH, NUM_SPEAKERS, FREQ_BINS, t)


class TestSyntheticAVDataset:
    def _ds(self):
        return SyntheticAVDataset(num_samples=10)

    def test_length(self):
        assert len(self._ds()) == 10

    def test_item_shapes(self):
        ds = self._ds()
        item = ds[0]
        assert set(item) == {"mixed_spec", "lip_frames", "clean_specs"}
        assert item["mixed_spec"].shape == (ds.freq_bins, ds.T)
        assert item["lip_frames"].shape == (ds.num_speakers * ds.num_frames, ds.frame_h, ds.frame_w)
        assert item["clean_specs"].shape == (ds.num_speakers, ds.freq_bins, ds.T)

    def test_lip_frames_in_unit_range(self):
        lips = self._ds()[3]["lip_frames"]
        assert lips.min() >= 0.0 and lips.max() <= 1.0

    def test_items_are_deterministic_per_index(self):
        ds = self._ds()
        a, b = ds[4], ds[4]
        assert all(torch.equal(a[k], b[k]) for k in a)

    def test_items_differ(self):
        ds = self._ds()
        assert not torch.equal(ds[0]["mixed_spec"], ds[1]["mixed_spec"])

    def test_dataloader_collates_batches(self):
        ds = self._ds()
        batch = next(iter(torch.utils.data.DataLoader(ds, batch_size=4)))
        assert batch["mixed_spec"].shape == (4, ds.freq_bins, ds.T)
        assert batch["lip_frames"].shape == (4, ds.num_speakers * ds.num_frames, ds.frame_h, ds.frame_w)
