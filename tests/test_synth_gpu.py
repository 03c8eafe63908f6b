"""GPU parity of the rows either side of the path (SURVEY 8f ranks 1, 3): avsep_synth_batch / avsep_eval_snr through
the C ABI against the reference's own items (tests/golden/synth_items.npz) and the oracle."""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "av-separation-transformer_b200"))
from oracle import synth_oracle as so   # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
WIDE_KW = dict(sample_rate=16000, duration=0.5, n_fft=256, hop_length=64, num_frames=10, frame_h=16, frame_w=24,
               speaker_freqs=(200.0, 330.0, 512.0))
# magnitudes reach ~130; fp32 FFT rounding differs between pocketfft and the in-kernel radix-2 transform
TOL_SPEC_REL = 2e-6
TOL_FRAMES = 2e-6


def _ds(**kw):
    from avsep_b200.dataset import SyntheticAVDataset
    return SyntheticAVDataset(**kw)


@pytest.mark.parametrize("cname,kw,idxs", [("default", {}, (0, 1, 7, 123)), ("wide", WIDE_KW, (3, 4))])
def test_synth_matches_reference_items(cname, kw, idxs):
    z = np.load(os.path.join(GOLD, "synth_items.npz"))
    ds = _ds(**kw)
    b = ds.batch(idxs)
    torch.cuda.synchronize()
    for i, idx in enumerate(idxs):
        for k in ("mixed_spec", "clean_specs"):
            ref = z[f"{cname}_{idx}_{k}"]
            got = b[k][i].cpu().numpy()
            assert got.shape == ref.shape
            err = np.abs(got - ref).max()
            assert err <= TOL_SPEC_REL * np.abs(ref).max() + 2e-5, (cname, idx, k, err, np.abs(ref).max())
        ref = z[f"{cname}_{idx}_lip_frames"]
        got = b["lip_frames"][i].cpu().numpy()
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() <= TOL_FRAMES, (cname, idx)
        assert np.array_equal(got == 0, ref == 0)          # zero border, same clip-to-zero pixels


def test_synth_against_oracle_larger_batch_and_item_interface():
    cfg = so.SynthConfig()
    ds = _ds()
    idxs = list(range(200, 232))
    b = ds.batch(idxs, want_clean=False)
    assert "clean_specs" not in b
    torch.cuda.synchronize()
    for i in (0, 13, 31):
        ref = so.synth_item(cfg, idxs[i])
        assert np.abs(b["mixed_spec"][i].cpu().numpy() - ref["mixed_spec"]).max() <= 3e-4
        assert np.abs(b["lip_frames"][i].cpu().numpy() - ref["lip_frames"]).max() <= TOL_FRAMES
    item = ds[5]
    ref = so.synth_item(cfg, 5)
    assert tuple(item["mixed_spec"].shape) == (257, 63) and tuple(item["lip_frames"].shape) == (50, 32, 32)
    assert tuple(item["clean_specs"].shape) == (2, 257, 63)
    assert np.abs(item["clean_specs"].cpu().numpy() - ref["clean_specs"]).max() <= 3e-4


def test_synth_feeds_the_forward_and_loud_errors():
    from avsep_b200 import AVSeparationTransformer
    ds = _ds()
    m = AVSeparationTransformer().cuda().eval()
    b = ds.batch(range(4))
    sep, masks = m(b["mixed_spec"], b["lip_frames"])
    assert tuple(sep.shape) == (4, 2, 257, 63) and torch.isfinite(sep).all()
    assert torch.allclose(sep, masks * b["mixed_spec"][:, None], atol=1e-4)
    bad = _ds(n_fft=500)
    with pytest.raises(RuntimeError, match="power of two"):
        bad.batch([0])


def test_eval_snr_matches_reference_scalars_and_oracle():
    from avsep_b200.engine import Engine, EngineConfig
    with open(os.path.join(GOLD, "synth_snr.json")) as f:
        gold = json.load(f)["snr"]
    eng = Engine(EngineConfig(257, 64, 4, 1, 1, 2, "bf16"), 0)
    cfg = so.SynthConfig()
    seps, tgs, mixes = [], [], []
    for idx_s in gold:
        idx = int(idx_s)
        item = so.synth_item(cfg, idx)
        tg = item["clean_specs"]
        rng = np.random.default_rng(100 + idx)
        seps.append((tg[::-1] * rng.uniform(0.7, 1.1, tg.shape) + rng.normal(0, 0.3, tg.shape)).astype(np.float32))
        tgs.append(tg); mixes.append(item["mixed_spec"])
    sep = torch.from_numpy(np.stack(seps)).cuda(); tg = torch.from_numpy(np.stack(tgs)).cuda()
    mx = torch.from_numpy(np.stack(mixes)).cuda()
    i_snr, o_snr, perm, si = eng.eval_snr(sep, tg, mx)
    torch.cuda.synchronize()
    for i, (idx_s, e) in enumerate(gold.items()):
        assert np.allclose(i_snr[i].cpu().numpy(), e["input_snr"], atol=2e-5)
        assert abs(float(o_snr[i]) - e["perm_snr"]) < 2e-5
        assert int(perm[i]) == 1 * 4 + 0                     # separated channels were swapped: perm = (1, 0)
        assert abs(float(si[i]) - float(so.si_snr_rows(seps[i][None], tgs[i][None])[0])) < 1e-3
    # three speakers, no mixture, identity best permutation, random data vs the oracle
    rng = np.random.default_rng(0)
    tg3 = rng.normal(0, 1, (5, 3, 33, 17)).astype(np.float32)
    sep3 = (tg3[:, [2, 0, 1]] + 0.1 * rng.normal(0, 1, tg3.shape)).astype(np.float32)
    i3, o3, p3, s3 = eng.eval_snr(torch.from_numpy(sep3).cuda(), torch.from_numpy(tg3).cuda(), None)
    assert i3 is None
    for b in range(5):
        assert abs(float(o3[b]) - so.permutation_snr(sep3[b], tg3[b])) < 2e-5
        assert int(p3[b]) == (1 * 16 + 2 * 4 + 0)            # target 0 <- channel 1, target 1 <- channel 2, target 2 <- channel 0
        assert abs(float(s3[b]) - float(so.si_snr_rows(sep3[b][None], tg3[b][None])[0])) < 1e-3
    with pytest.raises(RuntimeError, match="num_speakers"):
        eng.eval_snr(torch.zeros(1, 5, 4, 4).cuda(), torch.zeros(1, 5, 4, 4).cuda(), None)
    eng.close()


def test_evaluate_separation_mirror_runs_on_device():
    from avsep_b200 import AVSeparationTransformer, evaluate_separation
    ds = _ds(num_samples=8)
    m = AVSeparationTransformer().cuda().eval()
    in_snr, out_snr = evaluate_separation(m, ds, num_eval=8, batch_size=4)
    cfg = so.SynthConfig()
    ref_in = np.mean([so.input_snrs(it["mixed_spec"], it["clean_specs"]) for it in (so.synth_item(cfg, i) for i in range(8))])
    assert abs(in_snr - ref_in) < 1e-4
    assert np.isfinite(out_snr)


def _synth_item_matches_oracle(kw, idx):
    """One item of the device synthesis at geometry kw against the synthesis oracle; returns (dataset, batch)."""
    cfg = so.SynthConfig(**kw)
    ds = _ds(**kw)
    b = ds.batch([idx])
    torch.cuda.synchronize()
    ref = so.synth_item(cfg, idx)
    for k in ("mixed_spec", "lip_frames", "clean_specs"):
        got = b[k][0].cpu().numpy()
        assert got.shape == ref[k].shape, k
        assert np.abs(got - ref[k]).max() <= 2e-6 * max(1.0, np.abs(ref[k]).max()) + 2e-5, k
    return ds, b


def test_synth_and_snr_edge_geometries():
    """Single speaker, tiny FFT, one item, more video frames than fit evenly; SNR with one speaker."""
    kw = dict(sample_rate=4000, duration=0.25, n_fft=64, hop_length=16, num_frames=7, frame_h=8, frame_w=12,
              speaker_freqs=(300.0,))
    ds, b = _synth_item_matches_oracle(kw, 11)
    eng = ds.engine
    tg = b["clean_specs"]
    sep = (tg * 0.9).contiguous()
    i_snr, o_snr, perm, si = eng.eval_snr(sep, tg, b["mixed_spec"])
    assert abs(float(o_snr[0]) - so.permutation_snr(sep[0].cpu().numpy(), tg[0].cpu().numpy())) < 2e-5
    assert int(perm[0]) == 0
    assert abs(float(i_snr[0, 0]) - so.input_snrs(b["mixed_spec"][0].cpu().numpy(), tg[0].cpu().numpy())[0]) < 2e-5


def test_synth_at_the_largest_transform():
    """n_fft = 2048, whose analysis needs more than the default 48 KB of shared memory."""
    _synth_item_matches_oracle(dict(sample_rate=8000, duration=1.0, n_fft=2048, hop_length=512, num_frames=7,
                                    frame_h=8, frame_w=12, speaker_freqs=(300.0,)), 11)


def test_synth_scratch_growth_leaves_the_host_workspace_alone():
    """One handle serving both the host-buffer forward and the synthesis: growing the synthesis scratch must not
    touch the forward's workspace (regression: it used to free it)."""
    from avsep_b200 import AVSeparationTransformer, SyntheticAVDataset
    torch.manual_seed(0)
    model = AVSeparationTransformer(d_model=64, nhead=4, num_encoder_layers=1, num_fusion_layers=1).eval()
    g = torch.Generator().manual_seed(1)
    mixed = torch.rand(3, 257, 63, generator=g)
    frames = torch.rand(3, 50, 32, 32, generator=g)
    sep0, masks0 = (t.clone() for t in model(mixed, frames))          # CPU tensors -> avsep_forward_host
    ds = SyntheticAVDataset(engine=model.engine)
    ds.batch(range(2))
    ds.batch(range(24))                                               # scratch grows
    torch.cuda.synchronize()
    sep1, masks1 = model(mixed, frames)
    assert torch.equal(masks0, masks1) and torch.equal(sep0, sep1)
