"""GPU parity tests proper: the CUDA path (through the C ABI) against (a) the committed golden vectors produced by
the real reference, (b) the CPU oracle on the same seeded inputs, (c) size-independent properties at full size."""
import numpy as np
import pytest
import torch

from oracle import avsep_oracle as onp
from oracle import avsep_oracle_torch as otorch
from oracle.weights import CONFIGS, make_inputs, make_state_dict
from tests.helpers import (GOLDEN_CASES, STAGES, TOL, build_model, case_tensors, err_report, load_golden,
                           subsample_stage)

pytestmark = pytest.mark.gpu


def _run(model, mixed, frames):
    sep, masks = model(torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    return sep.cpu().numpy(), masks.cpu().numpy()


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_bf16_path_matches_reference_golden(name):
    z, meta = load_golden(name)
    cfg, P, mixed, frames = case_tensors(meta)
    model = build_model(cfg, P, "bf16")
    model.prepack()
    model.engine.set_debug(True)
    sep, masks = _run(model, mixed, frames)
    assert sep.shape == (meta["B"], cfg.num_speakers, cfg.freq_bins, meta["T"]) and masks.shape == sep.shape
    sf, st = meta["stride_f"], meta["stride_t"]
    rep = err_report(sep[:, :, ::sf, ::st], masks[:, :, ::sf, ::st], z["separated"], z["masks"], mixed[:, ::sf, ::st])
    stage_err = {}
    shapes = {"audio_embed": (meta["B"], meta["T"], cfg.d_model), "audio_enc": (meta["B"], meta["T"], cfg.d_model),
              "visual_pool": (meta["B"], meta["N"], 128), "visual_embed": (meta["B"], meta["N"], cfg.d_model),
              "visual_enc": (meta["B"], meta["N"], cfg.d_model), "fused": (meta["B"], meta["T"], cfg.d_model)}
    for k in STAGES:
        got = subsample_stage(model.engine.get_stage(k).reshape(shapes[k]))
        ref = z["stage_" + k]
        stage_err[k] = float(np.abs(got - ref).max() / max(1.0, np.abs(ref).max()))
    print(name, rep, stage_err)
    assert masks.min() >= 0.0 and masks.max() <= 1.0
    assert rep["masks"] < TOL["bf16"], (rep, stage_err)
    assert rep["separated_scaled"] < TOL["bf16"], (rep, stage_err)
    if meta["kind"] == "randn":
        assert rep["separated_abs"] < TOL["bf16"] * max(1.0, float(np.abs(mixed).max())), rep
    for k, v in stage_err.items():
        assert v < 5e-2, (k, v)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_tf32_path_matches_reference_golden(name):
    """fp32/TF32 path (north star: 1e-3): GEMMs on tcgen05 kind::tf32 with fp32 operands in HBM, attention and the
    CNN with bf16 hi/lo split contractions (fp32-grade), fp32 residual stream / LayerNorm / softmax."""
    z, meta = load_golden(name)
    cfg, P, mixed, frames = case_tensors(meta)
    model = build_model(cfg, P, "tf32")
    sep, masks = _run(model, mixed, frames)
    sf, st = meta["stride_f"], meta["stride_t"]
    rep = err_report(sep[:, :, ::sf, ::st], masks[:, :, ::sf, ::st], z["separated"], z["masks"], mixed[:, ::sf, ::st])
    print("tf32", name, rep)
    assert masks.min() >= 0.0 and masks.max() <= 1.0
    assert rep["masks"] < TOL["tf32"], rep
    assert rep["separated_scaled"] < TOL["tf32"], rep
    if meta["kind"] == "randn":     # unit-scale inputs: the north star's absolute bound on `separated` applies as is
        assert rep["separated_abs"] < TOL["tf32"] * max(1.0, float(np.abs(mixed).max())), rep


def test_against_live_oracle_other_seeds():
    cfg = CONFIGS["tiny2"]
    for seed in (21, 22):
        P = make_state_dict(cfg, seed=seed, gain=2.0)
        mixed, frames = make_inputs(cfg, 3, 40, 12, 16, 16, seed=seed, kind="randn")
        model = build_model(cfg, P, "bf16")
        sep, masks = _run(model, mixed, frames)
        sep_ref, masks_ref = onp.forward(P, cfg, mixed, frames)
        rep = err_report(sep, masks, sep_ref, masks_ref, mixed)
        assert rep["masks"] < TOL["bf16"] and rep["separated_scaled"] < TOL["bf16"], rep


def test_edge_shapes_batch1_short_sequences():
    cfg = CONFIGS["tiny"]
    P = make_state_dict(cfg, seed=31, gain=2.0)
    model = build_model(cfg, P, "bf16")
    for (B, T, N, Hh, Ww) in ((1, 1, 1, 8, 8), (1, 3, 2, 5, 7), (2, 130, 3, 16, 16), (1, 16, 64, 16, 16)):
        mixed, frames = make_inputs(cfg, B, T, N, Hh, Ww, seed=T, kind="randn")
        sep, masks = _run(model, mixed, frames)
        sep_ref, masks_ref = onp.forward(P, cfg, mixed, frames)
        rep = err_report(sep, masks, sep_ref, masks_ref, mixed)
        assert rep["masks"] < TOL["bf16"] and rep["separated_scaled"] < TOL["bf16"], ((B, T, N, Hh, Ww), rep)


def test_full_size_properties_and_batch_independence():
    """BASELINE.json configs[1] (B=256, default model): no op mixes utterances, so a shard of the batch must give
    bit-identical rows; separated == masks * mixed exactly; masks in [0,1]; spot-check rows against the CPU port."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=41, gain=2.0)
    B, T, N = 256, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=41, kind="dataset")
    model = build_model(cfg, P, "bf16")
    sep, masks = _run(model, mixed, frames)
    assert np.isfinite(sep).all() and masks.min() >= 0.0 and masks.max() <= 1.0
    assert np.array_equal(sep, masks * mixed[:, None])
    sub = slice(100, 132)
    sep_s, masks_s = _run(model, mixed[sub], frames[sub])
    assert np.array_equal(masks_s, masks[sub]) and np.array_equal(sep_s, sep[sub])
    idx = [0, 127, 255]
    sep_ref, masks_ref = otorch.forward(otorch.to_torch(P), cfg, torch.from_numpy(mixed[idx]), torch.from_numpy(frames[idx]))
    rep = err_report(sep[idx], masks[idx], sep_ref.numpy(), masks_ref.numpy(), mixed[idx])
    assert rep["masks"] < TOL["bf16"] and rep["separated_scaled"] < TOL["bf16"], rep


def test_more_tiles_than_sms_gives_the_same_rows():
    """B=700 utterances = 350 two-utterance tiles on 148 SMs: every CTA of the fused stack kernels walks several tiles
    (ring, barrier phases and stream offsets carried from tile to tile, input projection / K|V projection / decoder
    blocks included); any sub-batch computed alone must give bit-identical rows, and an odd batch leaves half a tile."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=43, gain=2.0)
    B, T, N = 701, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=43, kind="dataset")
    model = build_model(cfg, P, "bf16")
    sep, masks = _run(model, mixed, frames)
    assert np.isfinite(sep).all() and masks.min() >= 0.0 and masks.max() <= 1.0
    assert np.array_equal(sep, masks * mixed[:, None])
    for sub in (slice(0, 4), slice(296, 302), slice(690, 701)):
        sep_s, masks_s = _run(model, mixed[sub], frames[sub])
        assert np.array_equal(masks_s, masks[sub]) and np.array_equal(sep_s, sep[sub]), sub


def test_repeated_many_tile_forwards_are_stable():
    """Stress for ordering bugs between the kernel's roles that only show with several tiles per CTA and back-to-back
    graph replays (a ring-slot parity wait two phases behind hung 1 run in 3 here before the MMA role was made to
    observe the K|V bias block landing): 150 forwards of 1024 utterances, every result bit-identical to the first."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=44, gain=2.0)
    B, T, N = 1024, 63, 50
    mixed, frames = make_inputs(cfg, 64, T, N, 32, 32, seed=44, kind="dataset")
    model = build_model(cfg, P, "bf16")
    dev = torch.device("cuda")
    m = torch.from_numpy(mixed).to(dev).repeat(B // 64, 1, 1).contiguous()
    f = torch.from_numpy(frames).to(dev).repeat(B // 64, 1, 1, 1).contiguous()
    sep0, masks0 = model(m, f)
    sep0, masks0 = sep0.clone(), masks0.clone()
    assert torch.equal(masks0[:64], masks0[64:128])                  # the same utterances in other tiles of other CTAs
    for it in range(150):
        sep, masks = model(m, f)
        if it % 25 == 24:
            assert torch.equal(masks, masks0) and torch.equal(sep, sep0), it
    torch.cuda.synchronize()


def test_host_buffer_entry_point_matches_device_entry_point():
    cfg = CONFIGS["tiny2"]
    P = make_state_dict(cfg, seed=51, gain=2.0)
    mixed, frames = make_inputs(cfg, 4, 32, 10, 16, 16, seed=51, kind="randn")
    model = build_model(cfg, P, "bf16")
    sep_d, masks_d = _run(model, mixed, frames)
    sep_h, masks_h = model(torch.from_numpy(mixed).pin_memory(), torch.from_numpy(frames).pin_memory())
    assert not sep_h.is_cuda
    assert np.array_equal(sep_h.numpy(), sep_d) and np.array_equal(masks_h.numpy(), masks_d)


@pytest.mark.parametrize("chunk,lanes", [(3, 1), (3, 2), (4, 3), (16, 2)])
def test_host_path_chunks_and_lanes(chunk, lanes):
    """avsep_forward_host pipelines chunks of the batch over several compute lanes: same results as one device call."""
    cfg = CONFIGS["tiny2"]
    P = make_state_dict(cfg, seed=52, gain=2.0)
    mixed, frames = make_inputs(cfg, 10, 32, 10, 16, 16, seed=52, kind="randn")
    model = build_model(cfg, P, "bf16")
    sep_d, masks_d = _run(model, mixed, frames)
    model.engine.set_option("host_chunk", chunk)
    model.engine.set_option("host_lanes", lanes)
    for _ in range(3):      # eager, capture, replay
        sep_h, masks_h = model(torch.from_numpy(mixed).pin_memory(), torch.from_numpy(frames).pin_memory())
        assert np.array_equal(sep_h.numpy(), sep_d) and np.array_equal(masks_h.numpy(), masks_d)


def test_host_path_streaming_slots_overlap_safely():
    """avsep_forward_host_async on alternating slots: every batch of a stream equals its synchronous result, also when
    a slot is resubmitted without an explicit wait in between (the device-side ordering protects its buffers)."""
    cfg = CONFIGS["tiny2"]
    P = make_state_dict(cfg, seed=53, gain=2.0)
    model = build_model(cfg, P, "bf16")
    model.prepack()
    eng = model.engine
    eng.set_option("host_chunk", 4)
    batches = []
    for i in range(6):
        mixed, frames = make_inputs(cfg, 9, 32, 10, 16, 16, seed=100 + i, kind="randn")
        mt, ft = torch.from_numpy(mixed).pin_memory(), torch.from_numpy(frames).pin_memory()
        ref = eng.forward_host(mt, ft)
        batches.append((mt, ft, ref[0].clone(), ref[1].clone()))
    outs = [(torch.empty_like(b[2]).pin_memory(), torch.empty_like(b[3]).pin_memory()) for b in batches]
    for rounds in range(2):
        for i, (mt, ft, _, _) in enumerate(batches):
            eng.forward_host_async(mt, ft, outs[i][0], outs[i][1], i % 2)
        eng.host_wait(0)
        eng.host_wait(1)
        for (mt, ft, rs, rm), (os_, om) in zip(batches, outs):
            assert torch.equal(os_, rs) and torch.equal(om, rm)
            os_.zero_(); om.zero_()
    # slots 2 and 3 exist too (AVSEP_HOST_SLOTS = 4): the same batch through one of them, then an index past the end
    eng.forward_host_async(batches[1][0], batches[1][1], outs[1][0], outs[1][1], 3)
    eng.host_wait(3)
    assert torch.equal(outs[1][0], batches[1][2]) and torch.equal(outs[1][1], batches[1][3])
    for bad in (4, -1):
        with pytest.raises(RuntimeError, match="slot"):
            eng.forward_host_async(batches[0][0], batches[0][1], outs[0][0], outs[0][1], bad)


def test_submodule_dropins_match_oracle():
    """Reference tests drive the sub-modules directly (tests/test_model.py:77-179), incl. F=65, hd=16, N=10 -> T=50/20."""
    from avsep_b200 import AudioEncoder, CrossModalFusion, SeparationDecoder, VisualEncoder
    cfg = CONFIGS["tiny"]
    P = make_state_dict(cfg, seed=61, gain=2.0)
    mixed, frames = make_inputs(cfg, 2, 32, 10, 16, 16, seed=61, kind="randn")
    tt = lambda pre: {k[len(pre):]: torch.from_numpy(np.asarray(v)) for k, v in P.items() if k.startswith(pre)}
    ae = AudioEncoder(cfg.freq_bins, cfg.d_model, cfg.nhead, cfg.num_encoder_layers)
    ae.load_state_dict(tt("audio_encoder."))
    a = ae.cuda()(torch.from_numpy(mixed).cuda()).cpu().numpy()
    a_ref = onp.audio_encoder(P, cfg, mixed)
    assert a.shape == (2, 32, cfg.d_model) and np.abs(a - a_ref).max() < 5e-2 * max(1, np.abs(a_ref).max())
    ve = VisualEncoder(cfg.d_model, cfg.nhead, cfg.num_encoder_layers)
    ve.load_state_dict(tt("visual_encoder."))
    ve = ve.cuda()
    for target in (20, 32, 50):
        v = ve(torch.from_numpy(frames).cuda(), target_len=target).cpu().numpy()
        v_ref = onp.visual_encoder(P, cfg, frames, target)
        assert v.shape == (2, target, cfg.d_model) and np.abs(v - v_ref).max() < 5e-2 * max(1, np.abs(v_ref).max())
    fu = CrossModalFusion(cfg.d_model, cfg.nhead, cfg.num_fusion_layers)
    fu.load_state_dict(tt("fusion."))
    v32 = onp.visual_encoder(P, cfg, frames, 32)
    f = fu.cuda()(torch.from_numpy(a_ref).cuda(), torch.from_numpy(v32).cuda()).cpu().numpy()
    f_ref = onp.fusion(P, cfg, a_ref, v32)
    assert np.abs(f - f_ref).max() < 5e-2 * max(1, np.abs(f_ref).max())
    de = SeparationDecoder(cfg.d_model, cfg.freq_bins, cfg.num_speakers)
    de.load_state_dict(tt("decoder."))
    m = de.cuda()(torch.from_numpy(f_ref).cuda()).cpu().numpy()
    m_ref = onp.decoder_masks(P, cfg, f_ref)
    assert m.shape == (2, 2, cfg.freq_bins, 32) and np.abs(m - m_ref).max() < TOL["bf16"]
    assert m.min() >= 0 and m.max() <= 1


def test_errors_are_loud():
    cfg = CONFIGS["tiny"]
    P = make_state_dict(cfg, seed=1)
    model = build_model(cfg, P, "bf16")
    with pytest.raises(ValueError):
        model(torch.zeros(1, 64, 8, device="cuda"), torch.zeros(1, 4, 16, 16, device="cuda"))   # wrong freq_bins
    with pytest.raises(RuntimeError):
        model(torch.zeros(1, 65, 5001, device="cuda"), torch.zeros(1, 4, 16, 16, device="cuda"))  # > PE table


@pytest.mark.parametrize("option", ["use_graph", "two_stream", "pdl"])
@pytest.mark.parametrize("name", ["c1_dataset", "c3_long", "c4_scaled"])
def test_alternative_execution_paths_agree(name, option):
    """Every on/off execution option of the library (eager launches, one stream, plain stream order) must stay
    parity-green on each kernel path: the fused stack kernels (c1_dataset), the per-layer kernels with tcgen05
    attention (c3_long, T=1251) and with the add+LayerNorm kernel and unfused FFN (c4_scaled, d=512)."""
    z, meta = load_golden(name)
    cfg, P, mixed, frames = case_tensors(meta)
    model = build_model(cfg, P, "bf16")
    model.prepack()
    model.engine.set_option(option, 0)
    try:
        for _ in range(3):                       # 3 calls: eager warm-up, graph capture, graph replay
            sep, masks = _run(model, mixed, frames)
        sf, st = meta["stride_f"], meta["stride_t"]
        rep = err_report(sep[:, :, ::sf, ::st], masks[:, :, ::sf, ::st], z["separated"], z["masks"], mixed[:, ::sf, ::st])
        assert rep["masks"] < TOL["bf16"] and rep["separated_scaled"] < TOL["bf16"], (option, rep)
    finally:
        model.engine.set_option(option, 1)


def test_removed_options_are_unknown():
    """Names of retired A/B switches fail like any unknown option: the kernels they chose follow from the configuration
    and the shapes."""
    from avsep_b200.engine import Engine, EngineConfig
    eng = Engine(EngineConfig(**CONFIGS["tiny"].as_dict()), 0)
    try:
        for name in ("cnn_ig", "fuse_ln", "epilogue_tma", "cnn_tc", "attn_small", "attn_tc_min_len", "fuse_ffn",
                     "ffn_fused_min_rows", "fuse_stack", "fuse_proj", "fuse_kvp", "fuse_decoder"):
            with pytest.raises(RuntimeError, match="unknown option"):
                eng.set_option(name, 0)
    finally:
        eng.close()


@pytest.mark.parametrize("attn_tc", [0, 1])
def test_long_form_attention_paths_agree(attn_tc):
    """Long-form case (T=1251, N=500): the tcgen05 attention kernel (+ materialised K/V interpolation) and the
    mma.sync kernel (interpolation on load) are both parity-green against the reference golden."""
    z, meta = load_golden("c3_long")
    cfg, P, mixed, frames = case_tensors(meta)
    model = build_model(cfg, P, "bf16")
    model.prepack()
    model.engine.set_option("attn_tc", attn_tc)
    try:
        for _ in range(3):
            sep, masks = _run(model, mixed, frames)
        sf, st = meta["stride_f"], meta["stride_t"]
        rep = err_report(sep[:, :, ::sf, ::st], masks[:, :, ::sf, ::st], z["separated"], z["masks"], mixed[:, ::sf, ::st])
        assert rep["masks"] < TOL["bf16"] and rep["separated_scaled"] < TOL["bf16"], (attn_tc, rep)
    finally:
        model.engine.set_option("attn_tc", 1)


def test_graph_replay_is_bit_identical_to_eager():
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=71, gain=2.0)
    mixed, frames = make_inputs(cfg, 8, 63, 50, 32, 32, seed=71, kind="dataset")
    model = build_model(cfg, P, "bf16")
    m_t, f_t = torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda()
    model.prepack()
    model.engine.set_option("use_graph", 0)
    sep_e, masks_e = model(m_t, f_t)
    model.engine.set_option("use_graph", 1)
    outs = [model(m_t, f_t) for _ in range(4)]
    torch.cuda.synchronize()
    for sep_g, masks_g in outs:
        assert torch.equal(masks_g, masks_e) and torch.equal(sep_g, sep_e)
