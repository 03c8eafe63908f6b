"""Which kernels each forward path launches: one profiled forward per path, its label -> launch-count map pinned
against a table.  Whether a stage runs as a whole-stack kernel or as per-layer kernels, and whether the input
projections, the fusion K|V projection and the decoder run inside the stack kernels, follows from the configuration,
the precision, the sequence lengths and the debug flag."""
import pytest
import torch

from oracle import avsep_oracle as onp
from oracle.weights import CONFIGS, ModelConfig, make_inputs, make_state_dict
from tests.helpers import TOL, build_model, err_report

pytestmark = pytest.mark.gpu

# d = 256 with 3 speakers: the fusion stack kernel runs, but its fused decoder supports 1, 2 or 4 speakers only
D256_S3 = ModelConfig(257, 256, 4, 2, 2, 3)

FUSED = {"prep_audio": 1, "gemm.conv1d_0": 1, "visual_cnn": 1, "layer.visual_enc": 1, "layer.audio_enc": 1}

# name: (config, precision, B, T, N, frame side, debug, attn_tc, expected launches per profile label)
CASES = {
    # every stage in a stack kernel, input projections, K|V projection and decoder included
    "default": (CONFIGS["default"], "bf16", 8, 63, 50, 32, False, None, {**FUSED, "layer.fusion_decoder": 1}),
    # stage snapshots: projections, K|V rows and decoder outside the stack kernels
    "default_debug": (CONFIGS["default"], "bf16", 8, 63, 50, 32, True, None,
                      {**FUSED, "gemm.frame_proj": 1, "gemm.conv1d_2": 1, "lerp_kv": 1, "gemm.cross_kv": 1,
                       "layer.fusion": 1, "gemm.dec0": 1, "gemm.dec3_tail": 1}),
    # 100 audio frames do not fit the tile slot of 50 visual rows: K|V projection outside the visual stack
    "default_100_50": (CONFIGS["default"], "bf16", 8, 100, 50, 32, False, None,
                       {**FUSED, "lerp_kv": 1, "gemm.cross_kv": 1, "layer.fusion_decoder": 1}),
    # 300 audio frames exceed a stack tile: visual stack kernel, per-layer audio encoder and fusion (tcgen05 attention)
    "default_300_120_tc": (CONFIGS["default"], "bf16", 8, 300, 120, 32, False, 1,
                           {"visual_cnn": 1, "layer.visual_enc": 1, "prep_audio": 1, "gemm.conv1d_0": 1,
                            "gemm.conv1d_2": 1, "gemm.qkv": 2, "attn.self": 2, "gemm.out_proj": 4, "ffn.fused": 4,
                            "gemm.cross_kv": 1, "gemm.cross_q": 2, "lerp_kv": 2, "attn.cross": 2, "gemm.dec0": 1,
                            "gemm.dec3_tail": 1}),
    "d256_s3": (D256_S3, "bf16", 8, 63, 50, 32, False, None,
                {**FUSED, "layer.fusion": 1, "gemm.dec0": 1, "gemm.dec3_tail": 1}),
    # per-layer paths: d = 512 (residual add + LayerNorm as its own kernel), head dim 16, TF32
    "scaled": (CONFIGS["scaled"], "bf16", 8, 63, 50, 32, False, None,
               {"visual_cnn": 1, "gemm.frame_proj": 1, "prep_audio": 1, "gemm.conv1d_0": 1, "gemm.conv1d_2": 1,
                "gemm.qkv": 12, "attn.self": 12, "gemm.out_proj": 18, "gemm.ffn1": 18, "gemm.ffn2": 18,
                "add_layernorm": 38, "gemm.cross_kv": 1, "gemm.cross_q": 6, "attn.cross": 6, "gemm.dec0": 1,
                "gemm.dec3_tail": 1}),
    "tiny": (CONFIGS["tiny"], "bf16", 8, 63, 50, 16, False, None,
             {"visual_cnn": 1, "gemm.frame_proj": 1, "prep_audio": 1, "gemm.conv1d_0": 1, "gemm.conv1d_2": 1,
              "gemm.qkv": 2, "attn.self": 2, "gemm.out_proj": 3, "gemm.ffn1": 3, "gemm.ffn2": 3, "gemm.cross_kv": 1,
              "gemm.cross_q": 1, "attn.cross": 1, "gemm.dec0": 1, "gemm.dec3_tail": 1}),
    "default_tf32": (CONFIGS["default"], "tf32", 8, 63, 50, 32, False, None,
                     {"visual_cnn": 1, "gemm.frame_proj": 1, "prep_audio": 1, "gemm.conv1d_0": 1, "gemm.conv1d_2": 1,
                      "gemm.qkv": 4, "attn.self": 4, "gemm.out_proj": 6, "gemm.ffn1": 6, "gemm.ffn2": 6,
                      "gemm.cross_kv": 1, "gemm.cross_q": 2, "attn.cross": 2, "gemm.dec0": 1, "gemm.dec3_tail": 1}),
}


def _setup(cfg, prec, B, T, N, side, seed=71):
    P = make_state_dict(cfg, seed=seed, gain=2.0)
    mixed, frames = make_inputs(cfg, B, T, N, side, side, seed=seed, kind="dataset")
    return P, build_model(cfg, P, prec), mixed, frames


def _run(model, mixed, frames):
    sep, masks = model(torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    return sep.cpu().numpy(), masks.cpu().numpy()


@pytest.mark.parametrize("name", list(CASES))
def test_launches_per_path(name):
    cfg, prec, B, T, N, side, debug, attn_tc, want = CASES[name]
    P, model, mixed, frames = _setup(cfg, prec, B, T, N, side)
    model.prepack()
    eng = model.engine
    eng.set_debug(debug)
    if attn_tc is not None:
        eng.set_option("attn_tc", attn_tc)
    eng.set_profile(True)
    eng.profile_report(reset=True)
    _run(model, mixed, frames)
    got = {label: n for label, (n, _) in eng.profile_report(reset=True).items()}
    eng.set_profile(False)
    assert got == want, (name, got)
    assert eng.launch_count() == sum(want.values()), (name, eng.launch_count())


def test_d256_three_speakers_against_oracle():
    """The fused fusion stack followed by the per-layer decoder (debug off)."""
    P, model, mixed, frames = _setup(D256_S3, "bf16", 2, 63, 50, 32)
    sep, masks = _run(model, mixed, frames)
    sep_ref, masks_ref = onp.forward(P, D256_S3, mixed, frames)
    rep = err_report(sep, masks, sep_ref, masks_ref, mixed)
    assert rep["masks"] < TOL["bf16"] and rep["separated_scaled"] < TOL["bf16"], rep
