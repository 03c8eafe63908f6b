"""HBM rate of avsep_separate (SeparationDecoder.separate, model.py:210-220) at the benchmark shapes: algorithmic bytes
(masks in + mixture in + separated out = 4*F*T*(2S+1) per utterance) / device time, CUDA events, rotating buffer sets
larger than L2, against MEASURED_PEAKS.json's copy bandwidth where that file exists.  Also the shape of the 8-GPU root
rebuild (7 x 256).

Length arms (avsep_separate_varlen): every length full, and the seeded ragged batch of tools/waveform_varlen_bench.py
(T_b uniform in [16, 63]).  A ragged call reads masks and mixture only below each length and still writes the whole
padded output, so its algorithmic bytes are 4*F*(S+1)*sum(T_b) + 4*S*F*T*B.  Every line names the card and its power
limit."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(ROOT, "av-separation-transformer_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from avsep_b200.engine import Engine, EngineConfig   # noqa: E402
from varlen_bench import card_info   # noqa: E402

F, S, T = 257, 2, 63
eng = Engine(EngineConfig(F, 256, 4, 2, 2, S), 0)
peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
peak = json.load(open(peaks))["hbm_gbs"] if os.path.exists(peaks) else None
card, power_w = card_info(0)
st = torch.cuda.current_stream().cuda_stream
for B in (256, 1792):
    sets = [(torch.rand(B, S, F, T, device="cuda"), torch.randn(B, F, T, device="cuda"), torch.empty(B, S, F, T, device="cuda"))
            for _ in range(3)]
    assert torch.equal(eng.separate(sets[0][0], sets[0][1]), sets[0][0] * sets[0][1].unsqueeze(1))
    t_rag = np.random.default_rng(1).integers(16, T + 1, B).astype(np.int32)     # waveform_varlen_bench.py, seed 0
    arms = {"uniform": (None, T * B), "varlen_full": (torch.full((B,), T, dtype=torch.int32, device="cuda"), T * B),
            "varlen_ragged": (torch.from_numpy(t_rag).cuda(), int(t_rag.sum()))}
    for arm, (lens, frames_read) in arms.items():
        if lens is not None:
            want = sets[0][0] * sets[0][1].unsqueeze(1)
            want *= (torch.arange(T, device="cuda") < lens[:, None]).view(B, 1, 1, T)
            assert torch.equal(eng.separate(sets[0][0], sets[0][1], lengths=lens), want)

        def call(i):
            m, x, o = sets[i % 3]
            if lens is None:
                rc = eng.lib.avsep_separate(eng.h, m.data_ptr(), x.data_ptr(), B, T, o.data_ptr(), st)
            else:
                rc = eng.lib.avsep_separate_varlen(eng.h, m.data_ptr(), x.data_ptr(), lens.data_ptr(), B, T,
                                                   o.data_ptr(), st)
            assert rc == 0

        for i in range(6):
            call(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 60
        a.record()
        for i in range(n):
            call(i)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / n
        nbytes = 4 * F * (S + 1) * frames_read + 4 * S * F * T * B
        gbs = nbytes / ms / 1e6
        print(json.dumps({"kernel": "separate", "arm": arm, "B": B, "ms": round(ms, 4), "algorithmic_bytes": nbytes,
                          "gb_s": round(gbs, 1), "peak_gb_s": peak, "frac": round(gbs / peak, 3) if peak else None,
                          "card": card, "power_limit_w": power_w}), flush=True)
    del sets
