"""What a variable-length waveform batch costs and what it saves (avsep_stft_varlen -> avsep_forward_varlen ->
avsep_istft_varlen), default model, bf16, B = 256 one-second clips (L = 8000, n_fft 512, hop 128, T = 63, N = 50 lip
frames of 32 x 32).  Four arms, each timed as whole waveform-to-waveform steps, CUDA events after warm-up, repeated
interleaved:

  A  uniform: avsep_stft -> avsep_forward -> avsep_istft
  B  the varlen calls with every length full                     (B vs A: the overhead of the feature)
  C  the varlen calls on a seeded ragged batch: L_b = 128 (T_b - 1) + 64 with T_b uniform in [16, 63], and
     N_b = max(1, round(50 T_b / 63)); the analysis hands T_b to the forward on the device
  D  the same ragged batch as one uniform pipeline per distinct (L_b, N_b)  (C vs D: what the feature saves)

A, B and C rotate three input sets (so no step re-reads the previous step's inputs from L2).  D keeps one contiguous
input buffer per group: with ~48 groups, three sets per group would exceed the library's 64-entry CUDA-graph cache and
time graph captures instead of forwards.  D's inputs can therefore stay in L2 between steps while C's cannot: the
C / D ratio is biased in D's favour (against the feature).  Utterance-seconds count L_b / 8000 s per utterance.
For A, B and C the analysis and the inverse kernels are also timed on their own.
Prints one JSON line: card, power limit, per-arm ms per batch (median and min over the repeats) and utt-s/s, the
stand-alone kernel times, launch counts of A / B / C, and the largest |difference| between C's and D's valid regions.

  python tools/waveform_varlen_bench.py [--batch 256] [--steps 50] [--warmup 10] [--repeats 5] [--seed 0]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "av-separation-transformer_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from avsep_b200 import AVSeparationTransformer   # noqa: E402
from oracle.weights import CONFIGS, make_state_dict   # noqa: E402
from varlen_bench import card_info   # noqa: E402

L, NFFT, HOP, N, HW = 8000, 512, 128, 50, 32
T = 1 + L // HOP


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("waveform_varlen_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["default"]
    model = AVSeparationTransformer(**cfg.as_dict(), precision="bf16")
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in make_state_dict(cfg, seed=args.seed).items()})
    model = model.to(dev)
    model.prepack(dev)
    eng, lib, h = model.engine, model.engine.lib, model.engine.h
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    B, F, S = args.batch, cfg.freq_bins, cfg.num_speakers

    rng = np.random.default_rng(args.seed + 1)
    t_b = rng.integers(16, T + 1, B).astype(np.int32)
    l_b = (HOP * (t_b - 1) + 64).astype(np.int32)
    n_b = np.maximum(1, np.round(t_b * N / T)).astype(np.int32)
    utt_s_full, utt_s_ragged = float(B), float(l_b.sum()) / L

    g = torch.Generator(device=dev).manual_seed(args.seed + 2)
    sets = [(0.3 * torch.randn(B, L, device=dev, generator=g), torch.rand(B, N, HW, HW, device=dev, generator=g))
            for _ in range(3)]
    spec = torch.empty(B, F, T, dtype=torch.complex64, device=dev)
    mag = torch.empty(B, F, T, device=dev)
    sep = torch.empty(B, S, F, T, device=dev)
    masks = torch.empty_like(sep)
    out = torch.empty(B, S, L, device=dev)
    t_out = torch.empty(B, dtype=torch.int32, device=dev)
    full_l = torch.full((B,), L, dtype=torch.int32, device=dev)
    full_n = torch.full((B,), N, dtype=torch.int32, device=dev)
    rag_l, rag_n = torch.from_numpy(l_b).to(dev), torch.from_numpy(n_b).to(dev)

    def check(rc):
        if rc != 0:
            raise RuntimeError(lib.avsep_last_error(h).decode())

    counts = {}

    def count(stage):
        counts[stage] = int(lib.avsep_last_launch_count(h))

    def uniform(w, f, b, ll, nn, sp, mg, sp_s, sp_m, o):
        tt = 1 + ll // HOP
        check(lib.avsep_stft(h, w.data_ptr(), b, ll, NFFT, HOP, sp.data_ptr(), mg.data_ptr(), st))
        count("stft")
        check(lib.avsep_forward(h, mg.data_ptr(), f.data_ptr(), b, tt, nn, HW, HW, sp_s.data_ptr(), sp_m.data_ptr(),
                                None, 0, st))
        count("forward")
        check(lib.avsep_istft(h, sp.data_ptr(), sp_m.data_ptr(), b, S, tt, NFFT, HOP, ll, o.data_ptr(), st))
        count("istft")

    def varlen(i, lens, flens):
        w, f = sets[i % 3]
        check(lib.avsep_stft_varlen(h, w.data_ptr(), lens.data_ptr(), B, L, NFFT, HOP, spec.data_ptr(), mag.data_ptr(),
                                    t_out.data_ptr(), st))
        count("stft")
        check(lib.avsep_forward_varlen(h, mag.data_ptr(), f.data_ptr(), t_out.data_ptr(), flens.data_ptr(), B, T, N, HW,
                                       HW, sep.data_ptr(), masks.data_ptr(), None, 0, st))
        count("forward")
        check(lib.avsep_istft_varlen(h, spec.data_ptr(), masks.data_ptr(), lens.data_ptr(), B, S, T, NFFT, HOP, L,
                                     out.data_ptr(), st))
        count("istft")

    # D: one contiguous input / intermediate / output buffer set per distinct (L_b, N_b), built from input set 0
    groups = []
    w0, f0 = sets[0]
    for ll, nn in sorted(set(zip(l_b.tolist(), n_b.tolist()))):
        idx = np.nonzero((l_b == ll) & (n_b == nn))[0]
        it = torch.from_numpy(idx).to(dev)
        n, tt = len(idx), 1 + ll // HOP
        bufs = (w0.index_select(0, it)[:, :ll].contiguous(), f0.index_select(0, it)[:, :nn].contiguous(), n, ll, nn,
                torch.empty(n, F, tt, dtype=torch.complex64, device=dev), torch.empty(n, F, tt, device=dev),
                torch.empty(n, S, F, tt, device=dev), torch.empty(n, S, F, tt, device=dev),
                torch.empty(n, S, ll, device=dev))
        groups.append((idx, bufs))

    def grouped(i):
        for _, bufs in groups:
            uniform(*bufs)

    arms = {
        "A_uniform": lambda i: uniform(*sets[i % 3], B, L, N, spec, mag, sep, masks, out),
        "B_varlen_full": lambda i: varlen(i, full_l, full_n),
        "C_varlen_ragged": lambda i: varlen(i, rag_l, rag_n),
        "D_grouped_uniform": grouped,
    }
    launches = {}
    for name, fn in arms.items():
        for i in range(max(args.warmup, 6)):      # >= 2 uses of every (shape, buffer set): graphs captured
            fn(i)
        torch.cuda.synchronize()
        if name != "D_grouped_uniform":
            launches[name] = dict(counts)

    # C against D on the valid regions (input set 0 in both)
    varlen(0, rag_l, rag_n)
    grouped(0)
    torch.cuda.synchronize()
    # samples with a window sum below 1e-3 (the first few of each clip) divide by almost nothing: reported apart
    w2 = np.hanning(NFFT) ** 2
    wss = np.zeros((T - 1) * HOP + NFFT)
    for i in range(T):
        wss[i * HOP:i * HOP + NFFT] += w2
    solid = torch.from_numpy(wss[:L] > 1e-3).to(dev)
    max_diff = {"waves": 0.0, "waves_window_sum_above_1e-3": 0.0, "masks": 0.0}
    for idx, bufs in groups:
        it = torch.from_numpy(idx).to(dev)
        ll, tt = bufs[3], 1 + bufs[3] // HOP
        d = (out.index_select(0, it)[..., :ll] - bufs[9]).abs()
        max_diff["waves"] = max(max_diff["waves"], d.max().item())
        max_diff["waves_window_sum_above_1e-3"] = max(max_diff["waves_window_sum_above_1e-3"],
                                                      d[..., solid[:ll]].max().item())
        max_diff["masks"] = max(max_diff["masks"], (masks.index_select(0, it)[..., :tt] - bufs[8]).abs().max().item())
    zero_past = all(not out[b, :, l_b[b]:].any().item() and not masks[b, :, :, t_b[b]:].any().item() for b in range(B))

    # the analysis and the inverse kernels on their own, per arm (input set 0)
    w, _ = sets[0]
    kernels = {
        "A_uniform": (lambda: check(lib.avsep_stft(h, w.data_ptr(), B, L, NFFT, HOP, spec.data_ptr(), mag.data_ptr(), st)),
                      lambda: check(lib.avsep_istft(h, spec.data_ptr(), masks.data_ptr(), B, S, T, NFFT, HOP, L,
                                                    out.data_ptr(), st))),
    }
    for name, lens in (("B_varlen_full", full_l), ("C_varlen_ragged", rag_l)):
        kernels[name] = (
            lambda lens=lens: check(lib.avsep_stft_varlen(h, w.data_ptr(), lens.data_ptr(), B, L, NFFT, HOP,
                                                          spec.data_ptr(), mag.data_ptr(), t_out.data_ptr(), st)),
            lambda lens=lens: check(lib.avsep_istft_varlen(h, spec.data_ptr(), masks.data_ptr(), lens.data_ptr(), B, S,
                                                           T, NFFT, HOP, L, out.data_ptr(), st)))

    def timed(fn, steps):
        for i in range(2):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    times = {k: [] for k in arms}
    ktimes = {k: {"stft": [], "istft": []} for k in kernels}
    for _ in range(args.repeats):
        for name, fn in arms.items():
            times[name].append(timed(fn, args.steps))
        for name, (fs, fi) in kernels.items():
            ktimes[name]["stft"].append(timed(lambda i: fs(), 4 * args.steps))
            ktimes[name]["istft"].append(timed(lambda i: fi(), 4 * args.steps))

    card, power_w = card_info(0)
    res = {"tool": "waveform_varlen_bench", "card": card, "power_limit_w": power_w, "batch": B, "L": L, "n_fft": NFFT,
           "hop": HOP, "T": T, "N": N, "steps": args.steps, "repeats": args.repeats, "ragged_T_range": [16, T],
           "distinct_groups": len(groups), "utt_s_per_batch": {"full": utt_s_full, "ragged": round(utt_s_ragged, 3)},
           "arms": {}, "kernel_ms_median": {}}
    for name, ts in times.items():
        med = statistics.median(ts)
        us = utt_s_full if name in ("A_uniform", "B_varlen_full") else utt_s_ragged
        res["arms"][name] = {"ms_median": round(med, 4), "ms_min": round(min(ts), 4),
                             "utt_s_per_s": round(us / (med / 1000.0), 1)}
    for name, kt in ktimes.items():
        res["kernel_ms_median"][name] = {k: round(statistics.median(v), 4) for k, v in kt.items()}
    res["launch_count"] = launches
    res["max_abs_diff_C_vs_D_valid"] = max_diff
    res["C_zero_past_length"] = bool(zero_past)
    res["note"] = ("A, B, C rotate 3 input sets; D uses one buffer set per group (L2-resident between steps), which "
                   "favours D in the C / D ratio; stand-alone kernel times use input set 0")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
