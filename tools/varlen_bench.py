"""What a variable-length batch costs and what it saves (avsep_forward_varlen), default model, bf16, B = 256,
SyntheticAVDataset-shaped inputs.  Four arms, CUDA events after warm-up, repeated interleaved:

  A  uniform avsep_forward at T = 63, N = 50
  B  avsep_forward_varlen with every length full                       (B vs A: the overhead of the feature)
  C  avsep_forward_varlen on a seeded ragged batch: T_b uniform in [16, 63], N_b = max(1, round(T_b * 50 / 63))
  D  the same ragged batch as one avsep_forward per distinct (T_b, N_b)  (C vs D: what the feature saves)

A, B and C rotate three input sets (as bench.py does, so no step re-reads the previous step's inputs from L2).  D keeps
one contiguous input buffer per group: with ~48 groups, three sets per group would exceed the library's 64-entry
CUDA-graph cache and time graph captures instead of forwards.  D's inputs can therefore stay in L2 between steps
while C's cannot: the C / D ratio is biased in D's favour (against the feature).  Utterance-seconds count T_b / 63 s
per utterance.
Prints one JSON line: card, power limit, per-arm ms per batch (median and min over the repeats) and utt-s/s,
launch counts of A / B / C, and the largest |difference| between C's and D's valid regions.

  python tools/varlen_bench.py [--batch 256] [--steps 100] [--warmup 10] [--repeats 5] [--seed 0]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "av-separation-transformer_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from avsep_b200 import AVSeparationTransformer   # noqa: E402
from avsep_b200.synth import synthetic_batch     # noqa: E402
from oracle.weights import CONFIGS, make_state_dict   # noqa: E402

T, N, HW = 63, 50, 32


def card_info(index):
    name = torch.cuda.get_device_name(index)
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        return name, pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return name, float(out)
    except Exception:
        return name, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("varlen_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["default"]
    model = AVSeparationTransformer(**cfg.as_dict(), precision="bf16")
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in make_state_dict(cfg, seed=args.seed).items()})
    model = model.to(dev)
    model.prepack(dev)
    eng = model.engine
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    B, F, S = args.batch, cfg.freq_bins, cfg.num_speakers

    rng = np.random.default_rng(args.seed + 1)
    t_b = rng.integers(16, T + 1, B).astype(np.int32)
    n_b = np.maximum(1, np.round(t_b * N / T)).astype(np.int32)
    utt_s_full, utt_s_ragged = float(B), float(t_b.sum()) / T

    sets = [synthetic_batch(B, F, T, N, HW, HW, seed=1000 + i, device=dev) for i in range(3)]
    sep = torch.empty(B, S, F, T, device=dev)
    masks = torch.empty_like(sep)
    full_t = torch.full((B,), T, dtype=torch.int32, device=dev)
    full_n = torch.full((B,), N, dtype=torch.int32, device=dev)
    rag_t, rag_n = torch.from_numpy(t_b).to(dev), torch.from_numpy(n_b).to(dev)

    def check(rc):
        if rc != 0:
            raise RuntimeError(eng.lib.avsep_last_error(eng.h).decode())

    def uniform(mixed, frames, b, tt, nn, o_s, o_m):
        check(eng.lib.avsep_forward(eng.h, mixed.data_ptr(), frames.data_ptr(), b, tt, nn, HW, HW, o_s.data_ptr(),
                                    o_m.data_ptr(), None, 0, st))

    def varlen(i, lens, flens):
        m, f = sets[i % 3]
        check(eng.lib.avsep_forward_varlen(eng.h, m.data_ptr(), f.data_ptr(), lens.data_ptr(), flens.data_ptr(), B, T,
                                           N, HW, HW, sep.data_ptr(), masks.data_ptr(), None, 0, st))

    # D: one contiguous input / output buffer per distinct (T_b, N_b), built from input set 0
    groups = []
    m0, f0 = sets[0]
    for tt, nn in sorted(set(zip(t_b.tolist(), n_b.tolist()))):
        idx = np.nonzero((t_b == tt) & (n_b == nn))[0]
        it = torch.from_numpy(idx).to(dev)
        gm = m0.index_select(0, it)[:, :, :tt].contiguous()
        gf = f0.index_select(0, it)[:, :nn].contiguous()
        go = torch.empty(2, len(idx), S, F, tt, device=dev)
        groups.append((idx, tt, nn, gm, gf, go))

    def grouped(i):
        for idx, tt, nn, gm, gf, go in groups:
            uniform(gm, gf, len(idx), tt, nn, go[0], go[1])

    arms = {
        "A_uniform": lambda i: uniform(sets[i % 3][0], sets[i % 3][1], B, T, N, sep, masks),
        "B_varlen_full": lambda i: varlen(i, full_t, full_n),
        "C_varlen_ragged": lambda i: varlen(i, rag_t, rag_n),
        "D_grouped_uniform": grouped,
    }
    launches = {}
    for name, fn in arms.items():
        for i in range(max(args.warmup, 6)):      # >= 2 uses of every (shape, buffer set): graphs captured
            fn(i)
        torch.cuda.synchronize()
        if name != "D_grouped_uniform":
            launches[name] = eng.launch_count()

    # C against D on the valid regions (input set 0 in both)
    varlen(0, rag_t, rag_n)
    grouped(0)
    torch.cuda.synchronize()
    max_diff = 0.0
    for idx, tt, nn, gm, gf, go in groups:
        it = torch.from_numpy(idx).to(dev)
        for k, ref in ((0, sep), (1, masks)):
            d = (ref.index_select(0, it)[..., :tt] - go[k]).abs().max().item()
            max_diff = max(max_diff, d)
    padded_zero = all(not masks[b, :, :, t_b[b]:].any().item() for b in range(B))

    times = {k: [] for k in arms}
    for _ in range(args.repeats):
        for name, fn in arms.items():
            for i in range(2):
                fn(i)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                fn(i)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)

    card, power_w = card_info(0)
    res = {"tool": "varlen_bench", "card": card, "power_limit_w": power_w, "batch": B, "T": T, "N": N,
           "steps": args.steps, "repeats": args.repeats, "ragged_T_range": [16, T],
           "distinct_groups": len(groups), "utt_s_per_batch": {"full": utt_s_full, "ragged": round(utt_s_ragged, 3)},
           "arms": {}}
    for name, ts in times.items():
        med = statistics.median(ts)
        us = utt_s_full if name in ("A_uniform", "B_varlen_full") else utt_s_ragged
        res["arms"][name] = {"ms_median": round(med, 4), "ms_min": round(min(ts), 4),
                             "utt_s_per_s": round(us / (med / 1000.0), 1)}
    res["launch_count"] = launches
    res["max_abs_diff_C_vs_D_valid"] = max_diff
    res["C_zero_past_length"] = bool(padded_zero)
    res["note"] = ("A, B, C rotate 3 input sets; D uses one buffer per group (L2-resident between steps), which favours D "
                   "in the C / D ratio")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
