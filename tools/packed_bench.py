"""What the packed host path moves and how fast (avsep_forward_host_packed_async), default model, bf16, B = 256
one-second clips (T = 63, N = 50, 32 x 32 frames).  Every arm streams batches through two I/O slots the way bench.py's
e2e does (batch i on slot i % 2, its results waited for before the slot is used again) and rotates three input sets
whose ragged lengths differ, so a graph recapture per batch would show in the times:

  A  avsep_forward_host_async, padded uniform batches                    (bench.py's e2e)
  B  avsep_forward_host_packed_async with every length full              (B vs A: what unpack + pack cost)
  C  avsep_forward_host_packed_async on the varlen_bench.py ragged mix: T_b uniform in [16, 63],
     N_b = max(1, round(T_b * 50 / 63))                                  (C vs A: audio-seconds per second)
  D  the same ragged batches by the route that exists without packing: pinned padded H2D, avsep_forward_varlen,
     padded D2H, on two streams with a workspace each

Per arm: ms per batch (median and min over the repeats), audio-seconds per second (the sum of the clips' own
durations, T_b / 63 s each), H2D and D2H bytes per batch and the time those bytes take at the link rates measured in
the same run (pinned copies, both directions at once).  Also the device-only avsep_forward_packed against
avsep_forward_varlen on the ragged sets (CUDA events), and the unpack / pack kernels alone (per-launch event pairs of
the library's profiling mode) at full and ragged lengths, as bytes moved (reads + writes) per second against a
device-to-device cudaMemcpyAsync of the same byte count.  Prints one JSON line with the card name and power limit.

  python tools/packed_bench.py [--batch 256] [--steps 30] [--repeats 5] [--seed 0]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, os.path.join(ROOT, "av-separation-transformer_b200"), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from avsep_b200 import AVSeparationTransformer   # noqa: E402
from avsep_b200.synth import synthetic_batch     # noqa: E402
from oracle.weights import CONFIGS, make_state_dict   # noqa: E402
from varlen_bench import card_info               # noqa: E402

T, N, HW = 63, 50, 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("packed_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["default"]
    model = AVSeparationTransformer(**cfg.as_dict(), precision="bf16")
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in make_state_dict(cfg, seed=args.seed).items()})
    model = model.to(dev)
    model.prepack(dev)
    eng = model.engine
    B, F, S = args.batch, cfg.freq_bins, cfg.num_speakers
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def check(rc):
        if rc != 0:
            raise RuntimeError(eng.lib.avsep_last_error(eng.h).decode())

    # three input sets, each with its own ragged lengths
    sets = []
    for i in range(3):
        m, f = synthetic_batch(B, F, T, N, HW, HW, seed=1000 + i, device=dev)
        rng = np.random.default_rng(args.seed + 1 + i)
        t_b = rng.integers(16, T + 1, B).astype(np.int32)
        n_b = np.maximum(1, np.round(t_b * N / T)).astype(np.int32)
        mc, fc = m.cpu(), f.cpu()
        mp = torch.cat([mc[b, :, :t_b[b]].reshape(-1) for b in range(B)])
        fp = torch.cat([fc[b, :n_b[b]] for b in range(B)])
        sets.append(dict(m=m, f=f, hm=mc.pin_memory(), hf=fc.pin_memory(), t=t_b, n=n_b, hmp=mp.pin_memory(),
                         hfp=fp.pin_memory(), dmp=mp.to(dev), dfp=fp.to(dev), dt=torch.from_numpy(t_b).to(dev),
                         dn=torch.from_numpy(n_b).to(dev)))
    full_t, full_n = np.full(B, T, np.int32), np.full(B, N, np.int32)
    pad_out = B * S * F * T
    h_out = [(torch.empty(pad_out).pin_memory(), torch.empty(pad_out).pin_memory()) for _ in range(2)]

    def p(t):
        return t.data_ptr()

    def arm_a(i, slot):
        s = sets[i % 3]
        check(eng.lib.avsep_forward_host_async(eng.h, p(s["hm"]), p(s["hf"]), B, T, N, HW, HW, p(h_out[slot][0]),
                                               p(h_out[slot][1]), slot, st))

    def arm_packed(i, slot, full):
        s = sets[i % 3]
        hm, hf = (s["hm"], s["hf"]) if full else (s["hmp"], s["hfp"])
        t, n = (full_t, full_n) if full else (s["t"], s["n"])
        check(eng.lib.avsep_forward_host_packed_async(eng.h, p(hm), p(hf), t.ctypes.data, n.ctypes.data, B, T, N, HW,
                                                      HW, p(h_out[slot][0]), p(h_out[slot][1]), slot, st))

    # D: two streams, a workspace, device inputs and outputs each
    ws_bytes = eng.lib.avsep_workspace_bytes(eng.h, B, T, N, HW, HW)
    d_slots = []
    for _ in range(2):
        raw = torch.empty(ws_bytes + 1024, dtype=torch.uint8, device=dev)
        off = (-raw.data_ptr()) % 1024
        d_slots.append(dict(stream=torch.cuda.Stream(), raw=raw, ws=raw.data_ptr() + off,
                            m=torch.empty(B, F, T, device=dev), f=torch.empty(B, N, HW, HW, device=dev),
                            sep=torch.empty(pad_out, device=dev), masks=torch.empty(pad_out, device=dev)))

    def arm_d(i, slot):
        s, d = sets[i % 3], d_slots[slot]
        with torch.cuda.stream(d["stream"]):
            d["m"].copy_(s["hm"], non_blocking=True)
            d["f"].copy_(s["hf"], non_blocking=True)
            check(eng.lib.avsep_forward_varlen(eng.h, p(d["m"]), p(d["f"]), p(s["dt"]), p(s["dn"]), B, T, N, HW, HW,
                                               p(d["sep"]), p(d["masks"]), d["ws"], ws_bytes,
                                               C.c_void_p(d["stream"].cuda_stream)))
            h_out[slot][0].copy_(d["sep"], non_blocking=True)
            h_out[slot][1].copy_(d["masks"], non_blocking=True)

    def stream_run(fn, n):
        for i in range(n):
            slot = i % 2
            if fn is arm_d:
                fn(i, slot)          # stream order on the slot's stream keeps its buffers safe
                continue
            if i >= 2:
                eng.host_wait(slot)
            fn(i, slot)
        if fn is not arm_d:
            eng.host_wait(0)
            eng.host_wait(1)
        torch.cuda.synchronize()

    arms = {"A_uniform_host": arm_a, "B_packed_full": lambda i, s: arm_packed(i, s, True),
            "C_packed_ragged": lambda i, s: arm_packed(i, s, False), "D_padded_varlen_route": arm_d}
    for fn in arms.values():
        stream_run(fn, 12)             # every (set, slot) graph captured
    times = {k: [] for k in arms}
    for _ in range(args.repeats):
        for name, fn in arms.items():
            stream_run(fn, 2)
            t0 = time.perf_counter()
            stream_run(fn, args.steps)
            times[name].append((time.perf_counter() - t0) * 1e3 / args.steps)

    # correctness of the timed arms: C's last results per slot against avsep_forward_varlen's valid regions
    max_diff = 0.0
    for slot in range(2):
        i = args.steps - 2 + slot
        s = sets[i % 3]
        arm_packed(i, slot, False)
        eng.host_wait(slot)
        sep_v, masks_v = model(s["m"], s["f"], lengths=s["dt"], frame_lengths=s["dn"])
        nb = S * F * int(s["t"].sum())
        for k, ref in ((0, sep_v), (1, masks_v)):
            valid = torch.cat([ref[b, :, :, :s["t"][b]].reshape(-1) for b in range(B)]).cpu()
            max_diff = max(max_diff, (h_out[slot][k][:nb] - valid).abs().max().item())

    # link rates: pinned copies of one padded batch, both directions at once (the way the pipeline copies)
    cp_in, cp_out = torch.cuda.Stream(), torch.cuda.Stream()
    d_in = [torch.empty_like(sets[0]["hm"], device=dev), torch.empty_like(sets[0]["hf"], device=dev)]
    d_src = d_slots[0]

    def copy_round():
        with torch.cuda.stream(cp_in):
            d_in[0].copy_(sets[0]["hm"], non_blocking=True)
            d_in[1].copy_(sets[0]["hf"], non_blocking=True)
        with torch.cuda.stream(cp_out):
            h_out[0][0].copy_(d_src["sep"], non_blocking=True)
            h_out[0][1].copy_(d_src["masks"], non_blocking=True)

    h2d_pad = (sets[0]["hm"].numel() + sets[0]["hf"].numel()) * 4
    d2h_pad = 2 * pad_out * 4
    for _ in range(2):
        copy_round()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        copy_round()
    torch.cuda.synchronize()
    copy_s = (time.perf_counter() - t0) / 10
    h2d_rate, d2h_rate = h2d_pad / copy_s, d2h_pad / copy_s

    audio_s_full = float(B)
    audio_s_rag = statistics.mean(float(s["t"].sum()) / T for s in sets)
    h2d_rag = statistics.mean((F * int(s["t"].sum()) + HW * HW * int(s["n"].sum())) * 4 for s in sets)
    d2h_rag = statistics.mean(2 * S * F * int(s["t"].sum()) * 4 for s in sets)
    io = {"A_uniform_host": (h2d_pad, d2h_pad, audio_s_full), "B_packed_full": (h2d_pad, d2h_pad, audio_s_full),
          "C_packed_ragged": (h2d_rag, d2h_rag, audio_s_rag), "D_padded_varlen_route": (h2d_pad, d2h_pad, audio_s_rag)}
    card, power_w = card_info(0)
    res = {"tool": "packed_bench", "card": card, "power_limit_w": power_w, "batch": B, "T": T, "N": N,
           "steps": args.steps, "repeats": args.repeats,
           "link": {"h2d_gbs": round(h2d_rate / 1e9, 2), "d2h_gbs": round(d2h_rate / 1e9, 2),
                    "what": "pinned copies of one padded batch, both directions at once"},
           "arms": {}}
    for name, ts in times.items():
        med = statistics.median(ts)
        h2d, d2h, audio_s = io[name]
        ceil_ms = max(h2d / h2d_rate, d2h / d2h_rate) * 1e3
        res["arms"][name] = {"ms_median": round(med, 4), "ms_min": round(min(ts), 4),
                             "audio_s_per_s": round(audio_s / (med / 1e3), 1), "h2d_bytes": int(h2d),
                             "d2h_bytes": int(d2h), "link_ms": round(ceil_ms, 4),
                             "link_ceiling_audio_s_per_s": round(audio_s / (ceil_ms / 1e3), 1)}
    res["C_max_abs_diff_vs_varlen_valid"] = max_diff

    # device only: avsep_forward_packed against avsep_forward_varlen on the ragged sets (CUDA events)
    dsep, dmasks = torch.empty(pad_out, device=dev), torch.empty(pad_out, device=dev)
    vsep, vmasks = torch.empty(B, S, F, T, device=dev), torch.empty(B, S, F, T, device=dev)

    def dev_packed(i):
        s = sets[i % 3]
        check(eng.lib.avsep_forward_packed(eng.h, p(s["dmp"]), p(s["dfp"]), p(s["dt"]), p(s["dn"]), B, T, N, HW, HW,
                                           p(dsep), p(dmasks), None, 0, st))

    def dev_varlen(i):
        s = sets[i % 3]
        check(eng.lib.avsep_forward_varlen(eng.h, p(s["m"]), p(s["f"]), p(s["dt"]), p(s["dn"]), B, T, N, HW, HW,
                                           p(vsep), p(vmasks), None, 0, st))

    dev_arms = {"forward_packed": dev_packed, "forward_varlen": dev_varlen}
    dev_times = {k: [] for k in dev_arms}
    launches = {}
    for name, fn in dev_arms.items():
        for i in range(9):
            fn(i)
        torch.cuda.synchronize()
        launches[name] = eng.launch_count()
    for _ in range(args.repeats):
        for name, fn in dev_arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(100):
                fn(i)
            e1.record()
            torch.cuda.synchronize()
            dev_times[name].append(e0.elapsed_time(e1) / 100)
    res["device_only"] = {k: {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4)}
                          for k, v in dev_times.items()}
    res["launch_count"] = launches

    # unpack / pack alone: per-launch event pairs (profiling mode), full and ragged lengths, against a D2D copy
    full_dt = torch.full((B,), T, dtype=torch.int32, device=dev)
    full_dn = torch.full((B,), N, dtype=torch.int32, device=dev)
    kern = {}
    for label, lens_of in (("full", lambda s: (full_dt, full_dn, full_t, full_n)),
                           ("ragged", lambda s: (s["dt"], s["dn"], s["t"], s["n"]))):
        eng.set_profile(True)
        eng.profile_report(reset=True)
        reps = 20
        for i in range(reps):
            s = sets[i % 3]
            dt, dn, _, _ = lens_of(s)
            mp, fp = (s["m"], s["f"]) if label == "full" else (s["dmp"], s["dfp"])
            check(eng.lib.avsep_forward_packed(eng.h, p(mp), p(fp), p(dt), p(dn), B, T, N, HW, HW, p(dsep), p(dmasks),
                                               None, 0, st))
        rep = eng.profile_report(reset=True)
        eng.set_profile(False)
        t_sum = statistics.mean(float(lens_of(s)[2].sum()) for s in sets)
        n_sum = statistics.mean(float(lens_of(s)[3].sum()) for s in sets)
        moved = {"unpack": 2 * 4 * (F * t_sum + HW * HW * n_sum), "pack": 2 * 2 * 4 * S * F * t_sum}
        for k in ("unpack", "pack"):
            n_l, ms_tot = rep[k]
            ms = ms_tot / n_l
            nbytes = int(moved[k] // 2 // 4 * 4)
            a, b = torch.empty(nbytes, dtype=torch.uint8, device=dev), torch.empty(nbytes, dtype=torch.uint8, device=dev)
            for _ in range(3):
                b.copy_(a)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                b.copy_(a)
            e1.record()
            torch.cuda.synchronize()
            ms_copy = e0.elapsed_time(e1) / reps
            del a, b
            kern[f"{k}_{label}"] = {"ms": round(ms, 5), "bytes_moved": int(moved[k]),
                                    "tbs": round(moved[k] / (ms / 1e3) / 1e12, 3),
                                    "d2d_copy_ms": round(ms_copy, 5),
                                    "d2d_copy_tbs": round(2 * nbytes / (ms_copy / 1e3) / 1e12, 3),
                                    "rate_vs_d2d_copy": round(ms_copy / ms, 3)}
    res["kernels"] = kern
    print(json.dumps(res))


if __name__ == "__main__":
    main()
