"""Waveform to waveform in one call, on the device and from host buffers: default model, bf16, B = 256 one-second clips
(L = 8000 samples, n_fft 512, hop 128, T = 63), N = 50 lip frames of 32 x 32, pinned host buffers.  Four arms, timed in
one process and alternated over the repeats:

  a  the three-call device composition avsep_stft -> avsep_forward (on the magnitude) -> avsep_istft (on the masks)
  b  avsep_separate_waveforms (the STFT writes the Conv1d operand, masks-only decoder, masked inverse)
  c  avsep_forward_host_async streaming on two I/O slots: spectrogram + lip frames in, separated + masks out
  d  avsep_separate_waveforms_host_async streaming on two I/O slots: samples + lip frames in, waveforms + masks out
     (d0: the same without masks, so that only samples come back)

a and b rotate three device input sets (180 MB, more than the 126 MB L2) and are timed with CUDA events around `steps`
calls; c and d are timed with the host clock around `steps` calls that end in avsep_host_wait on both slots.  Reports,
per arm: ms per step (median and min over the repeats), utterance-seconds per second, bytes per step in each PCIe
direction (from the shapes), launches per call, and checks b == a and d == b bit for bit.  The GPU name and power
limit are read in the same run.  Prints one JSON line and, with --out, writes a markdown summary.

  python tools/waveform_host_bench.py [--batch 256] [--steps 40] [--warmup 5] [--repeats 5] [--out FILE]
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
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("waveform_host_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = CONFIGS["default"]
    model = AVSeparationTransformer(**cfg.as_dict(), precision="bf16")
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in make_state_dict(cfg, seed=args.seed).items()})
    model = model.to(dev)
    model.prepack(dev)
    eng, lib, h = model.engine, model.engine.lib, model.engine.h
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    B, F, S = args.batch, cfg.freq_bins, cfg.num_speakers

    def ok(rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {lib.avsep_last_error(h).decode()}")

    g = torch.Generator(device=dev).manual_seed(args.seed + 1)
    sets = [(0.3 * torch.randn(B, L, device=dev, generator=g), torch.rand(B, N, HW, HW, device=dev, generator=g))
            for _ in range(3)]
    spec = torch.empty(B, F, T, dtype=torch.complex64, device=dev)
    mag = torch.empty(B, F, T, device=dev)
    sep = torch.empty(B, S, F, T, device=dev)
    masks = torch.empty_like(sep)
    out_a = torch.empty(B, S, L, device=dev)
    out_b, masks_b = torch.empty_like(out_a), torch.empty_like(masks)

    def arm_a(k):
        w, lips = sets[k % 3]
        ok(lib.avsep_stft(h, w.data_ptr(), B, L, NFFT, HOP, spec.data_ptr(), mag.data_ptr(), st), "avsep_stft")
        n = eng.launch_count()
        ok(lib.avsep_forward(h, mag.data_ptr(), lips.data_ptr(), B, T, N, HW, HW, sep.data_ptr(), masks.data_ptr(), None,
                             0, st), "avsep_forward")
        n += eng.launch_count()
        ok(lib.avsep_istft(h, spec.data_ptr(), masks.data_ptr(), B, S, T, NFFT, HOP, L, out_a.data_ptr(), st),
           "avsep_istft")
        return n + eng.launch_count()

    def arm_b(k):
        w, lips = sets[k % 3]
        ok(lib.avsep_separate_waveforms(h, w.data_ptr(), lips.data_ptr(), None, None, B, L, N, HW, HW, NFFT, HOP,
                                        out_b.data_ptr(), masks_b.data_ptr(), None, 0, st), "avsep_separate_waveforms")
        return eng.launch_count()

    # host buffers: one input set, two output sets (one per slot)
    wave_h = sets[0][0].cpu().pin_memory()
    lips_h = sets[0][1].cpu().pin_memory()
    arm_b(0)
    _, mag0 = eng.stft(sets[0][0], NFFT, HOP)
    mag_h = mag0.cpu().pin_memory()
    sep_h = [torch.empty(B, S, F, T).pin_memory() for _ in range(2)]
    masks_h = [torch.empty(B, S, F, T).pin_memory() for _ in range(2)]
    wout_h = [torch.empty(B, S, L).pin_memory() for _ in range(2)]
    wmask_h = [torch.empty(B, S, F, T).pin_memory() for _ in range(2)]

    def arm_c(k):
        ok(lib.avsep_forward_host_async(h, mag_h.data_ptr(), lips_h.data_ptr(), B, T, N, HW, HW, sep_h[k % 2].data_ptr(),
                                        masks_h[k % 2].data_ptr(), k % 2, st), "avsep_forward_host_async")
        return eng.launch_count()

    def wave_host(with_masks):
        def arm(k):
            ok(lib.avsep_separate_waveforms_host_async(h, wave_h.data_ptr(), lips_h.data_ptr(), B, L, N, HW, HW, NFFT,
                                                       HOP, wout_h[k % 2].data_ptr(),
                                                       wmask_h[k % 2].data_ptr() if with_masks else None, k % 2, st),
               "avsep_separate_waveforms_host_async")
            return eng.launch_count()
        return arm

    def time_device(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            fn(k)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def time_host(fn, steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(steps):
            if k >= 2:
                eng.host_wait(k % 2)
            fn(k)
        eng.host_wait(0)
        eng.host_wait(1)
        return (time.perf_counter() - t0) * 1e3 / steps

    arms = {"a": (arm_a, time_device), "b": (arm_b, time_device), "c": (arm_c, time_host),
            "d": (wave_host(True), time_host), "d0": (wave_host(False), time_host)}
    launches = {}
    for name, (fn, timer) in arms.items():          # warm-up: every graph of every input set, both slots
        launches[name] = fn(0)
        timer(fn, max(args.warmup, 6))
    times = {name: [] for name in arms}
    for _ in range(args.repeats):
        for name, (fn, timer) in arms.items():
            times[name].append(timer(fn, args.steps))

    # results: b against a on the same inputs, d against b
    arm_a(0)
    arm_b(0)
    torch.cuda.synchronize()
    b_eq_a = bool(torch.equal(out_a, out_b) and torch.equal(masks, masks_b))
    wave_host(True)(0)
    eng.host_wait(0)
    d_eq_b = bool(torch.equal(wout_h[0], out_b.cpu()) and torch.equal(wmask_h[0], masks_b.cpu()))

    name, plimit = card_info(0)
    f4 = 4
    frames_b = B * N * HW * HW * f4
    pcie = {"a": (0, 0), "b": (0, 0),
            "c": (B * F * T * f4 + frames_b, 2 * B * S * F * T * f4),
            "d": (B * L * f4 + frames_b, B * S * L * f4 + B * S * F * T * f4),
            "d0": (B * L * f4 + frames_b, B * S * L * f4)}
    res = {"gpu": name, "power_limit_w": plimit, "batch": B, "steps": args.steps, "repeats": args.repeats,
           "b_equals_a": b_eq_a, "d_equals_b": d_eq_b, "arms": {}}
    for k in arms:
        med, lo = statistics.median(times[k]), min(times[k])
        res["arms"][k] = {"ms_median": round(med, 4), "ms_min": round(lo, 4),
                          "utt_s_per_s": round(B * (L / 8000.0) / (med * 1e-3)), "h2d_bytes": pcie[k][0],
                          "d2h_bytes": pcie[k][1], "launches_per_call": launches[k]}
    print(json.dumps(res))
    if args.out:
        labels = {"a": "device: avsep_stft -> avsep_forward -> avsep_istft",
                  "b": "device: avsep_separate_waveforms",
                  "c": "host, 2 slots: avsep_forward_host_async (spectrogram in, separated + masks out)",
                  "d": "host, 2 slots: avsep_separate_waveforms_host_async (samples in, waveforms + masks out)",
                  "d0": "host, 2 slots: avsep_separate_waveforms_host_async without masks (waveforms out)"}
        lines = [f"# Waveform path in one call: device and host-buffer rates ({name}, power limit "
                 f"{plimit if plimit is not None else 'unknown'} W)", "",
                 f"`python tools/waveform_host_bench.py --batch {B} --steps {args.steps} --repeats {args.repeats}`: "
                 "default model, bf16, one-second clips (L = 8000, n_fft 512, hop 128, T = 63), 50 lip frames of "
                 "32 x 32, pinned host buffers.  Arms alternated in one process; ms per step is the median (min) over "
                 "the repeats; bytes per step are computed from the shapes.", "",
                 "| arm | ms / step | utt-s/s | H2D MB / step | D2H MB / step | launches / call |",
                 "|---|---|---|---|---|---|"]
        for k, r in res["arms"].items():
            lines.append(f"| {k}: {labels[k]} | {r['ms_median']:.3f} ({r['ms_min']:.3f}) | {r['utt_s_per_s']:,} | "
                         f"{r['h2d_bytes'] / 1e6:.1f} | {r['d2h_bytes'] / 1e6:.1f} | {r['launches_per_call']} |")
        lines += ["", f"b equals a bit for bit: {b_eq_a}; d equals b bit for bit: {d_eq_b}.", "",
                  "Raw result line:", "", "```", json.dumps(res), "```", ""]
        with open(args.out, "w") as f:
            f.write("\n".join(lines))


if __name__ == "__main__":
    main()
