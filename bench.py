#!/usr/bin/env python
"""Benchmark of the hot path: AVSeparationTransformer.forward on SyntheticAVDataset-shaped input.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c3|c4] [--batch B] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one forward pass over one batch of B utterances per GPU.  Default workload = BASELINE.json configs[1]
(c2): default model (freq_bins=257, d_model=256, nhead=4, 2 encoder + 2 fusion layers, 2 speakers), bf16 operands,
B=256 one-second utterances per GPU (1 s @ 8 kHz: T=63 STFT frames, N=50 lip frames of 32x32).  The other configs of
BASELINE.json are selectable: c1 (same model, B=8), c3 (long form, 10 s @ 16 kHz: T=1251, N=500, B=32), c4 (scaled
model d=512, 8 heads, 6+6 layers, 3 speakers, B=256).

N = 1: `value` = forward with the inputs resident in HBM.
N > 1: `value` = the north-star data path (SURVEY 8e): the root (rank 0) holds the global batch, every rank pulls its
shard of the inputs over NVLink and runs the forward, and `separated` + `masks` (fp32) of the global batch end up in
the root's global buffers -- scatter and gather inside the timed region, executed by the copy engines on peer memory
(avsep_b200/sharded.py).  On the way back the ranks push either `separated` and `masks`, or -- once the traffic through
the root's NVLink ports would take longer than a forward (8 GPUs) -- `masks` and a ticket: the root then rebuilds the
remote rows of `separated` = masks x mixed from the mixture it holds (one fp32 multiply, bit-identical to what the rank
computed, checked in the run), which halves the bytes into the root.  `scatter_gather.wire` names the format used
(choose_wire; AVSEP_GATHER=both|masks overrides), the other one is timed beside it (`scatter_gather_two_tensors` /
`scatter_gather_masks_only`), as is the no-traffic variant (`sharded_no_traffic`).  Weak scaling: the per-GPU batch is fixed.
Prints ONE JSON line (rank 0).  Metric: separated utterance-seconds per second = B_total * clip seconds / time.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "av-separation-transformer_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "separated utterance-sec/sec"
UNIT = "utt-s/s"
DEFAULT_MODEL = dict(freq_bins=257, d_model=256, nhead=4, num_encoder_layers=2, num_fusion_layers=2, num_speakers=2)
SCALED_MODEL = dict(freq_bins=257, d_model=512, nhead=8, num_encoder_layers=6, num_fusion_layers=6, num_speakers=3)
# BASELINE.json configs; (T, N) follow dataset.py:63-65,114 (T = 1 + samples // hop, N = 25 fps x seconds x 2 speakers)
CONFIGS = {
    "c1": dict(name="configs[0]: demo default, B=8", model=DEFAULT_MODEL, batch=8, T=63, N=50, hw=32, seconds=1.0,
               cpu_sample=8, audio="1 s @ 8 kHz"),
    "c2": dict(name="configs[1]: default model, B=256 throughput batch", model=DEFAULT_MODEL, batch=256, T=63, N=50,
               hw=32, seconds=1.0, cpu_sample=32, audio="1 s @ 8 kHz"),
    "c3": dict(name="configs[2]: long form", model=DEFAULT_MODEL, batch=32, T=1251, N=500, hw=32, seconds=10.0,
               cpu_sample=4, audio="10 s @ 16 kHz"),
    "c4": dict(name="configs[3]: scaled model (d=512, 8 heads, 6+6 layers, 3 speakers)", model=SCALED_MODEL, batch=256,
               T=63, N=50, hw=32, seconds=1.0, cpu_sample=8, audio="1 s @ 8 kHz"),
}
# module-level view of the active config (tests and tools import these names)
MODEL = dict(DEFAULT_MODEL)
CLIP_SECONDS = 1.0
T_FRAMES, N_FRAMES, FRAME_HW = 63, 50, 32
CPU_SAMPLE_B = 32


def select_config(key):
    global MODEL, CLIP_SECONDS, T_FRAMES, N_FRAMES, FRAME_HW, CPU_SAMPLE_B
    c = CONFIGS[key]
    MODEL = dict(c["model"])
    CLIP_SECONDS, T_FRAMES, N_FRAMES, FRAME_HW, CPU_SAMPLE_B = c["seconds"], c["T"], c["N"], c["hw"], c["cpu_sample"]
    return c


def workload_name(batch, key="c2"):
    c, m = CONFIGS[key], CONFIGS[key]["model"]
    return (f"{c['name']} (F={m['freq_bins']},d={m['d_model']},H={m['nhead']},{m['num_encoder_layers']}+"
            f"{m['num_fusion_layers']} layers,S={m['num_speakers']}), B={batch}/GPU, {c['audio']} "
            f"(T={c['T']}, N={c['N']}, {c['hw']}x{c['hw']}), SyntheticAVDataset-shaped")


# ----------------------------------------------------------------------------------------------
# clocks: in-process NVML sampling on a thread (a 50 ms nvidia-smi loop misses a 13 ms timed region)
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.sm, self.mx, self.reasons = index, [], None, set()
        self.h, self.err, self._stop, self._thr = None, None, threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:                                  # pragma: no cover - no NVML on the build box
            self.err = f"NVML unavailable ({e})"

    def sample(self):
        if self.h is None:
            return
        try:
            self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            try:
                bits = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                bits = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for name, bit in self.REASONS:
                if bits & bit:
                    self.reasons.add(name)
        except Exception as e:                                  # pragma: no cover
            self.err = str(e)

    def start(self):
        def loop():
            while not self._stop.is_set():
                self.sample()
                time.sleep(0.001)
        self._stop.clear()
        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def report(self, how):
        out = {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx,
               "samples": len(self.sm), "reasons": sorted(self.reasons), "how": how}
        if self.err:
            out["note"] = self.err
        return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), tensor_burst=float(d["bf16_tflops"]),
                    tensor_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback")


def source_hash(files=None):
    """Identifies kernel sources of the build being timed.  files = None: every source of the library; a list: those
    files of csrc/ (profiles/traffic.json records, per kernel, the translation unit the kernel is compiled from -- its
    .cu file and common.cuh -- and the hash of both at capture time: the capture stays valid while that kernel's own
    sources are unchanged, and is reported as absent once they differ)."""
    h = hashlib.sha256()
    csrc = os.path.join(PKG, "csrc")
    names = sorted(os.listdir(csrc)) if files is None else sorted(files)
    for name in names:
        if name.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(csrc, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------------------------
# algorithmic work per kernel class, per forward of B utterances (SURVEY.md section 8d formulas; DESIGN.md section 4)
# ----------------------------------------------------------------------------------------------
def kernel_work(B, model=None, T=None, N=None):
    m = MODEL if model is None else model
    T = T_FRAMES if T is None else T
    N = N_FRAMES if N is None else N
    d, F, S = m["d_model"], m["freq_bins"], m["num_speakers"]
    Le, Lf = m["num_encoder_layers"], m["num_fusion_layers"]
    Ma, Mv = B * T, B * N
    rows_enc = Le * (Ma + Mv)
    cnn_per_frame = 2 * 256 * 32 * 9 + 2 * 64 * 64 * 288 + 2 * 16 * 128 * 576
    flops = {
        "gemm.conv1d_0": 2 * Ma * d * 3 * F, "gemm.conv1d_2": 2 * Ma * d * 3 * d,
        "gemm.qkv": rows_enc * 2 * 3 * d * d, "gemm.out_proj": (rows_enc + Lf * Ma) * 2 * d * d,
        "gemm.ffn1": (rows_enc + Lf * Ma) * 2 * 4 * d * d, "gemm.ffn2": (rows_enc + Lf * Ma) * 2 * 4 * d * d,
        "gemm.cross_q": Lf * Ma * 2 * d * d, "gemm.cross_kv": Mv * 2 * (Lf * 2 * d) * d,
        "attn.self": Le * B * 4 * d * (T * T + N * N), "attn.cross": Lf * B * 4 * d * T * T,
        "visual_cnn": Mv * cnn_per_frame, "gemm.frame_proj": Mv * 2 * 128 * d,
        "gemm.dec0": Ma * 2 * 2 * d * d, "gemm.dec3_tail": Ma * 2 * S * F * 2 * d,
    }
    base_total = sum(flops.values())
    # fused kernels = sums of the classes they contain (each class is still counted once in the total)
    flops["ffn.fused"] = flops["gemm.ffn1"] + flops["gemm.ffn2"]
    per_row_layer = 2 * 3 * d * d + 2 * d * d + 2 * 2 * 4 * d * d            # qkv + out_proj + ffn1 + ffn2 per row
    # round 2: the stack launches also carry their input projection (Conv1d #2 / frame_proj), the visual one the K|V
    # projection of the fusion layers (on the T interpolated rows), the fusion one the SeparationDecoder
    flops["layer.audio_enc"] = Le * (Ma * per_row_layer + B * 4 * d * T * T) + flops["gemm.conv1d_2"]
    flops["layer.visual_enc"] = Le * (Mv * per_row_layer + B * 4 * d * N * N) + flops["gemm.frame_proj"] + \
        Ma * 2 * (Lf * 2 * d) * d
    per_row_fus = 2 * d * d + 2 * d * d + 2 * 2 * 4 * d * d                  # q + out_proj + ffn1 + ffn2 per row
    flops["layer.fusion"] = Lf * (Ma * per_row_fus + B * 4 * d * T * T)
    flops["layer.fusion_decoder"] = flops["layer.fusion"] + flops["gemm.dec0"] + flops["gemm.dec3_tail"]
    bytes_ = {
        # x (fp32) + y (fp32) in, x (fp32) + normalised operand (bf16) out = 14 B per element
        "add_layernorm": 14 * d,      # per row; multiplied by the rows of the launches below
        # masks + separated fp32 out, mixed fp32 in, bf16 A operand in
        "gemm.dec3_tail": Ma * S * F * 8 + B * F * T * 4 + Ma * 2 * d * 2,
        "prep_audio": B * F * T * 4 + B * (T + 2) * ((F + 7) // 8 * 8) * 2,
    }
    ln_rows = (1 + 2 * Le) * Ma + (1 + 2 * Le) * Mv + 2 * Lf * Ma
    bytes_["add_layernorm"] = ln_rows * d * 14
    return flops, bytes_, base_total


ROOT_LINK_TBS = 1.0     # rank 0's NVLink ports with scatter and gather running at once: ~0.5 + 0.5 TB/s measured
                        # (tools/nvlink_probe.py, profiles/r2_nvlink_root_copy_rates_n8.txt)


def choose_wire(world, in_bytes_per_rank, out_bytes_per_rank, ms_forward, override=None):
    """Wire format of the gather: 'both' (separated + masks pushed) while the root's links carry a step's traffic in
    less than a forward, else 'masks' (the root rebuilds `separated`: half of the bytes into it, at the price of an
    HBM-bound pass over the remote rows on the root).  Measured: 2 GPUs 0.536 (both) vs 0.561 ms (masks); 8 GPUs 1.07 vs
    0.73 ms.  AVSEP_GATHER=both|masks overrides."""
    if override in ("both", "masks"):
        return override
    if override not in (None, "", "auto"):
        raise SystemExit("AVSEP_GATHER must be 'auto', 'masks' or 'both'")
    link_ms = (world - 1) * (in_bytes_per_rank + out_bytes_per_rank) / (ROOT_LINK_TBS * 1e12) * 1e3
    return "masks" if link_ms > ms_forward else "both"


def shard_bounds(rank, world, per_rank_batch):
    """[lo, hi) utterance indices of this rank's shard of the global batch (weak scaling: fixed per-rank batch)."""
    return rank * per_rank_batch, (rank + 1) * per_rank_batch


def throughput(world, per_rank_batch, ms_per_step, clip_seconds=None):
    """Whole-job utterance-seconds per second from the slowest rank's step time."""
    cs = CLIP_SECONDS if clip_seconds is None else clip_seconds
    return world * per_rank_batch * cs / (ms_per_step * 1e-3)


def max_over_ranks_cpu(x):
    """MAX all-reduce of a host scalar on the default process group (gloo in tests)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def total_flops(B):
    return kernel_work(B)[2]


DUMP_BYTES = 64 * 10**6       # --dump-outputs writes at most this many bytes in all


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes each (name, tensor) of one step's outputs as out_dir/<name>.npy in float32, so that two
    builds run with the same arguments (hence the same seeded inputs and weights) can be compared output for output.
    Whole utterances (dim 0) are kept; when all of them would exceed DUMP_BYTES, every array keeps the same seeded
    sample of utterances, in index order.  Returns the number of utterances written."""
    import numpy as np
    import torch
    n = arrays[0][1].shape[0]
    per_utt = sum(t[0].numel() * 4 for _, t in arrays)
    keep = min(n, (DUMP_BYTES - 1024 * len(arrays)) // per_utt)       # 1 KB per file for the .npy header
    idx = None if keep == n else torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, keep, replace=False)))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays:
        t = t.detach() if idx is None else t.detach()[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    return keep


# ----------------------------------------------------------------------------------------------
# the reference's own CPU implementation -- the ONLY place bench.py touches oracle/
# ----------------------------------------------------------------------------------------------
def make_cpu_reference(state):
    """Returns (kind, forward(mixed, frames)).  kind "reference": the UNMODIFIED reference modules staged under
    oracle/_ref by oracle/make_ref.py (model.py:227-276), eval mode, no_grad; kind "port": the oracle's restatement on
    the same torch CPU operators, used only when oracle/_ref is absent."""
    import torch
    from oracle import make_ref
    P = {k: v.detach().cpu() for k, v in state.items()}
    if make_ref.ref_available():
        ref = make_ref.load_reference_model_module()
        model = ref.AVSeparationTransformer(**MODEL)
        model.load_state_dict(P, strict=True)
        model.eval()

        def fwd(mixed, frames):
            with torch.no_grad():
                return model(mixed, frames)
        return "reference", fwd
    from oracle import avsep_oracle_torch as otorch
    from oracle.weights import ModelConfig
    cfg = ModelConfig(**MODEL)
    return "port", (lambda mixed, frames: otorch.forward(P, cfg, mixed, frames))


def cpu_reference_throughput(state, mixed, frames, min_seconds=10.0, max_reps=8):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind, fwd = make_cpu_reference(state)
    fwd(mixed, frames)            # warm-up
    times = []
    t_all = time.perf_counter()
    while len(times) < max_reps and (time.perf_counter() - t_all < min_seconds or len(times) < 3):
        t0 = time.perf_counter()
        fwd(mixed, frames)
        times.append(time.perf_counter() - t0)
    best = min(times)
    return mixed.shape[0] * CLIP_SECONDS / best, cores, best, len(times), kind


def build_state(seed=0, precision="bf16"):
    """Random-init weights of the architecture (torch default init, as the reference constructs them), with
    non-trivial BatchNorm statistics.  Uses only torch.nn parameter containers -- no kernels involved."""
    import torch
    from avsep_b200 import AVSeparationTransformer
    torch.manual_seed(seed)
    model = AVSeparationTransformer(**MODEL, precision=precision)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, buf in model.named_buffers():
            if name.endswith("running_mean"):
                buf.copy_(0.1 * torch.randn(buf.shape, generator=g))
            elif name.endswith("running_var"):
                buf.copy_(0.5 + torch.rand(buf.shape, generator=g))
    return model


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU forward on all host threads, a bounded sample of the workload."""
    if rank != 0:
        return
    import torch
    from avsep_b200.synth import synthetic_batch
    model = build_state()
    state = model.state_dict()
    mixed, frames = synthetic_batch(CPU_SAMPLE_B, MODEL["freq_bins"], T_FRAMES, N_FRAMES, FRAME_HW, FRAME_HW, seed=100)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    kind, fwd = make_cpu_reference(state)
    for _ in range(max(1, min(args.warmup, 3))):
        fwd(mixed, frames)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = fwd(mixed, frames)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [("separated", out[0]), ("masks", out[1])])
    value = args.steps * CPU_SAMPLE_B * CLIP_SECONDS / dt
    sample = (f"B={CPU_SAMPLE_B} utterances of the same workload per step (CPU throughput is flat beyond B~32); "
              + ("the unmodified reference modules (oracle/_ref, model.py:227-276), eval mode, no_grad" if kind == "reference"
                 else "oracle port on the same torch CPU operators (oracle/_ref not staged)"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.batch, args.config), "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's threads (and therefore its first-touch pinned host buffers) to the CPU cores local to its GPU,
    so that the e2e host<->device copies of 8 ranks do not all cross one socket.  Returns the core count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {w * 64 + b for w, word in enumerate(mask) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception as e:                                   # affinity is an optimisation, never a requirement
        sys.stderr.write(f"bench.py: NUMA binding skipped ({e})\n")
    return None


def run_ours(args, rank, local_rank, world):
    # Everything except the final JSON line goes to stderr (NCCL / torchrun print to stdout on their own).
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import ctypes as C
    import torch
    import torch.distributed as dist
    from avsep_b200.synth import synthetic_batch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cores = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = args.batch
    F, S = MODEL["freq_bins"], MODEL["num_speakers"]
    T, N, HW = T_FRAMES, N_FRAMES, FRAME_HW
    model = build_state().to(dev)
    model.prepack(dev)
    eng = model.engine
    stream = torch.cuda.current_stream()
    st = C.c_void_p(stream.cuda_stream)

    def fwd_raw(mixed, frames, sep, masks, b=None):
        rc = eng.lib.avsep_forward(eng.h, mixed.data_ptr(), frames.data_ptr(), mixed.shape[0] if b is None else b, T, N,
                                   HW, HW, sep.data_ptr(), masks.data_ptr(), None, 0, st)
        if rc != 0:
            raise RuntimeError(eng.lib.avsep_last_error(eng.h).decode())

    # rotating input sets: inputs + outputs + activations per step already exceed the 126 MB L2 at B=256; three distinct
    # input sets make sure no step re-reads the previous step's inputs from L2.
    n_sets = 3
    lo, hi = shard_bounds(rank, world, B)     # this rank's utterances of the global batch; seeds differ per shard
    sets = [synthetic_batch(hi - lo, F, T, N, HW, HW, seed=100003 * i + lo, device=dev) for i in range(n_sets)]
    sep = torch.empty((B, S, F, T), device=dev)
    masks = torch.empty_like(sep)

    def step(i):
        fwd_raw(sets[i % n_sets][0], sets[i % n_sets][1], sep, masks)

    def timed(fn, steps, warmup, sampler=None):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler is not None:
            sampler.start()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        barrier()
        if sampler is not None:
            sampler.stop()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    def phase(msg):       # AVSEP_BENCH_VERBOSE=1: progress markers on stderr (locating a failure in a multi-rank run)
        if os.environ.get("AVSEP_BENCH_VERBOSE"):
            torch.cuda.synchronize()
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for i in range(args.warmup):
        step(i)
    phase("warm-up done")
    launches_per_step = eng.launch_count()
    ms_sharded = timed(step, args.steps, 0, sampler)
    if world == 1 and args.dump_outputs:      # the later passes below overwrite sep / masks
        n_dumped = dump_outputs(args.dump_outputs, [("separated", sep), ("masks", masks)])
        print(f"bench.py: wrote separated, masks of the last timed step ({n_dumped} of {B} utterances) to "
              f"{args.dump_outputs}", file=sys.stderr)

    # ---- N > 1 headline: scatter from the root, forward, gather to the root (copy engines over NVLink peer memory) ----
    sharded_entry, sg = None, None
    if world > 1:
        from avsep_b200.sharded import PeerMemoryCuda, ShardedForward
        shapes = dict(mixed=(F, T), frames=(N, HW, HW), out=(S, F, T))
        # what crosses NVLink on the way back: "masks" (ranks push masks + a ticket, the root rebuilds the remote rows of
        # `separated` from the mixture it holds -- bit-identical, half of the bytes into the root) or "both" (separated
        # and masks pushed as two tensors); chosen by choose_wire from the traffic through the root.  Either way separated + masks (fp32) of the global batch end up in
        # the root's buffers inside the timed region; the other wire format is timed right after as a side entry.
        wire = choose_wire(world, 4 * B * (F * T + N * HW * HW), 4 * B * 2 * S * F * T, ms_sharded,
                           os.environ.get("AVSEP_GATHER"))
        other_wire = "both" if wire == "masks" else "masks"
        lanes = int(os.environ.get("AVSEP_COPY_LANES", "1"))
        sg = ShardedForward(PeerMemoryCuda(eng), fwd_raw, B, shapes, rank, world, n_input_sets=n_sets,
                            copy_lanes=lanes, gather=wire)
        if rank == 0:
            for s_i, (gm, gf) in enumerate(sg.root_in):
                for r in range(world):
                    m_r, f_r = synthetic_batch(B, F, T, N, HW, HW, seed=100003 * s_i + r * B, device=dev)
                    gm[r * B:(r + 1) * B].copy_(m_r)
                    gf[r * B:(r + 1) * B].copy_(f_r)
        barrier()

        def sg_timed(sg, steps, warmup):
            for i in range(warmup):
                sg.step(i)
            sg.finish()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
            e0.record(stream)
            for i in range(steps):
                sg.step(i)
                marks[i].record(stream)           # diagnostic only: forward-to-forward intervals of this rank
            if rank != 0:
                stream.wait_stream(sg.s_in)
                stream.wait_stream(sg.s_out)      # this rank's last push is inside its timed interval
            elif hasattr(sg, "s_rb"):
                stream.wait_stream(sg.s_rb)       # masks-only gather: the root's last rebuild is inside it too
            e1.record(stream)
            sg.finish()
            wall = time.perf_counter() - t0
            per = sorted(a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks))
            spread = {"median_step_ms": round(max_over_ranks(per[len(per) // 2]), 4),
                      "slowest_step_ms": round(max_over_ranks(per[-1]), 4)}
            return max_over_ranks(e0.elapsed_time(e1)) / steps, max_over_ranks(wall * 1e3) / steps, spread

        phase("sharded (no traffic) timed; scatter/gather buffers ready")
        # warm-up covers every (input set, output buffer) pair of the root: 3 x 2 CUDA graphs, the first two uses of a
        # pair run eagerly / capture (forward_cached), so 12 steps keep graph instantiation out of the timed region
        ms_sg, ms_sg_wall, sg_spread = sg_timed(sg, args.steps, max(args.warmup, 2 * 2 * n_sets))
        phase("scatter/gather timed")
        # verify the gathered result on the root: shard r of the last step == the root's own forward of those inputs
        def sg_verify(sgx):
            if rank != 0:
                return None
            i_last = args.steps - 1
            gm, gf = sgx.root_in[i_last % n_sets]
            gsep, gmasks = sgx.root_out[i_last & 1]
            ok = True
            for r in sorted({0, 1, world - 1}):
                fwd_raw(gm[r * B:(r + 1) * B], gf[r * B:(r + 1) * B], sep, masks)
                torch.cuda.synchronize()
                ok = ok and bool(torch.equal(gsep[r * B:(r + 1) * B], sep)) and \
                    bool(torch.equal(gmasks[r * B:(r + 1) * B], masks))
            return ok

        verified = sg_verify(sg)
        if rank == 0 and args.dump_outputs:      # the global batch gathered into the root's buffers by the last step
            gsep, gmasks = sg.root_out[(args.steps - 1) & 1]
            n_dumped = dump_outputs(args.dump_outputs, [("separated", gsep), ("masks", gmasks)])
            print(f"bench.py: wrote separated, masks of the last timed step ({n_dumped} of {world * B} utterances) "
                  f"to {args.dump_outputs}", file=sys.stderr)
        barrier()
        # side entry: the same step with the other wire format
        wire_what = {
            "masks": "ranks push masks + a ticket (avsep_flag_signal), the root waits in stream order (avsep_flag_wait) "
                     "and rebuilds the remote shards' separated = masks x mixed (avsep_separate, bit-identical)",
            "both": "ranks push separated and masks as two tensors"}
        other_entry = None
        if not os.environ.get("AVSEP_BENCH_ONE_WIRE"):
            sg_o = ShardedForward(PeerMemoryCuda(eng), fwd_raw, B, shapes, rank, world, n_input_sets=n_sets,
                                  copy_lanes=lanes, gather=other_wire)
            if rank == 0:
                for (gm, gf), (hm, hf) in zip(sg.root_in, sg_o.root_in):
                    hm.copy_(gm)
                    hf.copy_(gf)
            barrier()
            ms_o, ms_o_wall, spread_o = sg_timed(sg_o, args.steps, max(args.warmup, 2 * 2 * n_sets))
            ok_o = sg_verify(sg_o)
            barrier()
            ms_oo = max(ms_o, ms_o_wall)
            other_entry = {
                "wire": other_wire, "ms_per_step": round(ms_oo, 4), "value": throughput(world, B, ms_oo),
                "bytes_into_rank0_per_step": sg_o.bytes_out_per_step * (world - 1),
                "bytes_out_of_rank0_per_step": sg_o.bytes_in_per_step * (world - 1),
                "gathered_equals_local_forward": ok_o, "step_spread": spread_o,
                "what": "the headline's scatter -> forward -> gather step with the other wire format: "
                        + wire_what[other_wire]}
            phase("other wire format timed")
        sharded_entry = {"ms_per_step": round(ms_sharded, 4), "value": throughput(world, B, ms_sharded),
                         "what": "every rank's shard stays on its GPU: inputs generated per rank, outputs not gathered"}
        ms_per_step = max(ms_sg, ms_sg_wall)     # device time of the slowest rank; wall clock as the cross-rank check
    else:
        ms_per_step = ms_sharded
    value = throughput(world, B, ms_per_step)
    if rank == 0 and len(sampler.sm) < 5:
        # a short timed region can fall between NVML samples: probe the same steps for ~150 ms right after it
        sampler.start()
        t0 = time.perf_counter()
        i = 0
        while time.perf_counter() - t0 < 0.15:
            step(i)
            i += 1
            if i % 16 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        sampler.stop()
        clocks = sampler.report("NVML in-process, 1 ms period: timed region + the same steps for 150 ms right after it")
    elif rank == 0:
        clocks = sampler.report("NVML in-process, 1 ms period, during the timed region")
    else:
        clocks = None
    barrier()

    phase("headline done")
    # ---- python_api: the drop-in module call `model(mixed, frames)` (what a user of the reference writes) -------------
    def python_api_ms(bsz, steps):
        ms_in = [(m[:bsz].contiguous(), f[:bsz].contiguous()) for m, f in sets]
        keep = None
        for i in range(36):        # every (input set, output block) pair is seen often enough to be graph-captured
            keep = model(*ms_in[i % n_sets])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            out = model(*ms_in[i % n_sets])
        e1.record(stream)
        torch.cuda.synchronize()
        del out
        ms_py = e0.elapsed_time(e1) / steps
        o_s, o_m = torch.empty((bsz, S, F, T), device=dev), torch.empty((bsz, S, F, T), device=dev)
        for i in range(6):
            fwd_raw(ms_in[i % n_sets][0], ms_in[i % n_sets][1], o_s, o_m)
        torch.cuda.synchronize()
        e0.record(stream)
        for i in range(steps):
            fwd_raw(ms_in[i % n_sets][0], ms_in[i % n_sets][1], o_s, o_m)
        e1.record(stream)
        torch.cuda.synchronize()
        return ms_py, e0.elapsed_time(e1) / steps

    python_api = None
    if world == 1:
        python_api = {}
        for bsz in sorted({min(8, B), B}):
            ms_py, ms_c = python_api_ms(bsz, max(20, min(args.steps, 100)))
            python_api[f"B={bsz}"] = {"module_call_ms": round(ms_py, 4), "c_abi_ms": round(ms_c, 4),
                                      "ratio": round(ms_py / ms_c, 3), "value": throughput(1, bsz, ms_py)}

    # ---- e2e: the public host-buffer call; pinned inputs H2D and results D2H every step -----------------
    h_sets = [(m.cpu().pin_memory(), f.cpu().pin_memory()) for m, f in sets[:2]]
    h_out = [(torch.empty((B, S, F, T)).pin_memory(), torch.empty((B, S, F, T)).pin_memory()) for _ in range(2)]
    e2e_steps = max(4, min(args.steps, 20))

    def e2e_run(n):
        """n batches through the streaming host entry point: batch i goes to I/O slot i % 2, and its results are
        waited for (= are in the pinned host buffers) before that slot is submitted again."""
        for i in range(n):
            slot = i % 2
            if i >= 2:
                eng.host_wait(slot)
            eng.forward_host_async(h_sets[slot][0], h_sets[slot][1], h_out[slot][0], h_out[slot][1], slot)
        eng.host_wait(0)
        eng.host_wait(1)

    e2e_run(4)
    barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    # the synchronous call (one batch at a time, results on the host when it returns), for reference
    for _ in range(2):
        eng.forward_host(h_sets[0][0], h_sets[0][1], h_out[0][0], h_out[0][1])
    t0 = time.perf_counter()
    for i in range(4):
        eng.forward_host(h_sets[i % 2][0], h_sets[i % 2][1], h_out[0][0], h_out[0][1])
    e2e_sync_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_stream_value = world * B * CLIP_SECONDS * e2e_steps / e2e_s
    e2e_sync_value = world * B * CLIP_SECONDS * 4 / e2e_sync_s
    e2e_value = max(e2e_stream_value, e2e_sync_value)
    h2d = (h_sets[0][0].numel() + h_sets[0][1].numel()) * 4
    d2h = (h_out[0][0].numel() + h_out[0][1].numel()) * 4
    # host <-> device copy ceiling of this box, measured the way the e2e path copies (one cudaMemcpyAsync per buffer
    # per direction, both directions at once, every rank at the same time): names the link the e2e number sits on
    cp_in, cp_out = torch.cuda.Stream(), torch.cuda.Stream()
    d_in = [torch.empty_like(t, device=dev) for t in h_sets[0]]

    def copy_round():
        with torch.cuda.stream(cp_in):
            for d_t, h_t in zip(d_in, h_sets[0]):
                d_t.copy_(h_t, non_blocking=True)
        with torch.cuda.stream(cp_out):
            h_out[0][0].copy_(sep, non_blocking=True)
            h_out[0][1].copy_(masks, non_blocking=True)

    for _ in range(2):
        copy_round()
    barrier()
    t0 = time.perf_counter()
    for _ in range(6):
        copy_round()
    torch.cuda.synchronize()
    copy_s = max_over_ranks(time.perf_counter() - t0) / 6
    barrier()
    host_link = {"h2d_gbs_per_rank": round(h2d / copy_s / 1e9, 1), "d2h_gbs_per_rank": round(d2h / copy_s / 1e9, 1),
                 "bidirectional_copy_ms_per_step": round(copy_s * 1e3, 3), "ranks_concurrent": world,
                 "ceiling_value": world * B * CLIP_SECONDS / copy_s,
                 "what": "pinned-memory copies of one step's inputs and outputs, both directions at once, all ranks at once"}

    # ---- N > 1 side entries -----------------------------------------------------------------------------------------
    extras_multi = None
    if world > 1:
        extras_multi = {}
        # NCCL variant of the same data path (dist.scatter of the inputs, dist.gather of masks + separated, fp32)
        G = world * B
        sep2, masks2 = torch.empty_like(sep), torch.empty_like(masks)
        loc_m, loc_f = torch.empty((B, F, T), device=dev), torch.empty((B, N, HW, HW), device=dev)
        if rank == 0:
            gm, gf = sg.root_in[0]
            gsep, gmasks = sg.root_out[0]
            sc_m, sc_f = list(gm.view(world, B, F, T).unbind(0)), list(gf.view(world, B, N, HW, HW).unbind(0))
            ga_s, ga_m = list(gsep.view(world, B, S, F, T).unbind(0)), list(gmasks.view(world, B, S, F, T).unbind(0))
        else:
            sc_m = sc_f = ga_s = ga_m = None

        def nccl_step(i):
            dist.scatter(loc_m, sc_m, src=0)
            dist.scatter(loc_f, sc_f, src=0)
            fwd_raw(loc_m, loc_f, sep2, masks2)
            dist.gather(sep2, ga_s, dst=0)
            dist.gather(masks2, ga_m, dst=0)

        phase("e2e / copy rounds done")
        n_g = max(6, min(args.steps, 30))
        ms_nccl = timed(nccl_step, n_g, 3)
        phase("nccl scatter/gather done")
        extras_multi["nccl_scatter_gather_fp32"] = {
            "ms_per_step": round(ms_nccl, 4), "value": throughput(world, B, ms_nccl),
            "what": "same data path with dist.scatter / dist.gather (NCCL send/recv kernels, in stream order, no overlap)"}
        # strong scaling of configs[1] as BASELINE.md states it: B=256 in total, 256/N per GPU (no traffic)
        if B % world == 0 and B // world >= 1:
            bs = B // world
            o_s, o_m = torch.empty((bs, S, F, T), device=dev), torch.empty((bs, S, F, T), device=dev)
            ins = [(m[:bs].contiguous(), f[:bs].contiguous()) for m, f in sets]
            ms_strong = timed(lambda i: fwd_raw(ins[i % n_sets][0], ins[i % n_sets][1], o_s, o_m), 50, 6)
            extras_multi["strong_scaling_global_batch"] = {
                "global_batch": B, "per_gpu_batch": bs, "ms_per_step": round(ms_strong, 4),
                "value": throughput(world, bs, ms_strong),
                "what": "BASELINE.md reading of configs[1]: the fixed global batch split over the GPUs, outputs stay sharded"}
        phase("strong scaling done")
        sweep = {}
        for bs in (8, 64, 1024):                       # configs[4]: per-GPU batch sweep (no traffic), this N
            ins = [synthetic_batch(bs, F, T, N, HW, HW, seed=7 + lo, device=dev)]
            o_s, o_m = torch.empty((bs, S, F, T), device=dev), torch.empty((bs, S, F, T), device=dev)
            ms_b = timed(lambda i: fwd_raw(ins[0][0], ins[0][1], o_s, o_m), 30, 6)
            sweep[f"B={bs}"] = {"ms_per_step": round(ms_b, 4), "value": throughput(world, bs, ms_b)}
            del ins, o_s, o_m
        extras_multi["per_gpu_batch_sweep"] = sweep

    phase("multi-GPU extras done")
    # ---- per-kernel pass (same steps again, every launch bracketed by CUDA events on the launching stream) ----
    eng.set_profile(True)
    eng.profile_report(reset=True)
    prof_steps = max(2, min(args.steps, 10))
    for i in range(prof_steps):
        step(i)
    prof = eng.profile_report(reset=True)
    eng.set_profile(False)
    barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    flops, bytes_, flops_total = kernel_work(B)
    tot_ms = sum(v[1] for v in prof.values()) or 1.0
    breakdown = {}
    for label, (n, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        per_step_ms = ms / prof_steps
        entry = {"launches_per_step": n // prof_steps, "ms_per_step": round(per_step_ms, 4),
                 "share": round(ms / tot_ms, 4)}
        if label in flops and label != "gemm.dec3_tail":
            entry["tflops"] = round(flops[label] / (per_step_ms * 1e-3) / 1e12, 2)
            entry["frac_of_tensor_peak"] = round(entry["tflops"] / peaks["tensor_burst"], 4)
        if label in bytes_:
            entry["gbs"] = round(bytes_[label] / (per_step_ms * 1e-3) / 1e9, 1)
            entry["frac_of_hbm_peak"] = round(entry["gbs"] / peaks["hbm"], 4)
        breakdown[label] = entry
    # dominant kernel = the largest share among the classes with an algorithmic work figure
    top = next((k for k, v in breakdown.items() if "tflops" in v or "gbs" in v), next(iter(breakdown)))
    te = breakdown[top]
    # DRAM bytes per launch of the dominant kernel from the ncu --set full capture of THIS build (the capture records
    # the hash of the kernel sources it was taken from; a stale capture is not reported)
    traffic, traffic_note = None, "no ncu capture recorded for this build"
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        ent = tj.get("kernels", {}).get(top, {})
        if ent.get("src") and ent.get("src_hash") == source_hash(ent["src"]) and tj.get("batch") == B and \
                tj.get("config") == args.config:
            traffic = ent.get("traffic")
            traffic_note = tj.get("source") + "; valid for this build: " + " + ".join(ent["src"]) + " unchanged since the capture"
        else:
            traffic_note = "profiles/traffic.json was captured from different kernel sources / another workload"
    n_top = max(1, te["launches_per_step"])
    if "tflops" in te:
        roofline = {"kernel": top, "bound": "tensor", "achieved": te["tflops"], "peak": peaks["tensor_burst"],
                    "unit": "TFLOP/s", "frac": round(te["tflops"] / peaks["tensor_burst"], 4), "traffic": traffic,
                    "peak_source": peaks["source"] + " (burst bf16: every launch is timed alone, behind a spin kernel)",
                    "launch_ms": round(te["ms_per_step"] / n_top, 4),
                    "algorithmic_flops_per_launch": flops[top] / n_top}
    else:
        roofline = {"kernel": top, "bound": "hbm", "achieved": te["gbs"], "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": round(te["gbs"] / peaks["hbm"], 4), "traffic": traffic, "peak_source": peaks["source"],
                    "launch_ms": round(te["ms_per_step"] / n_top, 4),
                    "algorithmic_bytes_per_launch": bytes_[top] / n_top}
    roofline["traffic_source"] = traffic_note
    roofline["whole_step"] = {"model_tflops": round(flops_total / (ms_sharded * 1e-3) / 1e12, 2),
                              "frac_of_tensor_peak": round(flops_total / (ms_sharded * 1e-3) / 1e12 / peaks["tensor_burst"], 4)}

    cfg_entry = {"workload": workload_name(B, args.config), "config": args.config, "global_batch": world * B,
                 "rank_cpu_affinity_cores": numa_cores,
                 "l2": f"{n_sets} rotating input sets; per-step footprint (inputs+outputs+activations) > 126 MB L2"
                       if B * T >= 4096 else f"{n_sets} rotating input sets (small batch: the working set fits L2, as it does in use)"}
    if world > 1:
        cfg_entry["parallelism"] = (f"batch-sharded x{world}: inputs scattered from rank 0, separated+masks (fp32) gathered "
                                    "into rank 0's buffers inside the timed region, copy engines over NVLink peer memory; "
                                    "on the wire: " + wire_what[wire])
    else:
        cfg_entry["parallelism"] = "batch-sharded x1"
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": cfg_entry, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps,
                "api": ("avsep_forward_host_async on two I/O slots + avsep_host_wait" if e2e_stream_value >= e2e_sync_value
                        else "avsep_forward_host (one call per batch)") +
                       " (pinned host buffers; every step's H2D and D2H inside the timed region)",
                "streaming_value": e2e_stream_value, "sync_call_value": e2e_sync_value, "host_link": host_link},
        "gpu_launches": launches_per_step * args.steps,
        "gflop_per_step": flops_total / 1e9,
        "model_tflops": round(flops_total / (ms_sharded * 1e-3) / 1e12, 2),
        "roofline": roofline,
        "kernels": breakdown,
    }
    if python_api is not None:
        out["python_api"] = python_api
    if world > 1:
        out["sharded_no_traffic"] = sharded_entry
        if other_entry is not None:
            out["scatter_gather_masks_only" if other_wire == "masks" else "scatter_gather_two_tensors"] = other_entry
        out["scatter_gather"] = {
            "wire": wire,
            "ms_per_step_device": round(ms_sg, 4), "ms_per_step_wall": round(ms_sg_wall, 4),
            "step_spread": dict(sg_spread, what="forward-to-forward intervals inside the timed region, max over ranks "
                                                "(diagnostic: a one-off stall shows as slowest >> median)"),
            "bytes_out_of_rank0_per_step": sg.bytes_in_per_step * (world - 1),
            "bytes_into_rank0_per_step": sg.bytes_out_per_step * (world - 1),
            "rank0_egress_gbs": round(sg.bytes_in_per_step * (world - 1) / (ms_per_step * 1e-3) / 1e9, 1),
            "rank0_ingress_gbs": round(sg.bytes_out_per_step * (world - 1) / (ms_per_step * 1e-3) / 1e9, 1),
            "gathered_equals_local_forward": verified,
            "note": "the root's NVLink ports carry every other rank's inputs out and outputs in: once a step is shorter "
                    "than those transfers the 8-GPU value is bound by one GPU's NVLink bandwidth, not by the kernels"}
        out.update(extras_multi)
    if world == 1 and args.config in ("c1", "c2"):
        # The same workload waveform to waveform (SURVEY 8f rank 4): STFT of the 1 s mixture, forward on its magnitude,
        # masks applied to the complex mixture, inverse STFT -- three C-ABI calls per step, buffers preallocated.
        n_fft, hop, L = 2 * (F - 1), 128, int(8000 * CLIP_SECONDS)
        g = torch.Generator(device=dev).manual_seed(7)
        waves_in = [0.3 * torch.randn(B, L, device=dev, generator=g) for _ in range(n_sets)]
        spec = torch.empty(B, F, T, device=dev, dtype=torch.complex64)
        mag = torch.empty(B, F, T, device=dev)
        waves_out = torch.empty(B, S, L, device=dev)

        def wstep(i):
            frames = sets[i % n_sets][1]
            rc = eng.lib.avsep_stft(eng.h, waves_in[i % n_sets].data_ptr(), B, L, n_fft, hop, spec.data_ptr(),
                                    mag.data_ptr(), st)
            rc = rc or eng.lib.avsep_forward(eng.h, mag.data_ptr(), frames.data_ptr(), B, T, N, HW, HW, sep.data_ptr(),
                                             masks.data_ptr(), None, 0, st)
            rc = rc or eng.lib.avsep_istft(eng.h, spec.data_ptr(), masks.data_ptr(), B, S, T, n_fft, hop, L,
                                           waves_out.data_ptr(), st)
            if rc != 0:
                raise RuntimeError(eng.lib.avsep_last_error(eng.h).decode())

        w_steps = max(4, min(args.steps, 50))
        w_ms = timed(wstep, w_steps, 6)
        out["waveform_to_waveform"] = {"ms_per_step": round(w_ms, 4), "value": throughput(1, B, w_ms), "unit": UNIT,
                                       "steps": w_steps, "samples_per_utterance": L,
                                       "calls": "avsep_stft -> avsep_forward -> avsep_istft, inputs resident"}
    if world == 1 and args.config == "c2" and not args.no_sweep:
        sweep = {}
        for bs in (1, 8, 64, 1024):                    # configs[4]: per-GPU batch sweep
            ins = synthetic_batch(bs, F, T, N, HW, HW, seed=7, device=dev)
            o_s, o_m = torch.empty((bs, S, F, T), device=dev), torch.empty((bs, S, F, T), device=dev)
            ms_b = timed(lambda i: fwd_raw(ins[0], ins[1], o_s, o_m), 30, 6)
            sweep[f"B={bs}"] = {"ms_per_step": round(ms_b, 4), "value": throughput(1, bs, ms_b)}
        out["per_gpu_batch_sweep"] = sweep
    if world == 1 and not args.no_cpu_baseline:
        nb = min(CPU_SAMPLE_B, B)
        m_cpu, f_cpu = sets[0][0][:nb].cpu(), sets[0][1][:nb].cpu()
        v, cores, best, reps, kind = cpu_reference_throughput(model.state_dict(), m_cpu, f_cpu)
        out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                               "sample": f"first {nb} utterances of the same batch, best of {reps} forwards "
                                         f"({best * 1e3:.0f} ms each), "
                                         + ("the unmodified reference modules (oracle/_ref)" if kind == "reference"
                                            else "oracle port on torch CPU ops") + f", {cores} threads"}
    os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json config (default c2 = configs[1])")
    ap.add_argument("--batch", type=int, default=None, help="utterances per GPU per step (default: the config's)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's outputs as DIR/separated.npy and "
                         "DIR/masks.npy (float32, whole utterances; a fixed seeded sample of them above 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    cfg = select_config(args.config)
    if args.batch is None:
        args.batch = cfg["batch"]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # launched without torchrun: re-exec under torch.distributed.run, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__),
               "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup),
               "--config", args.config, "--batch", str(args.batch)] + \
              (["--no-cpu-baseline"] if args.no_cpu_baseline else []) + (["--no-sweep"] if args.no_sweep else []) + \
              (["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
