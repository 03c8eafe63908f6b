"""What variable-length batches cost on the multi-GPU path (avsep_b200/sharded.py, ShardedForward(varlen=True)).
Default model, bf16, B = 256 utterances per GPU (T = 63 audio frames, N = 50 lip frames of 32 x 32), one process per
GPU, both wire formats.  Three kinds of step, each timed as scatter -> forward -> gather steps after warm-up, CUDA
events on every rank, three rotating input sets:

  uniform        varlen=False, avsep_forward
  varlen_full    varlen=True with every length full (T_b = 63, N_b = 50): the overhead of carrying lengths
  varlen_ragged  varlen=True on the seeded ragged batch of tools/waveform_varlen_bench.py: T_b uniform in [16, 63],
                 N_b = max(1, round(50 T_b / 63)), over the global batch

The wire still moves padded tensors, so a ragged step moves the same bytes as a full one.  Rank 0 prints one JSON line
per (wire format, kind): card, power limit, per-rank mean ms per step, median and slowest step, utterances per second
of the slowest rank, and whether the root's buffers after the last step equal its own forward of the whole batch.

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/sharded_varlen_probe.py [steps]
"""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "av-separation-transformer_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
import bench  # noqa: E402
from avsep_b200.sharded import PeerMemoryCuda, ShardedForward  # noqa: E402
from avsep_b200.synth import synthetic_batch  # noqa: E402
from varlen_bench import card_info  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
STEPS = int(sys.argv[1]) if len(sys.argv) > 1 else 60
WARM = 6
B, F, S = 256, bench.MODEL["freq_bins"], bench.MODEL["num_speakers"]
T, N, HW = bench.T_FRAMES, bench.N_FRAMES, bench.FRAME_HW
model = bench.build_state().to(dev)
model.prepack(dev)
eng = model.engine
stream = torch.cuda.current_stream()
st = C.c_void_p(stream.cuda_stream)
shapes = dict(mixed=(F, T), frames=(N, HW, HW), out=(S, F, T))
card, power_w = card_info(local)

rng = np.random.default_rng(1)                     # tools/waveform_varlen_bench.py, seed 0: default_rng(seed + 1)
t_rag = rng.integers(16, T + 1, world * B).astype(np.int32)
n_rag = np.maximum(1, np.round(t_rag * N / T)).astype(np.int32)
LENGTHS = {"varlen_full": (np.full(world * B, T, np.int32), np.full(world * B, N, np.int32)),
           "varlen_ragged": (t_rag, n_rag)}


def check(rc):
    if rc != 0:
        raise RuntimeError(eng.lib.avsep_last_error(eng.h).decode())


def fwd_uniform(mixed, frames, sep, masks):
    check(eng.lib.avsep_forward(eng.h, mixed.data_ptr(), frames.data_ptr(), mixed.shape[0], T, N, HW, HW,
                                sep.data_ptr(), masks.data_ptr(), None, 0, st))


def fwd_varlen(mixed, frames, sep, masks, lens, flens):
    check(eng.lib.avsep_forward_varlen(eng.h, mixed.data_ptr(), frames.data_ptr(), lens.data_ptr(), flens.data_ptr(),
                                       mixed.shape[0], T, N, HW, HW, sep.data_ptr(), masks.data_ptr(), None, 0, st))


def run(kind, gather):
    varlen = kind != "uniform"
    sg = ShardedForward(PeerMemoryCuda(eng), fwd_varlen if varlen else fwd_uniform, B, shapes, rank, world,
                        n_input_sets=3, gather=gather, varlen=varlen)
    if rank == 0:
        for s_i, (gm, gf) in enumerate(sg.root_in):
            for r in range(world):
                m_r, f_r = synthetic_batch(B, F, T, N, HW, HW, seed=1 + s_i, device=dev)
                gm[r * B:(r + 1) * B].copy_(m_r)
                gf[r * B:(r + 1) * B].copy_(f_r)
            if varlen:
                lens, flens = LENGTHS[kind]
                sg.root_lens[s_i][0].copy_(torch.from_numpy(lens))
                sg.root_lens[s_i][1].copy_(torch.from_numpy(flens))
    torch.cuda.synchronize()
    dist.barrier()
    for i in range(WARM):
        sg.step(i)
    sg.finish()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(STEPS)]
    e0.record(stream)
    for i in range(STEPS):
        sg.step(i)
        marks[i].record(stream)
    if rank != 0:
        stream.wait_stream(sg.s_in)
        stream.wait_stream(sg.s_out)
    elif hasattr(sg, "s_rb"):
        stream.wait_stream(sg.s_rb)
    e1.record(stream)
    sg.finish()
    per = sorted(a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks))
    t = torch.tensor([e0.elapsed_time(e1) / STEPS, per[len(per) // 2], per[-1]], device=dev)
    every = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(every, t)
    if rank == 0:
        last = STEPS - 1
        gm, gf = sg.root_in[last % 3]
        lens = [x[:] for x in sg.root_lens[last % 3]] if varlen else []
        sep_w, masks_w = torch.empty_like(sg.root_out[0][0]), torch.empty_like(sg.root_out[0][1])
        (fwd_varlen if varlen else fwd_uniform)(gm, gf, sep_w, masks_w, *lens)
        torch.cuda.synchronize()
        sep_g, masks_g = sg.root_out[last & 1]
        same = bool(torch.equal(sep_g, sep_w)) and bool(torch.equal(masks_g, masks_w))
        ms = [round(float(x[0]), 4) for x in every]
        print(json.dumps({"tool": "sharded_varlen_probe", "card": card, "power_limit_w": power_w, "world": world,
                          "per_gpu_batch": B, "gather": gather, "kind": kind, "steps": STEPS,
                          "ms_per_step_per_rank": ms, "median_step_ms": [round(float(x[1]), 4) for x in every],
                          "slowest_step_ms": [round(float(x[2]), 4) for x in every],
                          "utt_per_s": round(world * B / (max(ms) * 1e-3)), "bytes_in_per_step": sg.bytes_in_per_step,
                          "bytes_out_per_step": sg.bytes_out_per_step, "root_equals_whole_batch_forward": same}),
              flush=True)
    for ptr in sg.ptr.values():       # peers unmap before the root frees
        if rank != 0:
            eng.lib.avsep_shared_close(eng.h, C.c_void_p(ptr))
    torch.cuda.synchronize()
    dist.barrier()
    for ptr in sg.ptr.values():
        if rank == 0:
            eng.lib.avsep_shared_free(eng.h, C.c_void_p(ptr))
    del sg
    torch.cuda.synchronize()
    dist.barrier()


for _ in range(int(os.environ.get("PROBE_REPEAT", "2"))):
    for gather in ("both", "masks"):
        for kind in ("uniform", "varlen_full", "varlen_ragged"):
            run(kind, gather)
dist.destroy_process_group()
