"""ShardedForward(varlen=True) on real peer memory (needs >= 2 GPUs; skipped on a one-GPU box): three input sets with
different per-utterance lengths and NaN in their padding, root outputs prefilled with NaN.  After every step, with
both tensors on the wire and with masks only (the root rebuilds `separated` with avsep_separate_varlen), the root's
buffers must hold what avsep_forward_varlen of the whole global batch gives on the root, bit for bit."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_sharded_gpu import _free_port

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from oracle.weights import CONFIGS, make_inputs, make_state_dict
        from tests.helpers import build_model
        from avsep_b200.sharded import PeerMemoryCuda, ShardedForward
        cfg = CONFIGS["default"]
        B, T, N, HW, n_sets = 6, 63, 50, 32, 3
        model = build_model(cfg, make_state_dict(cfg, seed=83, gain=2.0), "bf16", device=dev)
        model.prepack(dev)
        eng = model.engine
        shapes = dict(mixed=(cfg.freq_bins, T), frames=(N, HW, HW), out=(cfg.num_speakers, cfg.freq_bins, T))

        def fwd(mixed, frames, sep, masks, lengths, frame_lengths):
            eng.forward(mixed, frames, out=(sep, masks), lengths=lengths, frame_lengths=frame_lengths)

        rng = np.random.default_rng(84)
        glens = []
        for _ in range(n_sets):
            lens = rng.integers(1, T + 1, world * B).astype(np.int32)
            lens[0], lens[-1] = T, 1
            flens = np.maximum(1, np.round(lens * N / T)).astype(np.int32)
            glens.append((torch.from_numpy(lens), torch.from_numpy(flens)))
        results = {}
        for gather in ("both", "masks"):
            sf = ShardedForward(PeerMemoryCuda(eng), fwd, B, shapes, rank, world, n_input_sets=n_sets, gather=gather,
                                varlen=True)
            if rank == 0:
                for s_i, ((gm, gf), (gl, gfl)) in enumerate(zip(sf.root_in, sf.root_lens)):
                    m, f = make_inputs(cfg, world * B, T, N, HW, HW, seed=90 + s_i, kind="dataset")
                    lens, flens = glens[s_i]
                    for u in range(world * B):
                        m[u, :, lens[u]:] = np.nan
                        f[u, flens[u]:] = np.nan
                    gm.copy_(torch.from_numpy(m))
                    gf.copy_(torch.from_numpy(f))
                    gl.copy_(lens)
                    gfl.copy_(flens)
                for o_s, o_m in sf.root_out:
                    o_s.fill_(float("nan"))
                    o_m.fill_(float("nan"))
            torch.cuda.synchronize()
            dist.barrier()
            ok = True
            for i in range(7):
                sf.step(i)
                sf.finish()
                if rank == 0:
                    gm, gf = sf.root_in[i % n_sets]
                    gl, gfl = sf.root_lens[i % n_sets]
                    want_sep, want_masks = eng.forward(gm, gf, lengths=gl, frame_lengths=gfl)
                    got_sep, got_masks = sf.root_out[i & 1]
                    ok = ok and bool(torch.equal(got_sep, want_sep)) and bool(torch.equal(got_masks, want_masks))
                    ok = ok and bool(torch.isfinite(got_sep).all())
                dist.barrier()
            if rank == 0:
                results[gather] = (ok, sf.bytes_in_per_step, sf.bytes_out_per_step)
            dist.barrier()
        if rank == 0:
            out.update(results)
    finally:
        dist.destroy_process_group()


def test_varlen_scatter_forward_gather_two_gpus_both_wire_formats():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world, port = 2, _free_port()
    with mp.Manager() as m:
        out = m.dict()
        mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
        assert out["both"][0] is True and out["masks"][0] is True, dict(out)
        assert out["masks"][2] * 2 == out["both"][2]
        assert out["both"][1] == out["masks"][1] == 4 * 6 * (257 * 63 + 50 * 32 * 32 + 2)
