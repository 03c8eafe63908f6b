"""CPU, gloo: ShardedForward(varlen=True) -- per-utterance lengths through the scatter -> forward -> gather path.  Every
rank's forward must see its own shard of each input set's lengths, the root's masks-only rebuild must get the remote
shards' slice, and the root's buffers must end up equal to a forward of the whole batch, with NaN in the padding of the
inputs and in the root's outputs before the first step."""
import ctypes
import os

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_multirank_cpu import _free_port, _HostBackend

B, SHAPES, N_SETS = 3, dict(mixed=(5, 7), frames=(4, 2, 2), out=(2, 5, 7)), 3


class _VarlenHostBackend(_HostBackend):
    """_HostBackend plus the two calls a varlen ShardedForward makes: int32 views and the rebuild with lengths (which
    stores 0 past a length and never lets the padding into the product, like avsep_separate_varlen)."""

    def view_i32(self, ptr, shape):
        n = 1
        for s in shape:
            n *= s
        return torch.frombuffer((ctypes.c_int32 * n).from_address(ptr), dtype=torch.int32).view(*shape)

    def separate_varlen(self, masks_ptr, mixed_ptr, lens_ptr, n_utt, T, sep_ptr, stream):
        S, F = self.out_shape[0], self.out_shape[1]
        lens = self.view_i32(lens_ptr, (n_utt,)).clamp(1, T)
        self.rebuild_lens = getattr(self, "rebuild_lens", []) + [lens.tolist()]
        masks = self.view(masks_ptr, (n_utt, S, F, T))
        mixed = self.view(mixed_ptr, (n_utt, F, T))
        live = (torch.arange(T) < lens[:, None]).view(n_utt, 1, 1, T)
        self.view(sep_ptr, (n_utt, S, F, T)).copy_(torch.where(live, masks * mixed.unsqueeze(1), 0.0))


def _fake_forward_varlen(mixed, frames, sep, masks, lens, flens):
    """Per-utterance function of the first lens[b] frames / flens[b] lip frames only; 0 past lens[b]."""
    sep.zero_()
    masks.zero_()
    for b in range(mixed.shape[0]):
        tb, nb = int(lens[b]), int(flens[b])
        w = frames[b, :nb].mean()
        for s in range(sep.shape[1]):
            masks[b, s, :, :tb] = torch.sigmoid(mixed[b, :, :tb] * (s + 1) + w)
            sep[b, s, :, :tb] = masks[b, s, :, :tb] * mixed[b, :, :tb]


def _global_lengths(world):
    """Different lengths per input set (full, 1 and values in between), the same on every rank."""
    g = torch.Generator().manual_seed(7)
    T, N = SHAPES["mixed"][1], SHAPES["frames"][0]
    out = []
    for _ in range(N_SETS):
        lens = torch.randint(1, T + 1, (world * B,), generator=g, dtype=torch.int32)
        flens = torch.randint(1, N + 1, (world * B,), generator=g, dtype=torch.int32)
        lens[0], lens[-1], flens[1] = T, 1, N
        out.append((lens, flens))
    return out


def _worker(rank, world, port, out, lanes, gather, n_steps):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from avsep_b200.sharded import ShardedForward
    be = _VarlenHostBackend()
    be.out_shape = SHAPES["out"]
    seen = []

    def fwd(mixed, frames, sep, masks, lens, flens):
        assert lens.dtype == torch.int32 and flens.dtype == torch.int32 and lens.shape == (B,)
        seen.append((lens.tolist(), flens.tolist()))
        _fake_forward_varlen(mixed, frames, sep, masks, lens, flens)

    try:
        glens = _global_lengths(world)
        sf = ShardedForward(be, fwd, B, SHAPES, rank, world, n_input_sets=N_SETS, copy_lanes=lanes, gather=gather,
                            varlen=True)
        if rank == 0:
            assert len(sf.root_lens) == N_SETS and all(len(p) == 2 for p in sf.root_lens)
            g = torch.Generator().manual_seed(0)
            for (m, f), (l_v, fl_v), (lens, flens) in zip(sf.root_in, sf.root_lens, glens):
                m.copy_(torch.randn(m.shape, generator=g))
                f.copy_(torch.rand(f.shape, generator=g))
                for u in range(world * B):            # the padding holds NaN: it must never reach an output
                    m[u, :, lens[u]:] = float("nan")
                    f[u, flens[u]:] = float("nan")
                l_v.copy_(lens)
                fl_v.copy_(flens)
            for o_s, o_m in sf.root_out:
                o_s.fill_(float("nan"))
                o_m.fill_(float("nan"))
        dist.barrier()
        for i in range(n_steps):
            sf.step(i)
        sf.finish()
        lo, hi = rank * B, (rank + 1) * B
        want_seen = [(glens[i % N_SETS][0][lo:hi].tolist(), glens[i % N_SETS][1][lo:hi].tolist()) for i in range(n_steps)]
        out[f"seen_ok{rank}"] = seen == want_seen
        if rank == 0:
            ok = True
            for i in (n_steps - 2, n_steps - 1):         # the two steps still held by the double-buffered outputs
                m, f = sf.root_in[i % N_SETS]
                sep_ref, masks_ref = torch.empty(world * B, *SHAPES["out"]), torch.empty(world * B, *SHAPES["out"])
                _fake_forward_varlen(m, f, sep_ref, masks_ref, *glens[i % N_SETS])
                sep, masks = sf.root_out[i & 1]
                ok = ok and torch.equal(sep, sep_ref) and torch.equal(masks, masks_ref)
            out["ok"] = ok
            out["rebuild_ok"] = getattr(be, "rebuild_lens", []) == (
                [glens[i % N_SETS][0][B:].tolist() for i in range(n_steps)] if gather == "masks" and world > 1 else [])
            out["bytes"] = (sf.bytes_in_per_step, sf.bytes_out_per_step)
        dist.barrier()
    finally:
        be.close(unlink=(rank == 0))
        dist.destroy_process_group()


def _run(world, lanes, gather, n_steps):
    with mp.Manager() as m:
        out = m.dict()
        mp.spawn(_worker, args=(world, _free_port(), out, lanes, gather, n_steps), nprocs=world, join=True)
        return dict(out)


def test_varlen_scatter_gather_world_two_both_wire_formats_gloo():
    for gather in ("both", "masks"):
        out = _run(2, 1, gather, 5)
        assert out["ok"] and out["rebuild_ok"], (gather, out)
        assert out["seen_ok0"] and out["seen_ok1"], (gather, out)
        # the length shards (2 x B int32) ride with the inputs; the outputs stay padded tensors
        assert out["bytes"] == (4 * B * (35 + 16 + 2), 4 * B * (1 if gather == "masks" else 2) * 70), out


def test_varlen_masks_only_world_three_copy_lanes_gloo():
    """Two remote ranks, each transfer cut into three pieces (the length shards too): the rebuild covers both remote
    shards with their lengths in one call per step."""
    out = _run(3, 3, "masks", 8)
    assert out["ok"] and out["rebuild_ok"], out
    assert out["seen_ok0"] and out["seen_ok1"] and out["seen_ok2"], out
