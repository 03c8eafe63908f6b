"""Batch sharding of the forward path over the GPUs of one box, one process per GPU (SURVEY.md 8e).

No op of the model mixes utterances in eval mode (reference model.py: BatchNorm on running statistics :83-89,
attention per sample), so the batch shards with no collective inside the model.  What moves between GPUs is what the
north star names: the root's inputs are scattered, ``separated`` / ``masks`` are gathered.

    root (rank 0)                          rank r > 0
    -------------                          ----------
    global inputs  [sets][world*B, ...] -> pull own shard over NVLink      (copy stream, copy engine)
                                           forward on the local shard      (compute stream, libavsep kernels)
    global outputs [2][world*B, ...]    <- push separated + masks shard    (copy stream, copy engine)

The root's buffers come from ``avsep_shared_alloc`` (cudaMalloc + an inter-process handle); the other ranks map them
with ``avsep_shared_open`` and move data with ``avsep_copy_async`` -- peer-memory copies executed by the copy engines,
so the transfers of step i-1 / i+1 run under the kernels of step i without taking SMs from them (an NCCL send/recv
pair needs CTAs on both ends).  ``torch.distributed`` carries the 64-byte handles and the barriers, nothing else.
The root computes its own shard in place (zero copy).  Local input / output buffers are double buffered and ordered
with events; the root's output buffers are double buffered as well, so a consumer on the root can read step i-1 while
step i is being written.

``gather="masks"`` (SURVEY 8e: "gather only masks, the root recomputes separated = masks x mixed, which it already
holds") halves the bytes into the root: a rank pushes its ``masks`` shard only and then raises a ticket in the root's
memory (``avsep_flag_signal``, same stream, so it lands after the data); the root's rebuild stream waits for every
rank's ticket (``avsep_flag_wait``: a one-CTA kernel polling the root's own memory -- no host round trip, no
collective), runs ``avsep_separate`` over the remote shards -- one fp32 multiply per element, bit-identical to what
the remote decoder epilogue wrote -- and acknowledges with a ticket in every rank's memory, which is what a rank
waits for before it overwrites that output slot two steps later.  The root ends up with the same bytes in the same
buffers as with ``gather="both"``.

``varlen=True`` carries per-utterance lengths through the same path (a variable-length batch, avsep_forward_varlen):
the root holds two more int32 [world*B] buffers per input set, audio frames and lip frames per utterance, which every
rank pulls with the same copy calls as its inputs; the forward gets them as device tensors, and the masks-only rebuild
runs avsep_separate_varlen over the remote shards' slice of them, which stores 0 past each length without reading the
(possibly NaN) padding -- so both wire formats still leave the same bytes on the root.  The scatter and gather still
move padded tensors.

The memory backend is injected so that the bookkeeping (shard offsets, buffer rotation, ordering) is covered by
world_size-2 gloo tests on CPU (tests/test_multirank_cpu.py); on a GPU box the backend is the C ABI above.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import _lib

__all__ = ["shard_slices", "PeerMemoryCuda", "ShardedForward"]


def shard_slices(world: int, per_rank_batch: int):
    """[(lo, hi)] per rank: contiguous, disjoint shards that tile the global batch (weak scaling: fixed per-rank batch)."""
    return [(r * per_rank_batch, (r + 1) * per_rank_batch) for r in range(world)]


class _RawCuda:
    """Minimal __cuda_array_interface__ holder so that torch can view memory owned by libavsep."""

    def __init__(self, ptr: int, n: int, typestr: str = "<f4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class PeerMemoryCuda:
    """avsep_shared_alloc / avsep_shared_open / avsep_copy_async of one engine (one GPU, one process)."""

    def __init__(self, engine):
        self.eng = engine
        self.dev = torch.device("cuda", engine.device)

    def alloc(self, nfloats: int):
        ptr = C.c_void_p()
        handle = C.create_string_buffer(_lib.IPC_HANDLE_BYTES)
        self.eng._check(self.eng.lib.avsep_shared_alloc(self.eng.h, nfloats * 4, C.byref(ptr), handle), "avsep_shared_alloc")
        return int(ptr.value), bytes(handle.raw)

    def open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        self.eng._check(self.eng.lib.avsep_shared_open(self.eng.h, handle, C.byref(ptr)), "avsep_shared_open")
        return int(ptr.value)

    def view(self, ptr: int, shape) -> torch.Tensor:
        n = 1
        for s in shape:
            n *= int(s)
        return torch.as_tensor(_RawCuda(ptr, n), device=self.dev).view(*shape)

    def view_i32(self, ptr: int, shape) -> torch.Tensor:
        return torch.as_tensor(_RawCuda(ptr, _prod(shape), "<i4"), device=self.dev).view(*shape)

    def empty(self, shape) -> torch.Tensor:
        return torch.empty(*shape, device=self.dev, dtype=torch.float32)

    def copy(self, dst_ptr: int, src_ptr: int, nfloats: int, stream):
        self.eng._check(self.eng.lib.avsep_copy_async(self.eng.h, C.c_void_p(dst_ptr), C.c_void_p(src_ptr), nfloats * 4,
                                                      C.c_void_p(stream.cuda_stream)), "avsep_copy_async")

    def zero(self, ptr: int, nfloats: int):
        self.view(ptr, (nfloats,)).zero_()

    def _flag_array(self, ptrs):
        return (C.c_void_p * len(ptrs))(*[int(p) for p in ptrs])

    def signal(self, flag_ptrs, value: int, stream):
        self.eng._check(self.eng.lib.avsep_flag_signal(self.eng.h, self._flag_array(flag_ptrs), len(flag_ptrs),
                                                       value & 0xFFFFFFFF, C.c_void_p(stream.cuda_stream)),
                        "avsep_flag_signal")

    def wait(self, flag_ptrs, value: int, stream, timeout_s: float = 60.0):
        self.eng._check(self.eng.lib.avsep_flag_wait(self.eng.h, self._flag_array(flag_ptrs), len(flag_ptrs),
                                                     value & 0xFFFFFFFF, float(timeout_s),
                                                     C.c_void_p(stream.cuda_stream)), "avsep_flag_wait")

    def separate(self, masks_ptr: int, mixed_ptr: int, n_utt: int, T: int, sep_ptr: int, stream):
        self.eng._check(self.eng.lib.avsep_separate(self.eng.h, C.c_void_p(masks_ptr), C.c_void_p(mixed_ptr), n_utt, T,
                                                    C.c_void_p(sep_ptr), C.c_void_p(stream.cuda_stream)),
                        "avsep_separate")

    def separate_varlen(self, masks_ptr: int, mixed_ptr: int, lens_ptr: int, n_utt: int, T: int, sep_ptr: int, stream):
        self.eng._check(self.eng.lib.avsep_separate_varlen(self.eng.h, C.c_void_p(masks_ptr), C.c_void_p(mixed_ptr),
                                                           C.c_void_p(lens_ptr), n_utt, T, C.c_void_p(sep_ptr),
                                                           C.c_void_p(stream.cuda_stream)), "avsep_separate_varlen")

    # stream / event plumbing (torch is used for streams only)
    def stream(self):
        return torch.cuda.Stream(device=self.dev)

    def current_stream(self):
        return torch.cuda.current_stream(self.dev)

    def event(self):
        return torch.cuda.Event(enable_timing=False)

    def synchronize(self):
        torch.cuda.synchronize(self.dev)


class ShardedForward:
    """Root-scattered, root-gathered forward over ``world`` ranks.

    forward_fn(mixed, frames, sep, masks): runs the model on one shard (tensors of the backend's device), stream-ordered
    on the backend's current stream.  ``shapes``: dict with the per-utterance shapes ``mixed`` (F, T), ``frames``
    (N, H, W), ``out`` (S, F, T).

    ``varlen=True``: a variable-length batch.  ``root_lens[s] = (lengths, frame_lengths)`` are the root's int32
    [world*B] views of input set s's audio-frame and lip-frame counts, filled by the producer like ``root_in[s]``, and
    forward_fn is called as forward_fn(mixed, frames, sep, masks, lengths, frame_lengths) with int32 device tensors of
    the shard (buffers whose pointers stay fixed, so the forward's CUDA-graph keys do too).  With gather="masks" the
    root's rebuild of step i reads set s's lengths as it reads its mixture: both stay untouched until that rebuild is done.
    """

    def __init__(self, backend, forward_fn, per_rank_batch: int, shapes: dict, rank: int, world: int,
                 n_input_sets: int = 1, group=None, copy_lanes: int = 1, gather: str = "both", varlen: bool = False):
        if gather not in ("both", "masks"):
            raise ValueError("gather must be 'both' (separated + masks on the wire) or 'masks' (the root rebuilds separated)")
        self.gather, self.varlen = gather, bool(varlen)
        self.mem, self.fwd = backend, forward_fn
        self.B, self.rank, self.world, self.group = int(per_rank_batch), int(rank), int(world), group
        self.n_sets = int(n_input_sets)
        self.shapes = {k: tuple(int(x) for x in v) for k, v in shapes.items()}
        self.per = {k: _prod(v) for k, v in self.shapes.items()}        # floats per utterance
        self.lo, self.hi = shard_slices(world, self.B)[rank]
        G = world * self.B
        names = [f"in{s}.{k}" for s in range(self.n_sets) for k in ("mixed", "frames")] + \
                [f"out{o}.{k}" for o in range(2) for k in ("sep", "masks")]
        sizes = {n: G * self.per["mixed" if n.endswith("mixed") else "frames" if n.endswith("frames") else "out"]
                 for n in names}
        if self.varlen:                  # one int32 per utterance (the backend sizes buffers in 4-byte words)
            lens_names = [f"in{s}.{k}" for s in range(self.n_sets) for k in ("lens", "frame_lens")]
            names += lens_names
            sizes.update({n: G for n in lens_names})
        self.ptr = {}
        if rank == 0:
            handles = {}
            for n in names:
                self.ptr[n], handles[n] = self.mem.alloc(sizes[n])
            box = [handles]
        else:
            box = [None]
        if world > 1:
            dist.broadcast_object_list(box, src=0, group=group)
        if rank != 0:
            for n in names:
                self.ptr[n] = self.mem.open(box[0][n])
        # root: tensor views of the global buffers (what its producer fills / its consumer reads)
        self.root_in, self.root_out, self.root_lens = [], [], []
        if rank == 0:
            for s in range(self.n_sets):
                self.root_in.append((self.mem.view(self.ptr[f"in{s}.mixed"], (G,) + self.shapes["mixed"]),
                                     self.mem.view(self.ptr[f"in{s}.frames"], (G,) + self.shapes["frames"])))
                if self.varlen:
                    self.root_lens.append((self.mem.view_i32(self.ptr[f"in{s}.lens"], (G,)),
                                           self.mem.view_i32(self.ptr[f"in{s}.frame_lens"], (G,))))
            for o in range(2):
                self.root_out.append((self.mem.view(self.ptr[f"out{o}.sep"], (G,) + self.shapes["out"]),
                                      self.mem.view(self.ptr[f"out{o}.masks"], (G,) + self.shapes["out"])))
        else:
            B = self.B
            self.loc_in = [(self.mem.empty((B,) + self.shapes["mixed"]), self.mem.empty((B,) + self.shapes["frames"]))
                           for _ in range(2)]
            self.loc_out = [(self.mem.empty((B,) + self.shapes["out"]), self.mem.empty((B,) + self.shapes["out"]))
                            for _ in range(2)]
            if self.varlen:              # (lengths, frame_lengths) per slot: int32 views of one 2B-word buffer
                self.loc_lens = [tuple(self.mem.empty((2, B)).view(torch.int32)) for _ in range(2)]
            self.s_in, self.s_out = self.mem.stream(), self.mem.stream()
            # copy_lanes > 1: every transfer is cut into that many pieces on extra streams (more copy engines and more
            # requests in flight per rank; tools/nvlink_probe.py: the root's links carry more when both directions run)
            self.lanes = max(1, int(copy_lanes))
            self.x_in = [self.mem.stream() for _ in range(self.lanes - 1)]
            self.x_out = [self.mem.stream() for _ in range(self.lanes - 1)]
            self.ev_lane = [self.mem.event() for _ in range(2 * (self.lanes - 1))]
            self.ev_go = [self.mem.event() for _ in range(2)]
            self.ev_in_ready = [self.mem.event() for _ in range(2)]
            self.ev_fwd_done = [self.mem.event() for _ in range(2)]
            self.ev_out_free = [self.mem.event() for _ in range(2)]
            self.used = [False, False]
        self.bytes_in_per_step = 4 * self.B * (self.per["mixed"] + self.per["frames"] + (2 if self.varlen else 0))
        self.bytes_out_per_step = 4 * self.B * (1 if gather == "masks" else 2) * self.per["out"]
        self.count, self.last_ticket = 0, [0, 0]
        if gather == "masks" and world > 1:
            self._init_tickets()

    FLAG_STRIDE = 16       # floats: one 64-byte line per flag

    def _init_tickets(self):
        """arrived[r] lives in the root's memory (rank r raises it after its masks landed); ack lives in every other
        rank's memory (the root raises it after it rebuilt `separated` from that step's masks)."""
        if self.world > 17:
            raise ValueError("gather='masks' supports up to 17 ranks (16 flags per wait)")
        st = self.FLAG_STRIDE
        if self.rank == 0:
            self.arrived, h = self.mem.alloc(self.world * st)
            self.mem.zero(self.arrived, self.world * st)
            mine = ("arrived", h)
        else:
            self.ack, h = self.mem.alloc(st)
            self.mem.zero(self.ack, st)
            mine = ("ack", h)
        self.mem.synchronize()
        everyone = [None] * self.world
        dist.all_gather_object(everyone, mine, group=self.group)
        if self.rank == 0:
            self.peer_ack = [self.mem.open(everyone[r][1]) for r in range(1, self.world)]
            self.s_rb = self.mem.stream()
            self.ev_rebuilt = [self.mem.event() for _ in range(2)]
        else:
            self.arrived = self.mem.open(everyone[0][1])
        dist.barrier(group=self.group)          # every flag is zeroed and mapped before the first ticket

    # ---- one step: scatter -> forward -> gather, all enqueued asynchronously -------------------------------------
    def step(self, i: int):
        s_set, b = i % self.n_sets, i & 1
        if self.rank == 0:
            m, f = self.root_in[s_set]
            sep, masks = self.root_out[b]
            lens = [t[self.lo:self.hi] for t in self.root_lens[s_set]] if self.varlen else []
            self.fwd(m[self.lo:self.hi], f[self.lo:self.hi], sep[self.lo:self.hi], masks[self.lo:self.hi], *lens)
            self.count += 1
            if self.gather == "masks" and self.world > 1:
                # rebuild the remote shards' `separated` once their masks have landed, then free the slot for step + 2
                ticket, st, B = self.count, 4 * self.FLAG_STRIDE, self.B
                self.mem.wait([self.arrived + r * st for r in range(1, self.world)], ticket, self.s_rb)
                args = (self.ptr[f"out{b}.masks"] + 4 * B * self.per["out"],
                        self.ptr[f"in{s_set}.mixed"] + 4 * B * self.per["mixed"], (self.world - 1) * B,
                        self.shapes["mixed"][1], self.ptr[f"out{b}.sep"] + 4 * B * self.per["out"], self.s_rb)
                if self.varlen:          # past its length a remote row is 0, as the rank's decoder wrote it
                    self.mem.separate_varlen(args[0], args[1], self.ptr[f"in{s_set}.lens"] + 4 * B, *args[2:])
                else:
                    self.mem.separate(*args)
                self.mem.signal(self.peer_ack, ticket, self.s_rb)
                self.ev_rebuilt[b].record(self.s_rb)
            return
        comp = self.mem.current_stream()
        m, f = self.loc_in[b]
        sep, masks = self.loc_out[b]
        # scatter: this rank's shard of the root's inputs, once the forward that last read this buffer pair is done
        if self.used[b]:
            self.s_in.wait_event(self.ev_fwd_done[b])
        off = self.lo
        jobs = [(m.data_ptr(), self.ptr[f"in{s_set}.mixed"] + 4 * off * self.per["mixed"], self.B * self.per["mixed"]),
                (f.data_ptr(), self.ptr[f"in{s_set}.frames"] + 4 * off * self.per["frames"], self.B * self.per["frames"])]
        lens = list(self.loc_lens[b]) if self.varlen else []
        for t, k in zip(lens, ("lens", "frame_lens")):
            jobs.append((t.data_ptr(), self.ptr[f"in{s_set}.{k}"] + 4 * off, self.B))
        self._copy(self.s_in, self.x_in, 0, jobs)
        self.ev_in_ready[b].record(self.s_in)
        # forward on the shard, once its inputs have landed and the push that last read these outputs is done
        comp.wait_event(self.ev_in_ready[b])
        if self.used[b]:
            comp.wait_event(self.ev_out_free[b])
        self.fwd(m, f, sep, masks, *lens)
        self.ev_fwd_done[b].record(comp)
        # gather: push the shard's outputs into the root's global buffers
        self.s_out.wait_event(self.ev_fwd_done[b])
        self.count += 1
        if self.gather == "masks":
            if self.last_ticket[b]:      # the root has rebuilt `separated` from what this output slot held before
                self.mem.wait([self.ack], self.last_ticket[b], self.s_out)
            self._copy(self.s_out, self.x_out, 1, [
                (self.ptr[f"out{b}.masks"] + 4 * off * self.per["out"], masks.data_ptr(), self.B * self.per["out"])])
            self.mem.signal([self.arrived + 4 * self.FLAG_STRIDE * self.rank], self.count, self.s_out)
            self.last_ticket[b] = self.count
        else:
            self._copy(self.s_out, self.x_out, 1, [
                (self.ptr[f"out{b}.sep"] + 4 * off * self.per["out"], sep.data_ptr(), self.B * self.per["out"]),
                (self.ptr[f"out{b}.masks"] + 4 * off * self.per["out"], masks.data_ptr(), self.B * self.per["out"])])
        self.ev_out_free[b].record(self.s_out)
        self.used[b] = True

    def _copy(self, lead, extra, which, jobs):
        """jobs: [(dst_ptr, src_ptr, nfloats)] on the lead stream, or cut into len(extra) + 1 pieces each, one piece per
        stream; the lead stream ends up ordered after every piece."""
        if not extra:
            for dst, src, n in jobs:
                self.mem.copy(dst, src, n, lead)
            return
        k = len(extra) + 1
        self.ev_go[which].record(lead)
        for lane, st in enumerate([lead] + extra):
            if lane:
                st.wait_event(self.ev_go[which])
            for dst, src, n in jobs:
                lo, hi = (n * lane // k) & ~3, n if lane == k - 1 else (n * (lane + 1) // k) & ~3     # 16-byte pieces
                if hi > lo:
                    self.mem.copy(dst + 4 * lo, src + 4 * lo, hi - lo, st)
            if lane:
                ev = self.ev_lane[which * (k - 1) + lane - 1]
                ev.record(st)
                lead.wait_event(ev)

    def finish(self):
        """All enqueued scatters, forwards and gathers of every rank are complete when this returns."""
        self.mem.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)


def _prod(shape):
    n = 1
    for s in shape:
        n *= int(s)
    return n
