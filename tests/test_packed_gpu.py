"""Packed variable-length batches (avsep_forward_packed, avsep_forward_host_packed[_async]; forward_packed of Engine and
AVSeparationTransformer): utterances back to back with no padding give, bit for bit, the valid regions of the varlen
forward on the padded batch, on the device and through the chunked host-buffer pipeline."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.weights import CONFIGS, make_inputs, make_state_dict
from tests.helpers import build_model

pytestmark = pytest.mark.gpu

# (config, precision, B, T, N, frame H, frame W, attn_tc): the cases of test_varlen_gpu.py, plus 5 x 7 frames, whose
# blocks take the unpack kernel's scalar path
CASES = {
    "default_63_50": ("default", "bf16", 6, 63, 50, 32, 32, None),
    "default_100_80": ("default", "bf16", 4, 100, 80, 32, 32, None),
    "default_300_120_tc": ("default", "bf16", 3, 300, 120, 32, 32, 1),
    "tiny_40_12": ("tiny", "bf16", 5, 40, 12, 16, 16, None),
    "scaled_63_50": ("scaled", "bf16", 3, 63, 50, 32, 32, None),
    "default_tf32_63_50": ("default", "tf32", 3, 63, 50, 32, 32, None),
    "tiny_40_12_5x7": ("tiny", "bf16", 5, 40, 12, 5, 7, None),
}


def _setup(name, seed=81):
    cname, prec, B, T, N, hh, ww, attn_tc = CASES[name]
    cfg = CONFIGS[cname]
    P = make_state_dict(cfg, seed=seed, gain=2.0)
    mixed, frames = make_inputs(cfg, B, T, N, hh, ww, seed=seed, kind="dataset")
    model = build_model(cfg, P, prec)
    model.prepack()
    if attn_tc is not None:
        model.engine.set_option("attn_tc", attn_tc)
    return cfg, model, mixed, frames


def _ragged(B, T, N, seed):
    """Seeded lengths that include 1 and the maximum on both sides."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, T + 1, B).astype(np.int32)
    flens = rng.integers(1, N + 1, B).astype(np.int32)
    lens[0], flens[0] = 1, N
    lens[1], flens[1] = T, 1
    return lens, flens


def _pack(mixed, frames, lens, flens):
    mp = np.concatenate([mixed[b, :, :lens[b]].reshape(-1) for b in range(len(lens))])
    fp = np.concatenate([frames[b, :flens[b]] for b in range(len(lens))])
    return np.ascontiguousarray(mp), np.ascontiguousarray(fp)


def _varlen(model, mixed, frames, lens, flens):
    sep, masks = model(torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda(), lengths=lens,
                       frame_lengths=flens)
    torch.cuda.synchronize()
    return sep.cpu().numpy(), masks.cpu().numpy()


def _valid(x, lens):
    """Padded (B, S, F, T) -> the packed layout of its valid regions."""
    return np.concatenate([x[b, :, :, :lens[b]].reshape(-1) for b in range(len(lens))])


def _packed_dev(model, mp, fp, lens, flens, **kw):
    sep, masks = model.forward_packed(torch.from_numpy(mp).cuda(), torch.from_numpy(fp).cuda(), lens, flens, **kw)
    torch.cuda.synchronize()
    return sep.cpu().numpy(), masks.cpu().numpy()


def _abi_packed(eng, mp, fp, lens_d, flens_d, B, T, N, out):
    """avsep_forward_packed through the C ABI on device tensors (NULL length pointers when None)."""
    hh, ww = fp.shape[1:]
    rc = eng.lib.avsep_forward_packed(eng.h, mp.data_ptr(), fp.data_ptr(),
                                      None if lens_d is None else lens_d.data_ptr(),
                                      None if flens_d is None else flens_d.data_ptr(), B, T, N, hh, ww,
                                      out[0].data_ptr(), out[1].data_ptr(), None, 0,
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream))
    eng._check(rc, "avsep_forward_packed")
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", list(CASES))
def test_packed_equals_varlen_valid_regions(name):
    cfg, model, mixed, frames = _setup(name)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    lens, flens = _ragged(B, T, N, seed=82)
    sep_v, masks_v = _varlen(model, mixed, frames, lens, flens)
    mp, fp = _pack(mixed, frames, lens, flens)
    sep, masks = _packed_dev(model, mp, fp, lens, flens, max_len=T, max_frames=N)
    assert np.array_equal(sep, _valid(sep_v, lens)) and np.array_equal(masks, _valid(masks_v, lens)), name
    # default maxima (the batch's own) give the same bits here: the lengths include T and N
    sep_d, masks_d = _packed_dev(model, mp, fp, list(lens), torch.from_numpy(flens))
    assert np.array_equal(sep_d, sep) and np.array_equal(masks_d, masks), name


def test_null_lengths_give_forward_bytes_and_device_lengths_clamp():
    cfg, model, mixed, frames = _setup("default_63_50", seed=83)
    eng = model.engine
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    S, F = cfg.num_speakers, cfg.freq_bins
    sep_u, masks_u = model(torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda())
    out = torch.empty(2, B * S * F * T, device="cuda")
    _abi_packed(eng, torch.from_numpy(mixed).cuda().reshape(-1), torch.from_numpy(frames).cuda().reshape(B * N, *frames.shape[2:]),
                None, None, B, T, N, out)
    assert np.array_equal(out[0].cpu().numpy(), sep_u.cpu().numpy().reshape(-1))
    assert np.array_equal(out[1].cpu().numpy(), masks_u.cpu().numpy().reshape(-1))
    # out-of-range device lengths behave as the clamped values, which define the layout
    lens, flens = _ragged(B, T, N, seed=84)
    raw_t, raw_n = lens.copy(), flens.copy()
    raw_t[2], raw_t[3], raw_n[2], raw_n[3] = 0, T + 5, -3, N + 5
    lens[2], lens[3], flens[2], flens[3] = 1, T, 1, N
    mp, fp = _pack(mixed, frames, lens, flens)
    sep, masks = _packed_dev(model, mp, fp, lens, flens, max_len=T, max_frames=N)
    out = torch.full((2, B * S * F * T), np.nan, device="cuda")
    _abi_packed(eng, torch.from_numpy(mp).cuda(), torch.from_numpy(fp).cuda(), torch.from_numpy(raw_t).cuda(),
                torch.from_numpy(raw_n).cuda(), B, T, N, out)
    n = sep.size
    assert np.array_equal(out[0, :n].cpu().numpy(), sep) and np.array_equal(out[1, :n].cpu().numpy(), masks)
    assert torch.isnan(out[:, n:]).all()


@pytest.mark.parametrize("name", ["default_63_50", "tiny_40_12_5x7"])
def test_misaligned_views_and_canaries(name):
    cfg, model, mixed, frames = _setup(name, seed=85)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    lens, flens = _ragged(B, T, N, seed=86)
    mp, fp = _pack(mixed, frames, lens, flens)
    sep, masks = _packed_dev(model, mp, fp, lens, flens, max_len=T, max_frames=N)
    n = sep.size
    mbuf = torch.full((mp.size + 2,), np.nan, device="cuda")
    fbuf = torch.full((fp.size + 2,), np.nan, device="cuda")
    mbuf[1:1 + mp.size] = torch.from_numpy(mp).cuda()
    fbuf[1:1 + fp.size] = torch.from_numpy(fp.reshape(-1)).cuda()
    obuf = torch.full((2, n + 2), np.nan, device="cuda")
    out = (obuf[0, 1:1 + n], obuf[1, 1:1 + n])
    model.forward_packed(mbuf[1:1 + mp.size], fbuf[1:1 + fp.size].view(fp.shape), lens, flens, max_len=T,
                         max_frames=N, out=out)
    torch.cuda.synchronize()
    assert np.array_equal(out[0].cpu().numpy(), sep) and np.array_equal(out[1].cpu().numpy(), masks)
    assert torch.isnan(obuf[:, 0]).all() and torch.isnan(obuf[:, n + 1]).all()


@pytest.fixture(scope="module")
def default_b37():
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=87, gain=2.0)
    B, T, N = 37, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=87, kind="dataset")
    model = build_model(cfg, P, "bf16")
    model.prepack()
    lens, flens = _ragged(B, T, N, seed=88)
    mp, fp = _pack(mixed, frames, lens, flens)
    ref = _packed_dev(model, mp, fp, lens, flens, max_len=T, max_frames=N)
    return model, mp, fp, lens, flens, ref


@pytest.mark.parametrize("pinned", [True, False])
@pytest.mark.parametrize("lanes", [1, 2, 3])
@pytest.mark.parametrize("chunk", [1, 7, 0])
def test_host_packed_equals_device_packed(default_b37, chunk, lanes, pinned):
    model, mp, fp, lens, flens, (sep_ref, masks_ref) = default_b37
    eng = model.engine
    eng.set_option("host_chunk", chunk)
    eng.set_option("host_lanes", lanes)
    try:
        m, f = torch.from_numpy(mp), torch.from_numpy(fp)
        out = (torch.full((sep_ref.size,), np.nan), torch.full((sep_ref.size,), np.nan))
        if pinned:
            m, f, out = m.pin_memory(), f.pin_memory(), tuple(t.pin_memory() for t in out)
        sep, masks = model.forward_packed(m, f, lens, flens, max_len=63, max_frames=50, out=out)
        assert not sep.is_cuda
        assert np.array_equal(sep.numpy(), sep_ref) and np.array_equal(masks.numpy(), masks_ref), (chunk, lanes, pinned)
    finally:
        eng.set_option("host_chunk", 0)
        eng.set_option("host_lanes", 0)


def test_async_slots_with_long_then_short_batches():
    """Ragged batches of different lengths alternate through two slots (long ones, then short ones through the same
    slot), twice so that the second round replays captured graphs; each matches its synchronous result, so no stale
    staging or length buffer is read."""
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=89, gain=2.0)
    B, T, N = 40, 63, 50
    model = build_model(cfg, P, "bf16")
    model.prepack()
    eng = model.engine
    batches = []
    for k in range(4):
        mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=90 + k, kind="dataset")
        rng = np.random.default_rng(95 + k)
        lo, hi = (40, T) if k < 2 else (1, 12)
        lens = rng.integers(lo, hi + 1, B).astype(np.int32)
        flens = rng.integers(max(1, lo * N // T), max(1, hi * N // T) + 1, B).astype(np.int32)
        mp, fp = _pack(mixed, frames, lens, flens)
        ref = model.forward_packed(torch.from_numpy(mp), torch.from_numpy(fp), lens, flens, max_len=T, max_frames=N)
        n = ref[0].numel()
        io = (torch.from_numpy(mp).pin_memory(), torch.from_numpy(fp).pin_memory(),
              torch.full((n,), np.nan).pin_memory(), torch.full((n,), np.nan).pin_memory())
        batches.append((io, lens, flens, (ref[0].clone(), ref[1].clone())))
    for rnd in range(2):
        order = [(0, 0), (1, 1), (2, 0), (3, 1)]
        pending = {}
        for k, slot in order:
            if slot in pending:
                eng.host_wait(slot)
                done = pending.pop(slot)
                _check_async(batches[done], done, rnd)
            (m, f, s, ma), lens, flens, _ = batches[k]
            s.fill_(np.nan)
            ma.fill_(np.nan)
            eng.forward_host_packed_async(m, f, lens, flens, (s, ma), slot, max_len=T, max_frames=N)
            pending[slot] = k
        for slot, k in pending.items():
            eng.host_wait(slot)
            _check_async(batches[k], k, rnd)


def _check_async(batch, k, rnd):
    (_, _, s, ma), _, _, (sep_ref, masks_ref) = batch
    assert torch.equal(s, sep_ref) and torch.equal(ma, masks_ref), (k, rnd)


def test_b256_host_packed_equals_varlen():
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=99, gain=2.0)
    B, T, N = 256, 63, 50
    mixed, frames = make_inputs(cfg, B, T, N, 32, 32, seed=99, kind="dataset")
    model = build_model(cfg, P, "bf16")
    lens, flens = _ragged(B, T, N, seed=100)
    sep_v, masks_v = _varlen(model, mixed, frames, lens, flens)
    mp, fp = _pack(mixed, frames, lens, flens)
    for _ in range(3):      # eager, capture, replay
        sep, masks = model.forward_packed(torch.from_numpy(mp).pin_memory(), torch.from_numpy(fp).pin_memory(), lens,
                                          flens, max_len=T, max_frames=N)
        assert np.array_equal(sep.numpy(), _valid(sep_v, lens)) and np.array_equal(masks.numpy(), _valid(masks_v, lens))


def test_launch_count_is_the_forwards_plus_two():
    cfg, model, mixed, frames = _setup("default_63_50", seed=101)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    lens, flens = _ragged(B, T, N, seed=102)
    _varlen(model, mixed, frames, lens, flens)
    fwd = model.engine.launch_count()
    mp, fp = _pack(mixed, frames, lens, flens)
    for _ in range(3):      # eager, capture, replay
        _packed_dev(model, mp, fp, lens, flens, max_len=T, max_frames=N)
        assert model.engine.launch_count() == fwd + 2


def test_errors_fail_loudly():
    cfg, model, mixed, frames = _setup("tiny_40_12", seed=103)
    eng = model.engine
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    S, F = cfg.num_speakers, cfg.freq_bins
    hh, ww = frames.shape[2:]
    lens, flens = _ragged(B, T, N, seed=104)
    mp, fp = _pack(mixed, frames, lens, flens)
    m, f = torch.from_numpy(mp).pin_memory(), torch.from_numpy(fp).pin_memory()
    n = S * F * int(lens.sum())
    sep, masks = torch.empty(n).pin_memory(), torch.empty(n).pin_memory()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def host(lens_a, flens_a, ptrs=None, slot=None):
        ptrs = ptrs or (m.data_ptr(), f.data_ptr(), sep.data_ptr(), masks.data_ptr())
        la = np.ascontiguousarray(lens_a, np.int32)
        fa = np.ascontiguousarray(flens_a, np.int32)
        if slot is None:
            return eng.lib.avsep_forward_host_packed(eng.h, ptrs[0], ptrs[1], la.ctypes.data, fa.ctypes.data, B, T, N,
                                                     hh, ww, ptrs[2], ptrs[3], st)
        return eng.lib.avsep_forward_host_packed_async(eng.h, ptrs[0], ptrs[1], la.ctypes.data, fa.ctypes.data, B, T,
                                                       N, hh, ww, ptrs[2], ptrs[3], slot, st)

    assert host(lens, flens) == 0
    for bad_t, bad_n in (([0] + list(lens[1:]), flens), ([T + 1] + list(lens[1:]), flens),
                         (lens, [0] + list(flens[1:])), (lens, [N + 1] + list(flens[1:]))):
        assert host(bad_t, bad_n) != 0
        assert b"outside [1, T] / [1, N]" in eng.lib.avsep_last_error(eng.h)
    for k in range(4):
        ptrs = [m.data_ptr(), f.data_ptr(), sep.data_ptr(), masks.data_ptr()]
        ptrs[k] = None
        assert host(lens, flens, ptrs) != 0
    assert host(lens, flens, slot=4) != 0 and host(lens, flens, slot=-1) != 0
    d = lambda a: torch.from_numpy(a).cuda()
    assert eng.lib.avsep_forward_packed(eng.h, None, d(fp).data_ptr(), None, None, B, T, N, hh, ww, None, None, None, 0,
                                        st) != 0
    # Python: packed sizes against the lengths, length ranges, device lengths only with out= on CUDA inputs
    with pytest.raises(ValueError):
        model.forward_packed(m[:-1], f, lens, flens)
    with pytest.raises(ValueError):
        model.forward_packed(m, f[:-1], lens, flens)
    with pytest.raises(ValueError):
        model.forward_packed(m, f, lens, flens, out=(sep[:-1], masks[:-1]))
    with pytest.raises(ValueError):
        model.forward_packed(m, f, lens, flens, max_len=int(lens.max()) - 1)
    with pytest.raises(ValueError):
        model.forward_packed(m, f, [0] + list(lens[1:]), flens)
    with pytest.raises(ValueError):
        model.forward_packed(m, f, d(lens), d(flens), max_len=T, max_frames=N)
    with pytest.raises(ValueError):
        model.forward_packed(d(mp), d(fp), d(lens), d(flens), max_len=T, max_frames=N)
    with pytest.raises(ValueError):
        model.forward_packed(d(mp), d(fp), lens[:-1], flens)
    with pytest.raises(ValueError):
        model.forward_packed(d(mp).view(1, -1), d(fp), lens, flens)


def test_model_forward_packed_cpu_and_cuda_equal_padded_varlen():
    cfg, model, mixed, frames = _setup("default_63_50", seed=105)
    B, T, N = mixed.shape[0], mixed.shape[2], frames.shape[1]
    S, F = cfg.num_speakers, cfg.freq_bins
    lens, flens = _ragged(B, T, N, seed=106)
    sep_v, masks_v = _varlen(model, mixed, frames, lens, flens)
    specs = [torch.from_numpy(mixed[b, :, :lens[b]].copy()) for b in range(B)]
    frame_list = [torch.from_numpy(frames[b, :flens[b]].copy()) for b in range(B)]
    mp, fp = torch.cat([m.reshape(-1) for m in specs]), torch.cat(frame_list)
    for dev in ("cpu", "cuda"):
        sep, masks = model.forward_packed(mp.to(dev), fp.to(dev), torch.from_numpy(lens), list(flens))
        assert sep.device.type == dev
        seps = [x.view(S, F, t) for x, t in zip(torch.split(sep.cpu(), [S * F * int(t) for t in lens]), lens)]
        maskl = [x.view(S, F, t) for x, t in zip(torch.split(masks.cpu(), [S * F * int(t) for t in lens]), lens)]
        for b in range(B):
            assert np.array_equal(seps[b].numpy(), sep_v[b, :, :, :lens[b]]), (dev, b)
            assert np.array_equal(maskl[b].numpy(), masks_v[b, :, :, :lens[b]]), (dev, b)
    # device lengths with out= and fixed maxima: a graph replay per batch reads the lengths then in the buffers
    n = B * S * F * T
    out = (torch.empty(n, device="cuda"), torch.empty(n, device="cuda"))
    mbuf, fbuf = torch.zeros(B * F * T, device="cuda"), torch.zeros(B * N, *frames.shape[2:], device="cuda")
    lens_d, flens_d = torch.empty(B, dtype=torch.int32, device="cuda"), torch.empty(B, dtype=torch.int32, device="cuda")
    for k in range(4):
        lk, fk = _ragged(B, T, N, seed=107 + k)
        mpk, fpk = _pack(mixed, frames, lk, fk)
        mbuf[:mpk.size] = torch.from_numpy(mpk).cuda()
        fbuf[:fpk.shape[0]] = torch.from_numpy(fpk).cuda()
        lens_d.copy_(torch.from_numpy(lk))
        flens_d.copy_(torch.from_numpy(fk))
        model.forward_packed(mbuf, fbuf, lens_d, flens_d, max_len=T, max_frames=N, out=out)
        torch.cuda.synchronize()
        sv, mv = _varlen(model, mixed, frames, lk, fk)
        nk = S * F * int(lk.sum())
        assert np.array_equal(out[0][:nk].cpu().numpy(), _valid(sv, lk)), k
        assert np.array_equal(out[1][:nk].cpu().numpy(), _valid(mv, lk)), k
