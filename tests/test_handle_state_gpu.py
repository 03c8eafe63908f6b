"""State a handle keeps for itself: profiling brackets each kernel on the stream the kernel runs on, and everything a
handle allocates on the device goes with avsep_destroy."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.weights import CONFIGS, make_inputs, make_state_dict

pytestmark = pytest.mark.gpu


def test_profiling_times_the_launching_stream():
    """A fresh handle profiles an STFT on a non-blocking torch stream: the reported time is the kernel's, not that of
    an event pair on some other stream."""
    from avsep_b200.engine import Engine, EngineConfig
    eng = Engine(EngineConfig(**CONFIGS["tiny"].as_dict()), 0)
    B, L, n_fft, hop = 256, 8000, 2048, 128
    F, T = n_fft // 2 + 1, 1 + L // hop
    waves = torch.randn(B, L, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    spec = torch.empty(B, F, T, device="cuda", dtype=torch.complex64)
    mag = torch.empty(B, F, T, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())

    def stft():   # preallocated outputs: the call itself allocates nothing
        eng._check(eng.lib.avsep_stft(eng.h, waves.data_ptr(), B, L, n_fft, hop, spec.data_ptr(), mag.data_ptr(),
                                      C.c_void_p(s.cuda_stream)), "avsep_stft")

    eng.set_profile(True)
    # the first call loads the kernel and creates the handle's profiling events: host work that must not fall inside
    # the timed window below, which is to hold device work only
    stft()
    s.synchronize()
    eng.profile_report(reset=True)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s):
        torch.cuda._sleep(10_000_000)   # the GPU waits until the call is enqueued: the events then time device work only
        start.record()
        stft()
        end.record()
    end.synchronize()
    event_ms = start.elapsed_time(end)
    n, prof_ms = eng.profile_report()["other"]
    eng.close()
    assert n == 1
    assert prof_ms >= 0.5 * event_ms, (prof_ms, event_ms)


def test_handle_churn_leaves_no_device_memory_behind():
    """Create, use every buffer-owning path once, destroy, twenty times: the free device memory comes back to what it
    was after the first round (the first round also loads the kernels)."""
    from avsep_b200.engine import Engine, EngineConfig
    cfg = CONFIGS["default"]
    P = make_state_dict(cfg, seed=5, gain=2.0)
    B, T, N = 16, 63, 50
    S, F = cfg.num_speakers, cfg.freq_bins
    mixed, frames = make_inputs(cfg, B, T, N, seed=5, kind="dataset")
    mixed_d, frames_d = torch.from_numpy(mixed).cuda(), torch.from_numpy(frames).cuda()
    out_d = tuple(torch.empty(B, S, F, T, device="cuda") for _ in range(2))
    mixed_h, frames_h = torch.from_numpy(mixed).pin_memory(), torch.from_numpy(frames).pin_memory()
    out_h = [tuple(torch.empty(B, S, F, T).pin_memory() for _ in range(2)) for _ in range(2)]
    rng = np.random.default_rng(5)
    lens = rng.integers(1, T + 1, B).astype(np.int32)
    flens = rng.integers(1, N + 1, B).astype(np.int32)
    mixed_p = torch.from_numpy(np.concatenate([mixed[b, :, :lens[b]].reshape(-1) for b in range(B)])).pin_memory()
    frames_p = torch.from_numpy(np.concatenate([frames[b, :flens[b]] for b in range(B)])).pin_memory()
    out_p = tuple(torch.empty(S * F * int(lens.sum())).pin_memory() for _ in range(2))
    geom = dict(num_samples_audio=8000, duration=1.0, n_fft=512, hop_length=128, num_frames=25, frame_h=32,
                frame_w=32, num_speakers=S)
    g = torch.Generator("cuda").manual_seed(5)
    amps, freqs, phases = (torch.rand(B, S, device="cuda", dtype=torch.float64, generator=g) for _ in range(3))

    free = []
    for _ in range(20):
        eng = Engine(EngineConfig(**cfg.as_dict()), 0)
        eng.load_state(P)
        for _ in range(3):                      # eager, captured into a graph, replayed
            eng.forward(mixed_d, frames_d, out=out_d)
        for slot in (0, 1):
            eng.forward_host_async(mixed_h, frames_h, *out_h[slot], slot)
        for slot in (0, 1):
            eng.host_wait(slot)
        eng.forward_host_packed(mixed_p, frames_p, lens, flens, max_len=T, max_frames=N, out=out_p)
        eng.synth_batch(geom, amps, freqs, phases)
        eng.set_debug(True)
        eng.forward(mixed_d, frames_d, out=out_d)
        assert eng.get_stage("fused").size == B * T * cfg.d_model
        eng.close()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free.append(torch.cuda.mem_get_info()[0])
    lost_mb = [(free[0] - f) / 2**20 for f in free]
    assert max(lost_mb) <= 8, lost_mb
