"""The calling convention of the C ABI: every call runs on its handle's device and leaves the caller's current device as
it found it, and avsep_last_launch_count is the number of kernels the last call that enqueues device work enqueued.
Each entry point is driven through ctypes on buffers of the handle's device (cuda:0) and the stream of that device."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle.weights import CONFIGS, make_inputs, make_state_dict

pytestmark = pytest.mark.gpu

CFG = CONFIGS["default"]
B, T, N, HW = 4, 63, 50, 32            # the benchmark's clips: every forward stage runs in a stack kernel
L, NFFT, HOP = 8000, 512, 128          # their waveforms: 257 bins (the model's F), 63 frames (T)
TW = 1 + L // HOP
D, S, F = CFG.d_model, CFG.num_speakers, CFG.freq_bins
M = 256                                # rows of the kernel-hook problems
DEV = torch.device("cuda", 0)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _stream():
    return torch.cuda.current_stream(DEV).cuda_stream


def _rand(*shape, dtype=torch.float32, scale=1.0, seed=0):
    g = torch.Generator(DEV).manual_seed(seed)
    return (torch.randn(*shape, device=DEV, generator=g) * scale).to(dtype)


def _engine():
    from avsep_b200.engine import Engine, EngineConfig
    e = Engine(EngineConfig(**CFG.as_dict()), 0)
    e.load_state(make_state_dict(CFG, seed=21, gain=2.0))
    e.set_option("use_graph", 0)       # every forward runs eagerly unless a test turns graphs on
    return e


def _inputs():
    """Inputs on cuda:0, made once; every call below reads them and writes buffers of its own."""
    mixed, frames = make_inputs(CFG, B, T, N, HW, HW, seed=21, kind="dataset")
    rng = np.random.default_rng(21)
    lens, flens = rng.integers(1, T + 1, B).astype(np.int32), rng.integers(1, N + 1, B).astype(np.int32)
    mixed_p = np.concatenate([mixed[b, :, :lens[b]].reshape(-1) for b in range(B)])
    frames_p = np.concatenate([frames[b, :flens[b]] for b in range(B)])
    g = torch.Generator(DEV).manual_seed(22)
    return dict(
        mixed=torch.from_numpy(mixed).to(DEV), frames=torch.from_numpy(frames).to(DEV),
        mixed_h=torch.from_numpy(mixed).pin_memory(), frames_h=torch.from_numpy(frames).pin_memory(),
        lens=lens, flens=flens, lens_d=torch.from_numpy(lens).to(DEV), flens_d=torch.from_numpy(flens).to(DEV),
        mixed_p=torch.from_numpy(mixed_p).to(DEV), frames_p=torch.from_numpy(frames_p).to(DEV),
        mixed_ph=torch.from_numpy(mixed_p).pin_memory(), frames_ph=torch.from_numpy(frames_p).pin_memory(),
        rows_a=_rand(B, T, D, seed=1), rows_v=_rand(B, T, D, seed=2),
        masks=torch.rand(B, S, F, T, device=DEV, generator=g), targets=torch.rand(B, S, F, T, device=DEV, generator=g),
        amps=torch.rand(B, S, device=DEV, dtype=torch.float64, generator=g),
        freqs=200 + 800 * torch.rand(B, S, device=DEV, dtype=torch.float64, generator=g),
        phases=torch.rand(B, S, device=DEV, dtype=torch.float64, generator=g),
        waves=_rand(B, L, seed=3), wave_lens=torch.from_numpy(rng.integers(1, L + 1, B).astype(np.int32)).to(DEV),
        A=_rand(M, D, dtype=torch.bfloat16, seed=4), W=_rand(D, D, dtype=torch.bfloat16, scale=1 / 16, seed=5),
        W1=_rand(4 * D, D, dtype=torch.bfloat16, scale=1 / 16, seed=6),
        W2=_rand(D, 4 * D, dtype=torch.bfloat16, scale=1 / 32, seed=7), W3=_rand(D, 3 * D, dtype=torch.bfloat16,
                                                                                  scale=1 / 28, seed=8),
        b=_rand(D, seed=9), b4=_rand(4 * D, seed=10), x=_rand(M, D, scale=2, seed=11), gamma=_rand(D, seed=12),
        spec=torch.complex(_rand(B, F, TW, seed=16), _rand(B, F, TW, seed=17)),
        q=_rand(2 * 128, D, dtype=torch.bfloat16, seed=13), k=_rand(2 * 128, D, dtype=torch.bfloat16, seed=18),
        v=_rand(2 * 128, D, dtype=torch.bfloat16, seed=19), k_src=_rand(2 * 50, D, seed=14),
        v_src=_rand(2 * 50, D, seed=20),
        cnn_frames=torch.rand(8, HW, HW, device=DEV, generator=g),
        kv=_rand(B * T, CFG.num_fusion_layers * 2 * D, dtype=torch.bfloat16, seed=15),
    )


@pytest.fixture(scope="module")
def eng():
    e = _engine()
    yield e
    e.close()


@pytest.fixture(scope="module")
def inp():
    return _inputs()


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), device=DEV, dtype=dtype)


def _nan_host(*shape):
    return torch.full(shape, float("nan")).pin_memory()


def _trace():
    return torch.zeros(148 * 256, device=DEV, dtype=torch.int64)


def _flags(n, value):
    t = torch.full((16 * n,), value, dtype=torch.int32, device=DEV)
    return t, (C.c_void_p * n)(*[t.data_ptr() + 64 * i for i in range(n)])


class Calls:
    """One builder per C-ABI entry point that enqueues device work.  A builder allocates the call's outputs and returns
    (call, outputs): call() makes the one C-ABI call (and waits for a host-buffer call's results) and returns its
    status; outputs are the tensors it writes."""

    def __init__(self, eng, inp):
        self.lib, self.h, self.i = eng.lib, eng.h, inp
        self.st = int(inp["lens"].sum())

    def p(self, name):
        return self.i[name].data_ptr()

    def forward(self):
        sep, masks = _nan(B, S, F, T), _nan(B, S, F, T)
        return (lambda: self.lib.avsep_forward(self.h, self.p("mixed"), self.p("frames"), B, T, N, HW, HW,
                                               sep.data_ptr(), masks.data_ptr(), None, 0, _stream())), [sep, masks]

    def forward_varlen(self):
        sep, masks = _nan(B, S, F, T), _nan(B, S, F, T)
        return (lambda: self.lib.avsep_forward_varlen(self.h, self.p("mixed"), self.p("frames"), self.p("lens_d"),
                                                      self.p("flens_d"), B, T, N, HW, HW, sep.data_ptr(),
                                                      masks.data_ptr(), None, 0, _stream())), [sep, masks]

    def forward_packed(self):
        sep, masks = _nan(S * F * self.st), _nan(S * F * self.st)
        return (lambda: self.lib.avsep_forward_packed(self.h, self.p("mixed_p"), self.p("frames_p"), self.p("lens_d"),
                                                      self.p("flens_d"), B, T, N, HW, HW, sep.data_ptr(),
                                                      masks.data_ptr(), None, 0, _stream())), [sep, masks]

    def forward_host(self):
        sep, masks = _nan_host(B, S, F, T), _nan_host(B, S, F, T)
        return (lambda: self.lib.avsep_forward_host(self.h, self.p("mixed_h"), self.p("frames_h"), B, T, N, HW, HW,
                                                    sep.data_ptr(), masks.data_ptr(), _stream())), [sep, masks]

    def forward_host_async(self):
        sep, masks = _nan_host(B, S, F, T), _nan_host(B, S, F, T)
        return (lambda: self.lib.avsep_forward_host_async(self.h, self.p("mixed_h"), self.p("frames_h"), B, T, N, HW,
                                                          HW, sep.data_ptr(), masks.data_ptr(), 1, _stream())
                or self.lib.avsep_host_wait(self.h, 1)), [sep, masks]

    def forward_host_packed(self):
        sep, masks = _nan_host(S * F * self.st), _nan_host(S * F * self.st)
        return (lambda: self.lib.avsep_forward_host_packed(self.h, self.p("mixed_ph"), self.p("frames_ph"),
                                                           self.i["lens"].ctypes.data, self.i["flens"].ctypes.data, B,
                                                           T, N, HW, HW, sep.data_ptr(), masks.data_ptr(),
                                                           _stream())), [sep, masks]

    def forward_host_packed_async(self):
        sep, masks = _nan_host(S * F * self.st), _nan_host(S * F * self.st)
        return (lambda: self.lib.avsep_forward_host_packed_async(
            self.h, self.p("mixed_ph"), self.p("frames_ph"), self.i["lens"].ctypes.data, self.i["flens"].ctypes.data, B,
            T, N, HW, HW, sep.data_ptr(), masks.data_ptr(), 2, _stream()) or self.lib.avsep_host_wait(self.h, 2)), \
            [sep, masks]

    def audio_encoder(self):
        out = _nan(B, T, D)
        return (lambda: self.lib.avsep_audio_encoder(self.h, self.p("mixed"), B, T, out.data_ptr(), _stream())), [out]

    def visual_encoder(self):
        out = _nan(B, T, D)
        return (lambda: self.lib.avsep_visual_encoder(self.h, self.p("frames"), B, N, HW, HW, T, out.data_ptr(),
                                                      _stream())), [out]

    def fusion(self):
        out = _nan(B, T, D)
        return (lambda: self.lib.avsep_fusion(self.h, self.p("rows_a"), self.p("rows_v"), B, T, T, out.data_ptr(),
                                              _stream())), [out]

    def decoder(self):
        sep, masks = _nan(B, S, F, T), _nan(B, S, F, T)
        return (lambda: self.lib.avsep_decoder(self.h, self.p("rows_a"), self.p("mixed"), B, T, sep.data_ptr(),
                                               masks.data_ptr(), _stream())), [sep, masks]

    def synth_batch(self):
        from avsep_b200 import _lib
        geom = _lib.AvsepSynthConfig(L, 1.0, NFFT, HOP, 25, HW, HW, S)
        outs = [_nan(B, F, TW), _nan(B, S * 25, HW, HW), _nan(B, S, F, TW)]
        return (lambda: self.lib.avsep_synth_batch(self.h, C.byref(geom), B, self.p("amps"), self.p("freqs"),
                                                   self.p("phases"), None, *[o.data_ptr() for o in outs],
                                                   _stream())), outs

    def eval_snr(self):
        outs = [_nan(B, S, dtype=torch.float64), _nan(B, dtype=torch.float64),
                torch.zeros(B, dtype=torch.int32, device=DEV), _nan(B, dtype=torch.float64)]
        return (lambda: self.lib.avsep_eval_snr(self.h, self.p("masks"), self.p("targets"), self.p("mixed"), B, S, F, T,
                                                *[o.data_ptr() for o in outs], _stream())), outs

    def stft(self):
        outs = [_nan(B, F, TW, dtype=torch.complex64), _nan(B, F, TW)]
        return (lambda: self.lib.avsep_stft(self.h, self.p("waves"), B, L, NFFT, HOP, *[o.data_ptr() for o in outs],
                                            _stream())), outs

    def stft_varlen(self):
        outs = [_nan(B, F, TW, dtype=torch.complex64), _nan(B, F, TW), torch.zeros(B, dtype=torch.int32, device=DEV)]
        return (lambda: self.lib.avsep_stft_varlen(self.h, self.p("waves"), self.p("wave_lens"), B, L, NFFT, HOP,
                                                   *[o.data_ptr() for o in outs], _stream())), outs

    def istft(self):
        out = _nan(B, 1, L)
        return (lambda: self.lib.avsep_istft(self.h, self.p("spec"), None, B, 1, TW, NFFT, HOP, L, out.data_ptr(),
                                             _stream())), [out]

    def istft_varlen(self):
        out = _nan(B, 1, L)
        return (lambda: self.lib.avsep_istft_varlen(self.h, self.p("spec"), None, self.p("wave_lens"), B, 1, TW, NFFT,
                                                    HOP, L, out.data_ptr(), _stream())), [out]

    def separate(self):
        out = _nan(B, S, F, T)
        return (lambda: self.lib.avsep_separate(self.h, self.p("masks"), self.p("mixed"), B, T, out.data_ptr(),
                                                _stream())), [out]

    def separate_varlen(self):
        out = _nan(B, S, F, T)
        return (lambda: self.lib.avsep_separate_varlen(self.h, self.p("masks"), self.p("mixed"), self.p("lens_d"), B, T,
                                                       out.data_ptr(), _stream())), [out]

    def flag_signal(self):
        flags, arr = _flags(2, 0)
        return (lambda: self.lib.avsep_flag_signal(self.h, arr, 2, 3, _stream())), [flags]

    def flag_wait(self):
        flags, arr = _flags(2, 5)       # already raised: the wait returns at once
        return (lambda: self.lib.avsep_flag_wait(self.h, arr, 2, 5, 10.0, _stream())), [flags]

    def copy_async(self):
        out = _nan(B, F, T)
        return (lambda: self.lib.avsep_copy_async(self.h, out.data_ptr(), self.p("mixed"), out.numel() * 4,
                                                  _stream())), [out]

    def finalize_weights(self):
        return (lambda: self.lib.avsep_finalize_weights(self.h, _stream())), []

    def test_gemm(self):
        out = _nan(M, D)
        return (lambda: self.lib.avsep_test_gemm(self.h, self.p("A"), self.p("W"), self.p("b"), out.data_ptr(), M, D, D,
                                                 1, 0, _stream())), [out]

    def test_gemm_ln(self):
        x, out = self.i["x"].clone(), _nan(M, D, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_gemm_ln(self.h, self.p("A"), self.p("W"), self.p("b"), x.data_ptr(),
                                                    self.p("gamma"), self.p("b"), out.data_ptr(), M, D, D,
                                                    _stream())), \
            [x, out]

    def test_gemm_trace(self):
        out, trace = _nan(M, D), _trace()
        return (lambda: self.lib.avsep_test_gemm_trace(self.h, self.p("A"), self.p("W"), self.p("b"), out.data_ptr(),
                                                       None, None, None, M, D, D, 0, 0, trace.data_ptr(), _stream())), \
            [out]

    def test_ffn_fused(self):
        x, out = self.i["x"].clone(), _nan(M, D, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_ffn_fused(self.h, self.p("A"), self.p("W1"), self.p("b4"), self.p("W2"),
                                                      self.p("b"), 1, x.data_ptr(), self.p("gamma"), self.p("b"),
                                                      out.data_ptr(), M, _stream())), [x, out]

    def test_ffn_fused_trace(self):
        x, out, trace = self.i["x"].clone(), _nan(M, D, dtype=torch.bfloat16), _trace()
        return (lambda: self.lib.avsep_test_ffn_fused_trace(self.h, self.p("A"), self.p("W1"), self.p("b4"),
                                                            self.p("W2"), self.p("b"), 2, x.data_ptr(), self.p("gamma"),
                                                            self.p("b"), out.data_ptr(), M, trace.data_ptr(),
                                                            _stream())), [x, out]

    def test_conv1d(self):
        out = _nan(2 * 63, D)           # two utterances of 63 rows: A holds them with a halo row either side
        return (lambda: self.lib.avsep_test_conv1d(self.h, self.p("A"), self.p("W3"), self.p("b"), out.data_ptr(), 2,
                                                   63, D, D, _stream())), [out]

    def test_attention(self):
        out = _nan(2, 128, D, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_attention(self.h, self.p("q"), self.p("k"), self.p("v"), out.data_ptr(), 2,
                                                      4, 64, 128, 128, 0, _stream())), [out]

    def test_attention_lerp(self):     # 50 fp32 source rows interpolated to 128: two interpolations, then tcgen05
        out = _nan(2, 128, D, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_attention(self.h, self.p("q"), self.p("k_src"), self.p("v_src"),
                                                      out.data_ptr(), 2, 4, 64, 128, 128, 50, _stream())), [out]

    def test_add_layernorm(self):
        xo, out = _nan(M, D), _nan(M, D, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_add_layernorm(self.h, self.p("x"), self.p("x"), self.p("gamma"),
                                                          self.p("b"), xo.data_ptr(), out.data_ptr(), M, D,
                                                          _stream())), [xo, out]

    def test_visual_cnn(self):
        out = _nan(8, 128, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_visual_cnn(self.h, self.p("cnn_frames"), 8, HW, HW, out.data_ptr(),
                                                       _stream())), [out]

    def test_visual_cnn_trace(self):
        out, trace = _nan(8, 128, dtype=torch.bfloat16), _trace()
        return (lambda: self.lib.avsep_test_visual_cnn_trace(self.h, self.p("cnn_frames"), 8, out.data_ptr(),
                                                             trace.data_ptr(), _stream())), [out]

    def test_xformer_stack(self):
        out_x, out_op = _nan(B * T, D), _nan(B * T, D, dtype=torch.bfloat16)
        return (lambda: self.lib.avsep_test_xformer_stack(self.h, 0, self.p("rows_a"), None, B, T, out_x.data_ptr(),
                                                          out_op.data_ptr(), 1, None, _stream())), [out_x, out_op]

    def test_fusion_decoder(self):
        sep, masks = _nan(B, S, F, T), _nan(B, S, F, T)
        return (lambda: self.lib.avsep_test_fusion_decoder(self.h, self.p("rows_a"), self.p("kv"), B, T,
                                                           self.p("mixed"), sep.data_ptr(), masks.data_ptr(), None,
                                                           _stream())), \
            [sep, masks]


CALLS = [name for name in vars(Calls) if not name.startswith("_") and name != "p"]


def _ok(eng, rc):
    assert rc == 0, eng.lib.avsep_last_error(eng.h).decode()


def _profile_every_call(path):
    """Writes {name: [launch count, kernels the CUDA profiler recorded]} of one eager call of each entry point to
    path."""
    from torch.profiler import ProfilerActivity, profile
    eng = _engine()
    calls = Calls(eng, _inputs())
    got = {}
    for name in CALLS:
        build = getattr(calls, name)
        _ok(eng, build()[0]())             # loads the kernels and sizes the handle's buffers outside the profiled call
        _ok(eng, calls.forward()[0]())     # leaves a count of its own behind, which the call must not build on
        call, _ = build()
        torch.cuda.synchronize(DEV)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _ok(eng, call())
            torch.cuda.synchronize(DEV)
        kernels = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA
                   and not ev.name.startswith(("Memcpy", "Memset"))]      # copies are not kernels
        got[name] = [eng.launch_count(), kernels]
    eng.close()
    with open(path, "w") as f:
        json.dump(got, f)


@pytest.fixture(scope="module")
def profiled(tmp_path_factory):
    """The calls are profiled in a process of their own: once a torch.profiler session has run in a process, one
    started there some seconds later can record no CUDA events, which would break the other tests that profile."""
    path = tmp_path_factory.mktemp("profiled") / "counts.json"
    code = (f"import sys; sys.path[:0] = {[ROOT, os.path.join(ROOT, 'av-separation-transformer_b200')]!r}; "
            f"from tests.test_call_convention_gpu import _profile_every_call; _profile_every_call({str(path)!r})")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)
    return json.loads(path.read_text())


@pytest.mark.parametrize("name", CALLS)
def test_launch_count_is_the_kernels_the_call_enqueued(profiled, name):
    count, kernels = profiled[name]
    assert count == len(kernels), (name, count, kernels)


def test_host_forward_counts_the_same_eager_captured_and_replayed(eng, inp):
    """Two chunks of two utterances, each call after a forward of another shape: the eager call, the one that captures
    each chunk's graph and a replay report the same count."""
    calls = Calls(eng, inp)
    mixed = inp["mixed"][:2, :, :40].contiguous()
    sep, masks = _nan(2, S, F, 40), _nan(2, S, F, 40)
    eng.set_option("use_graph", 1)
    eng.set_option("host_chunk", 2)
    try:
        counts = []
        for _ in range(3):
            _ok(eng, eng.lib.avsep_forward(eng.h, mixed.data_ptr(), inp["frames"].data_ptr(), 2, 40, N, HW, HW,
                                           sep.data_ptr(), masks.data_ptr(), None, 0, _stream()))
            _ok(eng, calls.forward_host()[0]())
            counts.append(eng.launch_count())
    finally:
        eng.set_option("host_chunk", 0)
        eng.set_option("use_graph", 0)
    assert counts == [counts[0]] * 3 and counts[0] > 0, counts


def test_configuration_and_queries_leave_the_count(eng, inp):
    eng.set_debug(True)
    try:
        _ok(eng, Calls(eng, inp).forward()[0]())
    finally:
        eng.set_debug(False)
    want = eng.launch_count()
    assert want > 0

    def unchanged(what):
        assert eng.launch_count() == want, (what, eng.launch_count(), want)
    eng.set_option("host_lanes", 0)
    unchanged("set_option")
    eng.set_debug(False)
    unchanged("set_debug")
    eng.set_profile(False)
    unchanged("set_profile")
    eng.profile_report()
    unchanged("profile_report")
    assert eng.get_stage("fused").size == B * T * D
    unchanged("debug_get_stage")
    eng.host_wait(0)
    eng.host_wait(3)
    unchanged("host_wait")
    assert eng.lib.avsep_workspace_bytes(eng.h, B, T, N, HW, HW) > 0
    assert eng.lib.avsep_packed_workspace_bytes(eng.h, B, T, N, HW, HW) > 0
    unchanged("workspace sizes")
    eng.lib.avsep_last_error(eng.h)
    unchanged("last_error")


def _bytes(t):
    t = t.detach().cpu().contiguous()
    return (torch.view_as_real(t) if t.is_complex() else t).view(-1).view(torch.uint8)


def _run_with_current(eng, build, dev):
    """Makes one call with cuda:dev current; returns the bytes of its outputs and the device current after the call."""
    with torch.cuda.device(dev):
        call, outs = build()
        _ok(eng, call())
        after = torch.cuda.current_device()
        torch.cuda.synchronize(DEV)
    return [_bytes(o) for o in outs], after


def test_every_call_runs_on_the_handle_device_and_keeps_the_current_one(eng, inp):
    """The handle lives on cuda:0 and cuda:1 is current: each call gives the bytes it gives with cuda:0 current, and
    cuda:1 is still current afterwards."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    calls = Calls(eng, inp)
    for name in CALLS:
        want, _ = _run_with_current(eng, getattr(calls, name), 0)
        got, after = _run_with_current(eng, getattr(calls, name), 1)
        assert after == 1, name
        assert len(got) == len(want) and all(torch.equal(a, b) for a, b in zip(got, want)), name

    # a debug snapshot, read with either device current
    eng.set_debug(True)
    try:
        _ok(eng, calls.forward()[0]())
    finally:
        eng.set_debug(False)
    want = eng.get_stage("fused")
    with torch.cuda.device(1):
        got = eng.get_stage("fused")
        assert torch.cuda.current_device() == 1
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))

    # the report synchronises the handle's device, so the event pair of the call just made is in it
    eng.set_profile(True)
    try:
        eng.profile_report(reset=True)
        with torch.cuda.device(1):
            _ok(eng, calls.stft()[0]())
            report = eng.profile_report(reset=True)
            assert torch.cuda.current_device() == 1
    finally:
        eng.set_profile(False)
    assert report["other"][0] == 1, report
