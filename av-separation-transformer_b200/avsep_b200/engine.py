"""Thin Python owner of one ``avsep_handle``: weight upload and pointer marshalling for the C ABI.

PyTorch is used for device memory and streams only; every FLOP of the path runs in libavsep.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib

STAGE_NAMES = ("audio_embed", "audio_enc", "visual_pool", "visual_embed", "visual_enc", "fused")


@dataclass(frozen=True)
class EngineConfig:
    freq_bins: int
    d_model: int
    nhead: int
    num_encoder_layers: int
    num_fusion_layers: int
    num_speakers: int
    precision: str = "bf16"


def _prec_code(p: str) -> int:
    if p in ("bf16", "bfloat16"):
        return _lib.PREC_BF16
    if p in ("tf32", "fp32", "float32"):
        return _lib.PREC_TF32
    raise ValueError(f"unknown precision {p!r} (use 'bf16' or 'tf32')")


def expected_shapes(cfg: EngineConfig) -> dict:
    """state_dict contract of the reference module (SURVEY.md Appendix A): key -> shape."""
    d, F, S = cfg.d_model, cfg.freq_bins, cfg.num_speakers
    out = {
        "audio_encoder.input_proj.0.weight": (d, F, 3), "audio_encoder.input_proj.0.bias": (d,),
        "audio_encoder.input_proj.2.weight": (d, d, 3), "audio_encoder.input_proj.2.bias": (d,),
        "audio_encoder.pos_enc.pe": (1, 5000, d), "visual_encoder.pos_enc.pe": (1, 5000, d),
        "visual_encoder.frame_proj.weight": (d, 128), "visual_encoder.frame_proj.bias": (d,),
        "fusion.norm.weight": (d,), "fusion.norm.bias": (d,),
        "decoder.decoder.0.weight": (2 * d, d), "decoder.decoder.0.bias": (2 * d,),
        "decoder.decoder.3.weight": (S * F, 2 * d), "decoder.decoder.3.bias": (S * F,),
    }
    cin = 1
    for idx, cout in ((0, 32), (3, 64), (6, 128)):
        out[f"visual_encoder.conv.{idx}.weight"] = (cout, cin, 3, 3)
        out[f"visual_encoder.conv.{idx}.bias"] = (cout,)
        for k in ("weight", "bias", "running_mean", "running_var"):
            out[f"visual_encoder.conv.{idx + 1}.{k}"] = (cout,)
        cin = cout
    for pre in ("audio_encoder", "visual_encoder"):
        for l in range(cfg.num_encoder_layers):
            p = f"{pre}.transformer.layers.{l}"
            out.update({
                f"{p}.self_attn.in_proj_weight": (3 * d, d), f"{p}.self_attn.in_proj_bias": (3 * d,),
                f"{p}.self_attn.out_proj.weight": (d, d), f"{p}.self_attn.out_proj.bias": (d,),
                f"{p}.linear1.weight": (4 * d, d), f"{p}.linear1.bias": (4 * d,),
                f"{p}.linear2.weight": (d, 4 * d), f"{p}.linear2.bias": (d,),
                f"{p}.norm1.weight": (d,), f"{p}.norm1.bias": (d,),
                f"{p}.norm2.weight": (d,), f"{p}.norm2.bias": (d,),
            })
    for l in range(cfg.num_fusion_layers):
        p = f"fusion.layers.{l}"
        out.update({
            f"{p}.cross_attn.in_proj_weight": (3 * d, d), f"{p}.cross_attn.in_proj_bias": (3 * d,),
            f"{p}.cross_attn.out_proj.weight": (d, d), f"{p}.cross_attn.out_proj.bias": (d,),
            f"{p}.ff.0.weight": (4 * d, d), f"{p}.ff.0.bias": (4 * d,),
            f"{p}.ff.3.weight": (d, 4 * d), f"{p}.ff.3.bias": (d,),
            f"{p}.norm1.weight": (d,), f"{p}.norm1.bias": (d,),
            f"{p}.norm2.weight": (d,), f"{p}.norm2.bias": (d,),
        })
    return out


class Engine:
    """One C handle bound to one CUDA device."""

    def __init__(self, cfg: EngineConfig, device: int):
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = int(device)
        c = _lib.AvsepConfig(cfg.freq_bins, cfg.d_model, cfg.nhead, cfg.num_encoder_layers,
                             cfg.num_fusion_layers, cfg.num_speakers, _prec_code(cfg.precision), self.device)
        h = C.c_void_p()
        if self.lib.avsep_create(C.byref(c), C.byref(h)) != 0:
            raise RuntimeError("avsep_create: " + self.lib.avsep_last_error(None).decode())
        self.h = h
        self._keep = []
        self._len_bufs = {}   # ((method, name), stream) -> engine-owned int32 device buffer (stable graph key)

    def close(self):
        if getattr(self, "h", None):
            self.lib.avsep_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what}: {self.lib.avsep_last_error(self.h).decode()}")

    # ---- weights --------------------------------------------------------------------------------
    def load_state(self, state: dict, fill_missing: bool = False):
        """state: reference key -> torch tensor / numpy array.  Missing keys are an error unless
        ``fill_missing`` (stand-alone sub-modules), in which case neutral values are used."""
        want = expected_shapes(self.cfg)
        for key, shape in want.items():
            if key in state:
                v = state[key]
                arr = v.detach().to("cpu", torch.float32).contiguous().numpy() if isinstance(v, torch.Tensor) \
                    else np.ascontiguousarray(v, dtype=np.float32)
            elif fill_missing:
                neutral_one = key.endswith("running_var") or (key.endswith(".weight") and len(shape) == 1)
                arr = np.ones(shape, np.float32) if neutral_one else np.zeros(shape, np.float32)
            else:
                raise KeyError(f"state_dict is missing {key!r}")
            if tuple(arr.shape) != tuple(shape):
                raise ValueError(f"{key}: expected shape {shape}, got {tuple(arr.shape)}")
            shp = (C.c_int64 * len(shape))(*shape)
            self._check(self.lib.avsep_set_weight(self.h, key.encode(), arr.ctypes.data_as(C.c_void_p),
                                                  _lib.DTYPE_F32, shp, len(shape)), "avsep_set_weight")
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._check(self.lib.avsep_finalize_weights(self.h, C.c_void_p(stream)), "avsep_finalize_weights")

    # ---- helpers ---------------------------------------------------------------------------------
    def _dev_f32(self, t: torch.Tensor, name: str) -> torch.Tensor:
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{name} must be a torch.Tensor")
        if not t.is_cuda or t.device.index != self.device:
            raise RuntimeError(f"{name} must live on cuda:{self.device} (there is no CPU path)")
        if t.dtype != torch.float32:
            t = t.float()
        return t.contiguous()

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- shape contract (every entry point validates BEFORE a pointer reaches the C ABI: the library sizes its
    # copies and strides from the engine config, so a wrong F / d / batch would read or write out of bounds) ----
    def _check_inputs(self, what: str, mixed=None, frames=None, rows=None, rows2=None, out=None):
        """mixed (B,F,T) | frames (B,N,H,W) | rows / rows2 (B,L,d) | out = (separated, masks) (B,S,F,T).
        Returns (B, T, N, Hh, Ww) with None for the dims that were not given.  Raises ValueError."""
        cfg = self.cfg
        B = T = N = Hh = Ww = None
        if mixed is not None:
            if mixed.dim() != 3:
                raise ValueError(f"{what}: mixed_spec must be (B, freq_bins, T), got {tuple(mixed.shape)}")
            B, F, T = mixed.shape
            if F != cfg.freq_bins:
                raise ValueError(f"{what}: mixed_spec has {F} frequency bins, model expects {cfg.freq_bins}")
        if frames is not None:
            if frames.dim() != 4:
                raise ValueError(f"{what}: lip_frames must be (B, num_frames, H, W), got {tuple(frames.shape)}")
            Bf, N, Hh, Ww = frames.shape
            if B is not None and Bf != B:
                raise ValueError(f"{what}: batch size of mixed_spec ({B}) and lip_frames ({Bf}) differ")
            B = Bf
        for r in (rows, rows2):
            if r is None:
                continue
            if r.dim() != 3 or r.shape[2] != cfg.d_model:
                raise ValueError(f"{what}: expected (B, L, {cfg.d_model}) rows, got {tuple(r.shape)}")
            if B is not None and r.shape[0] != B:
                raise ValueError(f"{what}: batch sizes differ ({B} vs {r.shape[0]})")
            B = r.shape[0]
        if B is not None and B < 1:
            raise ValueError(f"{what}: empty batch")
        if out is not None:
            want = (B, cfg.num_speakers, cfg.freq_bins, T)
            for t in out:
                if tuple(t.shape) != want or t.dtype != torch.float32 or not t.is_contiguous():
                    raise ValueError(f"{what}: output buffers must be contiguous float32 {want}, got {tuple(t.shape)}")
        return B, T, N, Hh, Ww

    def _lengths(self, v, name: str, B: int, limit: int, what: str = "forward"):
        """Per-utterance lengths -> int32 device tensor (or None).  A list, numpy array or CPU integer tensor is
        validated here (B entries, 1 <= v <= limit) and copied into an engine-owned buffer of the current stream, so
        the pointer - and with it the CUDA-graph key - stays the same from call to call, and the copy is ordered after
        the previous call on that stream that read the buffer (one buffer per method, name and stream: calls on two
        streams never share one).  The copy goes through pinned memory and does not block the host.  An int32 tensor
        on the engine's device is passed through without reading it: the library clamps its values to [1, limit].
        ``what`` names the calling method in the error messages."""
        if v is None:
            return None
        if isinstance(v, torch.Tensor) and v.is_cuda:
            if v.device.index != self.device or v.dtype != torch.int32 or tuple(v.shape) != (B,) or not v.is_contiguous():
                raise ValueError(f"{what}: a device {name} tensor must be contiguous int32 ({B},) on cuda:{self.device}")
            return v
        a = v.numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        if a.shape != (B,):
            raise ValueError(f"{what}: {name} must have one entry per utterance ({B}), got shape {a.shape}")
        if a.dtype == np.bool_ or not np.issubdtype(a.dtype, np.integer):
            raise ValueError(f"{what}: {name} must hold integers, got {a.dtype}")
        if a.min() < 1 or a.max() > limit:
            raise ValueError(f"{what}: {name} must lie in [1, {limit}], got [{a.min()}, {a.max()}]")
        buf = self._stream_buf((what, name), B)
        # the pinned staging block is not reused before this copy has run (torch's host allocator records the stream)
        buf[:B].copy_(torch.from_numpy(a.astype(np.int32)).pin_memory(), non_blocking=True)
        return buf[:B]

    def _stream_buf(self, name, B: int) -> torch.Tensor:
        """Engine-owned int32 device buffer of at least B entries for ``name`` on the current stream."""
        key = (name, torch.cuda.current_stream(self.device).cuda_stream)
        buf = self._len_bufs.get(key)
        if buf is None or buf.numel() < B:
            buf = torch.empty(max(B, 256), dtype=torch.int32, device=torch.device("cuda", self.device))
            self._len_bufs[key] = buf
        return buf

    # ---- forward ---------------------------------------------------------------------------------
    def forward(self, mixed: torch.Tensor, frames: torch.Tensor, out=None, lengths=None, frame_lengths=None):
        """Device tensors in, device tensors out.  ``out=(separated, masks)`` reuses caller-owned (B,S,F,T) float32
        buffers: with fixed input and output buffers every call after the second is one CUDA-graph replay.

        Variable-length batch: ``lengths`` (B,) audio frames and ``frame_lengths`` (B,) lip frames per utterance, each
        left-aligned in the padded (T, N) inputs; None = all T / all N.  Utterance b's outputs [b, :, :, :lengths[b]]
        equal a forward of that utterance alone, the rest are 0, and the padding of the inputs is never read."""
        mixed = self._dev_f32(mixed, "mixed_spec")
        frames = self._dev_f32(frames, "lip_frames")
        B, T, N, Hh, Ww = self._check_inputs("forward", mixed=mixed, frames=frames, out=out)
        with torch.cuda.device(self.device):
            lens = self._lengths(lengths, "lengths", B, T)
            flens = self._lengths(frame_lengths, "frame_lengths", B, N)
        F, S = self.cfg.freq_bins, self.cfg.num_speakers
        if out is None:
            # one allocation for both outputs: the caching allocator then recycles a handful of blocks, so the
            # (inputs, outputs) pointer sets the library's CUDA-graph cache is keyed on repeat after a few calls
            both = torch.empty((2, B, S, F, T), device=mixed.device, dtype=torch.float32)
            sep, masks = both[0], both[1]
        else:
            sep, masks = out
            for t in out:
                if not t.is_cuda or t.device.index != self.device:
                    raise ValueError(f"forward: output buffers must live on cuda:{self.device}")
        if lens is None and flens is None:
            fn, what = self.lib.avsep_forward, "avsep_forward"
            args = (self.h, mixed.data_ptr(), frames.data_ptr(), B, T, N, Hh, Ww, sep.data_ptr(), masks.data_ptr(),
                    None, 0, self._stream())
        else:
            fn, what = self.lib.avsep_forward_varlen, "avsep_forward_varlen"
            args = (self.h, mixed.data_ptr(), frames.data_ptr(), None if lens is None else lens.data_ptr(),
                    None if flens is None else flens.data_ptr(), B, T, N, Hh, Ww, sep.data_ptr(), masks.data_ptr(),
                    None, 0, self._stream())
        if torch.cuda.current_device() == self.device:      # the library selects its device itself; only restore the
            rc = fn(*args)                                   # caller's when it differs
        else:
            with torch.cuda.device(self.device):
                rc = fn(*args)
        self._check(rc, what)
        return sep, masks

    @staticmethod
    def _host_f32(t: torch.Tensor, name: str) -> torch.Tensor:
        if not isinstance(t, torch.Tensor) or t.is_cuda:
            raise ValueError(f"{name} must be a CPU tensor")
        return t.contiguous().float()

    def forward_host(self, mixed: torch.Tensor, frames: torch.Tensor, sep: torch.Tensor = None,
                     masks: torch.Tensor = None):
        """CPU tensors in, CPU tensors out; H2D, kernels and D2H all inside the C call (pinned memory advised)."""
        mixed = self._host_f32(mixed, "mixed_spec")
        frames = self._host_f32(frames, "lip_frames")
        B, T, N, Hh, Ww = self._check_inputs("forward_host", mixed=mixed, frames=frames)
        F, S = self.cfg.freq_bins, self.cfg.num_speakers
        if sep is None:
            sep = torch.empty((B, S, F, T), dtype=torch.float32).pin_memory()
        if masks is None:
            masks = torch.empty((B, S, F, T), dtype=torch.float32).pin_memory()
        self._check_inputs("forward_host", mixed=mixed, out=(sep, masks))
        if sep.is_cuda or masks.is_cuda:
            raise ValueError("forward_host: output buffers must be CPU tensors")
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_forward_host(self.h, mixed.data_ptr(), frames.data_ptr(), B, T, N, Hh, Ww,
                                             sep.data_ptr(), masks.data_ptr(), self._stream())
        self._check(rc, "avsep_forward_host")
        return sep, masks

    def forward_host_async(self, mixed: torch.Tensor, frames: torch.Tensor, sep: torch.Tensor, masks: torch.Tensor,
                           slot: int):
        """Streaming form: enqueue one batch on I/O slot 0 .. 3 (AVSEP_HOST_SLOTS) and return; ``host_wait(slot)`` completes it.  All four
        tensors must be contiguous float32 CPU tensors (pinned for real overlap) that outlive the wait."""
        for t in (mixed, frames, sep, masks):
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError("forward_host_async: contiguous float32 CPU tensors required")
        B, T, N, Hh, Ww = self._check_inputs("forward_host_async", mixed=mixed, frames=frames, out=(sep, masks))
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_forward_host_async(self.h, mixed.data_ptr(), frames.data_ptr(), B, T, N, Hh, Ww,
                                                   sep.data_ptr(), masks.data_ptr(), int(slot), self._stream())
        self._check(rc, "avsep_forward_host_async")

    def host_wait(self, slot: int):
        self._check(self.lib.avsep_host_wait(self.h, int(slot)), "avsep_host_wait")

    def launch_count(self) -> int:
        return int(self.lib.avsep_last_launch_count(self.h))

    # ---- sub-modules -------------------------------------------------------------------------------
    def audio_encoder(self, mixed):
        mixed = self._dev_f32(mixed, "mixed_spec")
        B, T, _, _, _ = self._check_inputs("audio_encoder", mixed=mixed)
        out = torch.empty((B, T, self.cfg.d_model), device=mixed.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_audio_encoder(self.h, mixed.data_ptr(), B, T, out.data_ptr(), self._stream())
        self._check(rc, "avsep_audio_encoder")
        return out

    def visual_encoder(self, frames, target_len: int):
        frames = self._dev_f32(frames, "lip_frames")
        B, _, N, Hh, Ww = self._check_inputs("visual_encoder", frames=frames)
        if int(target_len) < 1:
            raise ValueError("visual_encoder: target_len must be >= 1")
        out = torch.empty((B, int(target_len), self.cfg.d_model), device=frames.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_visual_encoder(self.h, frames.data_ptr(), B, N, Hh, Ww, int(target_len),
                                               out.data_ptr(), self._stream())
        self._check(rc, "avsep_visual_encoder")
        return out

    def fusion(self, audio, visual):
        audio = self._dev_f32(audio, "audio")
        visual = self._dev_f32(visual, "visual")
        self._check_inputs("fusion", rows=audio, rows2=visual)
        B, T, d = audio.shape
        L = visual.shape[1]
        out = torch.empty_like(audio)
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_fusion(self.h, audio.data_ptr(), visual.data_ptr(), B, T, L, out.data_ptr(),
                                       self._stream())
        self._check(rc, "avsep_fusion")
        return out

    def decoder(self, fused, mixed):
        fused = self._dev_f32(fused, "fused")
        mixed = self._dev_f32(mixed, "mixed_spec")
        self._check_inputs("decoder", mixed=mixed, rows=fused)
        B, T, d = fused.shape
        if mixed.shape[2] != T:
            raise ValueError(f"decoder: fused has {T} frames, mixed_spec has {mixed.shape[2]}")
        F, S = self.cfg.freq_bins, self.cfg.num_speakers
        sep = torch.empty((B, S, F, T), device=fused.device, dtype=torch.float32)
        masks = torch.empty_like(sep)
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_decoder(self.h, fused.data_ptr(), mixed.data_ptr(), B, T, sep.data_ptr(),
                                        masks.data_ptr(), self._stream())
        self._check(rc, "avsep_decoder")
        return sep, masks

    def separate(self, masks, mixed, out=None):
        """avsep_separate: SeparationDecoder.separate (reference model.py:210-220), masks (B,S,F,T) x mixed (B,F,T)."""
        masks = self._dev_f32(masks, "masks")
        mixed = self._dev_f32(mixed, "mixed_spec")
        B, T, _, _, _ = self._check_inputs("separate", mixed=mixed, out=(masks,) if out is None else (masks, out))
        sep = torch.empty_like(masks) if out is None else out
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_separate(self.h, masks.data_ptr(), mixed.data_ptr(), B, T, sep.data_ptr(), self._stream())
        self._check(rc, "avsep_separate")
        return sep

    # ---- rows either side of the path --------------------------------------------------------------
    def synth_batch(self, geom: dict, amps, freqs, phases, noise=None, want_clean: bool = True):
        """avsep_synth_batch: device tensors amps/freqs/phases (B,S) float64, noise (B,S,nf,ph,pw) float32 or None.

        geom keys: num_samples_audio, duration, n_fft, hop_length, num_frames, frame_h, frame_w, num_speakers.
        Returns mixed_spec (B,F,T), lip_frames (B,S*nf,H,W), clean_specs (B,S,F,T) or None."""
        dev = torch.device("cuda", self.device)
        for t, dt in ((amps, torch.float64), (freqs, torch.float64), (phases, torch.float64)):
            if t.device != dev or t.dtype != dt or not t.is_contiguous():
                raise ValueError("synth_batch: amps/freqs/phases must be contiguous float64 tensors on the engine device")
        B, S = amps.shape
        if S != geom["num_speakers"] or freqs.shape != amps.shape or phases.shape != amps.shape:
            raise ValueError("synth_batch: amps/freqs/phases must be (B, num_speakers)")
        cfg = _lib.AvsepSynthConfig(geom["num_samples_audio"], float(geom["duration"]), geom["n_fft"],
                                    geom["hop_length"], geom["num_frames"], geom["frame_h"], geom["frame_w"], S)
        F, T = geom["n_fft"] // 2 + 1, 1 + geom["num_samples_audio"] // geom["hop_length"]
        nf, Hh, Ww = geom["num_frames"], geom["frame_h"], geom["frame_w"]
        if noise is not None:
            want = (B, S, nf, 3 * Hh // 4 - Hh // 4, 3 * Ww // 4 - Ww // 4)
            if tuple(noise.shape) != want or noise.dtype != torch.float32 or noise.device != dev or not noise.is_contiguous():
                raise ValueError(f"synth_batch: noise must be a contiguous float32 device tensor of shape {want}")
        mixed = torch.empty(B, F, T, device=dev)
        frames = torch.empty(B, S * nf, Hh, Ww, device=dev)
        clean = torch.empty(B, S, F, T, device=dev) if want_clean else None
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_synth_batch(self.h, C.byref(cfg), B, amps.data_ptr(), freqs.data_ptr(), phases.data_ptr(),
                                            noise.data_ptr() if noise is not None else None, mixed.data_ptr(),
                                            frames.data_ptr(), clean.data_ptr() if clean is not None else None,
                                            self._stream())
        self._check(rc, "avsep_synth_batch")
        return mixed, frames, clean

    def eval_snr(self, separated, targets, mixed=None):
        """avsep_eval_snr: per-utterance input SNRs (B,S), best-permutation output SNR (B), permutation code (B),
        SI-SNR (B); float64 dB, device tensors."""
        dev = torch.device("cuda", self.device)
        for t in (separated, targets) + ((mixed,) if mixed is not None else ()):
            if t.device != dev or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError("eval_snr: tensors must be contiguous float32 on the engine device")
        B, S, F, T = separated.shape
        if targets.shape != separated.shape or (mixed is not None and tuple(mixed.shape) != (B, F, T)):
            raise ValueError("eval_snr: shape mismatch")
        in_snr = torch.empty(B, S, device=dev, dtype=torch.float64) if mixed is not None else None
        out_snr = torch.empty(B, device=dev, dtype=torch.float64)
        perm = torch.empty(B, device=dev, dtype=torch.int32)
        si = torch.empty(B, device=dev, dtype=torch.float64)
        with torch.cuda.device(self.device):
            rc = self.lib.avsep_eval_snr(self.h, separated.data_ptr(), targets.data_ptr(),
                                         mixed.data_ptr() if mixed is not None else None, B, S, F, T,
                                         in_snr.data_ptr() if in_snr is not None else None, out_snr.data_ptr(),
                                         perm.data_ptr(), si.data_ptr(), self._stream())
        self._check(rc, "avsep_eval_snr")
        return in_snr, out_snr, perm, si

    def stft(self, waves, n_fft: int = 512, hop_length: int = 128, want_mag: bool = True, lengths=None):
        """avsep_stft: (B, L) float32 waveforms -> complex64 (B, F, T) with the framing of the reference's
        SyntheticAVDataset._stft (dataset.py:122-135) and, optionally, its float32 magnitude (the model input).

        Variable-length batch: ``lengths`` (B,) samples per utterance, each left-aligned in its row (see
        ``Engine._lengths`` for the accepted forms).  Utterance b's spec / mag [b, :, :T_b] with T_b = 1 + L_b // hop
        equal this call on ``waves[b, :L_b]`` alone and the rest is 0; samples past L_b are never read.  The call then
        returns (spec, mag, frame_lengths): frame_lengths is an int32 device tensor of the T_b, ready for
        ``forward(lengths=...)``.  It lives in an engine-owned buffer of the current stream (a stable pointer keeps the
        forward's CUDA graph cached) and is overwritten by the next such call on that stream."""
        dev = torch.device("cuda", self.device)
        if waves.device != dev or waves.dtype != torch.float32 or not waves.is_contiguous() or waves.dim() != 2:
            raise ValueError("stft: waves must be a contiguous float32 (B, L) tensor on the engine device")
        B, L = waves.shape
        F, T = n_fft // 2 + 1, 1 + L // hop_length
        spec = torch.empty(B, F, T, device=dev, dtype=torch.complex64)
        mag = torch.empty(B, F, T, device=dev, dtype=torch.float32) if want_mag else None
        with torch.cuda.device(self.device):
            if lengths is None:
                rc = self.lib.avsep_stft(self.h, waves.data_ptr(), B, L, n_fft, hop_length, spec.data_ptr(),
                                         mag.data_ptr() if want_mag else None, self._stream())
                self._check(rc, "avsep_stft")
                return spec, mag
            lens = self._lengths(lengths, "lengths", B, L, "stft")
            flens = self._stream_buf(("stft", "frame_lengths"), B)[:B]
            rc = self.lib.avsep_stft_varlen(self.h, waves.data_ptr(), lens.data_ptr(), B, L, n_fft, hop_length,
                                            spec.data_ptr(), mag.data_ptr() if want_mag else None, flens.data_ptr(),
                                            self._stream())
        self._check(rc, "avsep_stft_varlen")
        return spec, mag, flens

    def istft(self, spec, masks=None, length: int = None, n_fft: int = 512, hop_length: int = 128, lengths=None):
        """avsep_istft: complex64 (B, F, T) mixture spectrum (+ (B, S, F, T) float32 masks) -> (B, S, L) float32
        waveforms by weighted overlap-add; without masks the plain inverse, (B, 1, L).

        Variable-length batch: ``lengths`` (B,) output samples per utterance (forms as for ``stft``).  With
        T_b = min(T, 1 + L_b // hop), waves[b, :, :L_b] equal this call on spec[b, :, :T_b] and masks[b, :, :, :T_b]
        alone at length L_b, the rest is 0, and spectrum and mask columns past T_b are never read."""
        dev = torch.device("cuda", self.device)
        if spec.device != dev or spec.dtype != torch.complex64 or not spec.is_contiguous() or spec.dim() != 3:
            raise ValueError("istft: spec must be a contiguous complex64 (B, F, T) tensor on the engine device")
        B, F, T = spec.shape
        if F != n_fft // 2 + 1:
            raise ValueError("istft: spec has %d bins, n_fft=%d needs %d" % (F, n_fft, n_fft // 2 + 1))
        S = 1
        if masks is not None:
            if masks.device != dev or masks.dtype != torch.float32 or not masks.is_contiguous() or masks.dim() != 4:
                raise ValueError("istft: masks must be a contiguous float32 (B, S, F, T) tensor on the engine device")
            S = masks.shape[1]
            if (masks.shape[0], masks.shape[2], masks.shape[3]) != (B, F, T):
                raise ValueError("istft: masks / spec shape mismatch")
        L = (T - 1) * hop_length if length is None else int(length)
        waves = torch.empty(B, S, L, device=dev, dtype=torch.float32)
        with torch.cuda.device(self.device):
            if lengths is None:
                rc = self.lib.avsep_istft(self.h, spec.data_ptr(), masks.data_ptr() if masks is not None else None, B,
                                          S, T, n_fft, hop_length, L, waves.data_ptr(), self._stream())
                self._check(rc, "avsep_istft")
                return waves
            lens = self._lengths(lengths, "lengths", B, L, "istft")
            rc = self.lib.avsep_istft_varlen(self.h, spec.data_ptr(), masks.data_ptr() if masks is not None else None,
                                             lens.data_ptr(), B, S, T, n_fft, hop_length, L, waves.data_ptr(),
                                             self._stream())
        self._check(rc, "avsep_istft_varlen")
        return waves

    def set_option(self, name: str, value: int):
        """Execution options of avsep_set_option (include/avsep.h): 'use_graph', 'two_stream', 'pdl' (0/1), 'attn_tc'
        (0 never, 1 long sequences, 2 whenever usable), 'host_chunk', 'host_lanes' (0 = auto), 'profile_spin_us'.
        An unknown name raises RuntimeError."""
        self._check(self.lib.avsep_set_option(self.h, name.encode(), int(value)), "avsep_set_option")

    # ---- profiling -------------------------------------------------------------------------------
    def set_profile(self, on: bool):
        self._check(self.lib.avsep_set_profile(self.h, 1 if on else 0), "avsep_set_profile")

    def profile_report(self, reset: bool = True) -> dict:
        """label -> (launches, total_ms) accumulated since the last reset."""
        buf = C.create_string_buffer(1 << 16)
        self._check(self.lib.avsep_profile_report(self.h, buf, len(buf), 1 if reset else 0), "avsep_profile_report")
        out = {}
        for line in buf.value.decode().splitlines():
            label, n, ms = line.split()
            out[label] = (int(n), float(ms))
        return out

    # ---- debug -------------------------------------------------------------------------------------
    def set_debug(self, on: bool):
        self._check(self.lib.avsep_set_debug(self.h, 1 if on else 0), "avsep_set_debug")

    def get_stage(self, name: str) -> np.ndarray:
        n = C.c_size_t(0)
        self._check(self.lib.avsep_debug_get_stage(self.h, name.encode(), None, 0, C.byref(n)), "avsep_debug_get_stage")
        out = np.empty(n.value, dtype=np.float32)
        self._check(self.lib.avsep_debug_get_stage(self.h, name.encode(), out.ctypes.data_as(C.c_void_p), n.value,
                                                   C.byref(n)), "avsep_debug_get_stage")
        return out
