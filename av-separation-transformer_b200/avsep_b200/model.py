"""Host-side mirror of the reference's module interface for the forward path.

Same class names, constructor arguments, attribute tree and ``state_dict`` key set as
/root/reference/src/av_separation/model.py (AudioEncoder :22, VisualEncoder :67, CrossModalFusion :124,
SeparationDecoder :180, AVSeparationTransformer :227, PositionalEncoding :283), so
``load_state_dict(reference.state_dict())`` works and, for a given torch seed, a freshly constructed
module holds the same random-init weights as the reference would.  The torch.nn modules created here
are parameter containers only: ``forward`` never calls them -- it hands raw device pointers to
libavsep.so (hand-written sm_100a kernels) through the C ABI in include/avsep.h.

Semantics are the reference's eval mode (dropout off, BatchNorm running statistics).  Modules are
constructed in eval mode and ``train(True)`` raises: this build implements the forward path only.
"""
from __future__ import annotations

import math
import warnings

import torch
import torch.nn as nn

from .engine import Engine, EngineConfig

__all__ = ["AudioEncoder", "VisualEncoder", "CrossModalFusion", "CrossAttentionLayer", "SeparationDecoder",
           "AVSeparationTransformer", "PositionalEncoding"]


def _numbered(mods: dict) -> nn.ModuleDict:
    """Container whose children are named by the given indices (e.g. '0', '2'), like the sparse
    numbering nn.Sequential leaves after parameter-free layers."""
    return nn.ModuleDict({str(k): m for k, m in mods.items()})


def _encoder_stack(d_model: int, nhead: int, num_layers: int, dropout: float) -> nn.Module:
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        layer = nn.TransformerEncoderLayer(d_model=d_model, nhead=nhead, dim_feedforward=4 * d_model,
                                           dropout=dropout, batch_first=True, norm_first=True)
        return nn.TransformerEncoder(layer, num_layers=num_layers)


def _refresh_after_load(module, incompatible_keys):      # module-level so that torch.save(model) can pickle the hook
    module.refresh_weights()


class _InferenceOnly(nn.Module):
    """Shared behaviour: eval-only, lazily (re)built engine.

    The engine holds a prepacked copy of the weights.  It is rebuilt when the weights may have changed:
    ``load_state_dict`` / ``.to()`` / ``.cuda()`` / ``.float()`` (hooks below), any in-place update that bumps a
    tensor's autograd version counter (``p.copy_()``, ``p.add_()``, optimiser steps -- a ~10 us sum over a cached
    tensor list per forward), or an explicit ``refresh_weights()``.  Edits through ``p.data`` do not bump the
    counter: call ``refresh_weights()`` after them."""

    def _post_init(self):
        self._engine = None
        self._engine_sig = None
        self._tensors = None          # cached list of parameters + buffers (rebuilt when Parameter objects change)
        self._weights_epoch = 0
        self.host_device = getattr(self, "host_device", "cuda:0")
        self.register_load_state_dict_post_hook(_refresh_after_load)
        nn.Module.train(self, False)

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError(
                "avsep_b200 implements the inference forward path only (eval semantics: dropout off, BatchNorm "
                "running statistics); training is out of scope")
        return nn.Module.train(self, False)

    # -- engine management ---------------------------------------------------------------------
    def _engine_config(self) -> EngineConfig:  # pragma: no cover - overridden
        raise NotImplementedError

    def _state_prefix(self) -> str:
        return ""

    def refresh_weights(self):
        """Mark the prepacked weights stale (the next forward re-uploads them)."""
        self._weights_epoch += 1
        self._tensors = None
        return self

    def _apply(self, fn, *args, **kwargs):          # .to() / .cuda() / .float(): Parameter storage may be replaced
        out = super()._apply(fn, *args, **kwargs)
        if hasattr(self, "_weights_epoch"):
            self.refresh_weights()
        return out

    def _weights_sig(self, device_index: int):
        if self._tensors is None:
            self._tensors = [t for _, t in self.named_parameters()] + [t for _, t in self.named_buffers()]
        v = 0
        for t in self._tensors:
            v += t._version
        return (device_index, self._weights_epoch, v)

    def _get_engine(self, device: torch.device) -> Engine:
        if device.type != "cuda":
            raise RuntimeError("avsep_b200 runs on CUDA (sm_100a) only; there is no CPU fallback")
        index = device.index if device.index is not None else torch.cuda.current_device()
        sig = self._weights_sig(index)
        if self._engine is None or self._engine_sig != sig:
            if self._engine is not None:
                self._engine.close()
            eng = Engine(self._engine_config(), index)
            pre = self._state_prefix()
            state = {pre + k: v for k, v in self.state_dict().items()}
            eng.load_state(state, fill_missing=bool(pre))
            self._engine, self._engine_sig = eng, sig
        return self._engine

    def prepack(self, device="cuda"):
        """Fold/repack/upload the weights now (otherwise done lazily on the first forward)."""
        self._get_engine(torch.device(device))
        return self

    def _run(self, fn_name: str, *tensors, extra=()):
        """Route one call: CUDA tensors run in place; CPU tensors (how the reference's own tests call the modules,
        tests/test_model.py:77-179) are uploaded to ``host_device``, run there and come back as CPU tensors --
        the arithmetic is on the GPU either way (there is no CPU implementation)."""
        first = tensors[0]
        if first.is_cuda:
            return getattr(self._get_engine(first.device), fn_name)(*tensors, *extra)
        dev = torch.device(self.host_device)
        out = getattr(self._get_engine(dev), fn_name)(*[t.to(dev) for t in tensors], *extra)
        return tuple(o.cpu() for o in out) if isinstance(out, tuple) else out.cpu()

    # the engine owns a ctypes handle: never pickled / deep-copied, rebuilt lazily by the copy
    def __getstate__(self):
        state = self.__dict__.copy()
        state["_engine"] = None
        state["_engine_sig"] = None
        state["_tensors"] = None
        return state

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            new.__dict__[k] = None if k in ("_engine", "_engine_sig", "_tensors") else copy.deepcopy(v, memo)
        return new


class PositionalEncoding(nn.Module):
    """Sinusoidal table buffer ``pe`` (1, max_len, d) -- reference model.py:283-301.  In the fused path the
    table is added inside the GEMM epilogues; this module exists for the state_dict contract and for
    stand-alone use (plain torch add, not on the hot path)."""

    def __init__(self, d_model: int, dropout: float = 0.1, max_len: int = 5000):
        super().__init__()
        self.dropout = nn.Dropout(dropout)
        pos = torch.arange(0, max_len).unsqueeze(1).float()
        freq = torch.exp(torch.arange(0, d_model, 2).float() * (-math.log(10000.0) / d_model))
        table = torch.zeros(max_len, d_model)
        table[:, 0::2] = torch.sin(pos * freq)
        table[:, 1::2] = torch.cos(pos * freq)
        self.register_buffer("pe", table.unsqueeze(0))
        self.eval()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return x + self.pe[:, : x.size(1)]


class AudioEncoder(_InferenceOnly):
    """(B, freq_bins, T) -> (B, T, d_model).  Reference: model.py:22-60."""

    def __init__(self, freq_bins: int = 257, d_model: int = 256, nhead: int = 4, num_layers: int = 2,
                 dropout: float = 0.1, precision: str = "bf16"):
        super().__init__()
        self.freq_bins, self.d_model, self.nhead, self.num_layers = freq_bins, d_model, nhead, num_layers
        self.precision = precision
        self.input_proj = _numbered({0: nn.Conv1d(freq_bins, d_model, kernel_size=3, padding=1),
                                     2: nn.Conv1d(d_model, d_model, kernel_size=3, padding=1)})
        self.pos_enc = PositionalEncoding(d_model, dropout=dropout)
        self.transformer = _encoder_stack(d_model, nhead, num_layers, dropout)
        self._post_init()

    def _engine_config(self):
        return EngineConfig(self.freq_bins, self.d_model, self.nhead, self.num_layers, 1, 1, self.precision)

    def _state_prefix(self):
        return "audio_encoder."

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._run("audio_encoder", x)


class VisualEncoder(_InferenceOnly):
    """(B, num_frames, H, W) -> (B, target_len, d_model).  Reference: model.py:67-117."""

    def __init__(self, d_model: int = 256, nhead: int = 4, num_layers: int = 2, dropout: float = 0.1,
                 precision: str = "bf16"):
        super().__init__()
        self.d_model, self.nhead, self.num_layers, self.precision = d_model, nhead, num_layers, precision
        self.conv = _numbered({
            0: nn.Conv2d(1, 32, kernel_size=3, stride=2, padding=1), 1: nn.BatchNorm2d(32),
            3: nn.Conv2d(32, 64, kernel_size=3, stride=2, padding=1), 4: nn.BatchNorm2d(64),
            6: nn.Conv2d(64, 128, kernel_size=3, stride=2, padding=1), 7: nn.BatchNorm2d(128),
        })
        self.frame_proj = nn.Linear(128, d_model)
        self.pos_enc = PositionalEncoding(d_model, dropout=dropout)
        self.transformer = _encoder_stack(d_model, nhead, num_layers, dropout)
        self._post_init()

    def _engine_config(self):
        return EngineConfig(8, self.d_model, self.nhead, self.num_layers, 1, 1, self.precision)

    def _state_prefix(self):
        return "visual_encoder."

    def forward(self, frames: torch.Tensor, target_len: int) -> torch.Tensor:
        return self._run("visual_encoder", frames, extra=(target_len,))


class CrossAttentionLayer(nn.Module):
    """Parameter container for one fusion layer (reference model.py:152-173)."""

    def __init__(self, d_model: int, nhead: int, dropout: float = 0.1):
        super().__init__()
        self.cross_attn = nn.MultiheadAttention(d_model, nhead, dropout=dropout, batch_first=True)
        self.ff = _numbered({0: nn.Linear(d_model, 4 * d_model), 3: nn.Linear(4 * d_model, d_model)})
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)


class CrossModalFusion(_InferenceOnly):
    """audio (B,T,d) queries visual (B,T,d) -> (B,T,d).  Reference: model.py:124-149."""

    def __init__(self, d_model: int = 256, nhead: int = 4, num_layers: int = 2, dropout: float = 0.1,
                 precision: str = "bf16"):
        super().__init__()
        self.d_model, self.nhead, self.num_layers, self.precision = d_model, nhead, num_layers, precision
        self.layers = nn.ModuleList([CrossAttentionLayer(d_model, nhead, dropout) for _ in range(num_layers)])
        self.norm = nn.LayerNorm(d_model)
        self._post_init()

    def _engine_config(self):
        return EngineConfig(8, self.d_model, self.nhead, 1, self.num_layers, 1, self.precision)

    def _state_prefix(self):
        return "fusion."

    def forward(self, audio: torch.Tensor, visual: torch.Tensor) -> torch.Tensor:
        return self._run("fusion", audio, visual)


class SeparationDecoder(_InferenceOnly):
    """fused (B,T,d) -> masks (B,S,F,T) in [0,1]; ``separate`` applies them.  Reference: model.py:180-220."""

    def __init__(self, d_model: int = 256, freq_bins: int = 257, num_speakers: int = 2, dropout: float = 0.1,
                 precision: str = "bf16"):
        super().__init__()
        self.d_model, self.freq_bins, self.num_speakers, self.precision = d_model, freq_bins, num_speakers, precision
        self.decoder = _numbered({0: nn.Linear(d_model, 2 * d_model), 3: nn.Linear(2 * d_model, freq_bins * num_speakers)})
        self._post_init()

    def _engine_config(self):
        nhead = 1
        for cand in (64, 32, 16, 128):           # any legal head width; attention is unused by this sub-module
            if self.d_model % cand == 0:
                nhead = self.d_model // cand
                break
        return EngineConfig(self.freq_bins, self.d_model, nhead, 1, 1, self.num_speakers, self.precision)

    def _state_prefix(self):
        return "decoder."

    def forward(self, fused: torch.Tensor) -> torch.Tensor:
        B, T, _ = fused.shape
        ones = torch.ones((B, self.freq_bins, T), device=fused.device, dtype=torch.float32)
        return self._run("decoder", fused, ones)[1]

    def separate(self, masks: torch.Tensor, mixed_spec: torch.Tensor) -> torch.Tensor:
        # model.py:210-220 through avsep_separate; stand-alone use only -- in the full model the multiply is fused
        # into the decoder epilogue.  One fp32 multiply per element: bit-identical to the reference's product.
        return self._run("separate", masks, mixed_spec)


class AVSeparationTransformer(_InferenceOnly):
    """Drop-in for the reference's end-to-end model (model.py:227-276).

    forward(mixed_spec (B,F,T), lip_frames (B,N,H,W)) -> (separated, masks), both (B,S,F,T) fp32.
    CUDA tensors run through ``avsep_forward``; CPU tensors run through ``avsep_forward_host`` (host<->device
    copies inside the call) on ``self.host_device`` and come back as CPU tensors.
    ``precision`` ('bf16' | 'tf32') selects the tensor-core operand precision; it is not a reference argument.
    """

    def __init__(self, freq_bins: int = 257, d_model: int = 256, nhead: int = 4, num_encoder_layers: int = 2,
                 num_fusion_layers: int = 2, num_speakers: int = 2, dropout: float = 0.1, *,
                 precision: str = "bf16", host_device: str = "cuda:0"):
        super().__init__()
        self.config = EngineConfig(freq_bins, d_model, nhead, num_encoder_layers, num_fusion_layers, num_speakers,
                                   precision)
        self.host_device = host_device
        self.audio_encoder = AudioEncoder(freq_bins=freq_bins, d_model=d_model, nhead=nhead,
                                          num_layers=num_encoder_layers, dropout=dropout, precision=precision)
        self.visual_encoder = VisualEncoder(d_model=d_model, nhead=nhead, num_layers=num_encoder_layers,
                                            dropout=dropout, precision=precision)
        self.fusion = CrossModalFusion(d_model=d_model, nhead=nhead, num_layers=num_fusion_layers, dropout=dropout,
                                       precision=precision)
        self.decoder = SeparationDecoder(d_model=d_model, freq_bins=freq_bins, num_speakers=num_speakers,
                                         dropout=dropout, precision=precision)
        self._post_init()

    def _engine_config(self):
        return self.config

    def forward(self, mixed_spec: torch.Tensor, lip_frames: torch.Tensor, out=None, *, lengths=None,
                frame_lengths=None):
        """``out=(separated, masks)``: optional caller-owned output buffers (not a reference argument); with fixed
        input and output buffers the call is a single CUDA-graph replay.

        ``lengths`` / ``frame_lengths`` (not reference arguments; CUDA inputs only): per-utterance audio frames and lip
        frames of a variable-length batch, see ``Engine.forward``.  Utterance b then gives what the model gives on its
        first ``lengths[b]`` / ``frame_lengths[b]`` frames alone, and its outputs past ``lengths[b]`` are 0."""
        if mixed_spec.is_cuda:
            return self._get_engine(mixed_spec.device).forward(mixed_spec, lip_frames, out, lengths=lengths,
                                                               frame_lengths=frame_lengths)
        if lengths is not None or frame_lengths is not None:
            raise ValueError("forward: lengths / frame_lengths need CUDA inputs (the host-buffer path takes full "
                             "batches only)")
        eng = self._get_engine(torch.device(self.host_device))
        return eng.forward_host(mixed_spec, lip_frames, *(out or ()))

    def separate_waveforms(self, mixed_wave: torch.Tensor, lip_frames: torch.Tensor, n_fft: int = None,
                           hop_length: int = 128, *, lengths=None, frame_lengths=None):
        """Waveform in, waveforms out (not a reference method: the reference lists phase / iSTFT reconstruction as
        missing, README.md:140).  mixed_wave (B, L) float32 CUDA -> (B, S, L): complex STFT with the framing of
        SyntheticAVDataset._stft (dataset.py:122-135), forward on its magnitude, masks applied to the complex
        mixture, weighted overlap-add inverse.  Also returns the masks.

        ``lengths`` (B,) samples and ``frame_lengths`` (B,) lip frames per utterance (not reference arguments; forms as
        for ``forward``): utterance b, left-aligned in its rows, then gives what this method gives on
        ``mixed_wave[b, :lengths[b]]`` and ``lip_frames[b, :frame_lengths[b]]`` alone, and its waveforms and masks are
        0 past its lengths.  The per-utterance frame counts go from the analysis to the forward on the device."""
        if not mixed_wave.is_cuda:
            raise ValueError("separate_waveforms: mixed_wave must be a CUDA tensor")
        n_fft = 2 * (self.config.freq_bins - 1) if n_fft is None else n_fft
        eng = self._get_engine(mixed_wave.device)
        if lengths is None and frame_lengths is None:
            spec, mag = eng.stft(mixed_wave, n_fft, hop_length)
            _, masks = eng.forward(mag, lip_frames)
            return eng.istft(spec, masks, mixed_wave.shape[1], n_fft, hop_length), masks
        if not lip_frames.is_cuda:
            raise ValueError("separate_waveforms: lengths / frame_lengths need CUDA inputs")
        if mixed_wave.dim() != 2:
            raise ValueError(f"separate_waveforms: mixed_wave must be (B, L), got {tuple(mixed_wave.shape)}")
        B, L = mixed_wave.shape
        _, _, N, _, _ = eng._check_inputs("separate_waveforms", frames=lip_frames)
        with torch.cuda.device(eng.device):
            lens = eng._lengths(lengths, "lengths", B, L, "separate_waveforms")
            flens = eng._lengths(frame_lengths, "frame_lengths", B, N, "separate_waveforms")
        if lens is None:
            spec, mag = eng.stft(mixed_wave, n_fft, hop_length)
            t_lens = None
        else:
            spec, mag, t_lens = eng.stft(mixed_wave, n_fft, hop_length, lengths=lens)
        _, masks = eng.forward(mag, lip_frames, lengths=t_lens, frame_lengths=flens)
        return eng.istft(spec, masks, L, n_fft, hop_length, lengths=lens), masks

    @property
    def engine(self) -> Engine:
        """The live engine (after the first forward / prepack), for debug snapshots and launch counts."""
        return self._engine
