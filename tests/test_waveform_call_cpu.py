"""CPU: the one-call waveform entry points are declared in include/avsep.h and bound in _lib.py with the same arity,
and the model refuses a variable-length batch in host memory before it needs a device."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALLS = {"avsep_waveform_workspace_bytes": 8, "avsep_separate_waveforms": 17, "avsep_separate_waveforms_host": 13,
         "avsep_separate_waveforms_host_async": 14}


def _prototype_args(name):
    text = open(os.path.join(ROOT, "include", "avsep.h")).read()
    m = re.search(r"AVSEP_API[^;(]*?\b" + name + r"\s*\(([^;]*?)\)\s*;", text, re.S)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


@pytest.mark.parametrize("name", sorted(CALLS))
def test_header_and_binding_agree(name):
    from avsep_b200 import _lib
    args = _prototype_args(name)
    assert len(args) == CALLS[name] and args[0] == "avsep_handle* h"
    assert len(_lib.SIGNATURES[name][1]) == CALLS[name]
    if name != "avsep_waveform_workspace_bytes":
        assert args[-1] == "void* cuda_stream"


def test_host_arguments_are_full_batches_only():
    args = _prototype_args("avsep_separate_waveforms_host")
    assert not any("length" in a and "hop" not in a for a in args)
    assert any("slot" in a for a in _prototype_args("avsep_separate_waveforms_host_async"))


def test_cpu_waveforms_with_lengths_raise_before_any_device_work():
    from avsep_b200 import AVSeparationTransformer
    m = AVSeparationTransformer(freq_bins=65, d_model=64, nhead=4, num_encoder_layers=1, num_fusion_layers=1)
    with pytest.raises(ValueError, match="separate_waveforms"):
        m.separate_waveforms(torch.zeros(2, 1000), torch.zeros(2, 4, 16, 16), 128, 32, lengths=[1000, 500])
    with pytest.raises(ValueError, match="separate_waveforms"):
        m.separate_waveforms(torch.zeros(2, 1000), torch.zeros(2, 4, 16, 16), 128, 32, frame_lengths=[4, 2])
