"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol include/r433b.h
declares (no compute without a GPU); struct layouts in include/r433b_abi.h match the reference."""
import ctypes as C
import os
import re

import pytest

import refdata
from oracle import refh
from rtl_433_b200 import lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_and_exports_header_symbols():
    path = lib.build()
    L = C.CDLL(path)
    header = open(os.path.join(ROOT, "include", "r433b.h")).read()
    declared = set(re.findall(r"\b(r433b_[a-z_0-9]+)\s*\(", header)) - {"r433b_event_fn"}
    assert declared == set(lib.EXPORTS)
    for name in declared:
        assert getattr(L, name) is not None


def test_create_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(lib.R433Error):
        lib.Context(0)


def test_no_oracle_in_product():
    """The product must not import, link or call anything under oracle/."""
    pkg = os.path.join(ROOT, "rtl_433_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".hpp", ".h", ".c", ".cpp")):
                src = open(os.path.join(dp, f), errors="replace").read()
                assert "oracle" not in src.replace("the oracle", "").lower() or f == "synth.py", os.path.join(dp, f)
    out = os.popen(f"ldd {lib.LIB_PATH}").read()
    assert "r433ref" not in out and "r433oracle" not in out


def test_struct_layouts_match_reference():
    facts = refdata.recorded("abi_facts", refh.abi_facts)
    assert facts["sizeof_r_device"] == 152
    assert facts["sizeof_bitbuffer"] == 6604 == lib.BITBUFFER_DTYPE.itemsize
    assert facts["sizeof_pulse_data"] == 9672 == C.sizeof(lib.PulseData)
    assert facts["off_bits_per_row"] == lib.BITBUFFER_DTYPE.fields["bits_per_row"][1]
    assert facts["off_syncs_before_row"] == lib.BITBUFFER_DTYPE.fields["syncs_before_row"][1]
    assert facts["off_bb"] == lib.BITBUFFER_DTYPE.fields["bb"][1] == 204
    assert facts["off_pulse"] == lib.PulseData.pulse.offset
    assert facts["off_gap"] == lib.PulseData.gap.offset
    assert facts["off_ook_low_estimate"] == lib.PulseData.ook_low_estimate.offset
    assert facts["off_freq1_hz"] == lib.PulseData.freq1_hz.offset
    # r_device field offsets as laid out by include/r433b_abi.h on LP64
    assert (facts["off_modulation"], facts["off_short_width"], facts["off_decode_fn"], facts["off_priority"],
            facts["off_decode_events"], facts["off_decode_ctx"]) == (16, 20, 48, 64, 104, 136)
