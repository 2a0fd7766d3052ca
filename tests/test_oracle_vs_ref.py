"""CPU: the oracle restatement and the product's device functions against the unmodified reference (outputs of
oracle/_ref recorded in tests/golden/reference.json, tests/refdata.py) on seeded synthetic captures and on randomised
slicer inputs."""
import functools

import numpy as np
import pytest

import helpers
import refdata
from oracle import orc, refh
from rtl_433_b200 import lib, synth


@pytest.fixture(scope="module")
def devs():
    return lib.default_device_table()


@functools.lru_cache(None)
def slicer_ref():
    """The reference with its default devices, storing bitbuffers (recording runs only)."""
    r = refh.Ref(store_bitbuffers=True)
    r.register_defaults()
    r.L.refh_set_capture(r.h, 0, 1, 0)
    return r


def test_device_table_matches_reference():
    """protocol_num, modulation, widths, limits, tolerance and priority of every default device, in order."""
    table = lib.default_device_table()
    n, want = refdata.registered_devices("defaults")
    assert len(table) == n == 335
    assert helpers.digest(refdata.device_rows(table)) == want


@pytest.mark.parametrize("seed", [0, 1])
def test_ook_stream_all_devices(devs, seed):
    x = synth.ook_stream(seed, n_samples=1 << 19, n_bursts=4)
    want = refdata.ref_run(f"oracle_vs_ref/ook/{seed}", x, 2)
    assert len(want["packages"]) >= 4 and want["events"] > 1000
    o = orc.Oracle(store_bitbuffers=False, store_stages=True)
    o.add_devices(devs)
    assert not helpers.compare_fingerprint(want, o.run(x, 2), "oracle")
    hc = helpers.HostCore(store_bitbuffers=False, store_stages=True)
    hc.add_devices(devs)
    assert not helpers.compare_fingerprint(want, hc.run(x, 2), "device functions", floats=False)


@pytest.mark.parametrize("fpdm,freq", [(2, 868000000), (0, 433920000)])
def test_fsk_stream_all_devices(devs, fpdm, freq):
    x = synth.fsk_stream(1, n_samples=1 << 18, n_bursts=2)
    want = refdata.ref_run(f"oracle_vs_ref/fsk/{fpdm}/{freq}", x, 4, 1024000, freq, fpdm)
    assert any(p["type"] == 2 for p in want["packages"])
    o = orc.Oracle(store_bitbuffers=False, store_stages=True)
    o.add_devices(devs)
    assert not helpers.compare_fingerprint(want, o.run(x, 4, 1024000, freq, fpdm), "oracle")
    hc = helpers.HostCore(store_bitbuffers=False, store_stages=True)
    hc.add_devices(devs)
    assert not helpers.compare_fingerprint(want, hc.run(x, 4, 1024000, freq, fpdm), "device functions", floats=False)


def test_small_blocks_and_silence(devs):
    """32 KiB blocks (block-call semantics: eop flag, start_ago/end_ago, x[-1] int16 wrap) and a
    file that is constant 128/128 except for its bursts."""
    for xi, x in enumerate((synth.ook_stream(9, n_samples=1 << 18, n_bursts=3), synth.nice_flor_s_file()[: 46752 // 16 * 16])):
        for bb in (32768, 0):
            want = refdata.ref_run(f"oracle_vs_ref/small_blocks/{xi}/{bb}", x, 2, block_bytes=bb)
            o = orc.Oracle(store_bitbuffers=False, store_stages=True)
            o.add_devices(devs)
            assert not helpers.compare_fingerprint(want, o.run(x, 2, block_bytes=bb), "oracle")
            hc = helpers.HostCore(store_bitbuffers=False, store_stages=True)
            hc.add_devices(devs)
            assert not helpers.compare_fingerprint(want, hc.run(x, 2, block_bytes=bb), "device functions", floats=False)


def test_saturated_input_wraps_like_reference(devs):
    """I = Q = 255 gives an envelope of 32768, which the reference stores as int16 between
    blocks (src/baseband.c:167); a block boundary inside a saturated stretch exercises it."""
    x = synth.ook_stream(4, n_samples=1 << 16, n_bursts=0)
    x[2 * 16300:2 * 16500] = 255
    want = refdata.ref_run("oracle_vs_ref/saturated", x, 2, block_bytes=32768)
    hc = helpers.HostCore(store_bitbuffers=False, store_stages=True)
    hc.add_devices(devs)
    assert not helpers.compare_fingerprint(want, hc.run(x, 2, block_bytes=32768), "device functions", floats=False)
    o = orc.Oracle(store_bitbuffers=False, store_stages=True)
    o.add_devices(devs)
    assert not helpers.compare_fingerprint(want, o.run(x, 2, block_bytes=32768), "oracle")


def random_train(rng, kind):
    """Pulse trains that stress the slicers: nominal symbol mixes, long runs (row spill past
    1024 bits), many short rows (50-row overflow), zero widths, huge pulses."""
    n = int(rng.integers(1, 400))
    unit = int(rng.choice([12, 25, 50, 62, 100, 125, 250]))
    if kind == 0:
        pulse = rng.choice([unit, 2 * unit, 3 * unit], n) + rng.integers(-3, 4, n)
        gap = rng.choice([unit, 2 * unit, 4 * unit, 8 * unit], n) + rng.integers(-3, 4, n)
    elif kind == 1:  # long NRZ-like runs -> thousands of bits per row
        pulse = rng.integers(1, 40, n) * unit
        gap = rng.integers(1, 40, n) * unit
    elif kind == 2:  # many row breaks
        pulse = rng.choice([unit, 2 * unit], n)
        gap = rng.choice([unit, 20 * unit, 45 * unit], n, p=[0.5, 0.3, 0.2])
    else:
        pulse = rng.integers(0, 3000, n)
        gap = rng.integers(0, 30000, n)
        pulse[rng.integers(0, n)] = 400000
    gap[-1] = int(rng.integers(2500, 30000))
    return np.maximum(pulse, 0).astype(np.int32), np.maximum(gap, 0).astype(np.int32)


def test_slicers_on_random_pulse_trains(devs):
    """Every default device's slicer (all ten modulations + the FSK three) on random trains:
    device index order, event count and every bitbuffer byte must match the reference."""
    hc = helpers.HostCore(store_bitbuffers=True)
    hc.add_devices(devs)
    rng = np.random.default_rng(1234)
    total = 0
    for it in range(60):
        pulse, gap = random_train(rng, it % 4)
        for fsk, rate in ((0, 250000), (1, 1024000), (0, 1000000)):
            want = refdata.recorded(f"slicers/random/{it}/{fsk}/{rate}",
                                    lambda: helpers.events_digest(slicer_ref().slice_all(fsk, rate, pulse, gap)))
            got = hc.slice(2 if fsk else 1, rate, pulse, gap)
            assert helpers.events_digest(got) == want, (it, fsk, rate, want[0], len(got))
            total += want[0]
    assert total > 50000


def test_per_stage_functions():
    rng = np.random.default_rng(7)
    O = orc.lib()
    iq8 = rng.integers(0, 256, 2 * 5000, dtype=np.uint8)
    iq16 = rng.integers(-32767, 32768, 2 * 5000).astype(np.int16)
    for rf, of, src in (("refh_envelope_detect", "orc_envelope_cu8", iq8), ("refh_magnitude_est_cu8", "orc_magnitude_cu8", iq8),
                        ("refh_magnitude_est_cs16", "orc_magnitude_cs16", iq16)):
        def ref_stage():
            a = np.zeros(5000, np.uint16)
            getattr(refh.lib(), rf)(src.ctypes.data, a.ctypes.data, 5000)
            return helpers.digest(a)
        b = np.zeros(5000, np.uint16)
        getattr(O, of)(src.ctypes.data, b.ctypes.data, 5000)
        assert helpers.digest(b) == refdata.recorded(f"stage/{rf}", ref_stage)
    for cs16, src, lp in ((0, iq8, 0.1), (0, iq8, 0.2), (1, iq16, 0.2), (1, iq16, 0.1), (0, iq8, 25000.0), (1, iq16, 12.0)):
        def ref_fm():
            a = np.zeros(5000, np.int16)
            ca = np.zeros(2, np.int32)
            refh.lib().refh_demod_fm(cs16, src.ctypes.data, a.ctypes.data, 5000, 1024000 if cs16 else 250000, lp, ca.ctypes.data)
            return [helpers.digest(ca), helpers.digest(a)]
        b = np.zeros(5000, np.int16)
        cb = np.zeros(2, np.int32)
        O.orc_demod_fm(cs16, src.ctypes.data, b.ctypes.data, 5000, 1024000 if cs16 else 250000, lp, cb.ctypes.data)
        assert [helpers.digest(cb), helpers.digest(b)] == refdata.recorded(f"stage/refh_demod_fm/{cs16}/{lp}", ref_fm)
