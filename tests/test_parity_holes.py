"""CPU: the branches and slicers round 1 left untested, pinned against the compiled, unmodified reference.

* `pulse_slicer_piwm_raw` (src/pulse_slicer.c:597-657) and `pulse_slicer_nrzs` (:715-759): no default-enabled
  device uses them, so they are registered as CUSTOM devices (oracle/ref_harness.c: refh_register_custom) next to
  custom devices of every other modulation;
* the six-field "sample rate too low" check (src/pulse_slicer.c:79-84) at rates where single widths round to zero
  -- the defect ADVICE.md reported for protocols 198 / 270 at 250 kS/s (all 384 protocols incl. disabled ones);
* `pulse_data_shift` on the FSK train, more than 1200 FSK transitions inside one carrier, both FSK detectors
  (src/pulse_detect_fsk.c:110-114, :201-205, src/pulse_data.c:27-34);
* the 1200-pulse OOK end of package (src/pulse_detect.c:429-441);
* 2.048 MS/s cu8, OOK in a cs16 capture, FSK packages out of a cu8 capture.

For each: oracle/r433_oracle.c (the restatement the GPU tests compare with) and the product's own
__host__ __device__ functions (tests/host_core.cpp) must equal the reference bit for bit (its outputs recorded in
tests/golden/reference.json, tests/refdata.py).
"""
import numpy as np
import pytest

import helpers
import refdata
from oracle import orc
from rtl_433_b200 import lib, synth

# include/r_device.h:24-40
MOD = dict(OOK_MC=3, OOK_PCM=4, OOK_PPM=5, OOK_PWM=6, OOK_PIWM_RAW=8, OOK_DMC=9, OOK_OSV1=10, OOK_PIWM_DC=11,
           OOK_NRZS=12, OOK_RZI=13, FSK_PCM=16, FSK_PWM=17, FSK_MC=18)


def custom_devices():
    """Hand-made slicer parameter sets: every modulation, PIWM_RAW and NRZS several times."""
    def dev(mod, short, long_, reset, gap=0.0, sync=0.0, tol=0.0, prio=0):
        return dict(modulation=MOD[mod], short_width=float(short), long_width=float(long_), reset_limit=float(reset),
                    gap_limit=float(gap), sync_width=float(sync), tolerance=float(tol), priority=prio)
    return [
        dev("OOK_PIWM_RAW", 100, 450, 2000, tol=40), dev("OOK_PIWM_RAW", 250, 1200, 5000, tol=100),
        dev("OOK_PIWM_RAW", 48, 500, 1000, tol=20), dev("OOK_PIWM_RAW", 500, 4000, 12000, tol=240),
        dev("OOK_PIWM_RAW", 62, 130, 800, tol=30), dev("OOK_PIWM_RAW", 1, 40, 100, tol=1),
        dev("OOK_NRZS", 100, 100, 2000), dev("OOK_NRZS", 250, 250, 6000, tol=50), dev("OOK_NRZS", 50, 0, 1000),
        dev("OOK_NRZS", 1000, 1000, 20000), dev("OOK_NRZS", 2, 2, 60),
        dev("OOK_PWM", 100, 200, 1500, gap=600, tol=40), dev("OOK_PWM", 250, 500, 4000, sync=750),
        dev("OOK_PPM", 1000, 2000, 6000, gap=3000, tol=300), dev("OOK_PCM", 100, 100, 3000),
        dev("OOK_PCM", 50, 100, 2000, tol=20), dev("OOK_MC", 250, 0, 2000, tol=60), dev("OOK_DMC", 100, 200, 1500, tol=40),
        dev("OOK_PIWM_DC", 125, 250, 2000, tol=50), dev("OOK_OSV1", 1000, 0, 6000), dev("OOK_RZI", 100, 200, 2000),
        dev("FSK_PCM", 100, 100, 3000), dev("FSK_PWM", 100, 200, 1500, gap=600), dev("FSK_MC", 100, 0, 1500, tol=30),
        # widths that round to zero at low rates, one field at a time (the `ok` bits of SlicerParams)
        dev("OOK_PWM", 200, 400, 3000, gap=1000, tol=1), dev("OOK_PPM", 200, 400, 3000, sync=2),
        dev("OOK_RZI", 200, 400, 3000, gap=1, tol=1), dev("OOK_PIWM_RAW", 200, 900, 3000, gap=3),
        dev("OOK_NRZS", 200, 200, 3000, tol=2), dev("OOK_MC", 200, 0, 3000, gap=2), dev("OOK_DMC", 200, 400, 3000, sync=1, tol=60),
    ]


def symbol_train(rng, unit, n):
    """Widths on a grid of `unit` samples: what PIWM_RAW / NRZS / PCM-like slicers turn into long bit runs."""
    pulse = rng.integers(1, 9, n) * unit + rng.integers(-2, 3, n)
    gap = rng.integers(1, 9, n) * unit + rng.integers(-2, 3, n)
    for k in rng.integers(0, n, max(1, n // 12)):
        gap[k] = int(rng.choice([12, 25, 60])) * unit
    gap[-1] = 100 * unit
    return np.maximum(pulse, 0).astype(np.int32), np.maximum(gap, 0).astype(np.int32)


def assert_same_events(want, got, what):
    """`want`: helpers.events_digest() of the reference's events."""
    assert helpers.events_digest(got) == want, (what, want[0], len(got))


def slicing_ref(register):
    """The reference storing bitbuffers, devices registered by register(ref) (recording runs only)."""
    def setup(r):
        register(r)
        r.L.refh_set_capture(r.h, 0, 1, 0)
    return refdata.LiveRef(setup, store_bitbuffers=True)


def test_custom_slicers_piwm_raw_nrzs_and_rate_checks():
    from test_oracle_vs_ref import random_train
    devs = custom_devices()
    ref = slicing_ref(lambda r: [r.register_custom(**d) for d in devs])
    hc = helpers.HostCore(store_bitbuffers=True)
    hc.add_devices(devs)
    o = orc.Oracle(store_bitbuffers=True)
    o.add_devices(devs)
    rng = np.random.default_rng(4321)
    total = by_raw = by_nrzs = 0
    for it in range(48):
        if it % 2:
            pulse, gap = random_train(rng, it % 4)
        else:
            pulse, gap = symbol_train(rng, int(rng.choice([5, 12, 25, 62, 100, 256])), int(rng.integers(1, 300)))
        # 1 MS/s, the benchmark rates, and rates where short widths / limits / tolerances truncate to zero samples
        for fsk, rate in ((0, 250000), (1, 1024000), (0, 1000000), (0, 2048000), (0, 300000), (0, 20000), (1, 4000), (0, 700)):
            want = refdata.recorded(f"parity_holes/custom/{it}/{fsk}/{rate}",
                                    lambda: helpers.events_digest(ref.slice_all(fsk, rate, pulse, gap)))
            got = hc.slice(2 if fsk else 1, rate, pulse, gap)
            assert_same_events(want, got, ("device functions", it, fsk, rate))
            got_o = []
            for di in range(len(devs)):
                if (devs[di]["modulation"] >= 16) == bool(fsk):
                    got_o += [(di, bb) for bb in o.slice(di, rate, pulse, gap)]
            assert_same_events(want, got_o, ("oracle", it, fsk, rate))
            total += len(got)
            by_raw += sum(1 for d, _ in got if devs[d]["modulation"] == MOD["OOK_PIWM_RAW"])
            by_nrzs += sum(1 for d, _ in got if devs[d]["modulation"] == MOD["OOK_NRZS"])
    ref.close()
    assert total > 20000 and by_raw > 1000 and by_nrzs > 1000, (total, by_raw, by_nrzs)


def test_all_384_protocols_at_rates_where_widths_vanish():
    """Every protocol of the table, disabled ones included (klimalogg = NRZS; 198 / 270 have a 1 us tolerance
    that truncates to 0 samples at 250 kS/s: the reference then returns no events, src/pulse_slicer.c:79-84)."""
    from test_oracle_vs_ref import random_train
    ref = slicing_ref(lambda r: [r.register(p["protocol_num"]) for p in r.protocols()])
    devs = lib.default_device_table(include_disabled=True)  # the reference's protocols in order, checked here
    n, want = refdata.registered_devices("all")
    assert len(devs) == n >= 380
    assert helpers.digest(refdata.device_rows(devs)) == want
    assert any(d["modulation"] == MOD["OOK_NRZS"] for d in devs)
    hc = helpers.HostCore(store_bitbuffers=True)
    hc.add_devices(devs)
    rng = np.random.default_rng(99)
    total = 0
    for it in range(12):
        pulse, gap = random_train(rng, it % 4) if it % 3 else symbol_train(rng, 25, 120)
        for fsk, rate in ((0, 250000), (1, 250000), (0, 48000), (1, 1024000)):
            want = refdata.recorded(f"parity_holes/all_protocols/{it}/{fsk}/{rate}",
                                    lambda: helpers.events_digest(ref.slice_all(fsk, rate, pulse, gap)))
            assert_same_events(want, hc.slice(2 if fsk else 1, rate, pulse, gap), (it, fsk, rate))
            total += want[0]
    ref.close()
    assert total > 10000


def three_way(key, x, ss, rate, freq, fpdm=2, devices=None, block_bytes=0):
    """reference vs oracle vs the product's device functions on one stream; returns the oracle's result (equal to the
    reference's)."""
    want = refdata.ref_run(f"parity_holes/{key}", x, ss, rate, freq, fpdm, block_bytes, devices=devices)
    if devices is None:
        devices = lib.default_device_table()
    o = orc.Oracle(store_bitbuffers=False, store_stages=True)
    o.add_devices(devices)
    got = o.run(x, ss, rate, freq, fpdm, block_bytes)
    d = helpers.compare_fingerprint(want, got, "oracle")
    assert not d, "\n".join(d[:10])
    hc = helpers.HostCore(store_bitbuffers=False, store_stages=True)
    hc.add_devices(devices)
    d = helpers.compare_fingerprint(want, hc.run(x, ss, rate, freq, fpdm, block_bytes), "device functions", floats=False)
    assert not d, "\n".join(d[:10])
    return got


def test_ook_1200_pulse_end_of_package():
    """More than PD_MAX_PULSES pulses in one train: the detector returns a full package at pulse 1200 and the
    rest becomes a second one (src/pulse_detect.c:429-441)."""
    for seed, n, on, off in ((1, 1300, 200.0, 200.0), (2, 2500, 120.0, 80.0), (5, 1201, 400.0, 60.0)):
        x = synth.ook_train_stream(seed, n, on, off, n_samples=1 << 19)
        want = three_way(f"ook_1200/{seed}", x, 2, 250000, 433920000)
        sizes = [p["num_pulses"] for p in want["packages"] if p["type"] == 1]
        assert sizes[0] == 1200 and sum(sizes) >= n - 2, sizes
    # gaps the low-pass smears shut: the whole train is one OOK pulse whose ripple feeds the FSK sub-detector
    want = three_way("ook_1200/smeared", synth.ook_train_stream(3, 1201, 400.0, 44.0, n_samples=1 << 19), 2, 250000, 433920000)
    assert [p["type"] for p in want["packages"]] == [2]


@pytest.mark.parametrize("fpdm,freq", [(2, 868000000), (0, 433920000)])
def test_fsk_train_overflow_shifts_the_pulse_train(fpdm, freq):
    """More than 1200 FSK pulses inside one OOK pulse: pulse_data_shift drops the oldest 600 and adds the COUNT to
    `offset` (src/pulse_data.c:27-34; called at src/pulse_detect_fsk.c:114 and :205)."""
    x = synth.fsk_burst_stream(2, 2700)
    want = three_way(f"fsk_overflow/{fpdm}/{freq}/one", x, 4, 1024000, freq, fpdm)
    fsk = [p for p in want["packages"] if p["type"] == 2]
    assert fsk and 600 <= fsk[0]["num_pulses"] < 1200
    x = synth.fsk_burst_stream(5, 3900, bit_us=60.0)  # two shifts
    want = three_way(f"fsk_overflow/{fpdm}/{freq}/two", x, 4, 1024000, freq, fpdm)
    assert any(p["type"] == 2 for p in want["packages"])


def test_rates_and_formats_round_1_never_compared():
    # 2.048 MS/s cu8 OOK
    x = synth.ook_stream(61, n_samples=1 << 20, rate=2048000, n_bursts=4, kinds=("nice", "manchester"))
    want = three_way("rates/cu8_2048k", x, 2, 2048000, 433920000)
    assert len(want["packages"]) >= 2
    # OOK bursts inside a cs16 capture (magnitude_est_cs16 + the OOK state machine), 1.024 MS/s and 250 kS/s
    x = synth.cu8_to_cs16(synth.ook_stream(62, n_samples=1 << 19, rate=1024000, n_bursts=3, kinds=("nice", "manchester")))
    want = three_way("rates/cs16_ook_1024k", x, 4, 1024000, 433920000)
    assert sum(p["type"] == 1 for p in want["packages"]) >= 3
    x = synth.cu8_to_cs16(synth.ook_stream(63, n_samples=1 << 18, n_bursts=3, kinds=("nice", "manchester", "silvercrest")), gain=200)
    want = three_way("rates/cs16_ook_250k", x, 4, 250000, 433920000)
    assert sum(p["type"] == 1 for p in want["packages"]) >= 3
    # FSK packages out of a cu8 capture (baseband_demod_FM + both FSK detectors), 250 kS/s
    for freq in (433920000, 868000000):
        x = synth.fsk_burst_stream(64, 600, bit_us=400.0, n_samples=1 << 18, rate=250000, cu8=True, dev_hz=30e3)
        want = three_way(f"rates/cu8_fsk/{freq}", x, 2, 250000, freq)
        assert any(p["type"] == 2 for p in want["packages"])


def test_custom_devices_on_streams():
    """The custom PIWM_RAW / NRZS devices through the whole flow (detector + slicers), OOK and FSK captures."""
    devs = custom_devices()
    want = three_way("custom/ook", synth.ook_stream(71, n_samples=1 << 19, n_bursts=5), 2, 250000, 433920000, devices=devs)
    raw = [e for e in want["events"] if devs[e["dev"]]["modulation"] == MOD["OOK_PIWM_RAW"]]
    nrzs = [e for e in want["events"] if devs[e["dev"]]["modulation"] == MOD["OOK_NRZS"]]
    assert len(raw) > 20 and len(nrzs) > 20
    three_way("custom/fsk", synth.fsk_stream(72, n_samples=1 << 18, n_bursts=2), 4, 1024000, 868000000, devices=devs)
