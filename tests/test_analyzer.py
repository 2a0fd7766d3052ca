"""Pulse analyzer (SURVEY 8(f3)): r433b_analyze() -- histograms on the GPU (k_analyze), guess / RfRaw / text on the
host, trial demodulation on the GPU (k_slice_own) -- against pulse_analyzer() of the compiled reference
(src/pulse_analyzer.c:279-560; its answers recorded in tests/golden/reference.json by tests/refdata.py): the stderr
text, character for character (as a digest), and the bitbuffers of the trial demodulation.  The histogram functions
themselves are also run on the CPU through tests/host_core.cpp."""
import random

import numpy as np
import pytest

import helpers
import refdata
from rtl_433_b200 import lib, synth


def shaped_package(rng, kind, rate=250000):
    """pulse_data_t records that steer the analyzer into each of its branches."""
    pd = np.zeros(1, lib.PULSE_DATA_DTYPE)[0]
    pd["sample_rate"] = rate
    us = rate / 1e6

    def j(v):  # a little jitter, well inside the 20 % tolerance
        return max(1, int(v * us * (1 + rng.uniform(-0.04, 0.04))))
    pulses, gaps = [], []
    if kind == "single":
        pulses, gaps = [j(500)], [j(9000)]
    elif kind == "preamble":
        for _ in range(20):
            pulses.append(j(500)); gaps.append(j(500))
    elif kind == "ppm":
        for _ in range(4):
            for _b in range(24):
                pulses.append(j(500)); gaps.append(j(2000 if rng.random() < 0.5 else 4000))
            gaps[-1] = j(9000)
    elif kind == "pwm_fixed_gap":
        for _ in range(40):
            pulses.append(j(300 if rng.random() < 0.5 else 900)); gaps.append(j(600))
    elif kind == "pwm_fixed_period":
        for _ in range(40):
            w = 264 if rng.random() < 0.5 else 744
            pulses.append(j(w)); gaps.append(max(1, int((1000 - w) * us)))
    elif kind == "manchester":
        bits = [rng.randrange(2) for _ in range(48)]
        level = []
        for b in bits:
            level += [1, 0] if b else [0, 1]
        level = [1] + level + [0]
        runs, k = [], 0
        while k < len(level):
            m = k
            while m < len(level) and level[m] == level[k]:
                m += 1
            runs.append((level[k], m - k)); k = m
        if runs[0][0] == 0:
            runs = runs[1:]
        for q in range(0, len(runs) - 1, 2):
            pulses.append(j(500 * runs[q][1])); gaps.append(j(500 * runs[q + 1][1]))
    elif kind == "pwm_packets":
        for _ in range(5):
            for _b in range(16):
                pulses.append(j(300 if rng.random() < 0.5 else 900)); gaps.append(j(600))
            gaps[-1] = j(4000)
        gaps[10] = j(1800)
    elif kind == "pcm":
        for _ in range(60):
            pulses.append(j(100 * rng.choice([1, 1, 2, 3]))); gaps.append(j(100 * rng.choice([1, 1, 2, 3])))
    elif kind == "pwm_sync":
        for _ in range(3):
            pulses.append(j(2500)); gaps.append(j(600))
            for _b in range(20):
                pulses.append(j(300 if rng.random() < 0.5 else 900)); gaps.append(j(600))
    elif kind == "noclue":
        for _ in range(50):
            pulses.append(rng.randrange(20, 3000)); gaps.append(rng.randrange(20, 5000))
    elif kind == "many_bins":
        for i in range(300):
            pulses.append(int(10 * 1.3 ** (i % 24)) + 1); gaps.append(int(14 * 1.3 ** ((i * 7) % 24)) + 1)
    elif kind == "fsk_zero_bin":
        pulses.append(0); gaps.append(j(200))
        for _ in range(40):
            pulses.append(j(100 * rng.choice([1, 2, 3]))); gaps.append(j(100 * rng.choice([1, 2, 3])))
    n = min(len(pulses), 1200)
    pd["num_pulses"] = n
    pd["pulse"][:n] = pulses[:n]
    pd["gap"][:n] = gaps[:n]
    pd["ook_low_estimate"], pd["ook_high_estimate"] = rng.randrange(10, 300), rng.randrange(1000, 16000)
    return pd


KINDS = ["single", "preamble", "ppm", "pwm_fixed_gap", "pwm_fixed_period", "manchester", "pwm_packets", "pcm", "pwm_sync",
         "noclue", "many_bins", "fsk_zero_bin"]


def analyzed_by_reference(key, ref, pd, package_type):
    """[digest of pulse_analyzer()'s text, number and digest of the FNV-1a hashes of its trial demodulation's
    bitbuffers]"""
    def compute():
        text, hashes = ref.analyze(pd, package_type)
        return [helpers.digest(text), len(hashes), helpers.digest(hashes)]
    return refdata.recorded(key, compute)


def assert_analysis(want, text, bbs, what):
    assert helpers.digest(text) == want[0], f"{what}: the analyzer's text differs from the reference's:\n{text}"
    hashes = [fnv(bb) for bb in bbs]
    assert [len(hashes), helpers.digest(hashes)] == want[1:], f"{what}: trial demodulation differs"


def analyzer_matches_the_reference():
    ref = refdata.LiveRef(store_bitbuffers=False)
    ctx = lib.Context(0)
    ctx.set_devices(lib.default_device_table()[:8])
    try:
        rng = random.Random(17)
        # 1. hand-shaped packages through r433b_process_pulses, two sample rates, OOK and FSK typed
        ps = lib.Pulses()
        sent = []
        for rep in range(3):
            for kind in KINDS:
                rate = 250000 if rep != 1 else 1024000
                pd = shaped_package(rng, kind, rate)
                if rep == 2 and kind in ("pwm_fixed_gap", "pcm", "manchester", "pwm_sync", "fsk_zero_bin"):
                    pd["fsk_f2_est"], pd["fsk_f1_est"] = 3000, -2500
                ps.add(pd, stream=rep)
                sent.append(pd)
        ctx.process_pulses(ps)
        res = ctx.fetch()
        ctx.analyze()
        guesses = set()
        for i, pd in enumerate(sent):
            k = res["packages"][i]
            assert int(k["num_pulses"]) == int(pd["num_pulses"])
            want = analyzed_by_reference(f"analyzer/shaped/{i}", ref, ctx_pulse_data(ctx, i), int(k["type"]))
            a, g, text, bbs = ctx.analysis(i)
            assert_analysis(want, text, bbs, f"package {i}")
            guesses.add(int(g.modulation))
        assert {0, 3, 4, 5, 6, 16, 17, 18} <= guesses, guesses
        ps.close()
        # 2. packages k_detect finds in synthetic captures (levels, rssi, frequency estimates filled in)
        x = [synth.ook_stream(61, n_samples=1 << 19, n_bursts=4), synth.ook_stream(62, n_samples=1 << 19, n_bursts=4)]
        data = np.concatenate(x)
        ctx.process(data, np.array([0, x[0].nbytes, data.nbytes], np.uint64), lib.FMT_CU8, 250000, 433920000)
        res = ctx.fetch()
        ctx.analyze()
        assert res["n_packages"] >= 8
        demodulated = 0
        for i in range(res["n_packages"]):
            want = analyzed_by_reference(f"analyzer/capture/{i}", ref, ctx_pulse_data(ctx, i), int(res["packages"][i]["type"]))
            a, g, text, bbs = ctx.analysis(i)
            assert_analysis(want, text, bbs, f"capture package {i}")
            demodulated += len(bbs)
        assert demodulated >= 4
        y = synth.fsk_stream(7, n_samples=1 << 18, n_bursts=2).view(np.uint8)
        ctx.process(y, np.array([0, y.nbytes], np.uint64), lib.FMT_CS16, 1024000, 868000000)
        res = ctx.fetch()
        ctx.analyze()
        assert any(int(t) == 2 for t in res["packages"]["type"])
        for i in range(res["n_packages"]):
            want = analyzed_by_reference(f"analyzer/fsk/{i}", ref, ctx_pulse_data(ctx, i), int(res["packages"][i]["type"]))
            a, g, text, bbs = ctx.analysis(i)
            assert_analysis(want, text, bbs, f"fsk package {i}")
    finally:
        ref.close()
        ctx.close()


def ctx_pulse_data(ctx, i):
    """pulse_data_t of fetched package i as a numpy record (what the reference's analyzer is handed)."""
    pd = ctx.pulse_data(i)
    return np.frombuffer(bytes(pd), dtype=lib.PULSE_DATA_DTYPE)[0]


def fnv(bb):
    h = 1469598103934665603
    for b in np.ascontiguousarray(bb).tobytes():
        h = ((h ^ b) * 1099511628211) & 0xffffffffffffffff
    return h


@pytest.mark.gpu
def test_analyzer_matches_the_reference():
    analyzer_matches_the_reference()


def edge_cases_of_the_widening_rows():
    """Empty sets, a package without pulses, gates on loaded packages, call-order errors."""
    devices = lib.default_device_table()
    ctx = lib.Context(0)
    ref = refdata.LiveRef(lambda r: r.register_defaults(), store_bitbuffers=False)
    try:
        ctx.set_devices(devices)
        ps = lib.Pulses()
        ctx.process_pulses(ps)  # nothing loaded
        res = ctx.fetch()
        assert res["n_packages"] == 0 and res["n_events"] == 0
        ctx.analyze()
        empty = np.zeros(1, lib.PULSE_DATA_DTYPE)[0]
        empty["sample_rate"] = 250000
        ps.add(empty)  # a pulse_data_t without pulses: the analyzer says so, the slicers emit nothing
        rng = random.Random(2)
        full = shaped_package(rng, "ppm")
        ps.add(full)
        # without gates every event of the ppm package is the reference's, in order
        ctx.process_pulses(ps)
        ctx.fetch()
        pd1 = ctx_pulse_data(ctx, 1)
        want = [(e["dev"], e["hash"]) for e in helpers.gpu_stream_results(ctx, 0)["events"] if e["package"] == 1]

        def sliced_by_reference():
            ev = [[d, h] for d, h, _bb in ref.slice_pulse_data(pd1)]
            return [len(ev), helpers.digest(ev)]
        assert [len(want), helpers.digest(want)] == refdata.recorded("analyzer/edge/sliced", sliced_by_reference)
        ctx.set_gates(lib.default_gates(devices))
        ctx.process_pulses(ps)
        res = ctx.fetch()
        assert res["n_packages"] == 2
        got = helpers.gpu_stream_results(ctx, 0)
        kept = [(e["dev"], e["hash"]) for e in got["events"] if e["package"] == 1]
        assert not [e for e in got["events"] if e["package"] == 0]
        assert len(kept) + int(res["n_gated"]) == len(want) and res["n_gated"] > 0
        # the kept events are the reference's events the gates let through, in order
        it = iter(want)
        for dev, h in kept:
            for d2, h2 in it:
                if (d2, h2) == (dev, h):
                    break
            else:
                raise AssertionError("a stored event is not among the reference's events (in order)")
        ctx.analyze()
        a, g, text, bbs = ctx.analysis(0)
        assert text == "No pulses detected.\n" and g.modulation == 0 and len(bbs) == 0
        want = analyzed_by_reference("analyzer/edge/ppm", ref, pd1, 1)
        a, g, text, bbs = ctx.analysis(1)
        assert_analysis(want, text, bbs, "ppm package")
        assert g.modulation == 5
        ctx.set_gates(None)
        # call order: analyze needs a fetched batch
        x = synth.ook_stream(3, n_samples=1 << 17, n_bursts=1)
        ctx.process(x, np.array([0, x.nbytes], np.uint64), lib.FMT_CU8, 250000, 433920000)
        with pytest.raises(lib.R433Error):
            ctx.analyze()
        ctx.fetch()
        ctx.analyze()
        ps.close()
    finally:
        ref.close()
        ctx.close()


@pytest.mark.gpu
def test_edge_cases_of_the_widening_rows():
    edge_cases_of_the_widening_rows()


def analyzer_fuzz(n_packages=160, seed=31):
    """Random pulse trains of every shape the generator knows, plus unstructured ones with few distinct widths (the RfRaw
    B0 / B1 renderings, repeated groups, more than 32 groups, widths beyond 65535 us): text and trial demodulation
    against the reference."""
    rng = random.Random(seed)
    ref = refdata.LiveRef(store_bitbuffers=False)
    ctx = lib.Context(0)
    ctx.set_devices([])
    try:
        ps = lib.Pulses()
        for i in range(n_packages):
            r = rng.random()
            rate = rng.choice([250000, 250000, 1000000, 1024000, 48000])
            if r < 0.5:
                pd = shaped_package(rng, rng.choice(KINDS), rate)
            else:
                pd = np.zeros(1, lib.PULSE_DATA_DTYPE)[0]
                pd["sample_rate"] = rate
                n = rng.choice([2, 3, 7, 40, 200, 600, 1200])
                widths = [rng.choice([3, 10, 37, 120, 500, 2000, 70000]) for _ in range(rng.randrange(1, 5))]
                gapw = [rng.choice([5, 25, 100, 480, 3000, 20000, 90000]) for _ in range(rng.randrange(1, 6))]
                for k in range(n):
                    pd["pulse"][k] = max(0, int(rng.choice(widths) * (1 + rng.uniform(-0.03, 0.03))))
                    pd["gap"][k] = max(0, int(rng.choice(gapw) * (1 + rng.uniform(-0.03, 0.03))))
                    if rng.random() < 0.02:
                        pd["gap"][k] = rng.choice(gapw) * 9
                pd["num_pulses"] = n
            if rng.random() < 0.3:
                pd["fsk_f2_est"], pd["fsk_f1_est"] = rng.randrange(1, 9000), rng.randrange(-9000, 9000)
            ps.add(pd, stream=i % 3)
        ctx.process_pulses(ps)
        res = ctx.fetch()
        ctx.analyze()
        seen = set()
        for i in range(res["n_packages"]):
            a, g, text, bbs = ctx.analysis(i)
            if "this can't happen" in text:  # the reference exit(1)s there: the harness would not survive that package
                continue
            want = analyzed_by_reference(f"analyzer/fuzz/{seed}/{n_packages}/{i}", ref, ctx_pulse_data(ctx, i),
                                         int(res["packages"][i]["type"]))
            assert_analysis(want, text, bbs, f"package {i}")
            seen.add(int(g.modulation))
            if "+" in text.split("pdv/#")[-1].split("\n")[0]:
                seen.add("b0-groups")
        assert "b0-groups" in seen and len(seen) >= 6
        ps.close()
    finally:
        ref.close()
        ctx.close()


@pytest.mark.gpu
def test_analyzer_fuzz():
    analyzer_fuzz()


def analyzer_golden():
    """tests/golden/analyzer.json (recorded from the reference by tools/make_golden_pulse_io.py): text and trial
    demodulation without the compiled reference at hand."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "analyzer.json")) as f:
        cases = json.load(f)["cases"]
    ctx = lib.Context(0)
    ctx.set_devices([])
    try:
        ps = lib.Pulses()
        for c in cases:
            pd = np.zeros(1, lib.PULSE_DATA_DTYPE)[0]
            pd["sample_rate"] = c["rate"]
            pd["num_pulses"] = len(c["pulse"])
            pd["pulse"][:len(c["pulse"])] = c["pulse"]
            pd["gap"][:len(c["gap"])] = c["gap"]
            pd["fsk_f1_est"], pd["fsk_f2_est"] = c["fsk_f1_est"], c["fsk_f2_est"]
            ps.add(pd)
        ctx.process_pulses(ps)
        res = ctx.fetch()
        ctx.analyze()
        assert res["n_packages"] == len(cases)
        for i, c in enumerate(cases):
            assert int(res["packages"][i]["type"]) == c["type"]
            a, g, text, bbs = ctx.analysis(i)
            assert text == c["text"], f"{c['kind']} @ {c['rate']}"
            assert [str(fnv(bb)) for bb in bbs] == c["hashes"], c["kind"]
        ps.close()
    finally:
        ctx.close()


@pytest.mark.gpu
def test_analyzer_golden():
    analyzer_golden()
