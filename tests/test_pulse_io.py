"""Pulse-level I/O (SURVEY 8(f4)): `.ook` / RfRaw readers and `.ook` / VCD / logic.u8 writers of the product
(host functions of libr433b.so, rtl_433_b200/csrc/r433b_pulses.hpp) against the reference (what pulse_data_load,
rfraw_parse, pulse_data_dump, pulse_data_print_vcd and pulse_data_dump_raw of oracle/_ref return, recorded in
tests/golden/reference.json by tests/refdata.py) and against the committed golden fixture (tests/golden/pulse_io.json,
generated from the reference by tools/make_golden.py).  The -m gpu part sends loaded packages through k_slice and
compares every bitbuffer with run_ook_demods() / run_fsk_demods() of the reference on the same pulse_data_t."""
import json
import os
import random

import numpy as np
import pytest

import helpers
import refdata
from oracle import refh
from rtl_433_b200 import lib, synth

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "pulse_io.json")

INT_FIELDS = ["sample_rate", "num_pulses", "fsk_f1_est", "fsk_f2_est", "offset", "depth_bits", "start_ago", "end_ago",
              "ook_low_estimate", "ook_high_estimate"]
FLOAT_FIELDS = ["freq1_hz", "freq2_hz", "centerfreq_hz", "range_db", "rssi_db", "snr_db", "noise_db"]


def rfraw_b1(bins, codes):
    return "AAB1%02X" % len(bins) + "".join("%04X" % b for b in bins) + "".join("%02X" % c for c in codes) + "55"


def rfraw_b0(bins, codes, repeats):
    body = "%02X%02X" % (len(bins), repeats) + "".join("%04X" % b for b in bins) + "".join("%02X" % c for c in codes) + "55"
    return "AAB0%02X" % (len(body) // 2) + body


def ook_cases():
    """Texts that exercise every branch of pulse_data_load() and rfraw_parse()."""
    rng = random.Random(7)
    cases = {}
    cases["plain"] = ";pulse data\n;version 1\n;timescale 1us\n;received @0.1s\n;ook 4 pulses\n;freq1 433920123\n" \
                     "264 744\n744 264\n264 744\n264 6000\n;end\n"
    cases["two_packages"] = cases["plain"] + ";received @1s\n;fsk 3 pulses\n;freq1 -12000\n;freq2 25000\n100 100\n200 100\n100 9000\n;end\n"
    cases["no_end_no_newline"] = "500 1000\n1000 500\n500 20000"
    cases["crlf_and_blanks"] = ";x\r\n 500   1000 \r\n1000\t500\r\n500 20000\r\n;end\r\n"
    cases["negative_and_junk"] = "500 1000\n-5 10\n10 -5\nabc def\n\n700 800\n;end\n"
    cases["header_only"] = ";pulse data\n;version 1\n"
    cases["empty"] = ""
    cases["too_many"] = "".join("%d %d\n" % (100 + i % 7, 200 + i % 11) for i in range(1300)) + ";end\n"
    cases["rfraw_b1_line"] = rfraw_b1([300, 900, 9000], [0x81, 0x90, 0x81, 0x82]) + "\n"
    cases["rfraw_b0_repeats"] = rfraw_b0([250, 750, 8000], [0x81, 0x90, 0x90, 0x82], 3) + "\n"
    cases["rfraw_oldfmt"] = "AAB103012C03842328" + "0101100102" + "55\n"  # nibbles < 8 only: alternating pulse / gap
    cases["rfraw_plus_groups"] = rfraw_b1([300, 900], [0x81, 0x90]) + "+" + rfraw_b1([100, 5000], [0x80, 0x81]) + "\n"
    cases["rfraw_after_rows"] = "500 1000\n600 900\n" + rfraw_b1([300, 900, 9000], [0x81, 0x90, 0x82]) + "\n700 800\n;end\n"
    cases["rfraw_pulse_without_gap"] = "AAB1020100020088" + "55\n"  # ends on a pulse nibble: pulse[n] set, not counted
    cases["rfraw_two_pulses"] = "AAB102010002008889" + "9055\n"
    cases["rfraw_long_line"] = rfraw_b1([300, 900, 9000], [0x81 if rng.random() < 0.5 else 0x90 for _ in range(700)] + [0x82]) + "\n"
    cases["rfraw_full"] = rfraw_b1([300, 900, 9000], [0x81] * 1300) + "\n"
    cases["rfraw_bad_bins"] = "AAB109" + "0100" * 9 + "8155\n"
    cases["rfraw_truncated"] = "AAB1020100020081 9\n500 600\n"
    cases["rfraw_separators"] = "aa b1 02 01-00 02:00 81 90 55\n"
    lines = []
    for _ in range(60):
        r = rng.random()
        if r < 0.6:
            lines.append("%d %d" % (rng.randrange(0, 3000), rng.randrange(0, 30000)))
        elif r < 0.7:
            lines.append(";end" if rng.random() < 0.5 else ";freq1 %d" % rng.randrange(-50000, 50000))
        elif r < 0.8:
            lines.append(rfraw_b1([rng.randrange(50, 2000) for _ in range(3)], [0x80 | (rng.randrange(3) << 4) | rng.randrange(3) for _ in range(rng.randrange(1, 20))]))
        elif r < 0.9:
            lines.append("%d,%d" % (rng.randrange(0, 3000), rng.randrange(0, 3000)))
        else:
            lines.append("".join(rng.choice(" ;-+0123456789abAB\t") for _ in range(rng.randrange(0, 30))))
    cases["fuzz"] = "\n".join(lines) + "\n"
    return cases


RATES = [250000, 1000000, 1024000]


def pd_facts(pd):
    n = int(pd["num_pulses"])
    m = min(n + 1, 1200)
    d = {k: int(pd[k]) for k in ("sample_rate", "num_pulses", "fsk_f2_est")}
    d.update({k: float(pd[k]) for k in ("freq1_hz", "freq2_hz")})
    d["pulse"] = [int(v) for v in pd["pulse"][:m]]
    d["gap"] = [int(v) for v in pd["gap"][:m]]
    return d


def product_load(text, rate):
    ps = lib.Pulses()
    try:
        n = ps.load_ook(text, rate)
        assert n == len(ps)
        return [pd_facts(ps.get(i)) for i in range(n)]
    finally:
        ps.close()


def random_pulse_data(rng, fsk=False):
    pd = np.zeros(1, lib.PULSE_DATA_DTYPE)[0]
    n = rng.randrange(1, 60)
    pd["num_pulses"] = n
    pd["sample_rate"] = rng.choice([250000, 1000000, 1024000, 2048000, 48000])
    pd["offset"] = rng.randrange(0, 1 << 34)
    pd["depth_bits"] = rng.choice([8, 16])
    for i in range(n):
        pd["pulse"][i] = rng.randrange(0, 5000)
        pd["gap"][i] = rng.randrange(0, 50000)
    pd["fsk_f2_est"] = rng.randrange(1, 9000) if fsk else 0
    pd["fsk_f1_est"] = rng.randrange(-9000, 9000)
    pd["freq1_hz"] = 433.92e6 + rng.randrange(-60000, 60000)
    pd["freq2_hz"] = 433.92e6 + rng.randrange(-60000, 60000)
    pd["centerfreq_hz"] = 433.92e6
    pd["range_db"], pd["rssi_db"], pd["snr_db"], pd["noise_db"] = 42.1442, -rng.random() * 30, rng.random() * 30, -rng.random() * 40
    return pd


def ref_loaded(key, text, rate, cap=64):
    """digest of what pulse_data_load() reads out of `text`."""
    return refdata.recorded(key, lambda: helpers.digest([pd_facts(p) for p in refh.load_ook(text, rate, cap=cap)]))


def test_ook_and_rfraw_readers_match_the_reference():
    for name, text in ook_cases().items():
        for rate in RATES:
            got = product_load(text, rate)
            assert helpers.digest(got) == ref_loaded(f"pulse_io/load/{name}/{rate}", text, rate), f"case {name} @ {rate}"
    # the -y test-data path: rfraw_parse() into a zeroed struct
    ps = lib.Pulses()
    for name, text in ook_cases().items():
        if not name.startswith("rfraw"):
            continue
        line = text.split("\n")[0]

        def ref_rfraw():
            ref = refh.rfraw(line)
            return None if ref is None else helpers.digest(pd_facts(ref))
        ref = refdata.recorded(f"pulse_io/rfraw/{name}", ref_rfraw)
        ps.clear()
        n = ps.load_rfraw(line)
        assert n == (1 if ref is not None else 0), name
        if n:
            assert helpers.digest(pd_facts(ps.get(0))) == ref, name
    assert ps.load_rfraw("500 1000") == 0
    ps.close()


def random_ook_text(rng):
    lines = []
    for _ in range(rng.randrange(1, 80)):
        r = rng.random()
        if r < 0.55:
            lines.append("%d %d" % (rng.randrange(0, 3000), rng.randrange(0, 30000)))
        elif r < 0.65:
            lines.append(rng.choice([";end", ";freq1 %d" % rng.randrange(-50000, 50000), ";freq2 7", ";received @1s", ";", ";ook 3 pulses"]))
        elif r < 0.78:
            bins = [rng.randrange(50, 70000) for _ in range(rng.randrange(1, 9))]
            codes = [rng.choice([0x80, 0x00]) | (rng.randrange(len(bins)) << 4) | rng.randrange(len(bins)) for _ in range(rng.randrange(0, 40))]
            line = rfraw_b1(bins, codes) if rng.random() < 0.5 else rfraw_b0(bins, codes, rng.randrange(0, 5))
            if rng.random() < 0.2:
                line = line[:rng.randrange(4, len(line))]          # truncated
            if rng.random() < 0.2:
                line = line.lower().replace("aa", "a a", 1)         # separators, case
            if rng.random() < 0.15:
                line += "+" + rfraw_b1([100, 200], [0x81, 0x90])
            lines.append(line)
        elif r < 0.88:
            lines.append("%d%s%d" % (rng.randrange(0, 3000), rng.choice(",;:\t  x"), rng.randrange(-50, 3000)))
        else:
            lines.append("".join(rng.choice(" ;-+0123456789abAB\t.") for _ in range(rng.randrange(0, 40))))
    return rng.choice(["\n", "\r\n"]).join(lines) + rng.choice(["\n", ""])


def test_ook_reader_random_texts():
    """400 random pulse texts (rows, headers, whole / truncated / decorated RfRaw lines, junk): the same packages as
    pulse_data_load() reads out of them."""
    cases = []
    for seed in range(400):
        rng = random.Random(1000 + seed)
        text = random_ook_text(rng)
        cases.append((text, rng.choice(RATES)))
    want = refdata.recorded("pulse_io/random_texts", lambda: [helpers.digest([pd_facts(p) for p in refh.load_ook(text, rate, cap=128)])
                                                              for text, rate in cases])
    for seed, (text, rate) in enumerate(cases):
        assert helpers.digest(product_load(text, rate)) == want[seed], f"seed {seed}: {text!r}"


def test_writers_match_the_reference():
    rng = random.Random(11)
    for i in range(40):
        pd = random_pulse_data(rng, fsk=i % 3 == 0)
        # logic.u8: a window that cuts the package at both ends
        total = int(pd["pulse"][:pd["num_pulses"]].sum() + pd["gap"][:pd["num_pulses"]].sum())
        start = int(pd["offset"]) + total // 4 if i % 2 else max(0, int(pd["offset"]) - 100)
        length = max(1, min(total // 2 + 7, 200000))
        bits = 0x04 if pd["fsk_f2_est"] else 0x02

        def written():
            ref = refh.dump_ook(pd)
            assert ref.startswith(";received ")
            head = refh.dump_vcd(pd, "'", header=True)
            body = refh.dump_vcd(pd, "'")
            ref_head = head[:len(head) - len(body)]
            return {"ook": helpers.digest(ref[ref.index("\n") + 1:]), "vcd": [helpers.digest(refh.dump_vcd(pd, ch)) for ch in "'\""],
                    "date": ref_head.split("\n")[0][len("$date "):-len(" $end")], "vcd_header": helpers.digest(ref_head),
                    "logic_u8": helpers.digest(refh.dump_raw(pd, length, start, bits))}
        ref = refdata.recorded(f"pulse_io/writers/{i}", written)
        assert helpers.digest(lib.format_ook(pd)) == ref["ook"]
        assert lib.format_ook(pd, received="@1.5s").startswith(";received @1.5s\n")
        assert helpers.digest(lib.format_ook(pd, received="@1.5s")[len(";received @1.5s\n"):]) == ref["ook"]
        assert [helpers.digest(lib.format_vcd(pd, ch)) for ch in "'\""] == ref["vcd"]
        assert helpers.digest(lib.format_vcd_header(int(pd["sample_rate"]), ref["date"])) == ref["vcd_header"]
        assert helpers.digest(lib.dump_logic_u8(pd, length, start, bits)) == ref["logic_u8"]
    assert lib.format_ook_header() == ";pulse data\n;version 1\n;timescale 1us\n"
    assert lib.format_ook_header("now") == ";pulse data\n;version 1\n;timescale 1us\n;created now\n"


def test_dump_then_load_round_trip_like_the_reference():
    """pulse_data_dump() rounds to whole microseconds; loading that text back must give what the reference loads."""
    rng = random.Random(5)
    text = lib.format_ook_header("t")
    pds = [random_pulse_data(rng) for _ in range(8)]
    for pd in pds:
        text += lib.format_ook(pd, received="t")
    for rate in RATES:
        assert helpers.digest(product_load(text, rate)) == ref_loaded(f"pulse_io/round_trip/{rate}", text, rate)
    assert len(product_load(text, 250000)) == len(pds)


def test_golden_pulse_io():
    """The committed fixture (reference outputs recorded by tools/make_golden.py): readers and writers."""
    with open(GOLDEN) as f:
        g = json.load(f)
    for c in g["load"]:
        assert product_load(c["text"], c["rate"]) == c["packages"], c["name"]
    for c in g["dump"]:
        pd = np.zeros(1, lib.PULSE_DATA_DTYPE)[0]
        for k in INT_FIELDS:
            pd[k] = c["pd"][k]
        for k in FLOAT_FIELDS:
            pd[k] = np.float32(c["pd"][k])
        n = len(c["pd"]["pulse"])
        pd["pulse"][:n] = c["pd"]["pulse"]
        pd["gap"][:n] = c["pd"]["gap"]
        assert lib.format_ook(pd) == c["ook"]
        assert lib.format_vcd(pd, "'") == c["vcd"]


# ------------------------------------------------------------------------------- GPU -----------

def sliced_by_reference(ref, pd):
    return [(dev, h) for dev, h, _bb in ref.slice_pulse_data(pd)]


@pytest.mark.gpu
def test_loaded_packages_through_k_slice():
    """`.ook` text and RfRaw lines -> r433b_process_pulses -> every bitbuffer equal to the reference's slicers."""
    loaded_packages_through_k_slice()


def loaded_packages_through_k_slice():
    devices = lib.default_device_table()
    ctx = lib.Context(0)
    ctx.set_devices(devices)
    ref = refdata.LiveRef(lambda r: r.register_defaults(), store_bitbuffers=False)
    try:
        # packages k_detect finds in two synthetic captures, written as .ook text by the product
        x = [synth.ook_stream(s, n_samples=1 << 19, n_bursts=4) for s in (21, 22)]
        data = np.concatenate(x)
        ctx.process(data, np.array([0, x[0].nbytes, data.nbytes], np.uint64), lib.FMT_CU8, 250000, 433920000)
        ctx.fetch()
        texts = []
        for s in range(2):
            _pk, index = ctx.packages_of(s)
            assert len(index) >= 4
            texts.append(lib.format_ook_header("t") + "".join(lib.format_ook(ctx.pulse_data(gi), received="t") for gi in index))
        ps = lib.Pulses()
        for s, t in enumerate(texts):
            assert ps.load_ook(t, 250000, stream=s) >= 4
        # stream 2: RfRaw lines (1 MHz packages) between .ook rows of a 1.024 MHz file; stream 3: -y test data and
        # caller-built structs, one of them an FSK package (fsk_f2_est set -> run_fsk_demods)
        cases = ook_cases()
        mixed = cases["rfraw_after_rows"] + cases["plain"] + cases["rfraw_b0_repeats"] + ";end\n" + cases["rfraw_long_line"]
        ps.load_ook(mixed, 1024000, stream=2)
        ps.load_rfraw(cases["rfraw_b1_line"].strip(), stream=3)
        rng = random.Random(3)
        fsk_pd = random_pulse_data(rng, fsk=True)
        fsk_pd["sample_rate"] = 250000
        bits = [rng.randrange(2) for _ in range(200)]
        runs, k = [], 0
        while k < len(bits):
            j = k
            while j < len(bits) and bits[j] == bits[k]:
                j += 1
            runs.append((bits[k], (j - k) * 25))
            k = j
        if runs[0][0] == 0:
            runs = runs[1:]
        n = len(runs) // 2
        fsk_pd["num_pulses"] = n
        fsk_pd["pulse"][:] = 0
        fsk_pd["gap"][:] = 0
        for i in range(n):
            fsk_pd["pulse"][i] = runs[2 * i][1]
            fsk_pd["gap"][i] = runs[2 * i + 1][1]
        fsk_pd["gap"][n - 1] = 30000
        ps.add(fsk_pd, stream=3)
        ps.add(random_pulse_data(rng), stream=3)

        def loaded_by_reference():
            sets = [list(refh.load_ook(texts[0], 250000)), list(refh.load_ook(texts[1], 250000)),
                    list(refh.load_ook(mixed, 1024000)), [refh.rfraw(cases["rfraw_b1_line"].strip()), fsk_pd, ps.get(len(ps) - 1)]]
            return [[{"num_pulses": int(p["num_pulses"]), "sample_rate": int(p["sample_rate"]),
                      "pulse": helpers.digest(p["pulse"][:int(p["num_pulses"])]), "freq1_hz": float(p["freq1_hz"]),
                      "fsk_f2_est": int(p["fsk_f2_est"]), "events": helpers.digest(sliced_by_reference(ref, p))} for p in w]
                    for w in sets]
        want_sets = refdata.recorded("pulse_io/loaded_through_k_slice", loaded_by_reference)
        assert sum(len(w) for w in want_sets) == len(ps)
        assert len({p["sample_rate"] for w in want_sets for p in w}) >= 3

        ctx.process_pulses(ps)
        ctx.fetch()
        total_events = 0
        for s, want in enumerate(want_sets):
            got = helpers.gpu_stream_results(ctx, s)
            assert len(got["packages"]) == len(want)
            for li, (gp, wp) in enumerate(zip(got["packages"], want)):
                assert gp["num_pulses"] == wp["num_pulses"] and gp["sample_rate"] == wp["sample_rate"]
                assert helpers.digest(gp["pulse"][:gp["num_pulses"]].astype(np.int32)) == wp["pulse"]
                assert gp["freq1_hz"] == wp["freq1_hz"] and gp["fsk_f2_est"] == wp["fsk_f2_est"]
                mine = [(e["dev"], e["hash"]) for e in got["events"] if e["package"] == li]
                assert helpers.digest(mine) == wp["events"], f"stream {s} package {li}: {len(mine)} events differ from the reference's"
                total_events += len(mine)
        assert total_events > 1000
        assert ctx.counts()["events"] == total_events
        ps.close()
    finally:
        ref.close()
        ctx.close()
