"""Decoder length gates and the threaded replay (SURVEY 8(f1)).

CPU: the committed gate table (rtl_433_b200/data/gates_25.12.json, tools/probe_gates.py) against the compiled
reference decoders with inputs the generator never saw (their answers recorded in tests/golden/reference.json by
tests/refdata.py).  GPU / emulator: a gated run keeps exactly the events the
gate predicate lets through and counts the others per (package, device) and row class; with the reference's real
decoders behind r433b_dispatch_r_devices() every decoder's statistics and the decoded messages are those of a
pure-reference run -- gated or not, one thread or four."""
import ctypes as C
import json
import os
import random

import numpy as np
import pytest

import helpers
import refdata
from oracle import refh
from rtl_433_b200 import lib, synth

needs_ref = pytest.mark.skipif(not refh.available(), reason="oracle/_ref/libr433ref.so not built")
HERE = os.path.dirname(os.path.abspath(__file__))


def gate_table():
    with open(os.path.join(os.path.dirname(HERE), "rtl_433_b200", "data", "gates_25.12.json")) as f:
        return json.load(f)


def all_protocols_ref():
    L = refh.lib()
    L.refh_probe_gate.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_int)]
    L.refh_call_decoder.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    r = refh.Ref(store_bitbuffers=False)
    for i in range(L.refh_num_protocols(r.h)):
        r.register(i + 1)
    return L, r


def probe_reference_decoders(tab):
    """Per protocol: the gate a second probe (another seed) finds, its codes, and the distinct (single row, return
    value, output count) answers of the decoder to 40 hand-made bitbuffers below the committed gate (patterns the
    probe does not use: repeated rows and walking ones, what find_repeated_row() and preamble searches look for)."""
    L, r = all_protocols_ref()
    rng = random.Random(99)
    out = []
    for idx, d in enumerate(r.registered()):
        t = tab["gates"][str(d["protocol_num"])][0]
        code = (C.c_int * 2)()
        t2 = L.refh_probe_gate(r.h, idx, tab["max_bits"], 400, 12345, code)
        answers = set()
        for k in range(40 if t >= 2 else 0):
            bb = np.zeros(1, refh.BITBUFFER_DTYPE)
            rows = 1 if k % 3 == 0 else rng.randrange(2, 30)
            bb["num_rows"] = rows
            bb["free_row"] = rows
            for row in range(rows):
                bb["bits_per_row"][0][row] = rng.randrange(0, t)
                pat = [0xaa, 0x55, 0xff, 0x00, 0x2d, 0xd4, 0x80 >> (k % 8), rng.randrange(256)][k % 8]
                bb["bb"][0][row][:4] = pat
            n = C.c_int(0)
            ret = L.refh_call_decoder(r.h, idx, bb.ctypes.data, C.byref(n))
            answers.add((int(rows == 1), ret, n.value))
        out.append({"protocol_num": d["protocol_num"], "gate": t, "probe": t2, "code": [code[0], code[1]],
                    "answers": sorted(answers)})
    r.close()
    return out


def test_gate_table_holds_for_fresh_inputs():
    """A second probe with another seed never finds a shorter gate or another code than the committed table, and
    hand-made bitbuffers below each gate (patterns the probe does not use) are turned down with the table's code."""
    tab = gate_table()
    devs = lib.default_device_table(include_disabled=True)
    n, want = refdata.registered_devices("all")
    assert helpers.digest(refdata.device_rows(devs)) == want  # the reference's protocols in order
    assert len(devs) == n == len(tab["gates"])
    probed = refdata.recorded("gates/fresh_probe", lambda: probe_reference_decoders(tab))
    assert [p["protocol_num"] for p in probed] == [d["protocol_num"] for d in devs]
    n_gated_devices = 0
    for d, p in zip(devs, probed):
        t, c1, cn = tab["gates"][str(d["protocol_num"])]
        assert p["gate"] == t, f"protocol {d['protocol_num']}: the gate table changed; record the probe again"
        t2 = p["probe"]
        assert t2 >= t, f"protocol {d['protocol_num']}: gate {t} does not hold (fresh probe: {t2})"
        if t:
            assert tuple(p["code"]) == (c1, cn)
            n_gated_devices += 1
        if t < 2:
            continue
        assert p["answers"]
        for single, ret, n in p["answers"]:
            assert ret == (c1 if single else cn) and n == 0, (d["protocol_num"], single, ret)
    assert n_gated_devices > 300


def gate_predicate(bb, t):
    nr = int(bb["num_rows"])
    return nr >= 1 and int(bb["bits_per_row"][:nr].max()) < t


def gated_run_is_the_filtered_ungated_run():
    devices = lib.default_device_table()
    gates = lib.default_gates(devices)
    assert sum(1 for g in gates if g[0]) > 280
    ctx = lib.Context(0)
    try:
        streams = [synth.ook_stream(41, n_samples=1 << 18, n_bursts=3), synth.ook_stream(42, n_samples=1 << 18, n_bursts=3)]
        data = np.concatenate(streams)
        offs = np.array([0, streams[0].nbytes, data.nbytes], np.uint64)
        ctx.set_devices(devices)
        ctx.process(data, offs, lib.FMT_CU8, 250000, 433920000)
        full = ctx.fetch()
        assert full["n_gated"] == 0 and ctx.gated() == 0
        plain = [helpers.gpu_stream_results(ctx, s, store_bitbuffers=True) for s in range(2)]
        ctx.set_gates(gates)
        ctx.process(data, offs, lib.FMT_CU8, 250000, 433920000)
        res = ctx.fetch()
        kept = [helpers.gpu_stream_results(ctx, s, store_bitbuffers=True) for s in range(2)]
        pk = res["packages"]
        dropped_total = 0
        for s in range(2):
            want = [e for e in plain[s]["events"] if not gate_predicate(e["bitbuffer"], gates[e["dev"]][0])]
            got = kept[s]["events"]
            assert [(e["package"], e["dev"], e["hash"]) for e in got] == [(e["package"], e["dev"], e["hash"]) for e in want]
            assert len(got) < len(plain[s]["events"]) // 3  # most events are noise
            # per (package, device): the dropped events by row class
            index = [i for i in range(len(pk)) if pk["stream"][i] == s]
            count1, countn = {}, {}
            for e in plain[s]["events"]:
                if gate_predicate(e["bitbuffer"], gates[e["dev"]][0]):
                    tgt = count1 if int(e["bitbuffer"]["num_rows"]) == 1 else countn
                    tgt[(e["package"], e["dev"])] = tgt.get((e["package"], e["dev"]), 0) + 1
                    dropped_total += 1
            for li, gi in enumerate(index):
                row = res["pairs"][int(pk["first_pair"][gi]) // res["n_devices"]]  # the pair table is in device order
                for dv in np.nonzero(row["gated_single"] | row["gated_multi"])[0]:
                    assert int(row["gated_single"][dv]) == count1.get((li, int(dv)), 0)
                    assert int(row["gated_multi"][dv]) == countn.get((li, int(dv)), 0)
                assert int(row["gated_single"].sum()) == sum(v for (p, _d), v in count1.items() if p == li)
                assert int(row["gated_multi"].sum()) == sum(v for (p, _d), v in countn.items() if p == li)
        assert res["n_gated"] == dropped_total == ctx.gated()
        assert res["n_events"] + res["n_gated"] == full["n_events"]
        assert res["event_bytes"] < full["event_bytes"] // 2
        # the pipelined host path counts the same
        ctx.set_pipeline(4)
        big = np.concatenate([data] * 2)
        n = streams[0].nbytes
        ctx.process(big, np.arange(5, dtype=np.uint64) * n, lib.FMT_CU8, 250000, 433920000)
        r4 = ctx.fetch()
        assert r4["n_gated"] == 2 * dropped_total and r4["n_events"] == 2 * res["n_events"]
        assert ctx.stream_digest(0) == ctx.stream_digest(2) and ctx.stream_digest(1) == ctx.stream_digest(3)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_gated_run_is_the_filtered_ungated_run():
    gated_run_is_the_filtered_ungated_run()


def decoders_behind_gates_and_threads():
    """Reference decoders behind the GPU path: statistics and messages equal to a pure-reference run without gates,
    with gates, and with gates on four replay threads (four separately registered decoder sets)."""
    kinds = ("silvercrest", "nexus", "nice")
    files = [synth.ook_stream(50 + i, n_samples=1 << 18, n_bursts=3, kinds=kinds, decodable=True) for i in range(6)]
    r = refh.Ref(chain_decoders=True, store_bitbuffers=False)
    n = r.register_defaults()
    devs = r.registered()
    want_json, want_stats = [], np.zeros((n, 8), np.int64)
    for x in files:
        want_json.append(r.run(x, 2)["json"])
        want_stats += np.array([r.device_stats(i) for i in range(n)], np.int64)
        r.L.refh_reset_stats(r.h)
    assert sum(len(j) for j in want_json) >= 6
    data = np.concatenate(files)
    offs = np.arange(len(files) + 1, dtype=np.uint64) * files[0].nbytes
    ctx = lib.Context(0)
    ctx.set_devices(devs)
    workers = [refh.Ref(chain_decoders=True, store_bitbuffers=False) for _ in range(4)]
    for w in workers:
        assert w.register_defaults() == n
    timing = {}
    import time
    try:
        for mode in ("plain", "gated", "gated+threads"):
            ctx.set_gates(lib.default_gates(devs) if mode != "plain" else None)
            ctx.process(data, offs, lib.FMT_CU8, 250000, 433920000)
            res = ctx.fetch()
            if mode == "plain":
                plain_events = res["n_events"]
            else:
                assert res["n_events"] + res["n_gated"] == plain_events and res["n_gated"] > 2 * res["n_events"]
            if mode != "gated+threads":
                got_json, got_stats = [], np.zeros((n, 8), np.int64)
                timing[mode] = 0.0
                for s in range(len(files)):
                    ptrs = r.L.refh_begin_external_dispatch(r.h)
                    try:
                        t0 = time.perf_counter()
                        rc = ctx.L.r433b_dispatch_r_devices(ctx.h, C.byref(ctx._res), s, ptrs, n)
                        timing[mode] += time.perf_counter() - t0
                        assert rc == 0, ctx.L.r433b_last_error(ctx.h)
                        got_json.append([l for l in r.L.refh_json(r.h).decode().split("\n") if l])
                        got_stats += np.array([r.device_stats(i) for i in range(n)], np.int64)
                    finally:
                        r.L.refh_end_external_dispatch(r.h)
                assert got_json == want_json, mode
            else:
                sets = (C.c_void_p * len(workers))()
                for i, w in enumerate(workers):
                    sets[i] = w.L.refh_begin_external_dispatch(w.h)
                try:
                    t0 = time.perf_counter()
                    rc = ctx.L.r433b_dispatch_r_devices_parallel(ctx.h, C.byref(ctx._res), sets, n, len(workers))
                    timing[mode] = time.perf_counter() - t0
                    assert rc == 0, ctx.L.r433b_last_error(ctx.h)
                    got_stats = np.zeros((n, 8), np.int64)
                    per_worker = []
                    for w in workers:
                        got_stats += np.array([w.device_stats(i) for i in range(n)], np.int64)
                        per_worker.append([l for l in w.L.refh_json(w.h).decode().split("\n") if l])
                finally:
                    for w in workers:
                        w.L.refh_end_external_dispatch(w.h)
                # worker w replays streams w, w + 4, ... in order
                for wi in range(len(workers)):
                    assert per_worker[wi] == [l for s in range(wi, len(files), len(workers)) for l in want_json[s]]
            assert np.array_equal(got_stats, want_stats), mode
        assert int(want_stats[:, 0].sum()) > 5000
        # host-side cost of the replay with the reference's REAL decoders (SURVEY 8(f1)); recorded when the box lets us
        events = int(want_stats[:, 0].sum())
        report = {"decode_events": events, "files": len(files),
                  "seconds": {k: round(v, 4) for k, v in timing.items()},
                  "decode_events_per_s": {k: round(events / v) for k, v in timing.items() if v > 0},
                  "what": "r433b_dispatch_r_devices[_parallel] with the unmodified src/devices/*.c decoders (oracle/_ref): "
                          "plain = every event re-inflated and decoded, gated = events under the length gates booked from "
                          "their counts, gated+threads = 4 workers with their own decoder sets"}
        out = os.path.join(os.path.dirname(HERE), "gpurun_out")
        if os.path.isdir(out):
            with open(os.path.join(out, "dispatch_real_decoders.json"), "w") as f:
                json.dump(report, f, indent=1)
        print("dispatch with real decoders:", report["decode_events_per_s"])
    finally:
        for w in workers:
            w.close()
        r.close()
        ctx.close()


@pytest.mark.gpu
@needs_ref
def test_decoders_behind_gates_and_threads():
    decoders_behind_gates_and_threads()


def submit_wait_ping_pong():
    """Two contexts used alternately (r433b_submit / r433b_wait): batch k+1 is processed on a worker thread while the
    caller replays batch k; results equal those of plain process() + fetch()."""
    devices = lib.default_device_table()
    batches = [np.concatenate([synth.ook_stream(80 + 2 * k, n_samples=1 << 18, n_bursts=3),
                               synth.ook_stream(81 + 2 * k, n_samples=1 << 18, n_bursts=3)]) for k in range(3)]
    offs = np.array([0, batches[0].nbytes // 2, batches[0].nbytes], np.uint64)
    ctxs = [lib.Context(0), lib.Context(0)]
    try:
        want = []
        for c in ctxs:
            c.set_devices(devices)
            c.set_gates(lib.default_gates(devices))
        for b in batches:
            ctxs[0].process(b, offs, lib.FMT_CU8, 250000, 433920000)
            ctxs[0].fetch()
            want.append([ctxs[0].stream_digest(s) for s in range(2)])
        got = []
        ctxs[0].submit(batches[0], offs, lib.FMT_CU8, 250000, 433920000)
        for k in range(len(batches)):
            cur, nxt = ctxs[k % 2], ctxs[(k + 1) % 2]
            res = cur.wait()
            if k + 1 < len(batches):
                nxt.submit(batches[k + 1], offs, lib.FMT_CU8, 250000, 433920000)  # runs while batch k is replayed below
            assert res["n_packages"] >= 6
            events = []
            for s in range(2):
                cur.dispatch(s, lambda pk, dv, pd, bb: events.append(dv) or 0)
            assert len(events) == res["n_events"]
            got.append([cur.stream_digest(s) for s in range(2)])
        assert got == want
        with pytest.raises(lib.R433Error):
            ctxs[0].wait()
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.gpu
def test_submit_wait_ping_pong():
    submit_wait_ping_pong()
