"""-m gpu: the CUDA path (through the C ABI) against the oracle on the same seeded inputs.

Oracle = oracle/r433_oracle.c (CPU restatement) and the unmodified reference (oracle/_ref/libr433ref.so, its
outputs recorded in tests/golden/reference.json by tests/refdata.py).  Everything integer is compared
for equality: stage arrays, pulse widths, package headers, every bitbuffer (by FNV-1a of the
whole 6604-byte struct) in the reference's dispatch order.  The only floats on the path
(calc_rssi_snr, src/r_flow.c:35-64) are computed on the host with the reference's expressions and
compared for equality too (same libm, same box); tolerance would be 1 ULP if libm differed.
"""
import numpy as np
import pytest

import helpers
import refdata
from oracle import orc, refh
from rtl_433_b200 import lib, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def devices():
    return lib.default_device_table()


@pytest.fixture(scope="module")
def ctx(devices):
    c = lib.Context(0)
    c.set_devices(devices)
    yield c
    c.close()


def run_gpu(ctx, streams, fmt, rate, freq, fpdm=lib.FPDM_AUTO, block_bytes=0):
    lens = [s.nbytes for s in streams]
    padded = [(n + 15) // 16 * 16 for n in lens]
    # the ABI wants 16-byte aligned stream starts; stream i is exactly lens[i] bytes long only
    # when that is already a multiple of 16, so tests use such lengths
    assert lens == padded
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    data = np.concatenate([s.view(np.uint8).ravel() for s in streams]) if streams else np.zeros(0, np.uint8)
    # Without the stage dump the kernel computes FM on demand (only inside packages, filter state
    # rebuilt from the previous tile); with it, FM is computed for every tile.  Both must agree.
    ctx.process(data, offsets, fmt, rate, freq, fpdm, block_bytes, want_stages=False)
    ctx.fetch()
    on_demand = [helpers.gpu_stream_results(ctx, i) for i in range(len(streams))]
    ctx.process(data, offsets, fmt, rate, freq, fpdm, block_bytes, want_stages=True)
    ctx.fetch()
    out = []
    for i, s in enumerate(streams):
        r = helpers.gpu_stream_results(ctx, i)
        d = helpers.compare_results(r, on_demand[i], f"FM on demand vs every tile, stream {i}", stages=False)
        assert not d, "\n".join(d[:20])
        n = lens[i] // fmt
        r["am"], r["fm"] = ctx.copy_stage(i, n)
        out.append(r)
    return out


def oracle_for(devices, stages=True):
    o = orc.Oracle(store_bitbuffers=False, store_stages=stages)
    o.add_devices(devices)
    return o


def check(gpu, ref, tag):
    d = helpers.compare_results(ref, gpu, tag)
    assert not d, "\n".join(d[:20])


def test_ook_cu8_default_devices(ctx, devices):
    """BASELINE config 2 at test size: noisy 250 kS/s cu8 streams, all 335 default decoders."""
    streams = [synth.ook_stream(seed) for seed in range(6)]
    gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
    o = oracle_for(devices)
    for i, s in enumerate(streams):
        ref = o.run(s, 2)
        assert len(ref["packages"]) >= 8
        check(gpu[i], ref, f"ook seed {i}")


def test_fsk_cs16_minmax_and_classic(ctx, devices):
    """BASELINE config 3 at test size: 1.024 MS/s cs16 2-FSK, both FSK pulse detectors."""
    streams = [synth.fsk_stream(seed) for seed in range(3)]
    o = oracle_for(devices)
    for fpdm, freq in ((lib.FPDM_AUTO, 868000000), (lib.FPDM_CLASSIC, 433920000)):
        gpu = run_gpu(ctx, streams, lib.FMT_CS16, 1024000, freq, fpdm)
        for i, s in enumerate(streams):
            ref = o.run(s, 4, 1024000, freq, fpdm)
            assert any(p["type"] == 2 for p in ref["packages"])
            check(gpu[i], ref, f"fsk seed {i} fpdm {fpdm}")


def test_silence_and_reference_vectors(ctx, devices):
    """Constant 128/128 silence (the IIR sits on two different fixed points: the bracket rounds
    cannot collapse and must fall back to exact propagation), the reference's own Nice Flor-s
    vector (tests/rtl_tcp_serve.py) and the config-1 Silvercrest file."""
    def pad(x):
        n = (len(x) + 15) // 16 * 16
        return np.concatenate([x, np.full(n - len(x), 128, np.uint8)])
    streams = [pad(synth.nice_flor_s_file()), pad(synth.silvercrest_file()), pad(synth.silvercrest_file(noise_sigma=2.0)),
               np.full(4096 * 2, 128, np.uint8), np.zeros(0, np.uint8)]
    gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
    o = oracle_for(devices)
    for i, s in enumerate(streams):
        ref = o.run(s, 2) if len(s) else {"packages": [], "events": []}
        check(gpu[i], ref, f"vector {i}")
    # the decoder-facing bitbuffer of config 1: {33}7c2600020 x 4 from device 0 (Silvercrest)
    r = helpers.gpu_stream_results(ctx, 1, store_bitbuffers=True)
    bb = [e["bitbuffer"] for e in r["events"] if e["dev"] == 0][0]
    assert int(bb["num_rows"]) == 4
    assert [refh.row_hex(bb, k) for k in range(4)] == ["{33}7c2600020"] * 4


def test_fm_rebuild_after_constant_input(ctx, devices):
    """FM is computed on demand and its filter state rebuilt from the tile in front of a package.
    Over exactly constant input (digital silence between signals) the rebuild cannot converge --
    the two bracket ends sit on different fixed points of the floor map -- and the kernel has to
    walk forward from the last exact state instead.  cu8 and cs16, silence in front and in the
    middle, through run_gpu's on-demand / every-tile comparison and against the oracle."""
    a, b = synth.ook_stream(51, n_samples=1 << 18, n_bursts=3), synth.ook_stream(52, n_samples=1 << 18, n_bursts=3)
    quiet = np.full(2 * 5000, 128, np.uint8)
    o = oracle_for(devices)
    first = o.run(b, 2)["packages"][0]["offset"]
    assert first > 4096
    hushed = b.copy()
    hushed[: 2 * (first - 40)] = 128  # constant right up to the first pulse: the tile in front of it cannot help
    streams = [np.concatenate([quiet, a]), np.concatenate([a, quiet, quiet, b]), hushed, np.concatenate([a, hushed])]
    streams = [s[: len(s) // 16 * 16] for s in streams]
    gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
    for i, s in enumerate(streams):
        ref = o.run(s, 2)
        assert len(ref["packages"]) >= 2
        check(gpu[i], ref, f"constant cu8 {i}")
    f = synth.fsk_stream(53)
    zeros = np.zeros(2 * 7000, np.int16)
    streams = [np.concatenate([zeros, f]), np.concatenate([f, zeros, f])]
    streams = [s[: len(s) // 8 * 8] for s in streams]
    gpu = run_gpu(ctx, streams, lib.FMT_CS16, 1024000, 868000000)
    for i, s in enumerate(streams):
        ref = o.run(s, 4, 1024000, 868000000)
        assert any(p["type"] == 2 for p in ref["packages"])
        check(gpu[i], ref, f"constant cs16 {i}")


def check_recorded(gpu, want, tag):
    d = helpers.compare_fingerprint(want, gpu, tag)
    assert not d, "\n".join(d[:20])


def test_against_compiled_reference(ctx, devices):
    """Same comparison against the unmodified reference."""
    streams = [synth.ook_stream(100 + seed) for seed in range(2)]
    gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
    for i, s in enumerate(streams):
        check_recorded(gpu[i], refdata.ref_run(f"gpu_parity/ook/{i}", s, 2), f"ref ook {i}")
    streams = [synth.fsk_stream(100)]
    gpu = run_gpu(ctx, streams, lib.FMT_CS16, 1024000, 868000000)
    check_recorded(gpu[0], refdata.ref_run("gpu_parity/fsk", streams[0], 4, 1024000, 868000000, 2), "ref fsk")


def test_ragged_lengths_and_small_blocks(ctx, devices):
    """Streams of different lengths (incl. partial last tile/block) and a non-default block
    size: exercises the block-call emulation (eop flag, start_ago/end_ago, x[-1] int16 wrap)."""
    base = synth.ook_stream(7)
    cuts = [2 * 16 * 1000, 2 * 16 * 4097, 2 * 131072 + 2 * 16 * 3, 2 * 8 * 99991 // 16 * 16]
    streams = [base[:c].copy() for c in cuts]
    o = oracle_for(devices)
    for bb in (0, 32768):
        gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000, block_bytes=bb)
        for i, s in enumerate(streams):
            check(gpu[i], o.run(s, 2, block_bytes=bb), f"ragged {i} block {bb}")


def test_magnitude_mode_and_fixed_level(ctx, devices):
    streams = [synth.ook_stream(11), synth.ook_stream(12)]
    try:
        for kw in (dict(use_mag_est=1), dict(level_limit=-10.0), dict(min_level=-20.0, min_snr=6.0)):
            ctx.set_levels(**kw)
            gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
            o = oracle_for(devices)
            o.set_levels(**kw)
            for i, s in enumerate(streams):
                check(gpu[i], o.run(s, 2), f"levels {kw} {i}")
    finally:
        ctx.set_levels()


def test_pipelined_time_slices_identical(ctx, devices):
    """Host-input batches processed in overlapping time slices (detector and filter state carried
    between launches) must give exactly the single-launch result."""
    streams = [synth.ook_stream(20 + seed, n_samples=1 << 19, n_bursts=4) for seed in range(5)]
    o = oracle_for(devices, stages=False)
    refs = [o.run(s, 2) for s in streams]
    lens = [s.nbytes for s in streams]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    data = np.concatenate(streams)
    try:
        for groups in (3, 4, 16):
            ctx.set_pipeline(groups)
            ctx.process(data, offsets, lib.FMT_CU8, 250000, 433920000)
            ctx.fetch()
            assert ctx.timing()["detect_launches"] > 1
            for i in range(len(streams)):
                got = helpers.gpu_stream_results(ctx, i)
                d = helpers.compare_results(refs[i], got, f"pipeline {groups} stream {i}", stages=False)
                assert not d, "\n".join(d[:20])
    finally:
        ctx.set_pipeline(0)


def test_pipelined_ragged_files_on_a_uniform_stride(ctx, devices):
    """Capture files of different lengths padded to a common stride (captures.load_batches(uniform=True)) take the
    pipelined host path too: every stream ends -- and is flushed -- in the time slice that reaches its own end."""
    full = [synth.ook_stream(70 + seed, n_samples=1 << 19, n_bursts=4) for seed in range(5)]
    cuts = [len(full[0]), 2 * 16 * 20011, 2 * 131072 * 2, 2 * 16 * 9, 2 * (131072 * 3 + 16 * 77)]
    streams = [s[:c] for s, c in zip(full, cuts)]
    o = oracle_for(devices, stages=False)
    refs = [o.run(s, 2) for s in streams]
    stride = len(full[0])
    data = np.full(stride * len(streams), 0x5a, np.uint8)  # bytes behind a file's end must never be looked at
    for i, s in enumerate(streams):
        data[i * stride:i * stride + len(s)] = s
    offsets = np.arange(len(streams) + 1, dtype=np.uint64) * np.uint64(stride)
    lengths = np.array([len(s) for s in streams], np.uint64)
    try:
        for groups in (4, 16):
            ctx.set_pipeline(groups)
            ctx.process(data, offsets, lib.FMT_CU8, 250000, 433920000, lengths=lengths)
            ctx.fetch()
            assert ctx.timing()["detect_launches"] > 1
            for i in range(len(streams)):
                got = helpers.gpu_stream_results(ctx, i)
                d = helpers.compare_results(refs[i], got, f"ragged pipeline {groups} stream {i}", stages=False)
                assert not d, "\n".join(d[:20])
    finally:
        ctx.set_pipeline(0)


def test_cs8_input_is_cu8_plus_128(ctx, devices):
    """cs8 captures are converted to cu8 (+128, src/rtl_433.c:1830-1834) inside the load phase."""
    streams = [synth.ook_stream(31), synth.ook_stream(32)[: 2 * 16 * 40001]]
    o = oracle_for(devices, stages=False)
    lens = [s.nbytes for s in streams]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    as_cs8 = np.concatenate(streams) ^ np.uint8(0x80)  # the int8 bytes a .cs8 file would hold
    ctx.process(as_cs8, offsets, lib.FMT_CS8, 250000, 433920000)
    ctx.fetch()
    for i, s in enumerate(streams):
        d = helpers.compare_results(o.run(s, 2), helpers.gpu_stream_results(ctx, i), f"cs8 {i}", stages=False)
        assert not d, "\n".join(d[:20])


def test_fm_low_pass_override_and_wrapping_filter(ctx, devices):
    """-Y filter values: a cutoff in Hz, one in us, and a ratio above 0.5 whose feedback coefficient
    is negative -- the host can then no longer prove the int16 state never wraps, so the kernel
    variant that is exact by induction alone (up to 31 bracket rounds) runs."""
    streams = [synth.ook_stream(41, n_samples=1 << 19, n_bursts=4), synth.ook_stream(42, n_samples=1 << 19, n_bursts=4)]
    try:
        for lp in (25000.0, 12.0, 0.6):
            ctx.set_fm_low_pass(lp)
            gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
            o = oracle_for(devices)
            o.set_fm_low_pass(lp)
            for i, s in enumerate(streams):
                check(gpu[i], o.run(s, 2), f"fm_low_pass {lp} stream {i}")
    finally:
        ctx.set_fm_low_pass(0.0)


def test_priority_classes_stop_after_a_decode(ctx):
    """run_ook_demods(): a priority class only runs while no earlier class decoded something
    (src/r_api.c:444).  Same devices registered twice with priorities 0 and 5."""
    table = {d["protocol_num"]: d for d in lib.default_device_table(include_disabled=True)}
    devs = [dict(table[1]), dict(table[2], priority=5), dict(table[12]), dict(table[19], priority=10)]
    x = synth.ook_stream(5, n_samples=1 << 18, n_bursts=2, kinds=("silvercrest",), decodable=True)
    c = lib.Context(0)
    try:
        c.set_devices(devs)
        c.process(x, np.array([0, x.nbytes], np.uint64), lib.FMT_CU8, 250000, 433920000)
        c.fetch()
        seen = []
        c.dispatch(0, lambda pkg, dev, pd, bb: (seen.append((pkg, dev)), 1 if dev == 0 else 0)[1])
        assert seen and {d for _, d in seen} <= {0, 2}      # classes 5 and 10 never ran
        seen2 = []
        c.dispatch(0, lambda pkg, dev, pd, bb: (seen2.append((pkg, dev)), 0)[1])
        assert {d for _, d in seen2} == {0, 1, 2, 3}        # nobody decodes: every class runs
        order = [d for p, d in seen2 if p == seen2[0][0]]
        assert order == sorted(order, key=lambda d: (devs[d].get("priority", 0), d))
    finally:
        c.close()


def fresh_ctx(devs):
    c = lib.Context(0)
    c.set_devices(devs)
    return c


def test_custom_piwm_raw_and_nrzs_devices():
    """pulse_slicer_piwm_raw / pulse_slicer_nrzs (src/pulse_slicer.c:597-657, :715-759) have no default-enabled
    device: hand-made devices of every modulation (tests/test_parity_holes.py pins the oracle on the same set)."""
    from test_parity_holes import MOD, custom_devices
    devs = custom_devices()
    c = fresh_ctx(devs)
    try:
        o = oracle_for(devs)
        streams = [synth.ook_stream(71, n_samples=1 << 19, n_bursts=5), synth.ook_stream(73, n_samples=1 << 19, n_bursts=5)]
        gpu = run_gpu(c, streams, lib.FMT_CU8, 250000, 433920000)
        seen = set()
        for i, s in enumerate(streams):
            ref = o.run(s, 2)
            seen |= {devs[e["dev"]]["modulation"] for e in ref["events"]}
            check(gpu[i], ref, f"custom ook {i}")
        assert {MOD["OOK_PIWM_RAW"], MOD["OOK_NRZS"]} <= seen
        streams = [synth.fsk_stream(72, n_samples=1 << 18, n_bursts=2)]
        gpu = run_gpu(c, streams, lib.FMT_CS16, 1024000, 868000000)
        check(gpu[0], o.run(streams[0], 4, 1024000, 868000000), "custom fsk")
        # a rate at which single widths truncate to zero samples: the six-field check must silence those devices
        streams = [synth.ook_stream(74, n_samples=1 << 17, rate=48000, n_bursts=2, kinds=("nice", "manchester"))]
        gpu = run_gpu(c, streams, lib.FMT_CU8, 48000, 433920000)
        check(gpu[0], o.run(streams[0], 2, 48000, 433920000), "custom 48 kS/s")
    finally:
        c.close()


def test_all_protocols_including_disabled():
    """All 384 protocols (klimalogg = NRZS; 198 / 270: tolerance 1 us -> 0 samples at 250 kS/s, the reference's
    'sample rate too low' return, src/pulse_slicer.c:79-84)."""
    devs = lib.default_device_table(include_disabled=True)
    assert len(devs) >= 380
    c = fresh_ctx(devs)
    try:
        o = oracle_for(devs)
        streams = [synth.ook_stream(81, n_samples=1 << 19, n_bursts=4), synth.ook_stream(82, n_samples=1 << 19, n_bursts=4)]
        gpu = run_gpu(c, streams, lib.FMT_CU8, 250000, 433920000)
        for i, s in enumerate(streams):
            check(gpu[i], o.run(s, 2), f"all protocols {i}")
    finally:
        c.close()


def test_ook_1200_pulse_end_of_package(ctx, devices):
    """PD_MAX_PULSES reached inside a train (src/pulse_detect.c:429-441): through det_step() and through the
    GAP scan's own copy of that branch; different phases of the train against the tile grid."""
    streams = [synth.ook_train_stream(1, 1300, 200.0, 200.0), synth.ook_train_stream(2, 2500, 120.0, 80.0),
               synth.ook_train_stream(5, 1201, 400.0, 60.0), synth.ook_train_stream(3, 1201, 400.0, 44.0),
               synth.ook_train_stream(6, 1250, 180.0, 1900.0, n_samples=1 << 20, lead_us=9137.0)]
    gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, 433920000)
    o = oracle_for(devices)
    for i, s in enumerate(streams):
        ref = o.run(s, 2)
        if i != 3:
            assert [p["num_pulses"] for p in ref["packages"] if p["type"] == 1][0] == 1200
        check(gpu[i], ref, f"ook train {i}")


def test_fsk_train_overflow_shifts_the_pulse_train(ctx, devices):
    """> 1200 FSK pulses in one carrier: pulse_data_shift and its `offset += 600` (src/pulse_data.c:27-34,
    src/pulse_detect_fsk.c:114, :205), classic and minmax detectors, cs16 and cu8 captures."""
    o = oracle_for(devices)
    streams = [synth.fsk_burst_stream(2, 2700), synth.fsk_burst_stream(5, 3900, bit_us=60.0)]
    for fpdm, freq in ((lib.FPDM_AUTO, 868000000), (lib.FPDM_CLASSIC, 433920000)):
        gpu = run_gpu(ctx, streams, lib.FMT_CS16, 1024000, freq, fpdm)
        for i, s in enumerate(streams):
            ref = o.run(s, 4, 1024000, freq, fpdm)
            assert any(p["type"] == 2 and p["num_pulses"] >= 600 for p in ref["packages"])
            check(gpu[i], ref, f"fsk overflow {i} fpdm {fpdm}")
    streams = [synth.fsk_burst_stream(7, 2600, bit_us=200.0, n_samples=1 << 18, rate=250000, cu8=True, dev_hz=30e3)]
    for freq in (868000000, 433920000):
        gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, freq)
        ref = o.run(streams[0], 2, 250000, freq)
        assert any(p["type"] == 2 and p["num_pulses"] >= 600 for p in ref["packages"])
        check(gpu[0], ref, f"fsk overflow cu8 {freq}")


def test_rates_and_formats_round_1_never_compared(ctx, devices):
    """2.048 MS/s cu8, OOK in cs16 captures (two rates), FSK packages out of a cu8 capture (both detectors)."""
    o = oracle_for(devices)
    streams = [synth.ook_stream(61, n_samples=1 << 20, rate=2048000, n_bursts=4, kinds=("nice", "manchester"))]
    gpu = run_gpu(ctx, streams, lib.FMT_CU8, 2048000, 433920000)
    check(gpu[0], o.run(streams[0], 2, 2048000, 433920000), "2.048 MS/s cu8")
    streams = [synth.cu8_to_cs16(synth.ook_stream(62, n_samples=1 << 19, rate=1024000, n_bursts=3, kinds=("nice", "manchester")))]
    gpu = run_gpu(ctx, streams, lib.FMT_CS16, 1024000, 433920000)
    check(gpu[0], o.run(streams[0], 4, 1024000, 433920000), "cs16 OOK 1.024 MS/s")
    streams = [synth.cu8_to_cs16(synth.ook_stream(63, n_samples=1 << 18, n_bursts=3, kinds=("nice", "manchester", "silvercrest")), gain=200)]
    gpu = run_gpu(ctx, streams, lib.FMT_CS16, 250000, 433920000)
    check(gpu[0], o.run(streams[0], 4, 250000, 433920000), "cs16 OOK 250 kS/s")
    streams = [synth.fsk_burst_stream(64, 600, bit_us=400.0, n_samples=1 << 18, rate=250000, cu8=True, dev_hz=30e3)]
    for freq in (433920000, 868000000):
        gpu = run_gpu(ctx, streams, lib.FMT_CU8, 250000, freq)
        ref = o.run(streams[0], 2, 250000, freq)
        assert any(p["type"] == 2 for p in ref["packages"])
        check(gpu[0], ref, f"cu8 FSK {freq}")


def test_front_guesses_verified_and_repaired(devices, monkeypatch):
    """k_front starts every chunk from a GUESS of the AM filter state; a wrong guess must be caught -- inside a
    tile by the warp's verify / redo chain, at a tile start by k_detect's hand-over check and repair.
    R433B_SPOIL_FRONT makes the guesses wrong on purpose (1: the first chunk of every tile, 2: every chunk):
    stage arrays, packages and events must not change, and the counters must show that the paths ran."""
    streams = [synth.ook_stream(61, n_samples=1 << 17, n_bursts=2), synth.ook_stream(62, n_samples=(1 << 17) - 16 * 37, n_bursts=2)]
    o = oracle_for(devices)
    refs = [o.run(s, 2) for s in streams]
    for spoil in (1, 2):
        monkeypatch.setenv("R433B_SPOIL_FRONT", str(spoil))
        c = lib.Context(0)
        monkeypatch.delenv("R433B_SPOIL_FRONT")
        c.set_devices(devices)
        gpu = run_gpu(c, streams, lib.FMT_CU8, 250000, 433920000)
        tm = c.timing()
        c.close()
        for i in range(len(streams)):
            check(gpu[i], refs[i], f"spoil {spoil} stream {i}")
        tiles = sum((len(s) // 2 + 2047) // 2048 for s in streams)
        assert tm["front_repairs"] >= tiles - len(streams) - 2, tm
        if spoil == 2:
            assert tm["front_redone"] >= 20 * tiles, tm
