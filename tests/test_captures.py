"""Capture-file ingest (rtl_433_b200/captures.py): file-name metadata like file_info_parse_filename()
(src/fileformat.c:298), batching of ragged files, and -- on a GPU -- a replay of files on disk."""
import os

import numpy as np
import pytest

import refdata
from oracle import orc, refh
from rtl_433_b200 import captures, lib, synth

NAMES = ["g001_433.92M_250k.cu8", "x.cu8", "868M_1024k.cs16", "sdr_315M_1000k.cs8", "file_433920000Hz_250000sps.cu8",
         "am:s16:path/file.ext", "cs16:weird_2.4G_2048k.bin", "foo_868.3M_1MHz_2Msps.cs16", "a.b.c",
         "capture_433.92MHz_250ksps.cu8", "g5_915M_250k.complex16u", "iq:cu8:some/dir_1.2/file", "tx_10.k_433M.cu8",
         "data_433.5M_3200k.cf32", "noext_250k_433M", "dir.v2/rec_1024K_868.35m.CS16", "9.cu8", "a_12345.cu8"]


@pytest.mark.parametrize("name", NAMES)
def test_filename_metadata_matches_reference(name):
    want = refdata.recorded(f"parse_filename/{name}", lambda: refh.parse_filename(name))
    got = captures.parse_capture_name(name)
    assert got["sample_rate"] == want["sample_rate"]
    assert got["center_frequency"] == want["center_frequency"]
    if want["format"] is not None:
        assert got["format"] == want["format"]


def test_load_batches_groups_and_aligns(tmp_path):
    a = synth.nice_flor_s_file()
    b = synth.silvercrest_file()[:-6]          # not a multiple of 16 bytes
    c = synth.fsk_stream(1, n_samples=1 << 16, n_bursts=0)
    pa, pb, pc = tmp_path / "a_433.92M_250k.cu8", tmp_path / "b_250k.cu8", tmp_path / "c_868M_1024k.cs16"
    a.tofile(pa), b.tofile(pb), c.tofile(pc)
    batches = captures.load_batches([str(pa), str(pc), str(pb)])
    assert [(x["format"], x["sample_rate"], x["center_frequency"]) for x in batches] == [
        ("cu8", 250000, 433920000), ("cs16", 1024000, 868000000)]
    cu8 = batches[0]
    assert cu8["files"] == [str(pa), str(pb)]
    assert list(cu8["lengths"]) == [a.nbytes, b.nbytes]
    assert all(int(o) % 16 == 0 for o in cu8["offsets"])
    # cf32: 8 bytes per sample, 32-byte aligned starts (the device turns it into cs16 at half the size)
    f = (c.astype(np.float32) / np.float32(32768))[: 2 * 1001]
    pf = tmp_path / "f_868M_1024k.cf32"
    f.tofile(pf)
    (fb,) = captures.load_batches([str(pf), str(pf)])
    assert (fb["format"], fb["abi_format"], fb["sample_rate"]) == ("cf32", lib.FMT_CF32, 1024000)
    assert list(fb["lengths"]) == [f.nbytes, f.nbytes] and all(int(o) % 32 == 0 for o in fb["offsets"])
    assert bytes(cu8["data"][int(cu8["offsets"][1]):int(cu8["offsets"][1]) + b.nbytes]) == b.tobytes()


@pytest.mark.gpu
def test_replay_files_on_gpu(tmp_path):
    """Files of different lengths, formats and rates in one call; rows as rtl_433 prints them."""
    files = {"nice_433.92M_250k.cu8": synth.nice_flor_s_file(), "silver_250k.cu8": synth.silvercrest_file()[:-6],
             "silver_250k.cs8": synth.silvercrest_file() ^ np.uint8(0x80),
             "fsk_868M_1024k.cs16": synth.fsk_stream(2, n_samples=1 << 17, n_bursts=1)}
    paths = []
    for name, arr in files.items():
        arr.tofile(tmp_path / name)
        paths.append(str(tmp_path / name))
    lines = []
    summary = captures.replay(paths, protocols=[1, 169], out=lines.append)
    text = "\n".join(lines)
    assert "{52}e7a760b94372e" in text          # tests/http-rtltcp-test.sh:35
    assert text.count("{33}7c2600020 {33}7c2600020 {33}7c2600020 {33}7c2600020") >= 2   # cu8 and cs8 copy
    assert {s["file"]: s["packages"] for s in summary}[paths[3]] >= 1
    # against the oracle for the ragged cu8 file
    devs = [d for d in lib.default_device_table(include_disabled=True) if d["protocol_num"] in (1, 169)]
    o = orc.Oracle(store_bitbuffers=False)
    o.add_devices(devs)
    want = o.run(files["silver_250k.cu8"], 2)
    got = [s for s in summary if s["file"] == paths[1]][0]
    assert got["packages"] == len(want["packages"]) and got["events"] == len(want["events"])


def _make_sigmf(path, meta_name, meta, data, extra=()):
    import io
    import json
    import tarfile
    with tarfile.open(path, "w", format=tarfile.USTAR_FORMAT) as tar:
        for name, payload in [(meta_name, json.dumps(meta).encode())] + list(extra) + [(meta_name[:-4] + "data", data)]:
            ti = tarfile.TarInfo(name)
            ti.size = len(payload)
            tar.addfile(ti, io.BytesIO(payload))


def test_sigmf_container_like_the_reference(tmp_path):
    """rate / frequency / start of the sample data as sigmf_reader_open() finds them (src/sigmf.c:336-434)."""
    x = synth.nice_flor_s_file()
    meta = {"global": {"core:datatype": "cu8", "core:sample_rate": 250000, "core:version": "1.0.0", "core:recorder": "t"},
            "captures": [{"core:sample_start": 0, "core:frequency": 433920000}, {"core:sample_start": 10, "core:frequency": 868300000.0}],
            "annotations": []}
    cases = []
    p1 = str(tmp_path / "one.sigmf")
    _make_sigmf(p1, "rec.sigmf-meta", meta, x.tobytes())
    cases.append(p1)
    p2 = str(tmp_path / "two_streams.sigmf")
    m2 = dict(meta, **{"global": dict(meta["global"], **{"core:sample_rate": 1024000.0})})
    _make_sigmf(p2, "dir/a.sigmf-meta", m2, x.tobytes()[:1000], extra=[("dir/readme.txt", b"hello" * 300)])
    cases.append(p2)
    for p in cases:
        want = refdata.recorded(f"sigmf_open/{os.path.basename(p)}", lambda: refh.sigmf_open(p))
        got = captures.read_sigmf(p)
        assert want["rc"] == 0
        assert (got["sample_rate"], got["center_frequency"], got["data_offset"]) == (want["sample_rate"], want["center_frequency"], want["data_offset"])
        raw = open(p, "rb").read()
        assert got["data"].tobytes() == raw[want["data_offset"]:]  # the block loop reads to the end of the archive
    b = captures.load_batches(["sigmf:" + p1, str(tmp_path / "missing_250k.cu8")][:1])
    assert (b[0]["format"], b[0]["sample_rate"], b[0]["center_frequency"]) == ("cu8", 250000, 868300000)
    assert bytes(b[0]["data"][:x.nbytes]) == x.tobytes()
