"""Shared test helpers: result comparison, the CPU unit-test driver for the product's
__host__ __device__ functions (tests/host_core.cpp), reference device tables."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

from oracle import refh
from oracle.refh import BITBUFFER_DTYPE, Event, Package, _pkg_dict

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HOSTCORE_SO = os.path.join(HERE, "_build", "libhostcore.so")

PKG_INT_KEYS = ["type", "block", "offset", "sample_rate", "start_ago", "end_ago", "num_pulses", "ook_low_estimate",
                "ook_high_estimate", "fsk_f1_est", "fsk_f2_est", "pulse_count", "num_events"]
PKG_FLOAT_KEYS = ["freq1_hz", "freq2_hz", "centerfreq_hz", "range_db", "rssi_db", "snr_db", "noise_db",
                  "sample_file_pos"]


def compare_results(a, b, tag="", floats=True, stages=True):
    """Exact comparison of two result dicts (packages, events by hash, stage arrays).
    Returns a list of human-readable differences (empty == identical)."""
    diffs = []
    if len(a["packages"]) != len(b["packages"]):
        diffs.append(f"{tag} package count {len(a['packages'])} != {len(b['packages'])}")
    for i, (p, q) in enumerate(zip(a["packages"], b["packages"])):
        keys = PKG_INT_KEYS + (PKG_FLOAT_KEYS + ["depth_bits"] if floats else [])
        for k in keys:
            if p[k] != q[k]:
                diffs.append(f"{tag} package {i} {k}: {p[k]} != {q[k]}")
        if not np.array_equal(p["pulse"], q["pulse"]) or not np.array_equal(p["gap"], q["gap"]):
            diffs.append(f"{tag} package {i}: pulse/gap widths differ")
    if len(a["events"]) != len(b["events"]):
        diffs.append(f"{tag} event count {len(a['events'])} != {len(b['events'])}")
    bad = 0
    for i, (e, f) in enumerate(zip(a["events"], b["events"])):
        if (e["package"], e["dev"], e["hash"]) != (f["package"], f["dev"], f["hash"]):
            bad += 1
            if bad <= 3:
                diffs.append(f"{tag} event {i}: (pkg {e['package']}, dev {e['dev']}) vs (pkg {f['package']}, dev {f['dev']})"
                             f" hash {'same' if e['hash'] == f['hash'] else 'differs'}")
    if bad > 3:
        diffs.append(f"{tag} ... {bad} events differ in total")
    if stages:
        for k in ("am", "fm"):
            if k in a and k in b and not np.array_equal(a[k], b[k]):
                d = np.nonzero(a[k] != b[k])[0] if len(a[k]) == len(b[k]) else []
                diffs.append(f"{tag} stage {k} differs (len {len(a[k])} vs {len(b[k])}) first at {list(d[:3])}")
    return diffs


def digest(obj):
    """Short SHA-256 of an array (its bytes) or of a JSON-able value (numpy scalars as Python numbers)."""
    if isinstance(obj, np.ndarray):
        data = np.ascontiguousarray(obj).tobytes()
    else:
        data = json.dumps(obj, sort_keys=True, default=lambda v: v.item()).encode()
    return hashlib.sha256(data).hexdigest()[:16]


def fingerprint(res):
    """A result dict in the compact, exact form tests/golden/reference.json stores: package headers in full, widths,
    events and stage arrays as digests."""
    fp = {"packages": [dict({k: p[k] for k in PKG_INT_KEYS + PKG_FLOAT_KEYS + ["depth_bits"]},
                            widths=digest(np.concatenate([np.asarray(p["pulse"], np.int32), np.asarray(p["gap"], np.int32)])))
                       for p in res["packages"]],
          "events": len(res["events"]),
          "events_digest": digest(np.array([(e["package"], e["dev"], e["hash"]) for e in res["events"]],
                                           dtype=[("p", "<u4"), ("d", "<u4"), ("h", "<u8")]))}
    for k in ("am", "fm"):
        if k in res:
            fp[k] = digest(np.asarray(res[k], np.int16))
    return json.loads(json.dumps(fp, default=lambda v: v.item()))


def compare_fingerprint(want, got, tag="", floats=True, stages=True):
    """compare_results() for a recorded fingerprint `want` and a result dict `got`."""
    g = fingerprint(got)
    diffs = []
    if len(want["packages"]) != len(g["packages"]):
        diffs.append(f"{tag} package count {len(want['packages'])} != {len(g['packages'])}")
    for i, (p, q) in enumerate(zip(want["packages"], g["packages"])):
        for k in PKG_INT_KEYS + (PKG_FLOAT_KEYS + ["depth_bits"] if floats else []) + ["widths"]:
            if p[k] != q[k]:
                diffs.append(f"{tag} package {i} {k}: {p[k]} != {q[k]}")
    if (want["events"], want["events_digest"]) != (g["events"], g["events_digest"]):
        diffs.append(f"{tag} events differ: {want['events']} != {g['events']} or their digest")
    if stages:
        for k in ("am", "fm"):
            if k in want and k in g and want[k] != g[k]:
                diffs.append(f"{tag} stage {k} differs")
    return diffs


def events_digest(events):
    """[count, digest] of a slicer's output: [(device index, bitbuffer record)]."""
    return [len(events), digest(np.concatenate([np.frombuffer(np.uint32(d).tobytes() + bb.tobytes(), np.uint8)
                                                for d, bb in events]) if events else np.zeros(0, np.uint8))]


def default_devices():
    """The reference's default-enabled r_device table (335 entries) as dicts, from the committed
    data file (generated by tools/extract_devices.py from the reference)."""
    with open(os.path.join(ROOT, "rtl_433_b200", "data", "devices_25.12.json")) as f:
        return [d for d in json.load(f)["devices"] if d["disabled"] == 0]


def build_hostcore():
    src = os.path.join(HERE, "host_core.cpp")
    deps = [src] + [os.path.join(ROOT, "rtl_433_b200", "csrc", n) for n in
                    ("r433b_core.cuh", "r433b_slice.cuh", "r433b_host.hpp")]
    if os.path.exists(HOSTCORE_SO) and all(os.path.getmtime(HOSTCORE_SO) >= os.path.getmtime(d) for d in deps):
        return HOSTCORE_SO
    os.makedirs(os.path.dirname(HOSTCORE_SO), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-x", "c++", src,
                           "-o", HOSTCORE_SO])
    return HOSTCORE_SO


class DevDesc(C.Structure):
    _fields_ = [("modulation", C.c_uint32), ("short_width", C.c_float), ("long_width", C.c_float),
                ("reset_limit", C.c_float), ("gap_limit", C.c_float), ("sync_width", C.c_float),
                ("tolerance", C.c_float), ("priority", C.c_uint32)]

    @classmethod
    def of(cls, d):
        return cls(d["modulation"], d["short_width"], d["long_width"], d["reset_limit"], d.get("gap_limit", 0.0),
                   d.get("sync_width", 0.0), d.get("tolerance", 0.0), d.get("priority", 0))


class HostCore:
    """tests/host_core.cpp: the product's per-sample functions run sequentially on the CPU."""

    def __init__(self, store_bitbuffers=True, store_stages=False):
        L = C.CDLL(build_hostcore())
        L.hc_create.restype = C.c_void_p
        for n in ("hc_packages", "hc_events", "hc_bitbuffers"):
            getattr(L, n).restype = C.c_void_p
            getattr(L, n).argtypes = [C.c_void_p]
        for n, t in (("hc_pulse_pool", C.c_int32), ("hc_gap_pool", C.c_int32), ("hc_am", C.c_int16), ("hc_fm", C.c_int16)):
            getattr(L, n).restype = C.POINTER(t)
            getattr(L, n).argtypes = [C.c_void_p]
        for n in ("hc_num_packages", "hc_num_events", "hc_num_bitbuffers", "hc_num_stage"):
            getattr(L, n).restype = C.c_size_t
            getattr(L, n).argtypes = [C.c_void_p]
        L.hc_destroy.argtypes = [C.c_void_p]
        L.hc_set_capture.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.hc_set_levels.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float]
        L.hc_set_fm_low_pass.argtypes = [C.c_void_p, C.c_float]
        L.hc_add_device.argtypes = [C.c_void_p, C.POINTER(DevDesc)]
        L.hc_slice.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        L.hc_run_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32]
        self.L = L
        self.h = C.c_void_p(L.hc_create())
        L.hc_set_capture(self.h, int(store_bitbuffers), int(store_stages))

    def close(self):
        if self.h:
            self.L.hc_destroy(self.h)
            self.h = None

    def add_devices(self, devs):
        for d in devs:
            dd = DevDesc.of(d)
            self.L.hc_add_device(self.h, C.byref(dd))

    def set_levels(self, use_mag_est=0, level_limit=0.0, min_level=-12.1442, min_snr=9.0):
        self.L.hc_set_levels(self.h, use_mag_est, level_limit, min_level, min_snr)

    def set_fm_low_pass(self, v):
        self.L.hc_set_fm_low_pass(self.h, v)

    def slice(self, package_type, sample_rate, pulse, gap):
        """All registered devices on one pulse train -> [(dev, bitbuffer record)] in dispatch order."""
        pulse = np.ascontiguousarray(pulse, np.int32)
        gap = np.ascontiguousarray(gap, np.int32)
        L, h = self.L, self.h
        n = L.hc_slice(h, package_type, sample_rate, len(pulse), pulse.ctypes.data, gap.ctypes.data)
        if not n:
            return []
        ev = C.cast(L.hc_events(h), C.POINTER(Event))
        bbs = np.frombuffer((C.c_uint8 * (n * 6604)).from_address(L.hc_bitbuffers(h)), dtype=BITBUFFER_DTYPE).copy()
        return [(ev[i].dev, bbs[ev[i].bb_idx]) for i in range(n)]

    def run(self, iq, sample_size, samp_rate=250000, center_freq=433920000, fpdm=2, block_bytes=0):
        iq = np.ascontiguousarray(iq)
        L, h = self.L, self.h
        L.hc_run_stream(h, iq.ctypes.data, iq.nbytes, sample_size, samp_rate, center_freq, fpdm, block_bytes)
        npk, nev, nbb, nst = L.hc_num_packages(h), L.hc_num_events(h), L.hc_num_bitbuffers(h), L.hc_num_stage(h)
        pk = C.cast(L.hc_packages(h), C.POINTER(Package))
        npool = sum(pk[i].pulse_count for i in range(npk))
        if npool:
            pulses = np.ctypeslib.as_array(L.hc_pulse_pool(h), (npool,)).copy()
            gaps = np.ctypeslib.as_array(L.hc_gap_pool(h), (npool,)).copy()
        else:
            pulses = gaps = np.zeros(0, np.int32)
        packages = [_pkg_dict(pk[i], pulses, gaps) for i in range(npk)]
        ev = C.cast(L.hc_events(h), C.POINTER(Event))
        bbs = None
        if nbb:
            bbs = np.frombuffer((C.c_uint8 * (nbb * 6604)).from_address(L.hc_bitbuffers(h)), dtype=BITBUFFER_DTYPE).copy()
        events = [{"package": ev[i].package, "dev": ev[i].dev, "ret": ev[i].ret, "hash": ev[i].hash,
                   "bitbuffer": bbs[ev[i].bb_idx] if (bbs is not None and ev[i].bb_idx != 0xFFFFFFFF) else None}
                  for i in range(nev)]
        res = {"packages": packages, "events": events}
        if nst:
            res["am"] = np.ctypeslib.as_array(L.hc_am(h), (nst,)).copy()
            res["fm"] = np.ctypeslib.as_array(L.hc_fm(h), (nst,)).copy()
        return res


def _hostcore_lib():
    L = C.CDLL(build_hostcore())
    L.hc_collector_create.restype = C.c_void_p
    L.hc_collector_create.argtypes = [C.c_int]
    L.hc_collector_destroy.argtypes = [C.c_void_p]
    L.hc_collector_clear.argtypes = [C.c_void_p]
    L.hc_collector_count.restype = C.c_size_t
    L.hc_collector_count.argtypes = [C.c_void_p]
    L.hc_collector_events.restype = C.c_void_p
    L.hc_collector_events.argtypes = [C.c_void_p]
    L.hc_collector_bitbuffers.restype = C.c_void_p
    L.hc_collector_bitbuffers.argtypes = [C.c_void_p]
    return L


def gpu_stream_results(ctx, stream, store_bitbuffers=False):
    """Replay one stream of a fetched batch through r433b_dispatch() with a native collector
    (tests/host_core.cpp) -> the dict shape oracle.refh.Ref.run() returns."""
    L = _hostcore_lib()
    col = C.c_void_p(L.hc_collector_create(int(store_bitbuffers)))
    try:
        packages, index = ctx.packages_of(stream)
        local = {g: i for i, g in enumerate(index)}
        ctx.dispatch_native(stream, C.cast(L.hc_collect_cb, C.c_void_p).value, col)
        n = L.hc_collector_count(col)
        ev = C.cast(L.hc_collector_events(col), C.POINTER(Event))
        bbs = None
        if store_bitbuffers and n:
            bbs = np.frombuffer((C.c_uint8 * (n * 6604)).from_address(L.hc_collector_bitbuffers(col)),
                                dtype=BITBUFFER_DTYPE).copy()
        events = []
        for i in range(n):
            li = local[ev[i].package]
            packages[li]["num_events"] += 1
            events.append({"package": li, "dev": ev[i].dev, "ret": 0, "hash": ev[i].hash,
                           "num_rows": (ev[i].ret >> 16) & 0xffff, "max_bits": ev[i].ret & 0xffff,
                           "bitbuffer": bbs[ev[i].bb_idx] if bbs is not None else None})
        return {"packages": packages, "events": events}
    finally:
        L.hc_collector_destroy(col)
