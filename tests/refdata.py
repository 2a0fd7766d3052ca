"""Outputs of the unmodified reference (merbanan/rtl_433 25.12, compiled by oracle/Makefile into oracle/_ref) that the
tests compare with, stored in tests/golden/reference.json so that every comparison runs without the reference.

recorded(key, compute) returns the stored answer for `key`.  With R433B_RECORD_REFERENCE=1 it calls compute() instead
-- which asks the compiled reference -- stores the answer and rewrites the file when the process ends
(tools/record_reference.sh).  Large answers are stored as digests (helpers.digest, helpers.fingerprint): the
comparison stays exact."""
import atexit
import json
import os

import helpers

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference.json")
RECORD = os.environ.get("R433B_RECORD_REFERENCE") == "1"
_data = None


def _load():
    global _data
    if _data is None:
        _data = {}
        if os.path.exists(PATH):
            with open(PATH) as f:
                _data = json.load(f)
    return _data


def recorded(key, compute):
    data = _load()
    if RECORD:
        data[key] = json.loads(json.dumps(compute()))  # exactly what a later run reads back
    elif key not in data:
        raise KeyError(f"{key}: no recorded reference output in {PATH} (tools/record_reference.sh records it)")
    return data[key]


@atexit.register
def _save():
    if RECORD and _data is not None:
        with open(PATH, "w") as f:
            f.write("{\n" + ",\n".join(json.dumps(k) + ": " + json.dumps(_data[k], separators=(",", ":"))
                                       for k in sorted(_data)) + "\n}\n")


class LiveRef:
    """A refh.Ref constructed on first use, so that tests can name it in their compute() callbacks and only a
    recording run ever loads the compiled reference."""

    def __init__(self, setup=None, **kw):
        self._setup, self._kw, self._ref = setup, kw, None

    def __getattr__(self, name):
        if self._ref is None:
            from oracle import refh
            self._ref = refh.Ref(**self._kw)
            if self._setup:
                self._setup(self._ref)
        return getattr(self._ref, name)

    def close(self):
        if self._ref is not None:
            self._ref.close()
            self._ref = None


def ref_run(key, x, *args, devices=None, **kw):
    """Fingerprint of the reference's run over one capture: default devices, or `devices` registered as custom ones."""
    def compute():
        from oracle import refh
        r = refh.Ref(store_bitbuffers=False, store_stages=True)
        try:
            if devices is None:
                r.register_defaults()
            else:
                for d in devices:
                    r.register_custom(**d)
            return helpers.fingerprint(r.run(x, *args, **kw))
        finally:
            r.close()
    return recorded(key, compute)


DEVICE_KEYS = ("protocol_num", "modulation", "short_width", "long_width", "reset_limit", "gap_limit", "sync_width",
               "tolerance", "priority")


def device_rows(devs):
    return [[d[k] for k in DEVICE_KEYS] for d in devs]


def registered_devices(which):
    """[count, digest of device_rows()] of the reference's registered r_device table: 'defaults' (what it enables by
    default) or 'all' (every protocol, in protocol order)."""
    def compute():
        from oracle import refh
        r = refh.Ref(store_bitbuffers=False)
        try:
            if which == "defaults":
                r.register_defaults()
            else:
                for p in r.protocols():
                    r.register(p["protocol_num"])
            devs = r.registered()
            return [len(devs), helpers.digest(device_rows(devs))]
        finally:
            r.close()
    return recorded(f"registered/{which}", compute)
