#!/bin/sh
# Records what the unmodified reference answers to every question the tests put to it into
# tests/golden/reference.json (tests/refdata.py).  Needs oracle/_ref, which build() compiles when the reference's
# sources are at hand.  The -m gpu tests that ask the reference have emulator twins in tests/test_emu_parity.py,
# so a machine without a GPU records all of it.  Extra arguments go to pytest (e.g. one test file).
cd "$(dirname "$0")/.." || exit 1
[ -f oracle/_ref/libr433ref.so ] || { echo "oracle/_ref/libr433ref.so is missing: build it first" >&2; exit 1; }
R433B_RECORD_REFERENCE=1 exec python -m pytest -q -m "not gpu" "${@:-tests}"
