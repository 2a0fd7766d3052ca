"""CPU: the kernels' own source (k_detect, k_slice, k_cf32_to_cs16 and the C ABI around them) executed by
the SIMT emulator (tests/emu.py, tests/simt/) under the SAME parity tests the GPU suite runs on the B200:
every test function below is imported from the `-m gpu` modules and compares, through the C ABI, with the
oracle (and the recorded outputs of the compiled reference).  Two lane schedules (ascending here, descending in
test_emu_reverse_schedule) catch a missing __syncwarp() in either direction."""
import os

import numpy as np
import pytest

import emu
import helpers
from oracle import orc
from rtl_433_b200 import lib, synth


@pytest.fixture(scope="module", autouse=True)
def emulated_library():
    """rtl_433_b200.lib points at the emulated build for the tests of this module only."""
    old = (lib.LIB_PATH, lib._lib)
    emu.use()
    yield
    lib.LIB_PATH, lib._lib = old


from test_gpu_parity import (ctx, devices,  # noqa: E402,F401  (fixtures)
                             test_against_compiled_reference, test_all_protocols_including_disabled,
                             test_cs8_input_is_cu8_plus_128, test_custom_piwm_raw_and_nrzs_devices,
                             test_fm_low_pass_override_and_wrapping_filter, test_fm_rebuild_after_constant_input,
                             test_front_guesses_verified_and_repaired, test_fsk_cs16_minmax_and_classic,
                             test_fsk_train_overflow_shifts_the_pulse_train,
                             test_magnitude_mode_and_fixed_level, test_ook_1200_pulse_end_of_package,
                             test_ook_cu8_default_devices, test_pipelined_time_slices_identical,
                             test_pipelined_ragged_files_on_a_uniform_stride,
                             test_priority_classes_stop_after_a_decode, test_ragged_lengths_and_small_blocks,
                             test_rates_and_formats_round_1_never_compared, test_silence_and_reference_vectors)
import test_pulse_io  # noqa: E402


def test_emu_loaded_packages_through_k_slice():
    """r433b_process_pulses (SURVEY 8(f4)) under the emulator: the body of the -m gpu test."""
    test_pulse_io.loaded_packages_through_k_slice()


def test_emu_reverse_schedule(devices):
    """Lanes scheduled in descending order: a lane that reads shared or global memory another lane has not
    written yet (missing __syncwarp) shows up as a wrong result in one of the two orders."""
    import subprocess
    import sys
    code = ("import os,sys;sys.path.insert(0,%r);sys.path.insert(0,%r);import emu;emu.use();import numpy as np;"
            "import helpers;from oracle import orc;from rtl_433_b200 import lib,synth;"
            "devs=lib.default_device_table();c=lib.Context(0);c.set_devices(devs);o=orc.Oracle(store_bitbuffers=False);o.add_devices(devs);"
            "bad=0\n"
            "for x,fmt,rate,freq in ((synth.ook_stream(3,n_samples=1<<18,n_bursts=2),2,250000,433920000),"
            "(synth.fsk_stream(1,n_samples=1<<18,n_bursts=2).view(np.uint8),4,1024000,433920000),"
            "(synth.fsk_stream(2,n_samples=1<<18,n_bursts=2).view(np.uint8),4,1024000,868000000)):\n"
            "    c.process(x,np.array([0,x.nbytes],np.uint64),fmt,rate,freq);c.fetch();"
            "bad+=len(helpers.compare_results(o.run(x,fmt,rate,freq),helpers.gpu_stream_results(c,0),'rev',stages=False))\n"
            "sys.exit(1 if bad else 0)") % (os.path.dirname(os.path.abspath(__file__)), emu.ROOT)
    env = dict(os.environ, SIMT_REVERSE="1")
    assert subprocess.call([sys.executable, "-c", code], env=env) == 0


import test_gates  # noqa: E402


def test_emu_gated_run_is_the_filtered_ungated_run():
    """Decoder length gates in k_slice (SURVEY 8(f1)) under the emulator: the body of the -m gpu test."""
    test_gates.gated_run_is_the_filtered_ungated_run()


@test_gates.needs_ref
def test_emu_decoders_behind_gates_and_threads():
    test_gates.decoders_behind_gates_and_threads()


import test_analyzer  # noqa: E402


def test_emu_analyzer_matches_the_reference():
    """k_analyze / k_slice_own (SURVEY 8(f3)) under the emulator: the body of the -m gpu test."""
    test_analyzer.analyzer_matches_the_reference()


def test_emu_submit_wait_ping_pong():
    test_gates.submit_wait_ping_pong()


def test_emu_slice_v1_still_exact(devices):
    """R433B_SLICE_V1=1 keeps the round-1 formulation of the slicer kernel (lanes = devices on one package) for A/B
    timing; it has to stay exact too."""
    import subprocess
    import sys
    code = ("import os,sys;sys.path.insert(0,%r);sys.path.insert(0,%r);import emu;emu.use();import numpy as np;"
            "import helpers;from oracle import orc;from rtl_433_b200 import lib,synth;"
            "devs=lib.default_device_table();c=lib.Context(0);c.set_devices(devs);c.set_gates(lib.default_gates(devs));"
            "o=orc.Oracle(store_bitbuffers=False);o.add_devices(devs);"
            "x=synth.ook_stream(3,n_samples=1<<18,n_bursts=2);"
            "c.process(x,np.array([0,x.nbytes],np.uint64),2,250000,433920000);r=c.fetch();"
            "g=helpers.gpu_stream_results(c,0);w=o.run(x,2);gates=lib.default_gates(devs);"
            "keep=[(e['package'],e['dev'],e['hash']) for e in g['events']];"
            "c.set_gates(None);c.process(x,np.array([0,x.nbytes],np.uint64),2,250000,433920000);c.fetch();"
            "full=helpers.gpu_stream_results(c,0);"
            "bad=len(helpers.compare_results(w,full,'v1',stages=False));"
            "want=[(e['package'],e['dev'],e['hash']) for e in full['events'] if not (e['num_rows']>=1 and e['max_bits']<gates[e['dev']][0])];"
            "sys.exit(1 if bad or keep!=want or not keep else 0)") % (os.path.dirname(os.path.abspath(__file__)), emu.ROOT)
    env = dict(os.environ, R433B_SLICE_V1="1")
    assert subprocess.call([sys.executable, "-c", code], env=env) == 0


def test_emu_edge_cases_of_the_widening_rows():
    test_analyzer.edge_cases_of_the_widening_rows()


def test_emu_analyzer_fuzz():
    test_analyzer.analyzer_fuzz()


def test_emu_analyzer_golden():
    test_analyzer.analyzer_golden()
