"""The GPU parity tests run on a box WITHOUT a GPU: the engine's CUDA sources, unmodified, are compiled with g++
against a CPU emulation of the CUDA execution model (tests/emu: one fibre per CUDA thread, real barriers, shared
memory, shuffles) into tests/_build/libnrsc5_b200_emu.so, and the very test functions of tests/test_gpu_*.py are
run against that library.

What this proves and what it does not: the kernels' logic - indexing, work split, barrier placement (a missing or
divergent barrier deadlocks the emulator, which reports it instead of hanging a device), the host side of the C
ABI - is exercised bit for bit against the oracle on the CPU tier.  It says nothing about speed, and floating
point can differ from the GPU's in the last place (glibc's sincosf/atan2f, exact instead of approximate division),
so the `-m gpu` run of the same tests on a B200 remains the parity gate.  The emulator is test infrastructure: the
product library (nrsc5_b200/build.py, nvcc) has no CPU path.
"""
import os
import subprocess
import sys

import pytest

import common
import port

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))

pytestmark = pytest.mark.skipif(not port.available(), reason="oracle/_ref/liboracle.so not built")


@pytest.fixture(scope="module", autouse=True)
def emulated_engine():
    import build_emu
    from nrsc5_b200 import engine as eng
    so = build_emu.build()
    saved = (eng.lib_path, eng._lib)
    eng.lib_path = lambda: so
    eng._lib = None
    yield
    eng.lib_path, eng._lib = saved


import test_gpu_am as _am            # noqa: E402
import test_gpu_chain as _chain      # noqa: E402
import test_gpu_edge as _edge        # noqa: E402
import test_zz_gpu_l2 as _l2         # noqa: E402
import test_gpu_modes as _modes      # noqa: E402
import test_gpu_stages as _stages    # noqa: E402

# kernel-level
test_halfband_bit_exact = _stages.test_halfband_bit_exact
test_fft2048_matches_fp64 = _stages.test_fft2048_matches_fp64
test_viterbi_random_soft_bit_exact = _stages.test_viterbi_random_soft_bit_exact
test_viterbi_saturating_and_noisy = _stages.test_viterbi_saturating_and_noisy
test_viterbi_fast_path_and_fallback_agree = _stages.test_viterbi_fast_path_and_fallback_agree
test_viterbi_p1_length_bit_exact = _stages.test_viterbi_p1_length_bit_exact
test_rs_decode_bit_exact = _stages.test_rs_decode_bit_exact
test_viterbi_k9_equals_the_reference_decoder = _stages.test_viterbi_k9_equals_the_reference_decoder


def test_rs_beyond_the_correction_radius_equals_reference():
    nfail, ncorr = _stages.rs_beyond_radius(6000)         # (120 000 words on the B200)
    assert nfail > 5000


# whole chain, FM
test_synth_pdus_bit_exact = _chain.test_synth_pdus_bit_exact
test_mp3_p1_pids_p3_bit_exact = _chain.test_mp3_p1_pids_p3_bit_exact
test_service_modes_bit_exact = _modes.test_service_modes_bit_exact
test_mixed_service_modes_in_one_engine = _modes.test_mixed_service_modes_in_one_engine
test_chunked_push_matches_single_push = _chain.test_chunked_push_matches_single_push
test_drain_all_equals_per_stream_drain = _chain.test_drain_all_equals_per_stream_drain
test_endless_stream_is_trimmed_to_the_input_buffer = _chain.test_endless_stream_is_trimmed_to_the_input_buffer
test_cs16_input_equals_cu8_input = _chain.test_cs16_input_equals_cu8_input
test_multi_stream_independent = _chain.test_multi_stream_independent
test_pipelined_use_equals_synchronous_decode = _chain.test_pipelined_use_equals_synchronous_decode
test_pids_crc_verdicts_on_valid_frames = _chain.test_pids_crc_verdicts_on_valid_frames
# L2 framing on the device
test_l2_frames_equal_oracle = _l2.test_l2_frames_equal_oracle
test_l2_frames_mutated_equal_oracle = _l2.test_l2_frames_mutated_equal_oracle
test_l2_malformed_pdus_stay_in_bounds = _l2.test_l2_malformed_pdus_stay_in_bounds
test_l2_rare_branches = _l2.test_l2_rare_branches
test_l2_frames_of_sample_xz = _l2.test_l2_frames_of_sample_xz
test_chain_with_l2_on_device = _l2.test_chain_with_l2_on_device
test_mp3_chain_l2_records_follow_their_frames = _l2.test_mp3_chain_l2_records_follow_their_frames
test_am_chain_with_l2_on_device = _l2.test_am_chain_with_l2_on_device
test_am_rewind_repeats_the_decode = _l2.test_am_rewind_repeats_the_decode
test_mp3_chain_with_l2_content_in_p3_frames = _l2.test_mp3_chain_with_l2_content_in_p3_frames
test_service_mode_chain_l2_call_order = _l2.test_service_mode_chain_l2_call_order
# awkward inputs
test_dropout_and_reacquisition = _edge.test_dropout_and_reacquisition
test_stream_starting_mid_frame_mp3 = _edge.test_stream_starting_mid_frame_mp3
test_noise_only_and_short_inputs = _edge.test_noise_only_and_short_inputs
test_push_misuse_is_refused = _edge.test_push_misuse_is_refused
# whole chain, AM
test_am_pdus_bit_exact = _am.test_am_pdus_bit_exact
test_am_streams_independent_and_chunked = _am.test_am_streams_independent_and_chunked
test_am_cu8_input_bit_exact = _am.test_am_cu8_input_bit_exact


def test_reverse_thread_order_gives_the_same_results():
    """The same library with EMU_ORDER=reverse: threads of a block and blocks of a grid are scheduled from the last
    to the first.  A result that depended on the order in which threads run between two barriers would be a race
    on the GPU; a subset of the parity tests must pass unchanged.  (The order is fixed per process, hence the
    subprocess.)"""
    env = dict(os.environ, EMU_ORDER="reverse")
    sel = ("mp1_cfo-300_awgn12 or mp11 or ma3_noisy or viterbi_fast_path or (am_cu8_input_bit_exact and 2) or "
           "(l2_frames_equal_oracle and p1_fm_fixed_b) or mp3_chain_l2")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-k", sel, "-p", "no:cacheprovider"],
                       env=env, cwd=os.path.dirname(HERE), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout


# ---- the drop-in libnrsc5.so on the emulated engine: the reference's unmodified host side + our input seam, linked
# ---- against the emulator build of the engine instead of the CUDA one (same objects, other -l) ----
@pytest.fixture(scope="module")
def emulated_dropin(emulated_engine):
    import build_emu
    import test_dropin
    objdir = common.DROPIN_OBJDIR
    if not os.path.isdir(objdir):
        pytest.skip("drop-in objects not built (needs the reference tree at build time)")
    objs = sorted(os.path.join(objdir, f) for f in os.listdir(objdir) if f.endswith(".o"))
    so = os.path.join(HERE, "_build", "libnrsc5_emu.so")
    emu = build_emu.build()
    subprocess.run(["gcc", "-shared", "-o", so, *objs, emu, "-Wl,-rpath," + os.path.dirname(emu), "-lm", "-lpthread"], check=True)
    saved = test_dropin.DROPIN
    test_dropin.DROPIN = so
    yield so
    test_dropin.DROPIN = saved


@pytest.mark.parametrize("device_l2", [1])       # 0 (the reference's frame.c on the host) is the path the B200 run covers
def test_dropin_events_match_reference_on_sample_xz(emulated_dropin, device_l2):
    import test_dropin
    test_dropin.test_dropin_events_match_reference_on_sample_xz(device_l2)
    os.environ.pop("NRSC5_B200_DEVICE_L2", None)


@pytest.mark.parametrize("psmi,fmt,device_l2", [(1, "cs16", 0), (1, "cs16", 1), (2, "cu8", 1)])
def test_dropin_am_matches_reference_events(emulated_dropin, psmi, fmt, device_l2):
    import test_dropin
    os.environ["NRSC5_B200_DEVICE_L2"] = str(device_l2)
    try:
        test_dropin.test_dropin_am_matches_reference_events(psmi, fmt)
    finally:
        os.environ.pop("NRSC5_B200_DEVICE_L2", None)
