"""The drop-in libnrsc5.so (reference host side + our input seam + the B200 engine) driven through the
reference's PUBLIC API must deliver the events the unmodified reference delivers - same kinds, same order,
identical HDC audio packets - on support/sample.xz (golden: tests/golden/api_sample_xz.json, made by
tests/golden/make_golden_api.py with the unmodified reference)."""
import json
import os
import subprocess

import pytest

import common
import nrsc5_api

DROPIN = os.path.join(common.ROOT, "nrsc5_b200", "dropin", "_build", "libnrsc5.so")
PUBLIC_API = ["nrsc5_get_version", "nrsc5_service_data_type_name", "nrsc5_program_type_name", "nrsc5_open",
              "nrsc5_open_file", "nrsc5_open_pipe", "nrsc5_open_rtltcp", "nrsc5_close", "nrsc5_start", "nrsc5_stop",
              "nrsc5_set_mode", "nrsc5_set_bias_tee", "nrsc5_set_direct_sampling", "nrsc5_set_freq_correction",
              "nrsc5_get_frequency", "nrsc5_set_frequency", "nrsc5_get_gain", "nrsc5_set_gain", "nrsc5_set_auto_gain",
              "nrsc5_set_callback", "nrsc5_pipe_samples_cu8", "nrsc5_pipe_samples_cs16"]


def test_dropin_exports_the_public_api():
    if not os.path.exists(DROPIN):
        pytest.skip("drop-in not built (needs the reference tree at build time)")
    out = subprocess.run(["nm", "-D", "--defined-only", DROPIN], capture_output=True, text=True).stdout
    names = {ln.split()[-1] for ln in out.splitlines() if ln.strip()}
    for n in PUBLIC_API:
        assert n in names, n
    # and none of the reference's hot-path translation units were linked in
    for n in ("acquire_process", "sync_push", "decode_push_pm", "nrsc5_conv_decode_p1", "firdecim_q15_create"):
        assert n not in names, n


@pytest.mark.gpu
def test_dropin_events_match_reference_on_sample_xz(device_l2=0):
    """device_l2 = 1 (the library's default): L2 framing on the GPU, REC_L2 replayed by the seam; 0
    (NRSC5_B200_DEVICE_L2=0): the reference's own frame.c on the host - this test.  Both must deliver the
    reference's events (the device variant is run from tests/test_zz_gpu_l2.py and, emulated, from
    tests/test_emu_engine.py)."""
    if not os.path.exists(DROPIN):
        pytest.skip("drop-in not built")
    os.environ["NRSC5_B200_DEVICE_L2"] = str(device_l2)
    try:
        raw = common.load_sample()
        if raw is None:
            pytest.skip("sample.xz not available on this box")
        g = common.golden("api_sample_xz.json")
        got = nrsc5_api.run(DROPIN, raw.tobytes())
        want = g["events"]
        assert [e[0] for e in got] == [e[0] for e in want]                  # kinds and order
        for a, b in zip(got, want):
            if a[0] == "HDC":
                assert a == b                                               # program, length, payload digest
            elif a[0] == "SYNC":
                assert a[2:] == b[2:] and abs(a[1] - b[1]) < 0.05
            elif a[0] == "MER":
                assert abs(a[1] - b[1]) < 0.05 and abs(a[2] - b[2]) < 0.05
            elif a[0] == "BER":
                assert abs(a[1] - b[1]) < 2e-4
    finally:
        os.environ.pop("NRSC5_B200_DEVICE_L2", None)


@pytest.mark.gpu
def test_dropin_cs16_pipe_matches_reference_events():
    """nrsc5_pipe_samples_cs16 (input_push_cs16): the exactly decimated sample.xz must produce the events of
    the cu8 capture (the chain after the decimator is the same)."""
    if not os.path.exists(DROPIN):
        pytest.skip("drop-in not built")
    raw = common.load_sample()
    if raw is None:
        pytest.skip("sample.xz not available on this box")
    from nrsc5_b200 import engine as eng
    cs16 = eng.halfband_fm(raw[: raw.size & ~3])
    got = nrsc5_api.run(DROPIN, cs16.tobytes(), chunk=32768, cs16=True)
    want = common.golden("api_sample_xz.json")["events"]
    assert [e[0] for e in got] == [e[0] for e in want]
    assert [e for e in got if e[0] == "HDC"] == [e for e in want if e[0] == "HDC"]


@pytest.mark.gpu
@pytest.mark.parametrize("psmi,fmt", [(1, "cs16"), (2, "cs16"), (1, "cu8"), (2, "cu8")])
def test_dropin_am_matches_reference_events(psmi, fmt):
    """AM through the public API (nrsc5_set_mode(NRSC5_MODE_AM), nrsc5_pipe_samples_cs16 / _cu8): the drop-in and
    the unmodified reference library deliver the same events on a synthetic MA1 / MA3 capture (the reference's events:
    tests/golden/api_am.json, made by tests/golden/make_golden_api_am.py)."""
    import reftap
    from nrsc5_b200 import synth_am
    if not os.path.exists(DROPIN):
        pytest.skip("drop-in not built")
    cap = synth_am.make_am_ma1(nframes=8, seed=30 + psmi, lead_in=222, carrier=8000.0, unit=40.0, cfo_hz=0.5, psmi=psmi,
                               flags=(1, 0, 1, 0))
    if fmt == "cs16":
        data, kw = cap.cs16.tobytes(), dict(chunk=32768, cs16=True)
    else:
        data, kw = synth_am.am_to_cu8(cap.cs16).tobytes(), dict(chunk=32768)
    want = common.golden("api_am.json")[f"psmi{psmi}_{fmt}"]
    if reftap.available():
        live = json.loads(json.dumps(nrsc5_api.run(reftap.REF_SO, data, am=True, **kw)))
        assert live == want, "the reference library disagrees with the golden file"
    got = nrsc5_api.run(DROPIN, data, am=True, **kw)
    assert [e[0] for e in want].count("SYNC") == 1 and [e[0] for e in want].count("BER") >= 2
    assert [e[0] for e in got] == [e[0] for e in want]
    for a, b in zip(got, want):
        if a[0] == "SYNC":
            assert a[2:] == b[2:] and abs(a[1] - b[1]) < 0.05           # psmi, pli, hppi, aabi, rdbi
        elif a[0] == "BER":
            assert abs(a[1] - b[1]) < 1e-6
        else:
            assert a == b
