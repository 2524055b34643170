"""CPU tests pinning the oracle (the plain-C restatement in oracle/nrsc5_oracle.c)
against (1) the committed golden vectors produced by the unmodified reference
and (2) the reference's answers on further inputs, pinned by digest (tests/golden/reference_digests.json) and
recomputed by the reference itself (oracle/_ref/libnrsc5_ref.so) when it is present.
"""
import ctypes

import numpy as np
import pytest

import common
import port
import reftap
from nrsc5_b200 import synth

pytestmark = pytest.mark.skipif(not port.available(), reason="oracle/_ref/liboracle.so not built (run __graft_entry__.build())")


def _soft_fnv(log):
    return common.fnv1a32(b"".join(p["soft"].tobytes() for p in log.of(reftap.REC_SOFT_PM)))


@pytest.mark.parametrize("name", list(common.SYNTH_CASES))
def test_port_matches_golden_synth(name):
    g = common.golden("synth_fm.json")[name]
    cap = synth.make_fm_mp1(**common.SYNTH_CASES[name])
    if common.fnv1a32(cap.cu8[:1 << 20].tobytes()) != g["input_fnv"]:
        pytest.skip("numpy generator stream differs from the one the golden file was made with")
    log = port.decode(cap.cu8, want_soft=True)
    assert common.summarize(log) == g["events"]
    assert len(log.of(reftap.REC_SOFT_PM)) == g["soft_blocks"]
    assert _soft_fnv(log) == g["soft_fnv"]          # soft bits bit-identical to the reference
    # the receiver returns what the generator put in (sizes-independent round trip)
    got = [common.fnv1a32(b) for b in log.p1_frames]
    assert set(g["generated_p1_fnv"]) & set(got), "no generated frame was recovered"


def test_port_matches_golden_mp3():
    """MP3: 12 partitions per sideband, PX1 demap (incl. the unequalised block that reaches FINE sync),
    interleaver IV, P3 frames - everything the unmodified reference put into the golden file."""
    g = common.golden("synth_mp3.json")
    cap = synth.make_fm_mp3(**common.MP3_CASE)
    if common.fnv1a32(cap.cu8[:1 << 20].tobytes()) != g["input_fnv"]:
        pytest.skip("numpy generator stream differs from the one the golden file was made with")
    log = port.decode(cap.cu8, want_soft=True)
    assert common.summarize(log) == g["events"]
    assert _soft_fnv(log) == g["soft_fnv"]
    p3 = [common.fnv1a32(p["bits"]) for t, p in log.records if t == reftap.REC_FRAME and p["lc"] == 1]
    assert len(p3) >= 8 and set(p3) <= set(g["generated_p3_fnv"])     # round trip: only generated frames come out


@pytest.mark.parametrize("name", list(common.FM_MODE_CASES))
def test_port_matches_golden_service_modes(name):
    """MP2 (2304-bit P3 through interleaver IV with J=2, M=4), MP5 / MP6 (14 partitions per sideband in the Costas
    loops, the equaliser and the MER), MP11 (PX1 -> P3, PX2 -> P4 with the lower sideband's scale on both halves,
    sync.c:591-592): events, PDUs and soft bits identical to what the unmodified reference put into the golden file,
    and every P1 / P3 / P4 frame that comes out is one the generator put in."""
    g = common.golden("synth_fm_modes.json")[name]
    cap = synth.make_fm(**common.FM_MODE_CASES[name])
    if common.fnv1a32(cap.cu8[:1 << 20].tobytes()) != g["input_fnv"]:
        pytest.skip("numpy generator stream differs from the one the golden file was made with")
    log = port.decode(cap.cu8, want_soft=True)
    assert common.summarize(log) == g["events"]
    assert _soft_fnv(log) == g["soft_fnv"]
    for lc, key, least in ((0, "generated_p1_fnv", 2), (1, "generated_p3_fnv", 8 if g["generated_p3_fnv"] else 0),
                           (2, "generated_p4_fnv", 8 if g["generated_p4_fnv"] else 0)):
        got = [common.fnv1a32(p["bits"]) for t, p in log.records if t == reftap.REC_FRAME and p["lc"] == lc]
        assert len(got) >= least and set(got) <= set(g[key])


def _events_and_soft(log):
    return common.summarize(log), _soft_fnv(log)


@pytest.mark.parametrize("psmi", [2, 5, 11])
def test_port_matches_reference_live_service_modes(psmi):
    """The restatement against the unmodified reference on a capture that is not in the golden file (other seed,
    start block and noise), so that the pin does not rest on four inputs only."""
    cap = synth.make_fm(psmi=psmi, nframes=3, seed=100 + psmi, lead_in=1234, tail_blocks=2, cfo_hz=-150.0, noise_lsb=10.0,
                        start_bc=5)
    log = port.decode(cap.cu8, want_soft=True)
    common.assert_reference(f"fm_service_mode_psmi{psmi}", _events_and_soft(log),
                            lambda: _events_and_soft(reftap.decode(cap.cu8, want_soft=True)))


def test_port_matches_golden_sample():
    raw = common.load_sample()
    if raw is None:
        pytest.skip("sample.xz not available")
    g = common.golden("sample_xz.json")
    assert common.fnv1a32(raw[:1 << 20].tobytes()) == g["input_fnv"]
    log = port.decode(raw, want_soft=True)
    assert common.summarize(log) == g["events"]
    assert _soft_fnv(log) == g["soft_fnv"]
    kinds = [e[0] for e in g["events"]]
    # SURVEY §8c known answers
    assert kinds.count("S") == 2 and kinds.count("L") == 1 and kinds.count("M") == 10
    assert kinds.count("B") == 9 and kinds.count("F") == 9 and kinds.count("P") == 172


def test_port_cs16_matches_reference():
    """input_push_cs16: the reference and the restatement on the same pre-decimated FM capture."""
    cap = synth.make_fm_mp1(nframes=1, seed=21, lead_in=64, cfo_hz=50.0)
    cs16 = port.halfband_fm(cap.cu8[: cap.cu8.size & ~3])
    a = port.decode(cs16, want_soft=True)
    common.assert_reference("fm_cs16", _events_and_soft(a), lambda: _events_and_soft(reftap.decode(cs16, want_soft=True)))
    # and the decimator in front of it changes nothing: the cu8 capture gives the same PDUs
    c = port.decode(cap.cu8)
    assert [e for e in common.summarize(c) if e[0] in "FP"] == [e for e in common.summarize(a) if e[0] in "FP"]


def test_port_chunking_invariance():
    cap = synth.make_fm_mp1(nframes=1, seed=3, lead_in=10)
    a = port.decode(cap.cu8)
    b = port.decode(cap.cu8, chunk=32768)
    c = port.decode(cap.cu8, chunk=4 * 977)
    assert common.summarize(a) == common.summarize(b) == common.summarize(c)


def _records(log):
    """A decode's records, the reference tap's HDC records and the oracle's own PIDS CRC verdict left out, numpy
    arrays as bytes."""
    return [(t, {k: (v.tobytes() if isinstance(v, np.ndarray) else v) for k, v in r.items() if k != "crc_ok"})
            for t, r in log.records if t != reftap.REC_HDC]


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class TestAgainstReference:
    def test_full_chain_noisy(self):
        cap = synth.make_fm_mp1(nframes=1, seed=21, lead_in=123, cfo_hz=-150.0, noise_lsb=10.0)
        b = port.decode(cap.cu8, want_soft=True)
        common.assert_reference("fm_full_chain_noisy", _records(b), lambda: _records(reftap.decode(cap.cu8, want_soft=True)))

    def test_viterbi_k7_k9(self):
        rng = np.random.default_rng(1)
        soft7 = [rng.integers(-127, 128, 3 * n, dtype=np.int8) for n in (80, 2304, 4608)]
        soft9 = rng.integers(-1, 2, 3 * 3750, dtype=np.int8)
        e1, e23 = (0o561, 0o657, 0o711), (0o561, 0o753, 0o711)
        got = [port.viterbi(s).tobytes() for s in soft7]
        got += [port.viterbi(soft9, k=9, gens=e1).tobytes(), port.viterbi(soft9, k=9, gens=e23).tobytes()]

        def live():
            L = reftap.lib()
            outs = []
            for s in soft7:
                out = np.empty(s.size // 3, dtype=np.uint8)
                L.nrsc5_conv_decode_p3_p4(_ptr(s), _ptr(out), out.size)
                outs.append(out.tobytes())
            for f in (L.nrsc5_conv_decode_e1, L.nrsc5_conv_decode_e2_e3):
                out = np.empty(3750, dtype=np.uint8)
                f(_ptr(soft9), _ptr(out), 3750)
                outs.append(out.tobytes())
            return outs
        common.assert_reference("viterbi_k7_k9", got, live)

    def test_viterbi_saturation(self):
        # full-scale, perfectly consistent, unpunctured input drives the int16
        # path metrics into saturation between normalisations (SURVEY §7.3)
        rng = np.random.default_rng(5)
        u = rng.integers(0, 2, 4608, dtype=np.uint8)
        c = synth.conv_encode_tb(u).reshape(-1).astype(np.int16)
        s = ((2 * c - 1) * 127).astype(np.int8)
        got = port.viterbi(s)
        assert np.array_equal(got, u)

        def live():
            out = np.empty(4608, dtype=np.uint8)
            reftap.lib().nrsc5_conv_decode_p3_p4(_ptr(s), _ptr(out), 4608)
            return out.tobytes()
        common.assert_reference("viterbi_saturation", got.tobytes(), live)

    def test_halfband(self):
        rng = np.random.default_rng(2)
        cu8 = rng.integers(0, 256, 4 * 5000, dtype=np.uint8)
        cu8[:400] = 255                      # extremes
        cu8[400:800] = 0

        def live():
            L = reftap.lib()
            L.firdecim_q15_create.restype = ctypes.c_void_p
            L.halfband_q15_execute.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
            taps = (ctypes.c_float * 4)(0.6062333583831787, -0.13481467962265015, 0.032919470220804214, -0.00410953676328063)
            q = L.firdecim_q15_create(taps, 4)
            x = ((cu8.astype(np.int16) - 127) * 64).astype(np.int16)
            out = np.empty(2 * 5000, dtype=np.int16)
            for n in range(5000):
                L.halfband_q15_execute(q, _ptr(x[4 * n:]), _ptr(out[2 * n:]))
            return out.tobytes()
        common.assert_reference("halfband", port.halfband_fm(cu8).tobytes(), live)

    @staticmethod
    def _ref_rs(blocks):
        L = reftap.lib()
        L.init_rs_char.restype = ctypes.c_void_p
        L.decode_rs_char.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        rs = L.init_rs_char(8, 0x11D, 1, 1, 8)
        out = []
        for blk in blocks:
            ref = blk.copy()
            rc = L.decode_rs_char(rs, _ptr(ref), None, 0)
            out.append((rc, ref.tobytes()))
        return out

    @staticmethod
    def _port_rs(blocks):
        return [(rc, got.tobytes()) for rc, got in (port.rs_decode(blk) for blk in blocks)]

    def test_rs_decode(self):
        rng = np.random.default_rng(7)
        blocks = []
        for t in range(1500):
            hdr = np.frombuffer(synth.audio_pdu_header(rng=rng), dtype=np.uint8)
            blk = np.zeros(255, dtype=np.uint8)
            blk[254 - np.arange(96)] = hdr
            for p in rng.choice(255 if t % 3 == 0 else 96, t % 8, replace=False):
                blk[p if t % 3 == 0 else 254 - p] ^= rng.integers(1, 256)
            if t % 50 == 49:
                blk = rng.integers(0, 256, 255, dtype=np.uint8)
            blocks.append(blk)
        common.assert_reference("rs_decode", self._port_rs(blocks), lambda: self._ref_rs(blocks))

    def test_rs_decode_beyond_the_radius(self):
        """The words of tests/test_gpu_stages.py::test_rs_beyond_the_correction_radius_equals_reference (5..8 symbol
        errors): the oracle's decoder = the unmodified reference's decode_rs_char, including every mis-correction."""
        import test_gpu_stages
        blocks = test_gpu_stages._rs_words(np.random.default_rng(2024), 120000)
        got = self._port_rs(blocks)
        common.assert_reference("rs_decode_beyond_the_radius", got, lambda: self._ref_rs(blocks))
        assert sum(rc > 0 for rc, _ in got) > 50


def test_rs_roundtrip_without_reference():
    rng = np.random.default_rng(11)
    for ne in range(0, 6):
        hdr = np.frombuffer(synth.audio_pdu_header(rng=rng), dtype=np.uint8).copy()
        bad = hdr.copy()
        for p in rng.choice(96, ne, replace=False):
            bad[p] ^= rng.integers(1, 256)
        ok, fixed = port.fix_header(bad)
        if ne <= 4:
            assert ok == 1 and np.array_equal(fixed, hdr)
        else:
            assert ok == 0 or not np.array_equal(fixed, hdr)


def test_p1_sync_lost_predicate():
    rng = np.random.default_rng(4)
    good = synth.build_p1_frame_bits(rng, pci=synth.PCI_AUDIO, valid_header=True)
    assert port.p1_sync_lost(good) == (False, synth.PCI_AUDIO)
    bad = synth.build_p1_frame_bits(rng, pci=synth.PCI_AUDIO, valid_header=False)
    assert port.p1_sync_lost(bad) == (True, synth.PCI_AUDIO)
    fixed = synth.build_p1_frame_bits(rng, pci=synth.PCI_FIXED, valid_header=False)
    assert port.p1_sync_lost(fixed) == (False, synth.PCI_FIXED)


def test_pids_crc_verdict_restatements_agree():
    """oracle/nrsc5_oracle.c:orc_pids_crc12_ok (reference src/pids.c:52-86, 1032-1050) against the numpy restatement
    in nrsc5_b200/synth.py, on sample.xz's PIDS frames (143 of 172 valid) and on generated valid frames."""
    import numpy as np
    raw = common.load_sample()
    if raw is None:
        pytest.skip("sample.xz not available")
    log = port.decode(raw)
    frames = log.of(reftap.REC_PIDS)

    def verdict(packed):
        fb = np.unpackbits(np.frombuffer(packed, dtype=np.uint8))
        i = np.arange(80)
        p = fb[((i >> 3) << 3) + 7 - (i & 7)]
        return int(synth.pids_crc12(p) == int("".join(str(int(x)) for x in p[68:80]), 2))

    assert [p["crc_ok"] for p in frames] == [verdict(p["bits"]) for p in frames]
    assert sum(p["crc_ok"] for p in frames) == 143 and len(frames) == 172
    rng = np.random.default_rng(5)
    for _ in range(50):
        good = synth.pids_with_crc(rng.integers(0, 2, 80, dtype=np.uint8))
        assert verdict(np.packbits(good).tobytes()) == 1
