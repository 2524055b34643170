"""L2 framing (SURVEY §8 f1): the plain-C restatement oracle/nrsc5_oracle_l2.c against the UNMODIFIED reference
(frame.c observed through oracle/reftap_l2.c) and against the golden digests made from the reference."""
import pytest

import common
import port
import reftap
from common import golden, load_sample
from l2_cases import AM_BITS, L2_CASES, l2_digest, mutated_sequence, stress_sequences
from nrsc5_b200 import synth_l2

L2_TYPES = (1, 16, 17, 18, 19)


@pytest.mark.parametrize("name", sorted(L2_CASES))
def test_l2_oracle_equals_reference_on_generated_pdus(name):
    kw = L2_CASES[name]
    frames = synth_l2.make_l2_sequence(**kw)
    orc, lost = port.l2_frames(frames)
    assert l2_digest(orc.records) == golden("l2.json")[name]
    kinds = {t for t, _ in orc.records}
    assert {1, 16, 17, 18, 19} <= kinds
    if reftap.available():
        ref = reftap.l2_frames(frames, mode=1 if kw.get("nbits") in AM_BITS else 0)
        assert ref.records == orc.records                   # byte for byte, in call order


def test_l2_oracle_on_sample_xz():
    cu8 = load_sample()
    if cu8 is None:
        pytest.skip("sample.xz not present")
    l1 = port.decode(cu8)
    orc, lost = port.l2_frames(port.l1_to_l2_input(l1.records))
    dig = l2_digest(orc.records)
    assert dig == golden("l2.json")["sample_xz"]
    assert sum(1 for d in dig if d[0] == "K") == 522 and sum(1 for d in dig if d[0] == "S") == 8
    assert lost == 1                                        # the false-sync frame (its first header does not decode)


def test_l2_generator_covers_the_branches():
    frames = synth_l2.make_l2_sequence(**L2_CASES["p1_fm_fixed"])
    orc, lost = port.l2_frames(frames)
    pk = [r for t, r in orc.records if t == 19]
    assert any(r["flags"] for r in pk) and any(r["shape"] == 2 for r in pk) and any(r["shape"] == 3 for r in pk)
    assert {r["program"] for r in pk} >= {0, 1} and {r["stream_id"] for r in pk} == {0, 1}
    aas = [r["data"] for t, r in orc.records if t == 18]
    assert len(aas) > 20                                    # PSD messages and fixed-data subchannel messages
    # the subchannel messages (40 + 37 m + 11 s bytes, m-th message of subchannel s; FixedDataSource) got through the
    # CCC / block-marker / HDLC path, the one with the bad FCS (m = 1, s = 0) did not
    lens = {len(a) for a in aas}
    assert {40, 114, 51, 88, 125, 162} <= lens and 77 not in lens
    assert lost == 1


@pytest.mark.parametrize("block", range(4))
def test_l2_oracle_equals_reference_under_mutation(block):
    """Random byte errors in the PDUs (headers, locations, HEF, PSD, fixed-data tail): the restatement must take
    every early return and resynchronisation exactly as the unmodified reference's frame.c does."""
    for trial in range(12 * block, 12 * block + 12):
        frames, am = mutated_sequence(trial)
        orc, _ = port.l2_frames(frames)
        common.assert_reference(f"l2_mutation_{trial}", orc.records,
                                lambda: reftap.l2_frames(frames, mode=1 if am else 0).records)


@pytest.mark.parametrize("name", ["many_packets", "hdlc_overrun", "ev_overflow"])
def test_l2_oracle_equals_reference_on_stress_sequences(name):
    """Thousands of one-byte packets per frame; a PSD stream that overruns the 8212-byte HDLC buffer (frame.c:381-386)."""
    frames = stress_sequences()[name]
    orc, _ = port.l2_frames(frames)
    common.assert_reference(f"l2_stress_{name}", orc.records, lambda: reftap.l2_frames(frames).records)
    assert sum(1 for t, _ in orc.records if t == 19) >= 1000
