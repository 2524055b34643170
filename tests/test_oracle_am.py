"""CPU tests pinning the AM restatement (oracle/nrsc5_oracle_am.c) against the UNMODIFIED reference
(oracle/_ref/libnrsc5_ref.so, AM mode; pinned by digest in tests/golden/reference_digests.json) and the committed
golden file, on the synthetic MA1 and MA3 captures."""
import pytest

import common
import port
import reftap
from nrsc5_b200 import synth_am

pytestmark = pytest.mark.skipif(not port.available(), reason="oracle/_ref/liboracle.so not built")


@pytest.mark.parametrize("name", list(common.AM_CASES))
def test_am_port_matches_golden(name):
    g = common.golden("synth_am.json")[name]
    cap = synth_am.make_am_ma1(**common.AM_CASES[name])
    if common.fnv1a32(cap.cs16[:1 << 18].tobytes()) != g["input_fnv"]:
        pytest.skip("numpy generator stream differs from the one the golden file was made with")
    log = port.decode_am(cap.cs16)
    assert common.summarize(log) == g["events"]          # SYNC, PIDS, P1, P3, BER: values and order
    kinds = [e[0] for e in g["events"]]
    assert kinds.count("S") == 1 and kinds.count("B") >= 4 and kinds.count("P") >= 60


@pytest.mark.parametrize("psmi", [1, 2])
def test_am_port_matches_reference_and_is_chunking_invariant(psmi):
    cap = synth_am.make_am_ma1(nframes=9, seed=9, lead_in=1234, cfo_hz=-0.8, noise_lsb=5.0, psmi=psmi)
    a = port.decode_am(cap.cs16)
    b = port.decode_am(cap.cs16, chunk=16384)
    c = port.decode_am(cap.cs16, chunk=2 * 977)
    common.assert_reference(f"am_psmi{psmi}", common.summarize(a),
                            lambda: common.summarize(reftap.decode(cap.cs16, mode=reftap.MODE_AM)))
    assert common.summarize(a) == common.summarize(b) == common.summarize(c)
