"""Regenerates tests/golden/api_am.json: the synthetic AM MA1 / MA3 captures of
tests/test_dropin.py::test_dropin_am_matches_reference_events pushed through the PUBLIC API of the UNMODIFIED
reference library oracle/_ref/libnrsc5_ref.so (nrsc5_set_mode(NRSC5_MODE_AM), 32768-byte pushes).  Needs the
reference library; the JSON is committed.

    python tests/golden/make_golden_api_am.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import nrsc5_api  # noqa: E402
from nrsc5_b200 import synth_am  # noqa: E402


def main():
    out = {}
    for psmi in (1, 2):
        cap = synth_am.make_am_ma1(nframes=8, seed=30 + psmi, lead_in=222, carrier=8000.0, unit=40.0, cfo_hz=0.5, psmi=psmi,
                                   flags=(1, 0, 1, 0))
        for fmt in ("cs16", "cu8"):
            if fmt == "cs16":
                data, kw = cap.cs16.tobytes(), dict(chunk=32768, cs16=True)
            else:
                data, kw = synth_am.am_to_cu8(cap.cs16).tobytes(), dict(chunk=32768)
            out[f"psmi{psmi}_{fmt}"] = nrsc5_api.run(os.path.join(ROOT, "oracle", "_ref", "libnrsc5_ref.so"), data, am=True, **kw)
    json.dump(out, open(os.path.join(HERE, "api_am.json"), "w"), indent=0)
    print({k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    main()
