"""Shared helpers for the parity tests (test infrastructure)."""
import hashlib
import json
import lzma
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

SAMPLE = os.path.join(ROOT, "oracle", "_ref", "sample.xz")    # the reference's support/sample.xz, copied by build()
# every object of the drop-in libnrsc5.so but the engine (oracle/Makefile)
DROPIN_OBJDIR = os.path.join(ROOT, "oracle", "_ref", "dropin")


def fnv1a32(b: bytes) -> int:
    h = 0x811C9DC5
    for x in b:
        h = ((h ^ x) * 0x01000193) & 0xFFFFFFFF
    return h


def load_sample():
    if os.path.exists(SAMPLE):
        return np.frombuffer(lzma.open(SAMPLE).read(), dtype=np.uint8)
    return None


def golden(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


REF_DIGESTS = os.path.join(GOLDEN, "reference_digests.json")


def digest(value) -> str:
    """sha256 of repr(value): value is built from ints, Python floats, str, bytes, lists, tuples and dicts."""
    return hashlib.sha256(repr(value).encode()).hexdigest()


def assert_reference(key, got, live=None):
    """`got` must be what the unmodified reference computes for the same input.  The reference's answer is pinned by
    its digest in tests/golden/reference_digests.json (made by tests/golden/make_golden_digests.py), so the test
    needs no reference library; when oracle/_ref holds one, `live()` (the reference's answer, computed now) is checked
    against that digest as well.  With NRSC5_WRITE_REF_DIGESTS=1 the digest of live() is recorded instead."""
    import reftap
    with open(REF_DIGESTS) as f:
        table = json.load(f)
    if os.environ.get("NRSC5_WRITE_REF_DIGESTS") == "1":
        table[key] = digest(live())
        with open(REF_DIGESTS, "w") as f:
            json.dump(dict(sorted(table.items())), f, indent=0)
    elif live is not None and reftap.available():
        assert digest(live()) == table[key], f"{key}: the reference library disagrees with the committed digest"
    assert digest(got) == table[key], f"{key}: differs from the unmodified reference"


# the synthetic parity matrix (SURVEY §8d): name -> generator kwargs
SYNTH_CASES = {
    "mp1_clean": dict(nframes=2, seed=1234, lead_in=1777),
    "mp1_cfo120": dict(nframes=2, seed=77, lead_in=333, cfo_hz=120.0),
    "mp1_cfo-300_awgn12": dict(nframes=2, seed=77, lead_in=333, cfo_hz=-300.0, noise_lsb=12.0),
    "mp1_cfo2000_awgn20": dict(nframes=2, seed=77, lead_in=333, cfo_hz=2000.0, noise_lsb=20.0),
    "mp1_badhdr": dict(nframes=2, seed=9, lead_in=40, valid_header=False),
}


# MP3 (extended hybrid: 12 partitions per sideband, P3 on the PX1 partitions through interleaver IV)
MP3_CASE = dict(nframes=4, seed=11, lead_in=300, tail_blocks=2)


# the other FM service modes the reference tells apart (src/sync.c:343-357,537-595): MP2 (11 partitions per sideband,
# 2304-bit P3), MP5 / MP6 (14 partitions tracked and counted in the MER), MP11 (14 partitions, P3 on PX1, P4 on PX2)
FM_MODE_CASES = {
    "mp2": dict(psmi=2, nframes=4, seed=22, lead_in=300, tail_blocks=2, cfo_hz=50.0, noise_lsb=4.0),
    "mp5": dict(psmi=5, nframes=3, seed=25, lead_in=411, tail_blocks=2, cfo_hz=-80.0, noise_lsb=6.0),
    "mp6": dict(psmi=6, nframes=3, seed=26, lead_in=97, tail_blocks=2, noise_lsb=14.0),
    "mp11": dict(psmi=11, nframes=4, seed=31, lead_in=300, tail_blocks=2, cfo_hz=50.0, noise_lsb=4.0),
}


# AM hybrid MA1 (psmi 1) and all-digital MA3 (psmi 2), cs16 (SURVEY §8 a21); the *_noisy cases have a channel
# BER of about 1e-3 so that the K=9 Viterbi decoders correct real errors
AM_CASES = {
    "ma1_clean": dict(nframes=10, seed=3, lead_in=500),
    "ma1_cfo_awgn": dict(nframes=10, seed=4, lead_in=777, cfo_hz=1.5, noise_lsb=8.0),
    "ma1_noisy": dict(nframes=10, seed=8, lead_in=333, cfo_hz=-1.0, noise_lsb=120.0),
    "ma3_clean": dict(nframes=10, seed=5, lead_in=640, psmi=2),
    "ma3_noisy": dict(nframes=10, seed=6, lead_in=901, cfo_hz=-2.0, noise_lsb=120.0, psmi=2),
}


def summarize(log):
    """Digest a RefLog into a JSON-able summary (order-preserving)."""
    import reftap
    seq = []
    for ty, p in log.records:
        if ty == reftap.REC_FRAME:
            seq.append(["F", p["lc"], p["nbits"], fnv1a32(p["bits"])])
        elif ty == reftap.REC_PIDS:
            seq.append(["P", fnv1a32(p["bits"])])
        elif ty == reftap.REC_SYNC:
            flags = p.get("flags", [-1] * 4)
            seq.append(["S", round(p["freq_offset"], 3), p["psmi"]] + ([] if flags == [-1] * 4 else list(flags)))
        elif ty == reftap.REC_LOST_SYNC:
            seq.append(["L"])
        elif ty == reftap.REC_MER:
            seq.append(["M", round(p["lower"], 4), round(p["upper"], 4)])
        elif ty == reftap.REC_BER:
            seq.append(["B", round(p["cber"], 7)])
    return seq
