"""The reference's own end-to-end test (reference .github/workflows/ci.yml:30-42) on the drop-in library:

    nrsc5 -r sample -o sample.wav 0 2> sample.log ; grep -q "You're Listening to Q" sample.log
    cat sample | nrsc5 -r - -o sample.wav 0       ; same grep
    support/cli.py -r sample -o sample.wav 0      ; same grep

with `nrsc5` = the reference's UNMODIFIED command-line program (src/main.c + src/log.c, compiled where they lie by
oracle/Makefile, linked by tests/cli/build_cli.py, libao replaced by a byte-counting stand-in) against the drop-in libnrsc5.so, and
`support/cli.py` = the reference's unmodified Python CLI loading the drop-in through its own ctypes binding
(support/nrsc5.py:676-690).  This is the claim of BASELINE.json's north_star - "the CLI and Python bindings drop in
unchanged" - tested the way the reference tests itself.  Beyond the grep, every information line the CLI prints
(station, audio services, titles, artists, ...) must equal, in order, what the same program prints when linked
against the unmodified reference library.

CPU tier: the drop-in on the CPU emulation of the kernels (tests/emu), first 20 MB of the capture.
GPU tier: the real drop-in, whole capture; the binaries are linked by __graft_entry__.build() from oracle/_ref/.
"""
import os
import re
import subprocess
import sys

import pytest

import common

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "cli"))
sys.path.insert(0, os.path.join(HERE, "emu"))
import build_cli  # noqa: E402

BUILD = os.path.join(HERE, "_build")
GREP = "You're Listening to Q"
REF_SUPPORT = os.path.join(common.ROOT, "oracle", "_ref", "support")   # the reference's support/*.py, copied by build()


def info_lines(log: str):
    """The CLI's log without timestamps and without the lines that carry measured floats or build strings."""
    out = []
    for ln in log.splitlines():
        ln = re.sub(r"^\d\d:\d\d:\d\d ", "", ln)
        if re.match(r"(MER|BER|Synchronized|Lost synchronization|Audio bit rate|nrsc5 revision)", ln) or not ln.strip():
            continue
        out.append(ln)
    return out


@pytest.fixture(scope="module")
def sample_files(tmp_path_factory):
    raw = common.load_sample()
    if raw is None:
        pytest.skip("sample.xz not available")
    d = tmp_path_factory.mktemp("cli")
    full, part = d / "sample", d / "sample20"
    full.write_bytes(raw.tobytes())
    part.write_bytes(raw.tobytes()[:20_000_000])
    return str(full), str(part), str(d)


def run_cli(binary, sample, workdir, stdin=False):
    wav = os.path.join(workdir, "out.wav")
    if stdin:
        with open(sample, "rb") as f:
            r = subprocess.run([binary, "-r", "-", "-o", wav, "0"], stdin=f, capture_output=True, text=True, timeout=900)
    else:
        r = subprocess.run([binary, "-r", sample, "-o", wav, "0"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stderr


def control_binary():
    import reftap
    p = os.path.join(BUILD, "nrsc5_ref")
    if build_cli.available() and reftap.available():
        return build_cli.build(reftap.REF_SO, "ref")
    return p if os.path.exists(p) else None


@pytest.fixture(scope="module")
def emulated_cli():
    """libnrsc5.so = the drop-in's objects on the emulated engine, and the reference CLI linked against it."""
    import build_emu
    objdir = common.DROPIN_OBJDIR
    if not build_cli.available() or not os.path.isdir(objdir):
        pytest.skip("needs the reference tree (the CLI and the drop-in's host objects are compiled from it)")
    emu = build_emu.build()
    libdir = os.path.join(BUILD, "emu_lib")
    os.makedirs(libdir, exist_ok=True)
    so = os.path.join(libdir, "libnrsc5.so")
    objs = sorted(os.path.join(objdir, f) for f in os.listdir(objdir) if f.endswith(".o"))
    subprocess.run(["gcc", "-shared", "-o", so, *objs, emu, "-Wl,-rpath," + os.path.dirname(emu), "-lm", "-lpthread"], check=True)
    return build_cli.build(so, "emu"), libdir


def test_reference_cli_on_the_emulated_dropin(emulated_cli, sample_files):
    binary, _ = emulated_cli
    _, part, work = sample_files
    log = run_cli(binary, part, work)
    assert GREP in log                                              # ci.yml:35
    ctl = control_binary()
    assert ctl is not None
    assert info_lines(log) == info_lines(run_cli(ctl, part, work)) and len(info_lines(log)) >= 8


def test_reference_python_cli_on_the_emulated_dropin(emulated_cli, sample_files):
    """support/cli.py -r - (stdin), the reference's ctypes binding loading libnrsc5.so = the drop-in (ci.yml:41-42)."""
    _, libdir = emulated_cli
    _, part, work = sample_files
    if not os.path.exists(os.path.join(REF_SUPPORT, "cli.py")):
        pytest.skip("reference tree not present")
    env = dict(os.environ, PYTHONPATH=os.path.join(HERE, "cli", "stubs") + os.pathsep + REF_SUPPORT,
               LD_LIBRARY_PATH=libdir + os.pathsep + os.environ.get("LD_LIBRARY_PATH", ""))
    with open(part, "rb") as f:
        r = subprocess.run([sys.executable, os.path.join(REF_SUPPORT, "cli.py"), "-r", "-", "-o", os.path.join(work, "py.wav"), "0"],
                           stdin=f, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert GREP in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("stdin", [False, True])
def test_reference_cli_on_the_dropin(sample_files, stdin):
    """The real drop-in on the GPU, whole capture, from a file and from stdin (ci.yml:33-37)."""
    binary = os.path.join(BUILD, "nrsc5_dropin")
    if build_cli.available():
        binary = build_cli.build(os.path.join(common.ROOT, "nrsc5_b200", "dropin", "_build", "libnrsc5.so"), "dropin")
    if not os.path.exists(binary):
        pytest.skip("reference CLI not built (needs the reference tree at build time)")
    full, _, work = sample_files
    log = run_cli(binary, full, work, stdin=stdin)
    assert GREP in log
    assert log.count(GREP) == 8                                     # the capture's eight ID3 messages
    ctl = control_binary()
    if ctl is not None:
        assert info_lines(log) == info_lines(run_cli(ctl, full, work, stdin=stdin))
