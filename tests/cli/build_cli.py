"""Test infrastructure: links the reference's UNMODIFIED command-line program (reference src/main.c + src/log.c,
compiled against the reference's headers by oracle/Makefile into oracle/_ref/cli/) against a libnrsc5.so of our
choice - the drop-in (nrsc5_b200/dropin/_build/libnrsc5.so), the drop-in on the emulated engine, or the unmodified
reference library as the control - with a stand-in for libao (tests/cli/stubs).  Outputs go to tests/_build/
(git-ignored).  The reference's CMake does the same with nrsc5_static (reference src/CMakeLists.txt:96-110)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CLI_OBJS = [os.path.join(ROOT, "oracle", "_ref", "cli", f) for f in ("main.o", "log.o")]
OUTDIR = os.path.join(ROOT, "tests", "_build")


def available():
    return all(os.path.exists(p) for p in CLI_OBJS)


def build(lib_path: str, tag: str) -> str:
    """Returns the path of tests/_build/nrsc5_<tag>, the reference CLI linked against `lib_path`."""
    os.makedirs(OUTDIR, exist_ok=True)
    out = os.path.join(OUTDIR, "nrsc5_" + tag)
    srcs = [os.path.join(HERE, "stubs", "ao_stub.c")]
    deps = CLI_OBJS + srcs + [lib_path, os.path.join(HERE, "stubs", "ao", "ao.h")]
    if os.path.exists(out) and all(os.path.getmtime(p) <= os.path.getmtime(out) for p in deps):
        return out
    libdir = os.path.dirname(os.path.abspath(lib_path))
    rel = os.path.relpath(libdir, OUTDIR)
    cmd = ["gcc", "--std=gnu11", "-O2", "-w", "-I" + os.path.join(HERE, "stubs"), *CLI_OBJS, *srcs, "-o", out,
           os.path.abspath(lib_path), "-Wl,-rpath,$ORIGIN/" + rel, "-lm", "-lpthread"]
    subprocess.run(cmd, check=True)
    return out


if __name__ == "__main__":
    dropin = os.path.join(ROOT, "nrsc5_b200", "dropin", "_build", "libnrsc5.so")
    print(build(dropin, "dropin"))
