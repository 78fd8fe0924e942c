"""Build libdcb.so (CUDA kernels + C ABI) in-tree for sm_100a.

    python -m decombinator_b200.build [--force]
    python -m decombinator_b200.build --variants [--force]           every library of VARIANTS
    python -m decombinator_b200.build --variant NAME [-DFLAG=1 ...]   one variant (NAME from VARIANTS, or the flags given)

nvcc cross-compiles without a GPU; the built libraries are git-ignored.  A variant is the same sources, flags and link
with extra -D defines, written to build/libdcb_NAME.so; a process loads it in place of libdcb.so with DCB_LIB set.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdcb.so")
VARIANT_DIR = os.path.join(os.path.dirname(HERE), "build")
SYNTH_LIB = os.path.join(HERE, "libdcbsynth.so")   # the synthetic read generator alone (bench.py's reference arm maps only this + oracle/)
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SOURCES = ["decombine.cu", "collapse.cu", "tagset.cpp", "pack.cpp", "fastq.cpp", "group.cpp", "synth.cpp", "error.cpp"]

FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function", "-shared", "-Xptxas", "-v",
]


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


# Libraries the test suite loads besides libdcb.so (tests/test_gpu_halftag_capacity.py): the half-tag kernel's per-read
# candidate list and its two per-warp work lists shrunk, so that nearly every warp overflows every list and each pass-on
# branch runs on ordinary data.  The defaults are 12, 192 and 126 (csrc/decombine.cu).
VARIANTS = {
    "halfcap_tiny": {"DCB_HALF_CAP": 2, "DCB_HALF_WCAP": 32, "DCB_HALF_WCAP2": 12},
    "halfcap_small": {"DCB_HALF_CAP": 4, "DCB_HALF_WCAP": 64, "DCB_HALF_WCAP2": 30},
}


def needs_build(out=LIB):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(HERE), "include", "dcb.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def _command(out, defines=()):
    return ([NVCC] + FLAGS + ["-D%s" % d for d in defines] + ["-I", os.path.join(os.path.dirname(HERE), "include"), "-o", out]
            + sources() + ["-lpthread", "-lz"])


def _defines(defines):
    """{"NAME": value} or ["NAME=value", "-DNAME=value", ...] -> ["NAME=value", ...]"""
    if isinstance(defines, dict):
        return ["%s=%s" % (k, v) for k, v in defines.items()]
    return [d[2:] if d.startswith("-D") else d for d in defines]


def variant_path(name):
    return os.path.join(VARIANT_DIR, "libdcb_%s.so" % name)


def _variant_job(name, defines, force):
    """-> (output, command, Popen or None when the output is up to date)"""
    out = variant_path(name)
    cmd = _command(out, _defines(VARIANTS[name] if defines is None else defines))
    stamp = out + ".cmd"                       # the command that built it: other defines under the same name rebuild
    same = False
    if os.path.exists(stamp):
        with open(stamp) as fh:
            same = fh.read() == " ".join(cmd)
    if not force and same and not needs_build(out):
        return out, cmd, None
    os.makedirs(VARIANT_DIR, exist_ok=True)
    return out, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)


def _variant_wait(out, cmd, proc):
    if proc is None:
        return out
    log = proc.communicate()[0]
    if proc.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed building %s" % out)
    with open(out + ".cmd", "w") as fh:
        fh.write(" ".join(cmd))
    return out


def variant(name, defines=None, force=False):
    """build/libdcb_<name>.so: what build() compiles, with the -D defines given (default: VARIANTS[name]).  Skipped when
    the library is newer than every source and was built with the same command."""
    return _variant_wait(*_variant_job(name, defines, force))


def build_variants(force=False):
    """Every library of VARIANTS, compiled side by side."""
    jobs = [_variant_job(name, None, force) for name in VARIANTS]
    errors = []
    for job in jobs:                           # every compiler process is waited for, failed or not
        try:
            _variant_wait(*job)
        except RuntimeError as e:
            errors.append(e)
    if errors:
        raise errors[0]
    return [job[0] for job in jobs]


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    cmd = _command(LIB)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libdcb.so")
    with open(os.path.join(HERE, "build.log"), "w") as fh:
        fh.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    build_synth(force=True)
    return LIB


def build_synth(force=False):
    """libdcbsynth.so: csrc/synth.cpp alone (plain C++, no CUDA)."""
    src = [os.path.join(CSRC, "synth.cpp"), os.path.join(CSRC, "error.cpp")]
    if not force and os.path.exists(SYNTH_LIB) and all(os.path.getmtime(x) <= os.path.getmtime(SYNTH_LIB) for x in src):
        return SYNTH_LIB
    cmd = ["g++", "-O3", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(os.path.dirname(HERE), "include"), "-o", SYNTH_LIB] + src + ["-lpthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("g++ failed building libdcbsynth.so")
    return SYNTH_LIB


if __name__ == "__main__":
    force = "--force" in sys.argv
    if "--variant" in sys.argv:
        name = sys.argv[sys.argv.index("--variant") + 1]
        flags = [a for a in sys.argv[1:] if a.startswith("-D")]
        if not flags and name not in VARIANTS:
            sys.exit("unknown variant %r (known: %s); give its -D flags" % (name, ", ".join(VARIANTS)))
        print(variant(name, flags or None, force=force))
    elif "--variants" in sys.argv:
        print("\n".join(build_variants(force=force)))
    else:
        print(build(force=force, verbose=True))
