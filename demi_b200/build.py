"""Build the in-tree native libraries.

  demi_b200/libdemi_b200.so  — the CUDA engine + C ABI (nvcc, sm_100a only)
  oracle/liboracle.so        — the CPU oracle (gcc; test infrastructure only)

Both are git-ignored and travel to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "demi_b200", "csrc")
LIB = os.path.join(ROOT, "demi_b200", "libdemi_b200.so")
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "liboracle.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
]


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _sources(root, exts):
    out = []
    for d, _, files in os.walk(root):
        for f in files:
            if f.endswith(exts):
                out.append(os.path.join(d, f))
    return out


def source_id():
    """Hash of every source the engine library is built from: compiled into the library (demi_version) and
    recorded in profiles/*.json, so a profile taken from another build is recognised as stale."""
    import hashlib
    h = hashlib.sha1()
    srcs = _sources(CSRC, (".cu", ".cuh", ".h", ".hpp")) + _sources(os.path.join(ROOT, "include"), (".h",))
    for s in sorted(srcs):
        h.update(os.path.relpath(s, ROOT).encode())
        h.update(open(s, "rb").read())
    return h.hexdigest()[:12]


K1_SOURCES = ["demi_b200/csrc/lane_kernel.cuh", "demi_b200/csrc/machine.cuh", "demi_b200/csrc/fuzz_kernel.cuh",
              "demi_b200/csrc/models/models.cuh", "include/demi_limits.h"]


def k1_source_id():
    """Hash of the sources of the headline kernel alone (fuzz_lane_kernel / fuzz_kernel): what profiles/k1_profile.json
    is tied to, so work on the other kernels does not invalidate that capture."""
    import hashlib
    h = hashlib.sha1()
    for s in K1_SOURCES:
        h.update(s.encode())
        h.update(open(os.path.join(ROOT, s), "rb").read())
    return h.hexdigest()[:12]


def build_engine(force=False, verbose=False):
    srcs = _sources(CSRC, (".cu", ".cuh", ".h", ".hpp")) + _sources(os.path.join(ROOT, "include"), (".h",))
    if not force and _newer(LIB, srcs):
        return LIB
    cus = sorted(s for s in srcs if s.endswith(".cu"))
    cmd = ["nvcc"] + NVCC_FLAGS + ["-DDEMI_BUILD_ID=\"%s\"" % source_id(), "-DDEMI_K1_ID=\"%s\"" % k1_source_id()] + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + cus
    subprocess.check_call(cmd, cwd=ROOT)
    return LIB


def _cpu_stamp():
    """The oracle is compiled -march=native, so a library built on another machine (it travels with the
    gpurun snapshot) is rebuilt on the machine that runs it: model name + ISA flags identify the CPU."""
    import hashlib
    model, flags = "", ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and not model:
                model = line.split(":", 1)[1].strip()
            if line.startswith("flags") and not flags:
                flags = line.split(":", 1)[1].strip()
            if model and flags:
                break
    except OSError:
        pass
    return hashlib.sha1((model + "|" + flags).encode()).hexdigest()


ORACLE_STAMP = os.path.join(ORACLE_DIR, ".build_cpu")


def build_oracle(force=False, private=False):
    """Return the path of an oracle library built for this CPU.  private=True leaves the tree untouched: a missing
    or stale in-tree library is then built in a new temporary directory (bench.py may run from a read-only tree)."""
    srcs = _sources(ORACLE_DIR, (".c", ".h")) + _sources(os.path.join(ROOT, "include"), (".h",))
    srcs.append(os.path.join(ORACLE_DIR, "Makefile"))
    stamp = _cpu_stamp()
    same_cpu = os.path.exists(ORACLE_STAMP) and open(ORACLE_STAMP).read().strip() == stamp
    if not force and same_cpu and _newer(ORACLE_LIB, srcs):
        return ORACLE_LIB
    if private:
        import tempfile
        out = os.path.join(tempfile.mkdtemp(prefix="demi_oracle_"), "liboracle.so")
        subprocess.check_call(["make", "-B", "-C", ORACLE_DIR, "OUT=" + out, out], stdout=sys.stderr)
        return out
    # make's chatter goes to stderr: bench.py prints exactly one JSON line on stdout
    subprocess.check_call(["make", "-B", "-C", ORACLE_DIR, "liboracle.so"], stdout=sys.stderr)
    with open(ORACLE_STAMP, "w") as f:
        f.write(stamp + "\n")
    return ORACLE_LIB


if __name__ == "__main__":
    force = "--force" in sys.argv
    print(build_engine(force=force, verbose="-v" in sys.argv))
    print(build_oracle(force=force))
