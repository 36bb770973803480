"""Builds libust.so (sm_100a only) next to this file. Invoked by __graft_entry__.build()."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libust.so")
SOURCES = ["ust_stream.cu", "ust_kernels.cu", "ust_api.cu"]
DEPS = SOURCES + ["ust_dev.h", "ust_common.cuh", "ust_lut.h", os.path.join("..", "..", "include", "ust.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xcompiler", "-ffp-contract=off", "--fmad=false",
]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-shared", "-o", OUT] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    subprocess.check_call(cmd)
    return OUT


HOST_OUT = os.path.join(HERE, "libust_host.so")
HOST_SRC = os.path.join(HERE, "host", "upgrade.cpp")


def build_host(force=False):
    """libust_host.so: the C++ mirror of the reference's manager interface over the C ABI (links libust.so)."""
    deps = [HOST_SRC, os.path.join(HERE, "host", "upgrade.hpp"), OUT]
    if not force and os.path.exists(HOST_OUT) and all(os.path.getmtime(d) <= os.path.getmtime(HOST_OUT) for d in deps):
        return HOST_OUT
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-Wall", "-shared", "-o", HOST_OUT, HOST_SRC,
                           "-L" + HERE, "-lust", "-Wl,-rpath,$ORIGIN"])
    return HOST_OUT


def build_host_tests(root):
    """tests/host/_build/{upgrade_state_test,host_logic_test}: the reference's specs against the mirror."""
    tdir = os.path.join(root, "tests", "host")
    bdir = os.path.join(tdir, "_build")
    os.makedirs(bdir, exist_ok=True)
    common = ["g++", "-O1", "-std=c++17", "-Wall", "-Wno-unused-variable", "-I" + root]
    # rpaths relative to the executables, so that a built tree still runs after it is copied or moved
    link = ["-L" + HERE, "-lust_host", "-lust", "-Wl,-rpath,$ORIGIN/" + os.path.relpath(HERE, bdir)]
    oracle = os.path.join(root, "oracle")
    srcs = [os.path.join(tdir, f) for f in os.listdir(tdir) if f.endswith((".cpp", ".hpp"))] + [HOST_OUT]
    out = []
    for name, extra in (("upgrade_state_test", []),
                        ("host_logic_test", ["-L" + oracle, "-lust_oracle", "-Wl,-rpath,$ORIGIN/" + os.path.relpath(oracle, bdir)])):
        exe = os.path.join(bdir, name)
        if not os.path.exists(exe) or any(os.path.getmtime(x) > os.path.getmtime(exe) for x in srcs):
            subprocess.check_call(common + [os.path.join(tdir, name + ".cpp"), "-o", exe] + link + extra)
        out.append(exe)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_host(force="--force" in sys.argv))
