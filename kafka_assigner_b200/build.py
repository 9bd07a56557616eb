"""Build libkassign.so (hand-written CUDA for sm_100a) in-tree with nvcc. No JIT cache, no torch."""
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(CSRC, "libkassign.so")
SOURCES = ["kassign.cu"]
HEADERS = ["kassign_common.cuh", "kassign_stage.cuh", "kassign_order.cuh", "kassign_json.cuh", "kassign_plan.cuh",
           os.path.join("..", "..", "include", "kassign.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def cuda_tool(name):
    """Path of a CUDA toolkit program (nvcc, cuobjdump): PATH first, then $CUDA_HOME/bin, then /usr/local/cuda/bin,
    so that an account whose PATH lacks the toolkit still finds it."""
    homes = [os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"]
    for cand in [shutil.which(name)] + [os.path.join(h, "bin", name) for h in homes if h]:
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("%s not found: put the CUDA toolkit's bin/ on PATH or set CUDA_HOME "
                       "(libkassign.so has no CPU fallback)" % name)


HOST_DIR = os.path.join(_HERE, "host")
CLI = os.path.join(_HERE, "bin", "kafka-assignment-generator")
HOST_TEST = os.path.join(_HERE, "bin", "test_kafka_topic_assigner")
HOST_SOURCES = ["kafka_assignment_generator.cpp", "kassign_host.hpp", "test_kafka_topic_assigner.cpp"]


def build_host(force=False):
    """g++ the C++ host mirror + file-based CLI (reference flag surface) against libkassign.so."""
    deps = [os.path.join(HOST_DIR, f) for f in HOST_SOURCES] + [LIB, os.path.join(_HERE, "..", "include", "kassign.h")]
    if not force and os.path.exists(CLI) and all(os.path.getmtime(d) <= os.path.getmtime(CLI) for d in deps if os.path.exists(d)):
        return CLI
    os.makedirs(os.path.dirname(CLI), exist_ok=True)
    cmd = ["g++", "-O2", "-std=c++17", "-Wall", os.path.join(HOST_DIR, "kafka_assignment_generator.cpp"), "-L" + CSRC, "-lkassign",
           "-Wl,-rpath,$ORIGIN/../csrc", "-o", CLI]
    subprocess.check_call(cmd)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", os.path.join(HOST_DIR, "test_kafka_topic_assigner.cpp"), "-L" + CSRC,
                           "-lkassign", "-Wl,-rpath,$ORIGIN/../csrc", "-o", HOST_TEST])
    return CLI


def needs_build():
    if not os.path.exists(LIB):
        return True
    lib_m = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > lib_m for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every CUDA source into csrc/libkassign.so. Cross-compiles without a GPU."""
    if not force and not needs_build():
        return LIB
    cmd = [cuda_tool("nvcc")] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    subprocess.check_call(cmd, cwd=CSRC)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
