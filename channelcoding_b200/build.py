"""Build libccgpu.so (hand-written sm_100a CUDA kernels + the extern "C" ABI of include/ccgpu.h).

    python -m channelcoding_b200.build [--force]

nvcc cross-compiles without a GPU.  Objects go to channelcoding_b200/csrc/_obj/, the library to
channelcoding_b200/libccgpu.so (git-ignored, shipped to the GPU box by gpurun).  The min-sum kernel
instantiation groups (csrc/ms_shapes_generated.h) are compiled in parallel.
"""
import concurrent.futures
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj" + ("_" + os.environ["CCGPU_VARIANT"] if os.environ.get("CCGPU_VARIANT") else ""))
# CCGPU_VARIANT=<name> + CCGPU_EXTRA_FLAGS builds an experimental copy next to the product library
VARIANT = os.environ.get("CCGPU_VARIANT", "")
LIB = os.path.join(HERE, "libccgpu%s.so" % ("_" + VARIANT if VARIANT else ""))
NVCC = os.environ.get("NVCC", "nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xptxas", "-v"]
FLAGS += os.environ.get("CCGPU_EXTRA_FLAGS", "").split()


def _groups():
    with open(os.path.join(CSRC, "ms_shapes_generated.h")) as f:
        return int(re.search(r"#define CCGPU_MS_GROUPS (\d+)", f.read()).group(1))


def _units():
    units = [("api.o", "api.cu", []), ("ms_registry.o", "ms_registry.cu", []), ("ms_csr.o", "ms_csr.cu", []),
             ("gf_decode.o", "gf_decode.cu", []), ("chase.o", "chase.cu", []),
             ("osd.o", "osd.cu", []), ("gmd.o", "gmd.cu", []), ("abp.o", "abp.cu", []), ("ml.o", "ml.cu", []),
             ("group.o", "group.cc", [])]
    units.append(("ms_cyclic_cta.o", "ms_cyclic_cta_inst.cu", []))
    units.append(("ms_cyclic_lane.o", "ms_cyclic_lane_inst.cu", []))
    for g in range(_groups()):
        units.append(("ms_cyclic_g%d.o" % g, "ms_cyclic_inst.cu", ["-DCCGPU_GROUP=%d" % g]))
    return units


def _deps():
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".hpp", ".cuh", ".cu", ".cc"))]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "ccgpu.h"))
    deps.append(os.path.abspath(__file__))
    return deps


def _compile(unit):
    obj, src, extra = unit
    out = os.path.join(OBJ, obj)
    cmd = [NVCC] + ARCH + FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    return obj, r.returncode, r.stdout + r.stderr


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    newest = max(os.path.getmtime(d) for d in _deps())
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= newest:
        return LIB
    units = _units()
    logs = []
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(units), os.cpu_count() or 4)) as ex:
        for obj, rc, log in ex.map(_compile, units):
            logs.append("== %s\n%s" % (obj, log))
            if rc != 0:
                raise RuntimeError("nvcc failed for %s:\n%s" % (obj, log))
    with open(os.path.join(OBJ, "ptxas.log"), "w") as f:
        f.write("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    cmd = [NVCC] + ARCH + ["-shared", "-Xcompiler", "-pthread", "-o", LIB] + [os.path.join(OBJ, u[0]) for u in units]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


TOOLS_BIN = os.path.join(os.path.dirname(HERE), "tools", "_bin")


def build_tools(force=False):
    """the C++ host layer (include/cc/*.h) in use: the reference-style `benchmark` CLI and the C++
    test program, linked against libccgpu.so (g++; no CUDA code in these)."""
    root = os.path.dirname(HERE)
    os.makedirs(TOOLS_BIN, exist_ok=True)
    hdrs = [os.path.join(root, "include", "ccgpu.h"), os.path.join(root, "include", "cc", "codes.h"),
            os.path.join(root, "include", "cc", "simulation.h")]
    jobs = [(os.path.join(TOOLS_BIN, "benchmark"), os.path.join(root, "tools", "benchmark.cc")),
            (os.path.join(TOOLS_BIN, "uncoded"), os.path.join(root, "tools", "uncoded.cc")),
            (os.path.join(TOOLS_BIN, "bitflips"), os.path.join(root, "tools", "bitflips.cc")),
            (os.path.join(TOOLS_BIN, "host_layer_test"), os.path.join(root, "tests", "cpp", "host_layer_test.cc")),
            (os.path.join(TOOLS_BIN, "chase_test"), os.path.join(root, "tests", "cpp", "chase_test.cc")),
            (os.path.join(TOOLS_BIN, "osd_test"), os.path.join(root, "tests", "cpp", "osd_test.cc")),
            (os.path.join(TOOLS_BIN, "gmd_test"), os.path.join(root, "tests", "cpp", "gmd_test.cc")),
            (os.path.join(TOOLS_BIN, "abp_test"), os.path.join(root, "tests", "cpp", "abp_test.cc")),
            (os.path.join(TOOLS_BIN, "ml_test"), os.path.join(root, "tests", "cpp", "ml_test.cc"))]

    def one(job):
        out, src = job
        newest = max(os.path.getmtime(p) for p in hdrs + [src, LIB])
        if not force and os.path.exists(out) and os.path.getmtime(out) >= newest:
            return out
        cmd = ["g++", "-std=c++17", "-O1", "-Wall", "-I" + os.path.join(root, "include"), src, "-L" + HERE, "-lccgpu",
               "-Wl,-rpath,$ORIGIN/../../channelcoding_b200", "-pthread", "-o", out]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("g++ failed for %s:\n%s" % (src, r.stdout + r.stderr))
        return out
    with concurrent.futures.ThreadPoolExecutor(max_workers=4) as ex:
        return list(ex.map(one, jobs))


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
    if "--tools" in sys.argv:
        print(build_tools(force="--force" in sys.argv))
