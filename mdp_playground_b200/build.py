"""Build libmdpp_b200.so in-tree with nvcc for sm_100a (no torch involved).

    python -m mdp_playground_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmdpp_b200.so")
SOURCES = ["context.cu", "discrete.cu", "discrete_off.cu", "discrete_replay.cu",
           "discrete_philox_f64.cu", "discrete_philox_fast.cu",
           "discrete_philox_zig.cu", "continuous.cu",
           "render.cu", "grid.cu", "wrapper_tail.cu",
           "jit.cu", "qlearn.cu", "ars.cu"]
HEADERS = ["internal.h", "device_types.h", "philox.cuh", "discrete_kernels.cuh",
           "continuous_kernels.cuh", "ziggurat.cuh", "ziggurat_tables.h",
           "discrete_launch.h", "tabular_q.cuh", "../../include/mdpp_b200.h"]
# device-side sources embedded into the library for the NVRTC specialisation
EMBEDDED = ["discrete_kernels.cuh", "continuous_kernels.cuh", "device_types.h",
            "philox.cuh", "ziggurat.cuh",
            "../../include/mdpp_b200.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
    "-std=c++17", "-Xcompiler", "-fPIC",
    "-I", os.path.join(HERE, "..", "include"), "-I", os.path.join(HERE, "build"),
]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "--shared",
              "-cudart", "static", "-ldl"]
OBJ_DIR = os.path.join(HERE, "build")


def _newest_source_mtime():
    files = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    return max(os.path.getmtime(f) for f in files if os.path.exists(f))


def _run(cmd):
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout
                           + res.stderr)
    return res.stdout + res.stderr


def build(force=False, verbose=False):
    """Compile every .cu to an object (in parallel) and link the shared lib."""
    if (not force and os.path.exists(LIB)
            and os.path.getmtime(LIB) >= _newest_source_mtime()):
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ_DIR, exist_ok=True)
    with open(os.path.join(OBJ_DIR, "embedded_sources.inc"), "w") as f:
        for name in EMBEDDED:
            ident = os.path.basename(name).replace(".", "_")
            text = open(os.path.join(CSRC, name)).read()
            assert ")MDPPSRC\"" not in text
            f.write(f'static const char* kSrc_{ident} = R"MDPPSRC({text})MDPPSRC";\n')
    jobs = []
    for src in SOURCES:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [
            "-c", os.path.join(CSRC, src), "-o", obj]
        jobs.append((cmd, obj))
    with ThreadPoolExecutor(max_workers=len(jobs)) as pool:
        logs = list(pool.map(lambda j: _run(j[0]), jobs))
    log = "".join(logs)
    log += _run([nvcc] + LINK_FLAGS + [o for _, o in jobs] + ["-o", LIB])
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
