"""In-tree build of libhyperpose_b200.so (nvcc, sm_100a only).  `python -m hyperpose_b200.build`."""
from __future__ import annotations

import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libhyperpose_b200.so")
# binaries compiled from the drop-in together with the reference's headers / sources: kept out of git with the reference's builds,
# in a directory of their own (the rest of oracle/_ref is the checker, built from the reference alone by oracle/Makefile)
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "dropin")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-O2,-Wall", "-Xptxas", "-v"]
# bit-exact fp32 kernels (parser): never let nvcc contract a*b+c
EXACT_FLAGS = ["-fmad=false"]

# (source, extra flags)
SOURCES = [
    ("paf_parser.cu", EXACT_FLAGS),
    ("engine.cu", []),
    ("pifpaf_decoder.cu", EXACT_FLAGS),
    ("ppn_parser.cu", EXACT_FLAGS),
    ("common.cpp", []),
    ("handoff.cpp", []),
    ("pool.cpp", []),
]


def _newer(src_files, target):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in src_files)


def build(force: bool = False, verbose: bool = False) -> str:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(PKG, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(ROOT, "include", "hyperpose_b200.h"))
    objs = []
    rebuilt = False
    for src, extra in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        objs.append(o)
        if force or _newer([s] + headers, o):
            cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError(f"nvcc failed on {src}")
            with open(o + ".ptxas.txt", "w") as f:
                f.write(r.stderr)
            rebuilt = True
    if rebuilt or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-o", LIB] + objs  # static cudart (nvcc default); the driver API is reached via cudaGetDriverEntryPoint
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


def build_cpp_example(ref_root: str = "/root/reference") -> str | None:
    """Compiles the C++ drop-in (hyperpose_api/*.cpp) + examples/operator_api_b200.cpp against the reference's
    UNCHANGED public headers.  Needs the reference tree (headers are not copied into this repo); returns the
    binary path (oracle/_ref/dropin/operator_api_b200), or the one built earlier / None when the reference is absent."""
    exe = os.path.join(REF_BIN, "operator_api_b200")
    if not os.path.isdir(os.path.join(ref_root, "include", "hyperpose")):
        return exe if os.path.exists(exe) else None
    os.makedirs(REF_BIN, exist_ok=True)
    api = os.path.join(CSRC, "hyperpose_api")
    srcs = [os.path.join(api, "paf.cpp"), os.path.join(api, "tensorrt.cpp"), os.path.join(api, "pifpaf.cpp"), os.path.join(api, "pose_proposal.cpp"),
            os.path.join(ROOT, "examples", "operator_api_b200.cpp")]
    if _newer(srcs + [LIB], exe):
        cmd = ["g++", "-std=c++17", "-O2", "-DHP_B200_STANDALONE", "-I" + os.path.join(CSRC, "shim"), "-I" + os.path.join(ref_root, "include"),
               "-I" + os.path.join(ROOT, "include")] + srcs + ["-L" + PKG, "-lhyperpose_b200", "-Wl,-rpath,$ORIGIN/../../../hyperpose_b200", "-o", exe]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("C++ drop-in failed to compile against the reference headers")
    return exe


def build_stream_example(ref_root: str = "/root/reference", mock: bool = False) -> str | None:
    """examples/stream_api_b200.cpp: the reference's STREAM API on the drop-in.  The scheduler is the reference's own --
    include/hyperpose/stream/stream.hpp instantiated as it is, src/stream.cpp + src/thread_pool.cpp + src/logging.cpp compiled from
    the reference tree unchanged.  mock=True builds the CPU self-check variant (stand-in engine / parser, no GPU, no library)."""
    exe = os.path.join(REF_BIN, "stream_api_b200_mock" if mock else "stream_api_b200")
    if not os.path.isdir(os.path.join(ref_root, "include", "hyperpose")):
        return exe if os.path.exists(exe) else None
    os.makedirs(REF_BIN, exist_ok=True)
    api = os.path.join(CSRC, "hyperpose_api")
    ref = [os.path.join(ref_root, "src", f) for f in ("stream.cpp", "thread_pool.cpp", "logging.cpp")]
    srcs = [os.path.join(ROOT, "examples", "stream_api_b200.cpp")] + ref
    if not mock:
        srcs += [os.path.join(api, "paf.cpp"), os.path.join(api, "tensorrt.cpp")]
    if _newer([s for s in srcs if s.startswith(ROOT)] + ([] if mock else [LIB]) + [os.path.join(CSRC, "shim", "opencv2", "opencv.hpp")], exe):
        cmd = ["g++", "-std=c++17", "-O2", "-pthread", "-DHP_STREAM_MOCK" if mock else "-DHP_B200_STANDALONE", "-I" + os.path.join(CSRC, "shim"),
               "-I" + os.path.join(ref_root, "include"), "-I" + os.path.join(ref_root, "src"), "-I" + os.path.join(ROOT, "include")] + srcs
        if not mock:
            cmd += ["-L" + PKG, "-lhyperpose_b200", "-Wl,-rpath,$ORIGIN/../../../hyperpose_b200"]
        cmd += ["-o", exe]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("stream example failed to compile against the reference's stream sources")
    return exe


REFERENCE_EXAMPLES = ["operator_api_batched_images_paf.example", "operator_api_batched_images_pifpaf.example", "operator_api_batched_images_pose_proposal.example",
                      "stream_api_video_paf.example", "gen_serialized_engine.example", "cli"]


def build_reference_examples(ref_root: str = "/root/reference") -> dict | None:
    """The reference's OWN example programs, compiled UNMODIFIED from <ref>/examples/*.cpp (+ examples/utils.cpp) against the drop-in:
    the reference's unchanged headers, its unchanged src/{stream,thread_pool,logging,human,data}.cpp (scheduler, drawing, batching
    helpers), the B200 classes of hyperpose_api/*.cpp underneath, and the OpenCV / gflags stand-ins of csrc/shim (neither library
    exists in this image).  Nothing of the reference is copied: every source is compiled where it lies.  Returns {name: binary} in
    oracle/_ref/dropin/ref_build/, or the set built earlier / None where the reference tree is absent."""
    out_dir = os.path.join(REF_BIN, "ref_build")
    exes = {n: os.path.join(out_dir, n.replace(".example", "")) for n in REFERENCE_EXAMPLES}
    if not os.path.isdir(os.path.join(ref_root, "include", "hyperpose")):
        return exes if all(os.path.exists(e) for e in exes.values()) else None
    os.makedirs(out_dir, exist_ok=True)
    api = os.path.join(CSRC, "hyperpose_api")
    shim = os.path.join(CSRC, "shim")
    inc = ["-I" + shim, "-I" + os.path.join(ref_root, "include"), "-I" + os.path.join(ref_root, "src"), "-I" + os.path.join(ref_root, "examples"),
           "-I" + os.path.join(ROOT, "include")]
    common = [os.path.join(ref_root, "src", f) for f in ("stream.cpp", "thread_pool.cpp", "logging.cpp", "human.cpp", "data.cpp")]
    common += [os.path.join(ref_root, "examples", "utils.cpp")]
    common += [os.path.join(api, f) for f in ("paf.cpp", "tensorrt.cpp", "pifpaf.cpp", "pose_proposal.cpp")]
    shim_files = [os.path.join(dp, f) for dp, _, fs in os.walk(shim) for f in fs]
    objs = []
    for src in common:
        o = os.path.join(out_dir, ("ref_" if src.startswith(ref_root) else "b200_") + os.path.basename(src) + ".o")
        objs.append(o)
        if _newer([src] + shim_files + [os.path.join(ROOT, "include", "hyperpose_b200.h")], o):
            r = subprocess.run(["g++", "-std=c++17", "-O2", "-pthread", "-c"] + inc + [src, "-o", o], capture_output=True, text=True)
            if r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError(f"{src} failed to compile over the shim")
    for name, exe in exes.items():
        src = os.path.join(ref_root, "examples", name + ".cpp")
        if _newer([src, LIB] + objs, exe):
            cmd = ["g++", "-std=c++17", "-O2", "-pthread"] + inc + [src] + objs + ["-L" + PKG, "-lhyperpose_b200", "-Wl,-rpath,$ORIGIN/../../../../hyperpose_b200", "-o", exe]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError(f"reference example {name} failed to build unchanged against the drop-in")
    return exes


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
