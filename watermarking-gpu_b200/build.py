"""In-tree build of libwm_b200.so (hand-written sm_100a CUDA + the C ABI of include/wm_b200.h).

`python watermarking-gpu_b200/build.py [--force]`; also called by __graft_entry__.build().
nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libwm_b200.so")
SOURCES = [os.path.join(CSRC, f) for f in ("wm_api.cu", "wm_k_sweep.cu", "wm_k_stats.cu", "wm_k_apply.cu", "wm_k_detect.cu", "wm_k_nvfp.cu")]
DEPS = SOURCES + [os.path.join(CSRC, "wm_kernels.cuh"), os.path.join(CSRC, "wm_launch.h"), os.path.join(ROOT, "include", "wm_b200.h")]
OBJDIR = os.path.join(HERE, "build")

NVCC = os.environ.get("WM_NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-ccbin", "/usr/bin/g++",
         "-Xcompiler", "-fPIC"]
LINK_FLAGS = ["-shared", "-cudart", "static"]


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    # one translation unit per kernel family, compiled in parallel, then linked into the shared library
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJDIR, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJDIR, os.path.basename(src)[:-3] + ".o")
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    if verbose:
        for _, err in results:
            sys.stderr.write(err)
    cmd = [NVCC] + FLAGS + LINK_FLAGS + ["-o", LIB] + [o for o, _ in results]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return LIB


def build_facade_test(force=False):
    """C++ smoke/parity program over the Watermark façade (csrc/Watermark.hpp), linked against the .so."""
    return _build_cpp_test("test_facade", force)


def build_video_packed_test(force=False):
    """C++ program running processFramesInMemory (csrc/videoprocessingcontext.hpp) on packed BGR frames, linked against the .so."""
    return _build_cpp_test("test_video_packed", force)


def build_video_yuv422_test(force=False):
    """C++ program running processFramesInMemory (csrc/videoprocessingcontext.hpp) on packed YUYV frames, linked against the .so."""
    return _build_cpp_test("test_video_yuv422", force)


def build_video_y10_test(force=False):
    """C++ program running processFramesInMemory (csrc/videoprocessingcontext.hpp) on 10-bit luma frames, linked against the .so."""
    return _build_cpp_test("test_video_y10", force)


def build_video_v210_test(force=False):
    """C++ program running processFramesInMemory (csrc/videoprocessingcontext.hpp) on v210 frames, linked against the .so."""
    return _build_cpp_test("test_video_v210", force)


def _build_cpp_test(name, force):
    src = os.path.join(ROOT, "tests", "cpp", name + ".cpp")
    exe = os.path.join(ROOT, "tests", "cpp", name)
    if not os.path.exists(src):
        return None
    deps = [src, os.path.join(CSRC, "Watermark.hpp"), os.path.join(CSRC, "videoprocessingcontext.hpp"), LIB]
    if not force and os.path.exists(exe) and all(os.path.getmtime(d) <= os.path.getmtime(exe) for d in deps if os.path.exists(d)):
        return exe
    cmd = ["/usr/bin/g++", "-O2", "-std=c++20", "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", exe, src,
           "-L", HERE, "-lwm_b200", "-Wl,-rpath,$ORIGIN/../../watermarking-gpu_b200", "-ldl", "-lpthread", "-lrt"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    return exe


def build_generator(force=False):
    """tools/CommonRandomMatrix: the watermark-file generator (host-only C++)."""
    src = os.path.join(ROOT, "tools", "CommonRandomMatrix", "generate_w.cpp")
    exe = os.path.join(ROOT, "tools", "CommonRandomMatrix", "CommonRandomMatrix")
    if not os.path.exists(src):
        return None
    if not force and os.path.exists(exe) and os.path.getmtime(exe) >= os.path.getmtime(src):
        return exe
    r = subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-o", exe, src], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed:\n" + r.stdout + r.stderr)
    return exe


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_facade_test(force="--force" in sys.argv))
    print(build_video_packed_test(force="--force" in sys.argv))
    print(build_video_yuv422_test(force="--force" in sys.argv))
    print(build_video_y10_test(force="--force" in sys.argv))
    print(build_video_v210_test(force="--force" in sys.argv))
    print(build_generator(force="--force" in sys.argv))
