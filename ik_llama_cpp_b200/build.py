"""Build libb200q.so (sm_100a only) in-tree with nvcc.  `python -m ik_llama_cpp_b200.build [--force]`."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200q.so")
OBJDIR = os.path.join(HERE, "_obj")
SOURCES = ["b200q_decode_i0.cu", "b200q_decode_i1.cu", "b200q_decode_i2.cu", "b200q_decode_i3.cu", "b200q_wire.cu", "b200q_decode.cu", "b200q_gemm.cu", "b200q_reduce.cu", "b200q_api.cu"]
HEADERS = ["b200q_types.cuh", "b200q_internal.h", "b200q_wire.cuh", "b200q_codebooks.h", "b200q_decode_common.cuh", "b200q_decode_ring.cuh", "b200q_decode_inst.inc", os.path.join("..", "..", "include", "b200q.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_native(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJDIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        if force or _stale(obj, [os.path.join(CSRC, src)] + hdrs):
            cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB, *objs, "-cudart", "static", "-Xlinker", "--no-undefined"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


PLUG_SRC = os.path.join(HERE, "backend_plug", "ggml_b200_backend.cpp")
PLUG_LIB = os.path.join(HERE, "libggml_b200.so")
REFERENCE_ROOT = "/root/reference"


def build_backend_plug(force: bool = False, verbose: bool = False) -> str | None:
    """libggml_b200.so: the ggml-backend vtable + ggml-cuda.h symbols on top of libb200q.so.  It is compiled against the
    reference's headers where they lie, so it can only be (re)built where /root/reference exists; the GPU box gets the prebuilt file.
    Like the CUDA backend it replaces, it is a plug-in of ggml: the ggml_* core symbols it calls (ggml_backend_buffer_init, ggml_nbytes,
    the backend registry ...) stay UNDEFINED in the library and are resolved by the libggml of the process that loads it (llama-bench /
    llama-server in the reference; the test harness links the reference build for that).  Nothing under oracle/ is linked here."""
    if not os.path.isdir(REFERENCE_ROOT):
        return PLUG_LIB if os.path.exists(PLUG_LIB) else None
    if force or _stale(PLUG_LIB, [PLUG_SRC, LIB, os.path.join(os.path.dirname(HERE), "include", "b200q.h"), os.path.abspath(__file__)]):
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", PLUG_LIB, PLUG_SRC,
               f"-I{REFERENCE_ROOT}/ggml/include", f"-I{REFERENCE_ROOT}/ggml/src", f"-I{os.path.join(os.path.dirname(HERE), 'include')}",
               "-I/usr/local/cuda/include", "-DGGML_SHARED", "-DGGML_USE_CUDA", f"-L{HERE}", "-lb200q",
               "-L/usr/local/cuda/lib64", "-lcudart_static", "-ldl", "-lrt", "-lpthread", "-Wl,-rpath,$ORIGIN"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return PLUG_LIB


def build_backend_ops_test(force: bool = False) -> str | None:
    """tests/backend_ops/test_mul_mat_backend: test-backend-ops semantics through the real ggml-backend API."""
    root = os.path.dirname(HERE)
    exe = os.path.join(root, "tests", "backend_ops", "test_mul_mat_backend")
    src = exe + ".cpp"
    if not os.path.isdir(REFERENCE_ROOT):
        return exe if os.path.exists(exe) else None
    plug = build_backend_plug(force)
    ref_lib = os.path.join(root, "oracle", "_ref", "libggml_ref_avx2.so")
    if plug is None:
        return None
    if not os.path.exists(ref_lib):
        return None
    if force or _stale(exe, [src, plug]):
        # libraries by file name (-L/-l), found through RUNPATH: full paths on the link line would be recorded as absolute DT_NEEDED
        # entries, and the executable would not load once the tree is somewhere else
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, src, f"-I{REFERENCE_ROOT}/ggml/include", f"-I{REFERENCE_ROOT}/ggml/src",
                               f"-L{HERE}", "-lggml_b200", "-lb200q", f"-L{os.path.dirname(ref_lib)}", "-lggml_ref_avx2", "-lpthread", "-ldl",
                               "-Wl,-rpath,$ORIGIN/../../ik_llama_cpp_b200", "-Wl,-rpath,$ORIGIN/../../oracle/_ref"])
    return exe


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose=True))
    print(build_backend_plug(force="--force" in sys.argv, verbose=True))
    print(build_backend_ops_test(force="--force" in sys.argv))
