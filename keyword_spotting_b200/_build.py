"""Build-at-import of libkws_b200.so, the way the reference builds its ops
(octbit/op_compile.py:27-79: compile the sources next to the wrapper, then load
the .so) -- with nvcc for sm_100a instead of g++, and ctypes instead of
tf.load_op_library.  The library is built IN-TREE so it travels with the repo
snapshot; there is no CPU fallback: if it can neither be found nor built the
import fails loudly.
"""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libkws_b200.so")
SOURCES = ["api.cu", "posenc.cu", "octbit.cu", "octbit_tc.cu", "frontend.cu", "frontend_tc.cu", "frontend_dft.cu", "gru.cu", "gru_octbit.cu", "gru_tc.cu", "decode.cu", "stream.cu", "server.cu", "tc_debug.cu", "attention.cu", "attention_tc.cu"]
OBJ_DIR = os.path.join(HERE, "build")
_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]   # B200 only
NVCC_COMPILE_FLAGS = _ARCH + ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
NVCC_LINK_FLAGS = _ARCH + ["-shared", "-Xcompiler", "-fPIC"]


def _nvcc():
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    return cand if os.path.exists(cand) else None


def _inputs():
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    files.append(os.path.join(os.path.dirname(HERE), "include", "kws_b200.h"))
    return files


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > built for f in _inputs() if os.path.exists(f))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into keyword_spotting_b200/libkws_b200.so."""
    override = os.environ.get("KWS_B200_LIB")            # experiments: a library built elsewhere (same ABI)
    if override and not force:
        if not os.path.exists(override):
            raise ImportError("KWS_B200_LIB=%s does not exist" % override)
        return override
    if not force and not is_stale():
        return LIB_PATH
    nvcc = _nvcc()
    if nvcc is None:
        if os.path.exists(LIB_PATH):
            return LIB_PATH          # stale but usable (e.g. mtimes scrambled by a copy)
        raise ImportError("libkws_b200.so is not built and nvcc was not found; "
                          "keyword_spotting_b200 has no CPU fallback")
    # one nvcc -c per source, in parallel (objects cached under csrc/../build/ by mtime), then one link step
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [f for f in _inputs() if not f.endswith(".cu")]
    newest_header = max(os.path.getmtime(f) for f in headers if os.path.exists(f))
    log = []

    def compile_one(src):
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ_DIR, src[:-3] + ".o")
        if (not force and os.path.exists(obj) and os.path.getmtime(obj) > os.path.getmtime(path)
                and os.path.getmtime(obj) > newest_header):
            return obj, 0, ""
        cmd = [nvcc] + NVCC_COMPILE_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj + ".tmp"]
        proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if proc.returncode == 0:
            os.replace(obj + ".tmp", obj)
        return obj, proc.returncode, proc.stdout

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    for obj, rc, out in results:
        log.append(out)
        if rc != 0:
            raise ImportError("nvcc failed building %s:\n%s" % (obj, out))
    tmp = LIB_PATH + ".tmp.%d" % os.getpid()
    cmd = [nvcc] + NVCC_LINK_FLAGS + ["-o", tmp] + [r[0] for r in results]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise ImportError("nvcc failed linking libkws_b200.so:\n" + proc.stdout)
    if verbose:
        print("".join(log))
    os.replace(tmp, LIB_PATH)
    return LIB_PATH
