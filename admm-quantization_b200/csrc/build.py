"""Build libadmmq.so (sm_100a) in-tree:  python admm-quantization_b200/csrc/build.py

nvcc cross-compiles without a GPU.  The shared library lands in
admm-quantization_b200/lib/libadmmq.so (git-ignored; it travels to the GPU box with gpurun).
"""
import hashlib
import json
import os
import shutil
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OUT_DIR = os.path.join(PKG, "lib")
OBJ_DIR = os.path.join(PKG, "build")
SOURCES = ["api.cu", "project.cu", "contract.cu", "admm_loop.cu", "mttkrp_tc.cu", "tc_gemm.cu", "factorize.cu", "code_gemm.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC,-fvisibility=hidden", "--fmad=true", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(paths, extra=""):
    """sha256 over the CONTENT of the given files (sorted by name) and a flags string: what an object depends on."""
    h = hashlib.sha256(extra.encode())
    for p in sorted(paths):
        h.update(os.path.basename(p).encode() + b"\0")
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stale(target, digest):
    """An object is current when it exists and was built from exactly these contents (hash, not mtime)."""
    try:
        with open(target + ".sha256") as f:
            return not os.path.exists(target) or f.read().strip() != digest
    except OSError:
        return True


def build(verbose=False, force=False):
    os.makedirs(OUT_DIR, exist_ok=True)
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(PKG), "include", "admmq.h"))
    force = force or bool(os.environ.get("ADMMQ_FORCE_BUILD"))
    objs, procs, digests = [], [], {}
    ver = subprocess.run([nvcc, "--version"], stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[-1]
    for src in SOURCES:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        digests[src] = _digest([os.path.join(HERE, src)] + headers, " ".join(FLAGS) + ver)
        if force or _stale(obj, digests[src]):
            cmd = [nvcc] + FLAGS + ["-c", os.path.join(HERE, src), "-o", obj]
            procs.append((src, obj, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, obj, cmd, pr in procs:
        out, _ = pr.communicate()
        log.append(f"$ {' '.join(cmd)}\n{out}")
        if pr.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError(f"nvcc failed on {src}")
        with open(obj + ".sha256", "w") as f:
            f.write(digests[src])
    built = {src for src, _, _, _ in procs}
    for src in SOURCES:
        if src not in built:
            log.append(f"{src}: up to date (sha256 of source + headers + flags {digests[src][:16]})")
    lib = os.path.join(OUT_DIR, "libadmmq.so")
    if procs or not os.path.exists(lib):
        cmd = [nvcc, "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        log.append(f"$ {' '.join(cmd)}\n{r.stdout}")
        if r.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError("link failed")
    with open(os.path.join(OBJ_DIR, "manifest.json"), "w") as f:
        json.dump({"nvcc": ver, "flags": FLAGS, "sources": digests, "rebuilt": sorted(built), "forced": bool(force),
                   "lib_sha256": _digest([lib])}, f, indent=1)
    with open(os.path.join(OBJ_DIR, "build.log"), "a") as f:
        f.write(f"==== {time.ctime()}\n" + "\n".join(log) + "\n")
    if verbose:
        print("\n".join(log))
    return lib


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
