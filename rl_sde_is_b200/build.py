"""In-tree build of librlsde_b200.so (sm_100a) and of the C oracle (test infrastructure).

    python -m rl_sde_is_b200.build            # incremental
    python -m rl_sde_is_b200.build --force    # rebuild everything

nvcc cross-compiles without a GPU.  Every translation unit is compiled with
``-gencode arch=compute_100a,code=sm_100a -lineinfo`` and linked into
``rl_sde_is_b200/librlsde_b200.so`` (git-ignored, travels with gpurun snapshots).
"""
import argparse
import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
# A/B variants for kernel experiments: RLSDE_VARIANT=name RLSDE_NVCC_EXTRA="-DFOO=1" builds librlsde_b200_name.so
# from its own object directory; select it at run time with RLSDE_LIB_PATH.
VARIANT = os.environ.get("RLSDE_VARIANT", "")
# RLSDE_VARIANT_ONLY=prefix[,prefix]: only the translation units whose name starts with one of the prefixes are rebuilt
# with the variant's flags; all others are taken from the default build's object directory (fast A/B builds of one kernel)
VARIANT_ONLY = [p for p in os.environ.get("RLSDE_VARIANT_ONLY", "").split(",") if p]
BASE_OBJ_DIR = os.path.join(ROOT, "build", "obj")
OBJ_DIR = os.path.join(ROOT, "build", "obj" + ("_" + VARIANT if VARIANT else ""))
LIB_PATH = os.path.join(PKG_DIR, "librlsde_b200" + ("_" + VARIANT if VARIANT else "") + ".so")
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "librlsde_oracle.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr",
] + os.environ.get("RLSDE_NVCC_EXTRA", "").split()


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build librlsde_b200.so")
    return exe


def _headers_digest():
    h = hashlib.sha256()
    for d in (CSRC, os.path.join(ROOT, "include")):
        for f in sorted(os.listdir(d)):
            if f.endswith((".cuh", ".h")):
                with open(os.path.join(d, f), "rb") as fh:
                    h.update(f.encode())
                    h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile_one(args):
    src, obj, stamp, digest, verbose = args
    cmd = [_nvcc()] + NVCC_FLAGS + ["-I", CSRC, "-c", src, "-o", obj]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        return src, False, res.stdout + res.stderr
    with open(stamp, "w") as fh:
        fh.write(digest)
    return src, True, res.stdout + res.stderr


def build_cuda(force=False, verbose=False, jobs=None):
    os.makedirs(OBJ_DIR, exist_ok=True)
    digest_h = _headers_digest()
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))
    todo, objs = [], []
    for f in sources:
        src = os.path.join(CSRC, f)
        if VARIANT and VARIANT_ONLY and not any(f.startswith(p) for p in VARIANT_ONLY):
            objs.append(os.path.join(BASE_OBJ_DIR, f[:-3] + ".o"))      # shared with the default build (must be up to date)
            continue
        obj = os.path.join(OBJ_DIR, f[:-3] + ".o")
        stamp = obj + ".stamp"
        with open(src, "rb") as fh:
            digest = hashlib.sha256(fh.read() + digest_h.encode()).hexdigest()
        objs.append(obj)
        fresh = (not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == digest)
        if not fresh:
            todo.append((src, obj, stamp, digest, verbose))
    if todo:
        jobs = jobs or min(len(todo), os.cpu_count() or 4)
        print(f"[rlsde build] compiling {len(todo)} translation unit(s) with {jobs} job(s) ...", flush=True)
        with concurrent.futures.ThreadPoolExecutor(max_workers=jobs) as pool:
            for src, ok, log in pool.map(_compile_one, todo):
                if verbose and log.strip():
                    print(log)
                if not ok:
                    raise RuntimeError(f"nvcc failed on {src}:\n{log}")
    need_link = bool(todo) or not os.path.exists(LIB_PATH) or any(
        os.path.getmtime(o) > os.path.getmtime(LIB_PATH) for o in objs)
    if need_link:
        cmd = [_nvcc(), "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                             "-Xcompiler", "-fPIC", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
        print(f"[rlsde build] linked {LIB_PATH} ({os.path.getsize(LIB_PATH) / 1e6:.1f} MB)", flush=True)
    return LIB_PATH


def build_oracle(force=False):
    """Plain-C restatement used by tests / bench cpu_baseline only (see oracle/README.md)."""
    src = os.path.join(ORACLE_DIR, "rlsde_oracle.c")
    if not os.path.exists(src):
        return None
    if not force and os.path.exists(ORACLE_LIB) and os.path.getmtime(ORACLE_LIB) >= os.path.getmtime(src):
        return ORACLE_LIB
    cmd = ["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", ORACLE_LIB, src, "-lm"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + res.stdout + res.stderr)
    print(f"[rlsde build] built {ORACLE_LIB}", flush=True)
    return ORACLE_LIB


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--jobs", type=int, default=None)
    a = ap.parse_args()
    build_cuda(force=a.force, verbose=a.verbose, jobs=a.jobs)
    build_oracle(force=a.force)


if __name__ == "__main__":
    sys.exit(main())
