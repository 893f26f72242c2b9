"""Build recipe of libsgmm_b200.so (nvcc, sm_100a only, in-tree).

    python -m sgmm_b200.build            # or: __graft_entry__.build()

The library is a plain C-ABI shared object (include/sgmm.h); cudart is linked statically so the
only run-time dependency is the NVIDIA driver.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsgmm_b200.so")
SOURCES = ["sgmm_capi.cu", "sgmm_rollout.cu", "sgmm_spec256.cu", "sgmm_tc32.cu", "sgmm_ga.cu", "sgmm_peak.cu", "sgmm_prep.cu", "sgmm_account.cu", "sgmm_one.cu", "sgmm_exact256.cu", "sgmm_trace_pop.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--fmad=false",                       # no implicit a*b+c contraction: every FMA is written as one
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
    "-Xptxas", "-v",
    "-cudart", "static",
]


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libsgmm_b200.so cannot be built")
    return p


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "sgmm.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(src, obj, extra):
    cmd = [nvcc_path()] + NVCC_FLAGS[:-2] + extra + ["-c", "-o", obj, src]       # [:-2]: -cudart static is a link flag
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return src, " ".join(cmd) + "\n" + r.stdout, r.returncode


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every translation unit (in parallel, one object per .cu under csrc/build/, recompiled only when it or a
    header changed unless ``force``) and link libsgmm_b200.so."""
    if not force and not needs_build():
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    missing = [p for p in srcs if not os.path.exists(p)]
    if missing:
        raise RuntimeError("libsgmm_b200.so cannot be built, missing translation units: " + ", ".join(missing))
    extra = os.environ.get("SGMM_EXTRA_NVCC_FLAGS", "").split()      # debug builds, e.g. -DSGMM_TC32_WATCHDOG / -DSGMM_SPEC256_TRACE
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    stamp = os.path.join(objdir, "flags.txt")
    flags_now = " ".join(NVCC_FLAGS + extra)
    flags_same = os.path.exists(stamp) and open(stamp).read() == flags_now
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "sgmm.h"))
    hdr_time = max(os.path.getmtime(h) for h in headers)
    jobs, objs = [], []
    for src in srcs:
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        fresh = (not force and flags_same and os.path.exists(obj)
                 and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_time))
        if not fresh:
            jobs.append((src, obj))
    log_parts, failed = [], []
    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        for src, out, rc in ex.map(lambda j: _compile_one(j[0], j[1], extra), jobs):
            log_parts.append(out)
            if rc != 0:
                failed.append(src)
    link = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", LIB] + objs
    if not failed:
        r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        log_parts.append(" ".join(link) + "\n" + r.stdout)
        if r.returncode != 0:
            failed.append("link")
    log = os.path.join(HERE, "csrc", "build.log")
    with open(log, "w") as f:
        f.write("\n".join(log_parts))
    if verbose or failed:
        sys.stderr.write("\n".join(log_parts))
    if failed:
        raise RuntimeError(f"nvcc failed for {failed}; see {log}")
    with open(stamp, "w") as f:
        f.write(flags_now)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
