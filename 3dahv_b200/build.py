"""Build lib3dahv_b200.so in-tree with nvcc for sm_100a (no torch headers, plain C ABI).

    python 3dahv_b200/build.py [--force] [--verbose] [-DNAME[=VALUE] ... --out=path/to/variant.so]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib3dahv_b200.so")
SOURCES = ["ahv_api.cu", "ahv_so3.cu", "ahv_score_fp32.cu", "ahv_score_bwd.cu", "ahv_ascent.cu", "ahv_score_bwd_tc.cu", "ahv_score_tc.cu", "ahv_topk.cu", "ahv_topk_distinct.cu", "ahv_diag.cu", "ahv_exchange.cu", "ahv_lift.cu", "ahv_infonce.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "--fmad=true",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


STAMP = os.path.join(HERE, "build", "built_on.txt")


def _machine_id() -> str:
    import socket
    ids = []
    for path in ("/etc/machine-id", "/proc/sys/kernel/random/boot_id"):
        try:
            with open(path) as f:
                ids.append(f.read().strip())
        except OSError:
            ids.append("")
    return ":".join([socket.gethostname()] + ids)


def _write_stamp() -> None:
    with open(STAMP, "w") as f:
        f.write(_machine_id() + "\n")


def needs_build() -> bool:
    """Rebuild when the library is missing, older than any source, or was not produced on THIS machine (a
    prebuilt binary that travelled with a snapshot is never trusted by `build()`; the loader still uses it when
    nobody calls build first, which is what lets the GPU box run the library built in the build container)."""
    if not os.path.exists(LIB):
        return True
    try:
        with open(STAMP) as f:
            if f.read().strip() != _machine_id():
                return True
    except OSError:
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps.append(os.path.join(HERE, "..", "include", "ahv_b200.h"))
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, defines=(), out: str | None = None) -> str:
    """Product build: `build()` -> 3dahv_b200/lib3dahv_b200.so.  Experiment / diagnostics builds (scripts/ only):
    `build(defines=["AHV_STAGES=2"], out="experiments/variants/lib_stages2.so")` compile the same sources with
    extra -D flags into another file; the product loader never looks at those."""
    variant = out is not None
    lib_out = os.path.abspath(out) if variant else LIB
    if not variant and not force and not needs_build():
        return LIB
    flags = NVCC_FLAGS + [f"-D{d}" for d in defines]
    objs = []
    build_dir = os.path.join(HERE, "build", os.path.splitext(os.path.basename(lib_out))[0]) if variant else os.path.join(HERE, "build")
    os.makedirs(os.path.dirname(lib_out), exist_ok=True)
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [_nvcc(), *flags, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(build_dir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    cmd = [_nvcc(), "-shared", "-o", lib_out, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xcompiler", "-fvisibility=hidden"]
    subprocess.check_call(cmd)
    if not variant:
        _write_stamp()
    return lib_out


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, defines=defs, out=outs[0] if outs else None))
