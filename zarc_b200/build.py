"""Build libzarcgpu.so (product: nvcc, sm_100a) in-tree, and -- for the CPU test-suite only -- the
SIMT-emulator build of the very same kernel sources (tests/simt_emu/, g++)."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "zarc_b200", "csrc")
PRODUCT_SO = os.path.join(ROOT, "zarc_b200", "libzarcgpu.so")
EMU_DIR = os.path.join(ROOT, "tests", "simt_emu")
EMU_SO = os.path.join(EMU_DIR, "libzarcgpu_emu.so")
OBJ = os.path.join(ROOT, "build")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v",
]


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _deps_mtime():
    files = glob.glob(os.path.join(CSRC, "*")) + glob.glob(os.path.join(ROOT, "include", "*.h"))
    return max(os.path.getmtime(f) for f in files)


def _stale(target: str, extra: list[str] = ()) -> bool:
    if not os.path.exists(target):
        return True
    m = max([_deps_mtime()] + [os.path.getmtime(f) for f in extra])
    return os.path.getmtime(target) < m


def _into(target: str, make) -> None:
    """Run make(tmp) and move tmp over target: a process that loads the target while another one rebuilds it (the forked
    workers of bench.py's CPU arm, pytest-xdist) sees the old file or the new one, never half of one."""
    tmp = f"{target}.{os.getpid()}.tmp"
    try:
        make(tmp)
        os.replace(tmp, target)
    finally:
        if os.path.exists(tmp):
            os.unlink(tmp)


def build_product(force: bool = False, verbose: bool = False, target: str = PRODUCT_SO, objdir: str = OBJ, defines=()) -> str:
    """nvcc -> zarc_b200/libzarcgpu.so.  Cross-compiles without a GPU."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not force and not _stale(target):
        return target
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libzarcgpu.so (there is no CPU fallback)")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in _sources():
        o = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        objs.append(o)
        cmd = [nvcc, *NVCC_FLAGS, *[f"-D{d}" for d in defines], *os.environ.get("ZG_NVCC_EXTRA", "").split(), "-I", CSRC, "-c", src, "-o", o]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {os.path.basename(src)}\n{out}")
        if p.returncode:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(objdir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    _into(target, lambda tmp: subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp, *objs, "-lcudart"]))
    return target


def build_emu(force: bool = False, target: str = EMU_SO, objdir: str = os.path.join(OBJ, "emu"), defines=()) -> str:
    """g++ -DZG_EMU -> tests/simt_emu/libzarcgpu_emu.so (TEST INFRASTRUCTURE ONLY)."""
    emu_src = [os.path.join(EMU_DIR, "simt_emu.cpp")]
    if not force and not _stale(target, emu_src + [os.path.join(EMU_DIR, "simt_emu.h")]):
        return target
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    flags = ["-O2", "-g", "-std=c++17", "-fPIC", "-DZG_EMU", "-I", EMU_DIR, "-I", CSRC, "-Wall", "-Wno-unused-function",
             "-Wno-unknown-pragmas", "-Wno-unused-variable", "-Wno-sign-compare", "-Wno-stringop-overflow", "-Wno-maybe-uninitialized", "-Wno-array-bounds"]
    for src in _sources() + emu_src:
        o = os.path.join(objdir, os.path.basename(src).rsplit(".", 1)[0] + ".o")
        objs.append(o)
        cmd = ["g++", *flags, *[f"-D{d}" for d in defines], *os.environ.get("ZG_EMU_EXTRA", "").split(), "-x", "c++", "-c", src, "-o", o]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if out.strip():
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"g++ (emu) failed on {src}")
    _into(target, lambda tmp: subprocess.check_call(["g++", "-shared", "-o", tmp, *objs]))
    return target


# Rare-path builds: the same sources with tuning constants overridden (-DNAME=VALUE), each in its own directory under
# build/variants/, so that tests can force the paths the defaults take rarely (tests/test_encoder_edges_*.py).  They never
# touch libzarcgpu.so or libzarcgpu_emu.so.
VARIANTS = os.path.join(OBJ, "variants")


def _variant_dir(defines, kind: str) -> str:
    name = "_".join(d.replace("=", "-") for d in defines) or "default"
    return os.path.join(VARIANTS, kind, "".join(c if c.isalnum() or c in "-_" else "_" for c in name))


def build_emu_variant(defines, force: bool = False) -> str:
    d = _variant_dir(defines, "emu")
    return build_emu(force, target=os.path.join(d, "libzarcgpu_emu.so"), objdir=os.path.join(d, "obj"), defines=defines)


def build_product_variant(defines, force: bool = False) -> str:
    d = _variant_dir(defines, "product")
    return build_product(force, target=os.path.join(d, "libzarcgpu.so"), objdir=os.path.join(d, "obj"), defines=defines)


HOST_DIR = os.path.join(ROOT, "zarc_b200", "host")
HOST_BIN = os.path.join(ROOT, "zarc_b200", "zarc-b200")


def build_host(force: bool = False) -> str:
    """g++ -> zarc_b200/zarc-b200: the C++ host (Encoder/Decoder mirror, container format, CLI).  It binds
    libzarcgpu.so at run time (dlopen); no codec is linked into it."""
    srcs = [os.path.join(HOST_DIR, f) for f in ("zarc_host.cpp", "zarc_cli.cpp")]
    deps = glob.glob(os.path.join(HOST_DIR, "*")) + glob.glob(os.path.join(ROOT, "include", "*.h"))
    if not force and os.path.exists(HOST_BIN) and os.path.getmtime(HOST_BIN) >= max(os.path.getmtime(f) for f in deps):
        return HOST_BIN
    _into(HOST_BIN, lambda tmp: subprocess.check_call(["g++", "-O2", "-g", "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter",
                                                       "-Wno-missing-field-initializers", *srcs, "-o", tmp, "-ldl"]))
    return HOST_BIN


CORPUS_SO = os.path.join(ROOT, "tools", "libzarc_corpus.so")


def build_corpus_host(force: bool = False) -> str:
    """g++ -> tools/libzarc_corpus.so: the corpus generator alone, for the CPU reference arm of bench.py (which must
    not load the product library)."""
    src = os.path.join(ROOT, "tools", "corpus_host.cpp")
    deps = [src, os.path.join(CSRC, "corpus.cuh"), os.path.join(CSRC, "simt.h")]
    if not force and os.path.exists(CORPUS_SO) and os.path.getmtime(CORPUS_SO) >= max(os.path.getmtime(f) for f in deps):
        return CORPUS_SO
    _into(CORPUS_SO, lambda tmp: subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-DZG_EMU", "-I", EMU_DIR, "-I", CSRC,
                                                        "-Wno-unused-function", src, "-o", tmp]))
    return CORPUS_SO


if __name__ == "__main__":
    which = sys.argv[1:] or ["product"]
    if "product" in which:
        print(build_product(force="--force" in which, verbose="-v" in which))
    if "emu" in which:
        print(build_emu(force="--force" in which))
    if "host" in which:
        print(build_host(force="--force" in which))
    if "corpus" in which:
        print(build_corpus_host(force="--force" in which))
