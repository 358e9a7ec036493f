"""Builds libpxr.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["pxr_api.cu", "pxr_upload.cu", "pxr_ba.cu", "pxr_ba_block.cu", "pxr_refs.cu", "pxr_ka.cu", "pxr_synth.cu", "pxr_extract.cu", "pxr_problem.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "--expt-relaxed-constexpr",
         "-Xptxas", "-v"]
if os.environ.get("PXR_FM_WARPS"):
    FLAGS.append("-DPXR_FM_WARPS=" + os.environ["PXR_FM_WARPS"])


def _newer(src, obj):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    deps = [src] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(HERE, "..", "include", "pxr.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def compile_one(name, verbose):
    src = os.path.join(CSRC, name)
    obj = os.path.join(CSRC, name.replace(".cu", ".o"))
    if not _newer(src, obj):
        return name, "up to date"
    cmd = [NVCC] + FLAGS + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = os.path.join(CSRC, name.replace(".cu", ".ptxas.log"))
    with open(log, "w") as f:
        f.write(r.stderr)
    if r.returncode != 0:
        sys.stderr.write(r.stderr[-6000:])
        raise RuntimeError("nvcc failed for " + name)
    return name, "compiled"


def build(verbose=False):
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        for name, status in ex.map(lambda n: compile_one(n, verbose), srcs):
            if verbose:
                print("  %-16s %s" % (name, status))
    objs = [os.path.join(CSRC, s.replace(".cu", ".o")) for s in srcs]
    out = os.path.join(CSRC, "libpxr.so")
    if (not os.path.exists(out)) or any(os.path.getmtime(o) > os.path.getmtime(out) for o in objs):
        cmd = [NVCC, "-shared", "-o", out] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                     "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-lcudart", "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stderr[-4000:])
            raise RuntimeError("link failed")
    return out


def build_bindings(verbose=False):
    """bindings/_pxr_pybind*.so: the pybind11 binding of the C-ABI (host C++, g++).  Needs libpxr.so to link against.
    A machine without pybind11 / Python headers gets a warning, not a failed CUDA build."""
    import sysconfig
    src = os.path.join(HERE, "bindings", "pxr_pybind.cc")
    try:
        import pybind11
    except ImportError:
        sys.stderr.write("pybind11 not importable: bindings/_pxr_pybind is not built\n")
        return None
    out = os.path.join(HERE, "bindings", "_pxr_pybind" + sysconfig.get_config_var("EXT_SUFFIX"))
    deps = [src, os.path.join(HERE, "..", "include", "pxr.h"), os.path.join(CSRC, "libpxr.so")]
    if os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + pybind11.get_include(),
           "-I" + sysconfig.get_paths()["include"], src, "-o", out, "-L" + CSRC, "-lpxr", "-Wl,-rpath,$ORIGIN/../csrc"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write("bindings/_pxr_pybind did not build:\n" + r.stderr[-3000:])
        return None
    if verbose:
        print("  %-16s compiled" % "pxr_pybind.cc")
    return out


if __name__ == "__main__":
    print(build(verbose=True))
    print(build_bindings(verbose=True))
