"""Builds libagarcl_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libagarcl_b200.so")
SOURCES = ["sim_kernel.cu", "obs_kernel.cu", "ram_kernel.cu", "reset_kernel.cu", "episode_kernel.cu", "snapshot_kernel.cu", "archive_kernel.cu", "draw_kernel.cu", "bot_kernel.cu", "batch.cu", "mirror.cu", "layout.cpp", "host_util.cpp", "snapshot.cpp"]
HEADERS = ["device_math.cuh", "block_copy.cuh", "mode_rules.h", "sim_params.h", "sim_shared.cuh", "host_util.h", "mirror.h", os.path.join("..", "..", "include", "agarcl_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false",  # the reference host build has no FMA contraction (SURVEY Appendix A)
              "-ccbin", "g++", "-Xcompiler", "-fPIC", "-shared"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def pybind_module_path():
    import sysconfig
    return os.path.join(HERE, "agarcl" + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))


def build_pybind(force=False):
    """The reference's Python module `agarcl` (environment/bindings.cpp) over the C ABI: csrc/pybind_agarcl.cpp ->
    agarcl_b200/agarcl.<abi>.so, linked against libagarcl_b200.so next to it ($ORIGIN rpath)."""
    import sysconfig
    import pybind11
    out, src = pybind_module_path(), os.path.join(CSRC, "pybind_agarcl.cpp")
    deps = [src, LIB, os.path.join(HERE, "..", "include", "agarcl_b200.h")]
    if not force and os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    # the system g++ (what nvcc uses as -ccbin), NOT $CXX: the image's /opt/gcc links its own libstdc++ statically, which clashes with the
    # interpreter's at run time
    cmd = [os.environ.get("AGARCL_CXX", "g++"), "-O2", "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", "-I" + pybind11.get_include(),
           "-I" + sysconfig.get_paths()["include"], src, "-o", out, "-L" + HERE, "-lagarcl_b200", "-Wl,-rpath,$ORIGIN"]
    subprocess.check_call(cmd)
    return out


def nvcc_command(out, extra=(), verbose=False):
    """The nvcc command that compiles SOURCES into the shared library `out`: the product library, and the variants of
    tools/build_variant.sh (`extra`: more nvcc flags)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return [nvcc] + NVCC_FLAGS + list(extra) + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + [os.path.join(CSRC, f) for f in SOURCES]


def build(force=False, verbose=False):
    if force or needs_build():
        subprocess.check_call(nvcc_command(LIB, verbose=verbose))
    build_pybind(force)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
