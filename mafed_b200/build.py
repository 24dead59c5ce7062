"""Build the native code in-tree (sm_100a only):

* ``_lib/libmafed_distill.so`` -- the C ABI (``include/mafed_distill.h``) over the CUDA kernels.  Two translation
  units: ``distill_abi.cu`` (whole-program compiled: every ordinary launch) and ``distill_gate.cu`` (relocatable
  device code, device-linked with cudadevrt: the gated backward whose 1-CTA gate starts the real kernel from the
  device).  No torch anywhere in it.
* ``_lib/libmafed_teacher_gather.so`` -- the teacher-cache gather kernel (``csrc/teacher_gather.cu``) behind its own
  C ABI (``include/mafed_teacher_gather.h``), bound by ``mafed_b200.teacher_cache``.  A unit of its own, so the
  distillation library and its export list stay as they are.
* ``_lib/libmafed_cached_step.so`` -- the one-pass step that reads a replay batch's teacher rows straight from the
  teacher cache (``csrc/cached_step.cu``, the TMA-ring kernels of the distillation library with the cache's
  addressing) behind its own C ABI (``include/mafed_cached_step.h``), bound lazily by the torch extension.  A unit of
  its own for the same reason.
* ``_lib/mafed_torch_node*.so`` -- the torch extension (``csrc/torch_node.cpp``, host C++ only): the autograd node
  that turns one ``distill()`` into one call of the C ABI without Python on the hot path.
"""
import hashlib
import os
import shutil
import subprocess
import sysconfig

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
LIB_DIR = os.path.join(PKG, "_lib")
OBJ_DIR = os.path.join(LIB_DIR, "obj")
LIB_PATH = os.path.join(LIB_DIR, "libmafed_distill.so")
CSRC = os.path.join(PKG, "csrc")
SOURCES = [os.path.join(CSRC, "distill_abi.cu"), os.path.join(CSRC, "distill_gate.cu")]
HEADERS = [os.path.join(CSRC, n) for n in
           ("distill_common.cuh", "distill_ldg.cuh", "distill_tma.cuh", "distill_epilogue.cuh",
            "distill_comm.cuh", "distill_host.cuh", "distill_dispatch.cuh", "distill_gate.h")] + \
          [os.path.join(ROOT, "include", "mafed_distill.h")]

GATHER_SOURCE = os.path.join(CSRC, "teacher_gather.cu")
GATHER_HEADER = os.path.join(ROOT, "include", "mafed_teacher_gather.h")
GATHER_LIB_PATH = os.path.join(LIB_DIR, "libmafed_teacher_gather.so")
GATHER_STAMP_PATH = os.path.join(LIB_DIR, "gather.stamp")

CACHED_SOURCE = os.path.join(CSRC, "cached_step.cu")
CACHED_HEADER = os.path.join(ROOT, "include", "mafed_cached_step.h")
CACHED_LIB_PATH = os.path.join(LIB_DIR, "libmafed_cached_step.so")
CACHED_STAMP_PATH = os.path.join(LIB_DIR, "cached_step.stamp")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", *ARCH, "-lineinfo", "-Xcompiler", "-fPIC"]

EXT_NAME = "mafed_torch_node"
EXT_SOURCE = os.path.join(CSRC, "torch_node.cpp")
EXT_PATH = os.path.join(LIB_DIR, EXT_NAME + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-Wall", "-Wno-unused-function"]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA path cannot be built (there is no CPU fallback)")
    return exe


def _fingerprint(files, flags):
    """Hash of sources / headers and the compile flags (mtimes do not survive a copy to another box)."""
    h = hashlib.sha1(" ".join(flags).encode())
    for f in files:
        if os.path.exists(f):
            with open(f, "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()


def _stale(target, stamp, fingerprint):
    if not os.path.exists(target) or not os.path.exists(stamp):
        return True
    with open(stamp) as f:
        return f.read().strip() != fingerprint


STAMP_PATH = os.path.join(LIB_DIR, "build.stamp")
EXT_STAMP_PATH = os.path.join(LIB_DIR, "ext.stamp")


def is_stale():
    return _stale(LIB_PATH, STAMP_PATH, _fingerprint(SOURCES + HEADERS, NVCC_FLAGS))


def _run(cmds, verbose):
    """Run the commands concurrently; raise with the compiler output if one fails."""
    procs = [subprocess.Popen(c, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for c in cmds]
    outs = [p.communicate()[0] for p in procs]
    for c, p, out in zip(cmds, procs, outs):
        if p.returncode != 0:
            raise RuntimeError("command failed: " + " ".join(c) + "\n" + out)
        if verbose:
            print(out)


def build(force=False, verbose=False):
    """Compile libmafed_distill.so for sm_100a if missing or older than its sources."""
    fp = _fingerprint(SOURCES + HEADERS, NVCC_FLAGS)
    if not force and not _stale(LIB_PATH, STAMP_PATH, fp):
        return LIB_PATH
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    inc = ["-I", os.path.join(ROOT, "include"), "-I", CSRC]
    extra = ["-Xptxas=-v"] if verbose else []
    abi_o, gate_o, dlink_o = (os.path.join(OBJ_DIR, n) for n in ("distill_abi.o", "distill_gate.o", "distill_gate_dlink.o"))
    _run([[nvcc, *NVCC_FLAGS, *extra, *inc, "-c", SOURCES[0], "-o", abi_o],
          [nvcc, *NVCC_FLAGS, *extra, *inc, "-rdc=true", "-c", SOURCES[1], "-o", gate_o]], verbose)
    _run([[nvcc, *ARCH, "-Xcompiler", "-fPIC", "-dlink", gate_o, "-o", dlink_o, "-lcudadevrt"]], verbose)
    _run([[nvcc, *ARCH, "-shared", "-Xcompiler", "-fPIC", abi_o, gate_o, dlink_o, "-o", LIB_PATH, "-lcudadevrt"]], verbose)
    with open(STAMP_PATH, "w") as f:
        f.write(fp)
    return LIB_PATH


def build_teacher_gather(force=False, verbose=False):
    """Compile libmafed_teacher_gather.so for sm_100a if missing or older than its source."""
    fp = _fingerprint([GATHER_SOURCE, GATHER_HEADER], NVCC_FLAGS)
    if not force and not _stale(GATHER_LIB_PATH, GATHER_STAMP_PATH, fp):
        return GATHER_LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    extra = ["-Xptxas=-v"] if verbose else []
    _run([[_nvcc(), *NVCC_FLAGS, *extra, "-I", os.path.join(ROOT, "include"), "-shared", GATHER_SOURCE,
           "-o", GATHER_LIB_PATH]], verbose)
    with open(GATHER_STAMP_PATH, "w") as f:
        f.write(fp)
    return GATHER_LIB_PATH


def build_cached_step(force=False, verbose=False):
    """Compile libmafed_cached_step.so for sm_100a if missing or older than its source or the kernel headers."""
    fp = _fingerprint([CACHED_SOURCE, CACHED_HEADER] + HEADERS, NVCC_FLAGS)
    if not force and not _stale(CACHED_LIB_PATH, CACHED_STAMP_PATH, fp):
        return CACHED_LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    extra = ["-Xptxas=-v"] if verbose else []
    _run([[_nvcc(), *NVCC_FLAGS, *extra, "-I", os.path.join(ROOT, "include"), "-I", CSRC, "-shared", CACHED_SOURCE,
           "-o", CACHED_LIB_PATH]], verbose)
    with open(CACHED_STAMP_PATH, "w") as f:
        f.write(fp)
    return CACHED_LIB_PATH


def build_torch_ext(force=False, verbose=False):
    """Compile the torch extension (host C++ against the torch headers; it dlopens libmafed_distill.so)."""
    from torch.utils import cpp_extension as ce
    import torch
    inc = [f"-I{p}" for p in ce.include_paths()] + [f"-I{sysconfig.get_paths()['include']}",
                                                    f"-I{os.path.join(ROOT, 'include')}"]
    cuda_home = os.environ.get("CUDA_HOME") or "/usr/local/cuda"
    inc.append(f"-I{os.path.join(cuda_home, 'include')}")
    libdir = ce.library_paths()[0]
    flags = CXX_FLAGS + [f"-D_GLIBCXX_USE_CXX11_ABI={int(torch.compiled_with_cxx11_abi())}",
                         f"-DTORCH_EXTENSION_NAME={EXT_NAME}", "-DTORCH_API_INCLUDE_EXTENSION_H"]
    fp = _fingerprint([EXT_SOURCE, os.path.join(ROOT, "include", "mafed_distill.h"), CACHED_HEADER],
                      flags + [torch.__version__])
    if not force and not _stale(EXT_PATH, EXT_STAMP_PATH, fp):
        return EXT_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cxx = shutil.which("g++") or "g++"
    cmd = [cxx, *flags, *inc, EXT_SOURCE, "-o", EXT_PATH, f"-L{libdir}", "-ltorch", "-ltorch_cpu", "-ltorch_python",
           "-lc10", "-lc10_cuda", "-ltorch_cuda", "-ldl", f"-Wl,-rpath,{libdir}"]
    _run([cmd], verbose)
    with open(EXT_STAMP_PATH, "w") as f:
        f.write(fp)
    return EXT_PATH


if __name__ == "__main__":
    import sys
    force, verbose = "--force" in sys.argv, "-v" in sys.argv
    print(build(force=force, verbose=verbose))
    print(build_teacher_gather(force=force, verbose=verbose))
    print(build_cached_step(force=force, verbose=verbose))
    if "--no-ext" not in sys.argv:
        print(build_torch_ext(force=force, verbose=verbose))
