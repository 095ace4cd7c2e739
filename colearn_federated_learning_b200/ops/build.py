"""In-tree build of the sm_100a extension (``_colearn_C*.so`` next to this file).

``nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo`` for every ``.cu`` (they do not include
torch headers, so each compiles in seconds), ``g++`` for ``bindings.cpp``, one link step.  The
result is git-ignored but travels with the gpurun snapshot; ``__graft_entry__.build()`` calls
:func:`build_all`.  Objects are cached under ``csrc/_obj`` keyed by source mtime+flags.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
import sysconfig
from concurrent.futures import ThreadPoolExecutor
from typing import List

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
EXT_NAME = "_colearn_C"
EMUL_NAME = "_colearn_emul"     # CPU emulator of the conv kernels (tests on boxes without a GPU)
HOST_NAME = "_colearn_host"     # native CPU executor of the MLP local fit (devices / boxes without a GPU)
SIMT_NAME = "_colearn_simt"     # the persistent-MLP CUDA kernels compiled for the CPU through csrc/host_shim.h (tests)

CU_SOURCES = ["mlp_persistent.cu", "mlp_generic.cu", "elementwise.cu", "comm.cu", "gemm_tcgen05.cu", "convnet.cu"]
CPP_SOURCES = ["bindings.cpp"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo",
              "--use_fast_math", "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
# --use_fast_math would change expf/logf/division semantics in the loss kernels; keep IEEE there.
NVCC_FLAGS.remove("--use_fast_math")


def ext_path() -> str:
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    return os.path.join(HERE, EXT_NAME + suffix)


def _nvcc() -> str:
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else (shutil.which("nvcc") or "nvcc")


def _stamp(src: str, flags: List[str]) -> str:
    h = hashlib.sha1()
    with open(src, "rb") as f:
        h.update(f.read())
    for dep in ("colearn_kernels.h", "mlp_v2.inc", "conv_ops.cuh", "conv_bindings.inc", "client_desc.inc"):
        with open(os.path.join(CSRC, dep), "rb") as f:
            h.update(f.read())
    h.update(" ".join(flags).encode())
    return h.hexdigest()[:16]


def _run(cmd: List[str], log_name: str) -> None:
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    with open(os.path.join(OBJ, log_name + ".log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError(f"build step failed: {' '.join(cmd)}\n{proc.stdout}")


def _cxx_setup():
    import torch
    from torch.utils import cpp_extension as ce

    cuda_home = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    inc = [f"-I{p}" for p in ce.include_paths(device_type="cuda")] + [f"-I{sysconfig.get_paths()['include']}", f"-I{CSRC}",
                                                                       f"-I{os.path.join(cuda_home, 'include')}"]
    flags = ["-O2", "-std=c++17", "-fPIC", "-DTORCH_API_INCLUDE_EXTENSION_H",
             f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}", "-Wno-deprecated-declarations"]
    return ce, cuda_home, inc, flags


def emul_path() -> str:
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    return os.path.join(HERE, EMUL_NAME + suffix)


def build_emul(force: bool = False) -> str:
    """g++-only build of ``csrc/conv_emul.cpp`` (the conv kernels' bodies run on the CPU).  Links against the CPU
    libtorch only, so it loads on a box without a CUDA driver."""
    ce, _, inc, flags = _cxx_setup()
    os.makedirs(OBJ, exist_ok=True)
    out = emul_path()
    src = os.path.join(CSRC, "conv_emul.cpp")
    cxx_flags = flags + [f"-DTORCH_EXTENSION_NAME={EMUL_NAME}"]
    obj = os.path.join(OBJ, f"conv_emul.cpp.{_stamp(src, cxx_flags)}.o")
    if force or not os.path.exists(obj) or not os.path.exists(out):
        for name in os.listdir(OBJ):
            if name.startswith("conv_emul.cpp.") and name.endswith(".o"):
                os.remove(os.path.join(OBJ, name))
        _run(["g++", *cxx_flags, *inc, "-c", src, "-o", obj], "conv_emul.cpp")
        link = ["g++", "-shared", obj, "-o", out]
        for d in ce.library_paths(device_type="cpu"):
            link += [f"-L{d}", f"-Wl,-rpath,{d}"]
        link += ["-lc10", "-ltorch_cpu", "-ltorch", "-ltorch_python"]
        _run(link, "link_emul")
    return out


def host_path() -> str:
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    return os.path.join(HERE, HOST_NAME + suffix)


def build_host(force: bool = False) -> str:
    """g++-only build of ``csrc/mlp_host.cpp`` (worker-side local SGD for devices without a GPU).  No CUDA headers or
    libraries are involved; portable ``-O3`` (no ``-march=native``: the in-tree ``.so`` travels between boxes)."""
    ce, _, inc, flags = _cxx_setup()
    os.makedirs(OBJ, exist_ok=True)
    out = host_path()
    src = os.path.join(CSRC, "mlp_host.cpp")
    cxx_flags = [f for f in flags if f != "-O2"] + ["-O3", "-fno-math-errno", "-fopenmp-simd", f"-DTORCH_EXTENSION_NAME={HOST_NAME}"]
    h = hashlib.sha1(open(src, "rb").read() + " ".join(cxx_flags).encode()).hexdigest()[:16]
    obj = os.path.join(OBJ, f"mlp_host.cpp.{h}.o")
    if force or not os.path.exists(obj) or not os.path.exists(out):
        for name in os.listdir(OBJ):
            if name.startswith("mlp_host.cpp.") and name.endswith(".o"):
                os.remove(os.path.join(OBJ, name))
        _run(["g++", *cxx_flags, *[i for i in inc if "cuda" not in i.lower() or "torch" in i.lower()], "-c", src, "-o", obj], "mlp_host.cpp")
        link = ["g++", "-shared", obj, "-o", out, "-pthread"]
        for d in ce.library_paths(device_type="cpu"):
            link += [f"-L{d}", f"-Wl,-rpath,{d}"]
        link += ["-lc10", "-ltorch_cpu", "-ltorch", "-ltorch_python"]
        _run(link, "link_host")
    return out


def simt_path() -> str:
    suffix = sysconfig.get_config_var("EXT_SUFFIX") or ".so"
    return os.path.join(HERE, SIMT_NAME + suffix)


def build_simt_emul(force: bool = False) -> str:
    """g++ build of ``csrc/simt_emul.cpp``: ``mlp_persistent.cu`` + ``mlp_v2.inc`` + ``mlp_generic.cu`` — the kernel sources themselves —
    compiled for the CPU with one OS thread per CUDA thread (``csrc/host_shim.h``).  Needs C++20 (``std::barrier``) and
    the CUDA headers, no GPU and no CUDA libraries."""
    ce, cuda_home, inc, flags = _cxx_setup()
    os.makedirs(OBJ, exist_ok=True)
    out = simt_path()
    src = os.path.join(CSRC, "simt_emul.cpp")
    cxx_flags = [f for f in flags if f not in ("-O2", "-std=c++17")] + ["-O1", "-std=c++20", "-pthread", "-Wno-unknown-pragmas",
                                                                        f"-DTORCH_EXTENSION_NAME={SIMT_NAME}"]
    sources = ["simt_emul.cpp", "simt_mlp.cpp", "simt_mlp_generic.cpp", "simt_elementwise.cpp", "simt_comm.cpp", "simt_convnet.cpp", "simt_gemm.cpp"]
    h = hashlib.sha1()
    for dep in sources + ["host_shim.h", "mlp_persistent.cu", "mlp_generic.cu", "client_desc.inc", "mlp_v2.inc", "elementwise.cu", "comm.cu", "convnet.cu", "gemm_tcgen05.cu", "tcgen05_host_model.h", "conv_bindings.inc", "colearn_kernels.h", "conv_ops.cuh"]:
        with open(os.path.join(CSRC, dep), "rb") as f:
            h.update(f.read())
    h.update(" ".join(cxx_flags).encode())
    stamp = h.hexdigest()[:16]
    objs = [os.path.join(OBJ, f"{src}.{stamp}.simt.o") for src in sources]
    if force or not all(os.path.exists(o) for o in objs) or not os.path.exists(out):
        for name in os.listdir(OBJ):
            if name.endswith(".simt.o"):
                os.remove(os.path.join(OBJ, name))
        with ThreadPoolExecutor(max_workers=6) as pool:
            list(pool.map(lambda so: _run(["g++", *cxx_flags, *inc, "-c", os.path.join(CSRC, so[0]), "-o", so[1]], so[0]), zip(sources, objs)))
        link = ["g++", "-shared", *objs, "-o", out, "-pthread"]
        for d in ce.library_paths(device_type="cpu"):
            link += [f"-L{d}", f"-Wl,-rpath,{d}"]
        link += ["-lc10", "-ltorch_cpu", "-ltorch", "-ltorch_python"]
        _run(link, "link_simt")
    return out


def build_all(force: bool = False, verbose: bool = True) -> str:
    ce, cuda_home, inc, base_cxx = _cxx_setup()

    os.makedirs(OBJ, exist_ok=True)
    out = ext_path()
    objs, jobs = [], []

    for src in CU_SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ, f"{src}.{_stamp(path, NVCC_FLAGS)}.o")
        objs.append(obj)
        if force or not os.path.exists(obj):
            jobs.append(([_nvcc(), *NVCC_FLAGS, "-I", CSRC, "-c", path, "-o", obj], src))

    cxx_flags = base_cxx + [f"-DTORCH_EXTENSION_NAME={EXT_NAME}"]
    for src in CPP_SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(OBJ, f"{src}.{_stamp(path, cxx_flags)}.o")
        objs.append(obj)
        if force or not os.path.exists(obj):
            jobs.append((["g++", *cxx_flags, *inc, "-c", path, "-o", obj], src))

    if jobs:
        if verbose:
            print(f"[colearn build] compiling {len(jobs)} translation unit(s) for sm_100a", file=sys.stderr)
        with ThreadPoolExecutor(max_workers=min(8, len(jobs))) as pool:
            list(pool.map(lambda j: _run(j[0], j[1]), jobs))

    if jobs or force or not os.path.exists(out):
        lib_dirs = ce.library_paths(device_type="cuda")
        link = ["g++", "-shared", *objs, "-o", out]
        for d in lib_dirs:
            link += [f"-L{d}", f"-Wl,-rpath,{d}"]
        link += [f"-L{os.path.join(cuda_home, 'lib64')}", "-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda",
                 "-ltorch", "-ltorch_python", "-lcudart"]
        _run(link, "link")
        if verbose:
            print(f"[colearn build] linked {out}", file=sys.stderr)
    # drop stale cached objects (every source edit leaves one behind)
    keep = {os.path.basename(o) for o in objs}
    for name in os.listdir(OBJ):
        if name.endswith(".o") and name not in keep and not name.startswith(("conv_emul.cpp.", "mlp_host.cpp.")) and not name.endswith(".simt.o"):
            os.remove(os.path.join(OBJ, name))
    build_host(force=force)      # the CPU executor ships with every build (CPU-only boxes: `--host` builds it alone)
    return out


def main(argv=None) -> int:
    """``python -m colearn_federated_learning_b200.ops.build [--emul | --host] [--force]`` / ``colearn-build-kernels``.

    ``--host`` builds only the CPU executor (no nvcc needed: edge devices), ``--emul`` only the conv-kernel emulator."""
    argv = sys.argv[1:] if argv is None else argv
    force = "--force" in argv
    if "--simt" in argv:
        print(build_simt_emul(force=force))
    elif "--emul" in argv:
        print(build_emul(force=force))
    elif "--host" in argv:
        print(build_host(force=force))
    else:
        print(build_all(force=force))
    return 0


if __name__ == "__main__":
    sys.exit(main())
