"""Build liblhn.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Used by __graft_entry__.build() and runnable by hand:  python -m litehandnet_b200.build
Each translation unit is compiled in parallel, then linked into litehandnet_b200/lib/liblhn.so.
nvcc cross-compiles without a GPU.
"""
import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIB = os.path.join(LIBDIR, "liblhn.so")
SOURCES = ["lhn_heatmap.cu", "lhn_heatmap_team_launch.cu", "lhn_heatmap_team_f32.cu", "lhn_heatmap_team_bf16.cu",
           "lhn_heatmap_team_f16.cu", "lhn_loss_render.cu", "lhn_loss_multi.cu", "lhn_backward.cu", "lhn_loss_grad.cu", "lhn_simdr.cu", "lhn_simdr_heads.cu", "lhn_metrics.cu", "lhn_exchange.cu", "lhn_region.cu", "lhn_host.cu"]
HEADERS = [os.path.join(CSRC, "lhn_common.cuh"), os.path.join(CSRC, "lhn_exchange.cuh"), os.path.join(CSRC, "lhn_heatmap.cuh"), os.path.join(CSRC, "lhn_heatmap_team.cuh"), os.path.join(HERE, "..", "include", "lhn.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr"]
if os.environ.get("LHN_TRACE") == "1":      # phase timestamps in the team kernel (profiles/probes/trace_run.py)
    NVCC_FLAGS.append("-DLHN_TRACE")


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _digest(paths):
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for p in paths:
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _compile_one(nvcc, src, verbose):
    obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
    stamp = obj + ".sha"
    dig = _digest([os.path.join(CSRC, src)] + HEADERS)
    if os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
        return obj, False
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    if verbose:
        sys.stderr.write(r.stderr)
    with open(stamp, "w") as f:
        f.write(dig)
    return obj, True


EXT_SRC = os.path.join(CSRC, "ext", "lhn_torch_ext.cpp")
EXT_NAME = "lhn_torch_ext"


def ext_path():
    import sysconfig
    return os.path.join(LIBDIR, EXT_NAME + sysconfig.get_config_var("EXT_SUFFIX"))


def build_ext(verbose=False):
    """The torch-extension shim (csrc/ext/lhn_torch_ext.cpp): plain g++ against torch's headers, linked to liblhn.so
    through an $ORIGIN rpath, built in-tree next to it (no JIT cache: the file travels with the snapshot)."""
    import sysconfig
    import torch
    from torch.utils import cpp_extension as ce
    out = ext_path()
    stamp = out + ".sha"
    dig = _digest([EXT_SRC, os.path.join(HERE, "..", "include", "lhn.h")]) + torch.__version__
    if os.path.exists(out) and os.path.exists(stamp) and open(stamp).read() == dig:
        return out
    cuda_home = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    inc = [f"-I{p}" for p in ce.include_paths()] + [f"-I{sysconfig.get_paths()['include']}", f"-I{cuda_home}/include"]
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-fvisibility=hidden", f"-DTORCH_EXTENSION_NAME={EXT_NAME}",
           "-DTORCH_API_INCLUDE_EXTENSION_H", f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}"] + inc + \
          [EXT_SRC, "-o", out, f"-L{LIBDIR}", "-llhn", "-Wl,-rpath,$ORIGIN"] + \
          [f"-L{p}" for p in ce.library_paths()] + ["-lc10", "-lc10_cuda", "-ltorch_cpu", "-ltorch_cuda", "-ltorch", "-ltorch_python",
                                                   f"-L{cuda_home}/lib64", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"torch extension shim failed to build:\n{r.stdout}\n{r.stderr}")
    if verbose:
        sys.stderr.write(r.stderr)
    with open(stamp, "w") as f:
        f.write(dig)
    return out


def build(verbose=False, force=False):
    os.makedirs(OBJDIR, exist_ok=True)
    if force:
        for f in os.listdir(OBJDIR):
            os.remove(os.path.join(OBJDIR, f))
    nvcc = _nvcc()
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(lambda s: _compile_one(nvcc, s, verbose), SOURCES))
    objs = [o for o, _ in results]
    if any(changed for _, changed in results) or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    build_ext(verbose)
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
