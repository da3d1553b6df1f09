"""Build libgnn_decode_b200.so in-tree with nvcc for sm_100a (no torch headers involved)."""
import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
LIB_DIR = os.path.join(_PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libgnn_decode_b200.so")
SOURCES = ["gd_graph.cu", "gd_options.cu", "gd_lean.cu", "gd_decode.cu", "gd_decode_light.cu", "gd_streamed.cu", "gd_streamed_tma.cu", "gd_propagate.cu", "gd_host.cu", "gd_pipeline.cu", "gd_sampler.cu", "gd_eval.cu",
           "gd_backward.cu", "gd_backward_light.cu", "gd_backward_nbp.cu", "gd_loss.cu", "gd_p2p.cu", "gd_optim.cu", "gd_bench.cu"]
# GD_EXTRA_NVCC: extra flags for developer builds (e.g. -DGD_VTAB_DEBUG, -Xptxas -v)
NVCC_FLAGS = os.environ.get("GD_EXTRA_NVCC", "").split() + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
                                                             "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def is_stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    deps.append(os.path.join(os.path.dirname(_PKG), "include", "gnn_decode.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile every CUDA source (one object each, in parallel, rebuilt only when stale) and link
    them into one shared library.  Returns the library path."""
    if not force and not is_stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    obj_dir = os.path.join(LIB_DIR, "obj")
    os.makedirs(obj_dir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    headers.append(os.path.join(os.path.dirname(_PKG), "include", "gnn_decode.h"))
    t_hdr = max(os.path.getmtime(h) for h in headers)
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), t_hdr):
            return obj, ""
        cmd = [_nvcc()] + flags + ["-c", src, "-o", obj]
        res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), res.stdout + res.stderr))
        return obj, res.stdout + res.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_one, sources()))
    cmd = [_nvcc(), "-shared", "-o", LIB_PATH] + [o for o, _ in results]
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (" ".join(cmd), res.stdout + res.stderr))
    if verbose:
        print("".join(log for _, log in results))
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
