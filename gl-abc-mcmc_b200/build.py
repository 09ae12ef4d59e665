"""In-tree build of the CUDA extension: nvcc -> gl-abc-mcmc_b200/csrc/libglabc.so (sm_100a only).

The .so is git-ignored but travels to the GPU box with the repo snapshot; nothing is JIT-compiled
at import time.  `python -m gl-abc-mcmc_b200.build` is not spellable (hyphen), use
`python -c "import __graft_entry__ as g; g.build()"`.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
SOURCES = ["abi.cu", "diag.cu", "step_global.cu", "step_global_d1.cu", "step_global_d2.cu", "step_global_d3.cu",
           "step_global_d4.cu", "step_isir.cu", "step_isir_d1.cu", "step_isir_d2.cu", "step_isir_d3.cu", "step_isir_d4.cu",
           "step_mala.cu", "step_mala_d1.cu", "step_mala_d2.cu", "step_mala_d3.cu", "step_mala_d4.cu",
           "kde.cu", "resample.cu", "step_aglmcmc.cu", "flow.cu", "flow_train.cu", "step_generic.cu", "user_model.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v",
              "--expt-relaxed-constexpr", "-I", os.path.join(ROOT, "include")]
LIB = os.path.join(CSRC, "libglabc.so")


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _deps():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))] + \
           [os.path.join(ROOT, "include", "glabc.h")]


def _embed_dist_device():
    """csrc/dist_device_src.inc: the text of dist_device.cuh as a C++ raw string literal.  user_model.cu hands it to
    NVRTC as a named header, so the user-model kernels compile the same distribution code as the built-in ones and the
    library needs no file of the tree at run time."""
    with open(os.path.join(CSRC, "dist_device.cuh")) as f:
        text = f.read()
    assert ')GLABC_DIST"' not in text
    out = os.path.join(CSRC, "dist_device_src.inc")
    body = 'R"GLABC_DIST(' + text + ')GLABC_DIST"\n'
    if not os.path.exists(out) or open(out).read() != body:
        with open(out, "w") as f:
            f.write(body)


def build(force=False, verbose=False, variant=None, extra_flags=()):
    """`variant` builds csrc/libglabc.<variant>.so with `extra_flags` (kernel experiments; select it
    at run time with GLABC_LIB=<path>)."""
    lib_path = LIB if variant is None else os.path.join(CSRC, f"libglabc.{variant}.so")
    newest = max(os.path.getmtime(p) for p in _deps())
    if not force and os.path.exists(lib_path) and os.path.getmtime(lib_path) >= newest:
        return lib_path
    nvcc = _nvcc()
    _embed_dist_device()
    logs = {}
    tag = "" if variant is None else "." + variant

    def compile_one(src):
        obj = os.path.join(CSRC, src[:-3] + tag + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-c", os.path.join(CSRC, src), "-o", obj]
        p = subprocess.run(cmd, capture_output=True, text=True)
        logs[src] = p.stderr + p.stdout
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{logs[src]}")
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    # -cudart static (nvcc default): the library loads on a box without a GPU or libcudart.so
    p = subprocess.run([nvcc, "-shared", "-o", lib_path, *objs, "-Xcompiler", "-fvisibility=hidden", "-ldl"], capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError("link failed:\n" + p.stderr)
    with open(os.path.join(CSRC, f"ptxas{tag}.log"), "w") as f:
        for src in SOURCES:
            f.write(f"==== {src}\n{logs[src]}\n")
    if verbose:
        for src in SOURCES:
            sys.stderr.write(logs[src])
    return lib_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
