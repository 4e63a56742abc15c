"""In-tree build of libe2e_asr_b200.so (hand-written sm_100a CUDA + the C ABI) and of libe2e_asr_b200_tc.so, the
tcgen05 tensor-core kernels it links against (found next to it through its $ORIGIN run path).

``nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo`` cross-compiles without a
GPU; the resulting shared object lives next to the sources (``lib/``), is
git-ignored, and travels to the GPU box with the repo snapshot.
"""
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libe2e_asr_b200.so")
TC_LIB_PATH = os.path.join(LIB_DIR, "libe2e_asr_b200_tc.so")
SOURCES = ["abi.cu", "ctc_posterior.cu", "prefix_score.cu", "prefix_lazy.cu", "beam_step.cu", "attention_full.cu", "lstm_step.cu", "conv_split.cu",
           "conv_igemm_host.cu", "lstm_seq.cu", "encoder_post.cu",
           "beam_wide.cu"]
TC_SOURCES = ["conv_igemm.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "beam_select.cuh"), os.path.join(CSRC, "conv_igemm.cuh"), os.path.join(CSRC, "softplus_lut.inc"), os.path.join(CSRC, "softplus_poly.inc"), os.path.join(_HERE, "..", "include", "e2e_asr_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--expt-extended-lambda", "-Xcompiler", "-fPIC", "-shared"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def stale():
    if not os.path.exists(LIB_PATH) or not os.path.exists(TC_LIB_PATH):
        return True
    built = min(os.path.getmtime(LIB_PATH), os.path.getmtime(TC_LIB_PATH))
    deps = [os.path.join(CSRC, s) for s in SOURCES + TC_SOURCES] + HEADERS
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False):
    """Compile the extension if missing or older than its sources.  Returns the path.
    The translation units are compiled concurrently (one nvcc per .cu), then linked."""
    if not force and not stale():
        return LIB_PATH
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libe2e_asr_b200.so")
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(LIB_DIR, exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"] + (["-Xptxas", "-v"] if verbose else [])
    with tempfile.TemporaryDirectory(prefix="e2e_build_") as tmp:
        def compile_one(src):
            obj = os.path.join(tmp, src.replace(".cu", ".o"))
            proc = subprocess.run([nvcc] + compile_flags + ["-c", "-o", obj, src], cwd=CSRC, capture_output=True, text=True)
            return src, obj, proc
        with ThreadPoolExecutor(max_workers=min(len(SOURCES) + len(TC_SOURCES), os.cpu_count() or 1)) as pool:
            done = list(pool.map(compile_one, SOURCES + TC_SOURCES))
        failed = [(src, proc) for src, _, proc in done if proc.returncode != 0]
        if failed:
            raise RuntimeError("nvcc failed:\n" + "\n".join(src + ":\n" + proc.stdout + proc.stderr for src, proc in failed))
        if verbose:
            for src, _, proc in done:
                print(proc.stderr)
        objs = {src: obj for src, obj, _ in done}

        def link(path, srcs, extra):
            out_tmp = path + ".tmp%d" % os.getpid()
            proc = subprocess.run([nvcc] + NVCC_FLAGS + ["-o", out_tmp] + [objs[s] for s in srcs] + extra, cwd=CSRC,
                                  capture_output=True, text=True)
            if proc.returncode != 0:
                raise RuntimeError("nvcc link failed:\n" + proc.stdout + proc.stderr)
            os.replace(out_tmp, path)                      # atomic: a concurrent loader never sees a half-written library
        link(TC_LIB_PATH, TC_SOURCES, [])
        link(LIB_PATH, SOURCES, ["-L" + LIB_DIR, "-le2e_asr_b200_tc", "-Xlinker", "-rpath=$ORIGIN"])
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
