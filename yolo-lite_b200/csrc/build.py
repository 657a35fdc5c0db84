"""Build libyl11.so (sm_100a only) in-tree with nvcc; no JIT cache, no torch extension machinery.

    python yolo-lite_b200/csrc/build.py [--force]

Object files go to yolo-lite_b200/csrc/build/, the library to yolo-lite_b200/yololite/lib/libyl11.so.
nvcc cross-compiles without a GPU, so this also is the CPU-side "does it build" check.
"""
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
SOURCES = ["runtime.cu", "conv.cu", "conv_tc.cu", "conv_chain.cu", "dwpw_tc.cu", "conv_direct.cu", "layout.cu", "pool.cu", "attention.cu",
           "decode.cu", "nms.cu", "preprocess.cu", "c3k2_fused.cu", "c3k2_tc.cu", "stem_fused.cu", "metrics.cu", "tta.cu", "embed.cu",
           "cocoeval.cu"]
HEADERS = [HERE / "common.cuh", HERE / "conv_tc.cuh", HERE.parents[1] / "include" / "yl11.h"]
OUT_DIR = HERE.parent / "yololite" / "lib"
LIB = OUT_DIR / "libyl11.so"
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--use_fast_math", "-Xptxas", "-v"]
# nms.cu and decode.cu need IEEE arithmetic (bit-exact IoU / accurate expf), tta.cu ATen's bilinear arithmetic, embed.cu
# keeps denormal activations in its sums, cocoeval.cu is bit-exact fp64 against numpy: no fast-math
NO_FAST_MATH = {"nms.cu", "decode.cu", "preprocess.cu", "metrics.cu", "tta.cu", "embed.cu", "cocoeval.cu"}


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; libyl11 cannot be built")
    return exe


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def _compile(src: str, force: bool) -> Path:
    obj = HERE / "build" / (src[:-3] + ".o")
    if force or _stale(obj, [HERE / src, *HEADERS]):
        flags = [f for f in FLAGS if not (src in NO_FAST_MATH and f == "--use_fast_math")]
        cmd = [_nvcc(), *ARCH, *flags, "-c", str(HERE / src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        (HERE / "build" / (src[:-3] + ".log")).write_text(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    return obj


def build(force: bool = False, verbose: bool = True) -> Path:
    (HERE / "build").mkdir(exist_ok=True)
    OUT_DIR.mkdir(parents=True, exist_ok=True)
    with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(lambda s: _compile(s, force), SOURCES))
    if force or _stale(LIB, objs):
        cmd = [_nvcc(), *ARCH, "-shared", "-o", str(LIB), *map(str, objs), "-lcudart_static", "-ldl", "-lrt",
               "-lpthread"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print(f"[yl11] built {LIB} ({LIB.stat().st_size // 1024} KiB)")
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
