"""Sweep of kModelWarpNodes (dq_kernels.cuh), the node budget of one model inside a dq_solve_models launch.

The budget is a compile-time constant of the library, not an option, so the sweep builds one library per value from a
copy of the sources and runs scripts/models_bench.py against each:

  python scripts/models_budget_sweep.py build OUTDIR [EXP ...]   # needs nvcc only; default exponents 12 14 16 18
  python scripts/models_budget_sweep.py run OUTDIR               # on the GPU: models_bench.py once per library

Each library is OUTDIR/libdequan_b200_<EXP>.so with kModelWarpNodes = 2^EXP; the tree itself is not modified."""
import glob
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dequan_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
PATTERN = r"constexpr unsigned long long kModelWarpNodes = 1ull << \d+;"


def build(outdir, exps):
    os.makedirs(outdir, exist_ok=True)
    procs = []
    for e in exps:
        src = tempfile.mkdtemp(prefix=f"dq_budget_{e}_")
        for f in glob.glob(os.path.join(CSRC, "*")):
            shutil.copy(f, src)
        k = os.path.join(src, "dq_kernels.cuh")
        text = open(k).read()
        assert len(re.findall(PATTERN, text)) == 1, "kModelWarpNodes not found"
        open(k, "w").write(re.sub(PATTERN, f"constexpr unsigned long long kModelWarpNodes = 1ull << {e};", text))
        out = os.path.join(outdir, f"libdequan_b200_{e}.so")
        cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
               "-I" + os.path.join(ROOT, "include"), "-I" + src, "-shared", "-o", out,
               os.path.join(src, "dq_api.cu"), os.path.join(src, "dq_compile.cpp"), os.path.join(src, "dq_formats.cpp")]
        procs.append((subprocess.Popen(cmd), src, out))
    for p, src, out in procs:
        if p.wait() != 0:
            sys.exit(f"build of {out} failed")
        shutil.rmtree(src)
        print("built", out)


def run(outdir):
    libs = sorted(glob.glob(os.path.join(outdir, "libdequan_b200_*.so")), key=lambda p: int(re.findall(r"_(\d+)\.so$", p)[0]))
    for lib in libs:
        e = int(re.findall(r"_(\d+)\.so$", lib)[0])
        print(f"== kModelWarpNodes = 2^{e}", flush=True)
        code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
                "from dequan_b200 import api; api.LIB_PATH = %r\n"
                "import models_bench; models_bench.main()") % (ROOT, os.path.join(ROOT, "scripts"), os.path.abspath(lib))
        subprocess.run([sys.executable, "-c", code], check=True)


if __name__ == "__main__":
    if len(sys.argv) < 3 or sys.argv[1] not in ("build", "run"):
        sys.exit(__doc__)
    if sys.argv[1] == "build":
        build(sys.argv[2], [int(x) for x in sys.argv[3:]] or [12, 14, 16, 18])
    else:
        run(sys.argv[2])
