"""Build a variant of libdsoft.so with extra nvcc defines (kernel A/B arms on one board):

    python scripts/build_variant.py variant -DNAME=VALUE   # prints the path of libdsoft_variant.so (out_dir below)
    DSOFT_LIB=<that path> python bench.py ...               # that build instead of the in-tree one
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dinosoft_b200._build as b  # noqa: E402

name, defs = sys.argv[1], sys.argv[2:]
out_dir = os.path.join(ROOT, "gpurun_variants")
os.makedirs(out_dir, exist_ok=True)
out = os.path.join(out_dir, f"libdsoft_{name}.so")
cmd = [b._nvcc(), *b.NVCC_FLAGS, *defs, "-o", out, *[os.path.join(b.CSRC, s) for s in b.SOURCES]]
subprocess.run(cmd, check=True)
print(out)
