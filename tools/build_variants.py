#!/usr/bin/env python3
"""Build variants of libtrpl_b200.so into build/variants/ (git-ignored) for A/B runs:
    python tools/build_variants.py name[:-DFLAG=1,...] ...  [head[@rev]]
`name` builds the working tree with the given extra nvcc flags; the only flag that selects other
code is -DTRPL_DEBUG=1 (device-side checks, e.g. `debug:-DTRPL_DEBUG=1`).  `head` builds the kernel
sources of git HEAD (or of `rev`) as the baseline."""
import os
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bayesian_inference_trpl_b200 import _lib

OUT = os.path.join(ROOT, "build", "variants")
os.makedirs(OUT, exist_ok=True)


def build(spec):
    name, _, flags = spec.partition(":")
    flags = [f for f in flags.split(",") if f]
    inc = os.path.dirname(_lib.SRC)
    src = _lib.SRC
    tmp = None
    if name.startswith("head"):
        rev = name.partition("@")[2] or "HEAD"
        tmp = tempfile.mkdtemp()
        for f in os.listdir(inc):
            data = subprocess.run(["git", "-C", ROOT, "show", "%s:bayesian_inference_trpl_b200/csrc/%s" % (rev, f)],
                                  capture_output=True)
            if data.returncode == 0:
                open(os.path.join(tmp, f), "wb").write(data.stdout)
        src = os.path.join(tmp, "trpl_kernels.cu")
        name = "head"
    out = os.path.join(OUT, "libtrpl_%s.so" % name)
    cmd = ["/usr/local/cuda/bin/nvcc"] + _lib.NVCC_FLAGS + flags + ["-I", _lib.INCLUDE, "-o", out, src]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    with ThreadPoolExecutor(4) as ex:
        for o in ex.map(build, sys.argv[1:]):
            print("built", o)
