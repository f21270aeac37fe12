"""TEST INFRASTRUCTURE ONLY: compiles the product's CUDA sources against the SIMT
emulator (cpusim.h) with g++, so kernel logic can be exercised without a GPU.

Output: tests/cpusim/_build/libnutsb200_sim.so.  Never shipped, never loaded by the
nuts333_b200 package (which only ever loads nuts333_b200/_lib/libnutsb200.so).
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
if str(ROOT) not in sys.path:                 # (run as a script)
    sys.path.insert(0, str(ROOT))
from nuts333_b200.build import HEADERS, SOURCES  # noqa: E402

CSRC = ROOT / "nuts333_b200" / "csrc"
OUT = HERE / "_build" / "libnutsb200_sim.so"
# the product library's own sources and headers: an edit to any of them rebuilds the emulated one too
DEPS = SOURCES + HEADERS + [HERE / "cpusim.h", Path(__file__).resolve()]


def build_sim(force: bool = False, sanitize: str | None = None) -> Path:
    out = OUT if not sanitize else OUT.with_name(f"libnutsb200_sim_{sanitize}.so")
    if not force and out.exists() and all(d.stat().st_mtime <= out.stat().st_mtime for d in DEPS):
        return out
    out.parent.mkdir(parents=True, exist_ok=True)
    cmd = ["g++", "-std=c++17", "-O1", "-g", "-fPIC", "-shared", "-pthread", "-DNUTSB_CPUSIM",
           "-DCPUSIM_IMPLEMENTATION", "-Wall", "-Wno-unused-function", "-Wno-unknown-pragmas",
           "-I", str(HERE), "-x", "c++", str(CSRC / "nutsb_lib.cu"), "-o", str(out)]
    if sanitize:
        cmd[1:1] = [f"-fsanitize={sanitize}", "-fno-omit-frame-pointer"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("cpusim build failed:\n" + r.stderr)
    if r.stderr.strip():
        sys.stderr.write(r.stderr)
    return out


if __name__ == "__main__":
    print(build_sim(force=True, sanitize=sys.argv[1] if len(sys.argv) > 1 else None))
