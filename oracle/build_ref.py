#!/usr/bin/env python3
"""Build oracle/_ref/libkdme_ref.so from the reference's own kernel text.

TEST INFRASTRUCTURE ONLY (see oracle/kdme_oracle.c header).

The reference's hot-path kernels use nothing from OpenCV/OpenNI except
``GpuMat::data``, so their text compiles for the host behind a small shim
(SURVEY.md 8(c)).  This script reads the cited line ranges from the sources
WHERE THEY LIE in a checkout of the reference -- $KDME_REFERENCE_ROOT, else a
directory named ``reference`` beside this repository's checkout -- concatenates
shim + text + drivers in memory and pipes the translation unit to
``g++ -x c++ -``.  The only output is ``oracle/_ref/libkdme_ref.so``
(git-ignored).  No reference source is written into this repository; where no
reference checkout is found nothing is built and the committed golden vectors
(tests/golden/ref_golden.npz) stand in for the reference.

The reference's own build system (two MSVC .props files) is not run.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("KDME_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.dirname(HERE)), "reference")
OUT_DIR = os.path.join(HERE, "_ref")
OUT = os.path.join(OUT_DIR, "libkdme_ref.so")

# (file, first line, last line, sha256 of the whole file at survey time)
RANGES = [
    ("JointBilateralFilter/JointBilateralFilter.cu", 3, 83,
     "f090094cac182aeb9d600e54ed61cc514875fa3e860feca1e7c0c545c345a385"),
    ("EdgeRefinedSuperpixel/EdgeRefinedSuperpixel.cu", 103, 205,
     "ef72d9fc489a674a458234e30bcd222afb6a302db3b79a5f3bba768619a0ae11"),
    ("MarkovRandomField/MarkovRandomField.cu", 3, 40,
     "032667abea302c33667fadb0ca847a440ba5be3d3def20cc23f1317f163d5182"),
    ("Projection_GPU/Projection_GPU.cu", 213, 246,
     "7b810ed18aa43e9fefe86819aba7e69e2ac89aacc452751ad09e2cf4b5f1e2ac"),
    ("ArrayBuffer/ArrayBuffer.cu", 9, 22,
     "221c6a62eede11af55778f4ffbd44ca08e4e75cc7a9f57a2a4c27b6cb889ee98"),
    ("ArrayBuffer/Buffer2D.cu", 13, 50,
     "6401c779b467f64215feb98a8e1b6440542e94d6f87a5efd0c725bab2a809fc3"),
    ("ArrayBuffer/Buffer2D.cu", 59, 70, None),
    ("ArrayBuffer/Buffer2D.cu", 79, 89, None),
    ("ArrayBuffer/Buffer2D.cu", 97, 113, None),
    ("ArrayBuffer/Buffer2D.cu", 123, 140, None),
]


def available() -> bool:
    return os.path.isdir(REF) and all(os.path.isfile(os.path.join(REF, r[0])) for r in RANGES)


def build(verbose: bool = True) -> str | None:
    """Returns the path of the built library, or None when the reference checkout is absent."""
    if not available():
        if verbose:
            print(f"[build_ref] reference checkout {REF} not present; keeping any prebuilt {OUT}")
        return OUT if os.path.isfile(OUT) else None
    parts = [open(os.path.join(HERE, "ref_shim_pre.h"), encoding="utf-8").read()]
    for rel, lo, hi, sha in RANGES:
        raw = open(os.path.join(REF, rel), "rb").read()
        if sha is not None and hashlib.sha256(raw).hexdigest() != sha:
            raise RuntimeError(f"{rel}: reference file changed since the survey; re-check line ranges")
        lines = raw.decode("utf-8", errors="replace").splitlines()
        parts.append(f"\n/* ---- {rel}:{lo}-{hi} (read in place) ---- */\n")
        parts.append("\n".join(lines[lo - 1:hi]) + "\n")
    parts.append(open(os.path.join(HERE, "ref_shim_post.h"), encoding="utf-8").read())
    tu = "".join(parts)
    os.makedirs(OUT_DIR, exist_ok=True)
    cmd = ["g++", "-x", "c++", "-std=c++17", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math",
           "-fPIC", "-shared", "-fvisibility=hidden", "-w", "-", "-o", OUT]
    res = subprocess.run(cmd, input=tu.encode("utf-8"), capture_output=True)
    if res.returncode != 0:
        sys.stderr.write(res.stderr.decode("utf-8", errors="replace"))
        raise RuntimeError("g++ failed on the reference kernel text")
    if verbose:
        print(f"[build_ref] built {OUT}")
    return OUT


if __name__ == "__main__":
    build()
