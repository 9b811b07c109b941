#!/usr/bin/env python
"""Build the UNMODIFIED reference programs into baseline/_ref/ (git-ignored, travels to the GPU box).

The reference (/root/reference) is five CMake C++ programs on LibTorch + MPI + OpenCV C++.  The image has LibTorch
(inside the torch wheel) but no MPI and no OpenCV C++, so the sources are compiled AS THEY ARE (copied byte for byte
into baseline/_ref/src, sha256 recorded) against two tiny stand-ins kept in baseline/shim/: a single-node MPI subset
over POSIX shm (mpi.h / egmpi.c / mpirun) and a header-only opencv2/opencv.hpp that synthesises CIFAR-shaped images.
`pip install /root/reference` was tried first, as prescribed, and fails (no setup.py / pyproject) -- see README.md.

    python baseline/build_ref.py --ref <reference checkout> [--only cifar_event,...]
"""
from __future__ import annotations
import argparse, hashlib, json, os, shutil, subprocess, sys, time

HERE = os.path.dirname(os.path.abspath(__file__))
PROGRAMS = {  # binary name -> source relative to the reference root
    "cifar_event": "dcifar10/event/event.cpp",
    "cifar_spevent": "dcifar10/spevent/spevent.cpp",
    "mnist_event": "dmnist/event/event.cpp",
    "mnist_decent": "dmnist/decent/decent.cpp",
    "mnist_cent": "dmnist/cent/cent.cpp",
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True, help="checkout of the reference programs")
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default=os.path.join(HERE, "_ref"))
    a = ap.parse_args()
    import torch
    tdir = os.path.dirname(torch.__file__)
    out, shim = a.out, os.path.join(HERE, "shim")
    src_root = os.path.join(out, "src")
    os.makedirs(os.path.join(out, "bin"), exist_ok=True)
    if os.path.isdir(src_root):
        shutil.rmtree(src_root)
    shutil.copytree(a.ref, src_root, ignore=shutil.ignore_patterns(".git"))
    log = {"when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), "torch": torch.__version__, "programs": {}}
    subprocess.check_call(["gcc", "-O2", "-c", "-fPIC", os.path.join(shim, "egmpi.c"), "-o", os.path.join(out, "egmpi.o")])
    names = [n for n in PROGRAMS if not a.only or n in a.only.split(",")]
    rc = 0
    for name in names:
        src = os.path.join(src_root, PROGRAMS[name])
        sha = hashlib.sha256(open(src, "rb").read()).hexdigest()
        same = sha == hashlib.sha256(open(os.path.join(a.ref, PROGRAMS[name]), "rb").read()).hexdigest()
        # LibTorch >= 2.x needs C++17 (the reference's CMake says 14; the sources compile unchanged under 17)
        # `-include fstream`: the MNIST mains use std::ofstream without including <fstream> (older LibTorch headers pulled it
        # in transitively); a command-line include keeps the sources untouched
        cmd = ["g++", "-O2", "-std=c++17", "-w", "-include", "fstream", "-D_GLIBCXX_USE_CXX11_ABI=%d" % int(torch._C._GLIBCXX_USE_CXX11_ABI),
               "-I", shim, "-isystem", os.path.join(tdir, "include"),
               "-isystem", os.path.join(tdir, "include", "torch", "csrc", "api", "include"),
               src, os.path.join(out, "egmpi.o"), "-o", os.path.join(out, "bin", name),
               "-L", os.path.join(tdir, "lib"), "-Wl,-rpath," + os.path.join(tdir, "lib"), "-Wl,--no-as-needed",
               "-ltorch", "-ltorch_cpu", "-lc10", "-lpthread", "-lrt"]
        t0 = time.time()
        p = subprocess.run(cmd, capture_output=True, text=True)
        log["programs"][name] = {"source": PROGRAMS[name], "sha256": sha, "identical_to_reference": same,
                                 "rc": p.returncode, "seconds": round(time.time() - t0, 1), "stderr_tail": p.stderr[-2000:]}
        print(f"[build_ref] {name}: rc={p.returncode} ({time.time()-t0:.0f}s) identical={same}")
        if p.returncode:
            print(p.stderr[-3000:])
            rc = 1
    shutil.copy(os.path.join(shim, "mpirun"), os.path.join(out, "bin", "mpirun"))
    json.dump(log, open(os.path.join(out, "BUILD_LOG.json"), "w"), indent=1)
    shutil.copy(os.path.join(out, "BUILD_LOG.json"), os.path.join(HERE, "BUILD_LOG.json"))
    return rc


if __name__ == "__main__":
    sys.exit(main())
