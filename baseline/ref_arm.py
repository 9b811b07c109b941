"""`bench.py --impl reference`: time the UNMODIFIED reference (baseline/_ref, built by baseline/build_ref.py).

What runs: the reference's own `main()` of dcifar10/event (or dcifar10/spevent) -- byte-identical source, sha256 in
baseline/_ref/BUILD_LOG.json -- started the way its README says (`mpirun -np N ./event <file_write> <thres_type>
<value>`, /root/reference/dcifar10/README.md) through the shm MPI stand-in of baseline/shim (no MPI on the image).
Nothing of eventgrad_b200 is imported or loaded on this path.

* dense D-PSGD (the headline config) = the reference's documented equivalence knob: non-adaptive threshold 0
  (`<thres_type>=0 <constant>=0`, /root/reference/dmnist/event/README.md:59-60) -> every tensor is sent every step.
* The program hard-codes 20 epochs x 196 steps and has no step-count option, so it is run with `file_write=1`
  (it then appends `pass_num, loss` + std::endl to train<rank>.txt every step, event.cpp:271-273) and this harness
  timestamps the lines: K steps = time between line W+1 and line W+K+1 on each rank, MAX over ranks.  The process
  group is then stopped (exact pids).  The timed region therefore contains everything the reference does per step:
  data loading (synthetic imread stub + its own pad/flip/crop transforms), forward, backward, the per-tensor
  norm/Put/average loop, optimizer step, its own log writes.  That is an END-TO-END number; the reference has no
  device (CPU only, event.cpp:39), so `value` and `e2e.value` are the same measurement.
"""
from __future__ import annotations

import json
import os
import signal
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "_ref")


def _unavailable(why: str) -> int:
    print(json.dumps({"impl": "reference", "unavailable": why}), flush=True)
    return 0


def _ensure_built(binary: str) -> str | None:
    # the reference sources are not part of this repository: the binaries are built ahead of time, never here
    path = os.path.join(REF, "bin", binary)
    if os.path.exists(path) and os.path.exists(os.path.join(REF, "bin", "mpirun")):
        return None
    return (f"baseline/_ref/bin/{binary} is not built "
            "(python baseline/build_ref.py --ref <reference checkout> --only " + binary + ")")


def _count_lines(path: str) -> int:
    try:
        with open(path, "rb") as f:
            return f.read().count(b"\n")
    except OSError:
        return 0


def run(args) -> int:
    # under torchrun every rank executes bench.py: only rank 0 drives the reference job
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    N, K, W = int(args.gpus), int(args.steps), int(args.warmup)
    algo = getattr(args, "algo", "dpsgd")
    if algo == "cent":
        return _unavailable("the reference has no CIFAR all-reduce program (cent is MNIST-only and its dataset path is "
                            "a hard-coded AFS location)")
    binary = "cifar_spevent" if algo == "spevent" else "cifar_event"
    why = _ensure_built(binary)
    if why:
        return _unavailable(why)
    if algo == "dpsgd":
        prog_args = ["1", "0", "0"]
    elif algo == "event":
        prog_args = ["1", "1", str(args.horizon)]
    else:
        prog_args = ["1", "1", str(args.horizon), str(int(args.topk))]
    gb = 256                                 # hard-coded in the reference (event.cpp:31), split over the ranks
    if getattr(args, "global_batch", 256) != 256 or getattr(args, "scaling", "strong") != "strong":
        return _unavailable("the reference hard-codes global batch 256, strong scaling (event.cpp:31,91)")
    work = tempfile.mkdtemp(prefix="egref_")
    cmd = [sys.executable, os.path.join(REF, "bin", "mpirun"), "-np", str(N), os.path.join(REF, "bin", binary)] + prog_args
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    env.pop("OMP_NUM_THREADS", None)          # torchrun exports 1; let the launcher give each rank ncpu/N threads
    budget_s = float(os.environ.get("EGREF_BUDGET_S", "2400"))
    log = open(os.path.join(work, "stdout.txt"), "w")
    t_launch = time.perf_counter()
    proc = subprocess.Popen(cmd, cwd=work, env=env, stdout=log, stderr=subprocess.STDOUT, start_new_session=True)
    files = [os.path.join(work, f"train{r}.txt") for r in range(N)]
    t_start = [None] * N
    t_end = [None] * N
    first_line = None
    try:
        while True:
            now = time.perf_counter()
            for r in range(N):
                if t_end[r] is not None:
                    continue
                n = _count_lines(files[r])
                if n >= 1 and first_line is None:
                    first_line = now
                if t_start[r] is None and n >= W + 1:
                    t_start[r] = now
                if t_start[r] is not None and n >= W + K + 1:
                    t_end[r] = now
            if all(t is not None for t in t_end):
                break
            if proc.poll() is not None:
                tail = open(os.path.join(work, "stdout.txt")).read()[-300:].replace("\n", " | ")
                return _unavailable(f"reference job exited rc={proc.returncode} before {W + K + 1} steps: {tail}")
            if now - t_launch > budget_s:
                done = min(_count_lines(f) for f in files)
                return _unavailable(f"reference reached only {done} of {W + K + 1} steps in {budget_s:.0f} s")
            time.sleep(0.002)
    finally:
        if proc.poll() is None:
            proc.send_signal(signal.SIGTERM)       # the launcher stops its ranks (exact pids) and unlinks its shm
            try:
                proc.wait(timeout=20)
            except subprocess.TimeoutExpired:
                os.killpg(proc.pid, signal.SIGKILL)  # the session/process group WE created above
        log.close()
    # whole-job time for K steps = slowest rank
    seconds = max(t_end[r] - t_start[r] for r in range(N))
    # with a 2 ms poll the resolution is ~0.3 % of a >= 0.6 s region
    value = gb * K / seconds
    losses = []
    try:
        losses = [float(l.split(",")[1]) for l in open(files[0]).read().strip().splitlines()[:W + K + 1]]
    except Exception:
        pass
    build = {}
    try:
        build = json.load(open(os.path.join(REF, "BUILD_LOG.json")))["programs"].get(binary, {})
    except Exception:
        pass
    ncpu = len(os.sched_getaffinity(0))
    out = {
        "metric": "images/sec, CIFAR-10 ResNet (reference topology) D-PSGD ring gossip training step",
        "value": value, "unit": "images/s", "n_gpus": N, "steps": K, "warmup": W,
        "ms_per_step": seconds / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic", "impl": "reference",
        "reference_class": "unmodified reference source (sha256 below) built against the wheel's LibTorch with the "
                           "in-repo shm MPI + OpenCV stand-ins (baseline/shim); CPU only -- the reference hard-wires "
                           "torch::kCPU (dcifar10/event/event.cpp:39), it has no GPU path",
        "config": {"model": "ResNet<BasicBlock>({2,2,2,2},10) as the reference builds it (86 tensors, 17444682 params)",
                   "global_batch": gb, "per_gpu_batch": gb // N, "seq_len": None, "image": "3x32x32",
                   "parallelism": f"{N} MPI ranks (CPU processes), ring gossip via MPI_Put",
                   "algorithm": algo, "program": f"{binary} {' '.join(prog_args)}",
                   "optimizer": "SGD lr=1e-2 momentum=0.9", "cpu_cores": ncpu,
                   "omp_threads_per_rank": max(1, ncpu // N),
                   "timing": "host clock on the reference's own per-step train<rank>.txt lines, max over ranks",
                   "source_sha256": build.get("sha256"), "identical_to_reference": build.get("identical_to_reference")},
        "gpu_launches": 0,
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "CPU program: the timed region already contains its data loading and loss read"},
        "startup_s": (first_line - t_launch) if first_line else None,
        "loss_first_last": [losses[0], losses[-1]] if losses else None,
    }
    print(json.dumps(out), flush=True)
    return 0
