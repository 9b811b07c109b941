#!/usr/bin/env python
"""Headline benchmark (driver contract).

Metric (BASELINE.json): images/sec, whole job, device-timed, max over ranks, for the CIFAR-10
ResNet D-PSGD training step -- the dcifar10/event configuration of the reference
(/root/reference/dcifar10/event/event.cpp:29-42, :91, :196-200): ResNet{2,2,2,2} exactly as the
reference builds it (12 BasicBlocks, 86 tensors, 17 444 682 parameters), GLOBAL batch 256 split
over the ranks (strong scaling), SGD lr 1e-2 momentum 0.9, ring gossip with both neighbours every
step.  Default algorithm = dense D-PSGD (every tensor pushed every step -- the most communication
the reference ever does); `--algo event|spevent|cent` times the other programs.

    python bench.py --gpus N --steps K --warmup W         (torchrun launches N ranks for N>1)

One JSON line on rank 0.  `value` is timed on the device (CUDA events) over K whole training steps
(forward, backward, fused exchange+average+SGD) with inputs already resident; `e2e` repeats the
measurement through the public Trainer API with, every step, the H2D copy of that step's uint8
batch from pinned host memory, GPU decode/augmentation, and a D2H read of the loss.
`--dump-outputs DIR` writes what the last device-timed step computed as DIR/<name>.npy; the inputs are seeded, so
two builds run with the same arguments can be compared output for output.
The headline runs at the reference's precision (fp32, TF32 off) with the Trainer's DEFAULT execution
switches (on a GPU: NHWC + fused BN kernels, whole-step CUDA graph, overlapped pushes for N >= 2) -- the
same configuration `python -m eventgrad_b200.cli.cifar_event` uses; bf16 / tf32 rows ride along under
`other_dtypes`.  `--impl reference` times the unmodified reference C++ program (baseline/).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference", "nccl", "refport"],
                   help="ours: fused p2p kernels | nccl: batched torch.distributed baseline | refport: reference-"
                        "structured per-tensor port (host sync per tensor) | reference: the unmodified reference C++ programs (baseline/_ref, CPU + shm MPI shim)")
    p.add_argument("--algo", default="dpsgd", choices=["dpsgd", "event", "spevent", "cent"])
    p.add_argument("--model", default="resnet18")
    p.add_argument("--global-batch", type=int, default=256)
    p.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    p.add_argument("--dtype", default="fp32", choices=["bf16", "fp32", "tf32"],
                   help="compute dtype of forward/backward. fp32 (default) = IEEE fp32 with TF32 OFF, the reference's "
                        "precision (event.cpp:279); the exchange / optimizer kernels are fp32 in every mode")
    p.add_argument("--conv-tc", default="auto", choices=["auto", "on", "off"],
                   help="fp32 only: 3x3 convolutions on the tcgen05 tensor cores at fp32 accuracy (csrc/conv_tc.cu; "
                        "auto = on) or cuDNN's SIMT fp32 kernels (off)")
    p.add_argument("--also", default="fp32_cudnn,bf16,tf32",
                   help="extra dtypes measured after the headline (device-timed only) and reported under "
                        "`other_dtypes` in the same JSON line; '' to skip")
    p.add_argument("--sync-mode", default="iter", choices=["iter", "async"])
    p.add_argument("--horizon", type=float, default=1.0)
    p.add_argument("--topk", type=float, default=10.0)
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--overlap", default="auto", choices=["auto", "on", "off"],
                   help="split step: pushes on a side stream overlapping forward/backward "
                        "(auto = on for N >= 2: measured 2.65 vs 2.83 ms/step at N=2, 1.95 vs 2.22 at N=4, "
                        "1.89 vs 2.09 at N=8)")
    p.add_argument("--ce-push", action="store_true", help="copy-engine push in the split step (decent + overlap)")
    p.add_argument("--double-buffer", action=argparse.BooleanOptionalAction, default=None,
                   help="fused (non-split) decent step: two inbox slots, no WAR ack (default on where it applies)")
    p.add_argument("--no-channels-last", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--out", default="")
    p.add_argument("--profile", default="", help="write a torch.profiler kernel table of a few e2e steps here")
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="after the timed steps, write what the last one computed (loss, a fixed seeded sample of the "
                        "updated parameters, the BatchNorm running statistics) as DIR/<name>.npy in float32")
    return p.parse_args()


DUMP_PARAM_SAMPLE = 1 << 22          # parameters written by --dump-outputs over all ranks (16 MB of float32)


def dump_outputs(tr, out_dir, rank, world):
    """Write what the last step handed its caller as float32 .npy files: the loss it returned, the updated
    parameters (a fixed, seeded sample of their concatenation in named_parameters() order) and the BatchNorm
    running statistics.  The inputs are seeded, so two builds run with the same arguments compare file by file."""
    import numpy as np
    import torch
    params = torch.cat([p.detach().reshape(-1) for p in tr.model.parameters()]).float().cpu()
    k = DUMP_PARAM_SAMPLE // world
    if params.numel() > k:
        idx = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))[:k].sort().values
        params = params[idx]
    stats = [b.detach().reshape(-1).float() for b in tr.model.buffers() if b.is_floating_point()]
    arrays = {"loss": tr.last_loss.detach().float().reshape(1).cpu(), "params_sample": params,
              "bn_running_stats": torch.cat(stats).cpu() if stats else torch.zeros(0)}
    sfx = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + sfx + ".npy"), a.numpy().astype(np.float32))
    return sorted(name + sfx + ".npy" for name in arrays)


def reference_arm(args):
    # The unmodified reference, built by baseline/build_ref.py into baseline/_ref (shm MPI + OpenCV stand-ins); none of
    # this repo's package is imported on this path.  Details: baseline/ref_arm.py, baseline/README.md.
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "baseline"))
    import ref_arm
    return ref_arm.run(args)


def measure(args, env, dtype, want_e2e, src, sample_clocks, dump_dir=""):
    """One Trainer at `dtype`: device-timed K steps (+ optionally the end-to-end loop).  Returns a dict.
    `fp32_cudnn` = fp32 with the tensor-core convolutions switched off (cuDNN's SIMT fp32 kernels, NCHW).
    With `dump_dir`, what the last device-timed step computed is written there before anything else runs."""
    conv_tc = {"auto": None, "on": True, "off": False}[args.conv_tc]
    if dtype == "fp32_cudnn":
        dtype, conv_tc = "fp32", False
    import torch
    from eventgrad_b200.config import preset
    from eventgrad_b200.engine.trainer import Trainer
    from eventgrad_b200.utils.clocks import NvmlClockSampler
    from eventgrad_b200.utils.dist import barrier, max_over_ranks, sum_over_ranks
    N = env.world
    gb = args.global_batch if args.scaling == "strong" else args.global_batch * N
    per_rank = max(1, gb // N)
    algo = {"dpsgd": "decent", "event": "event", "spevent": "spevent", "cent": "cent"}[args.algo]
    backend = {"ours": "p2p", "nccl": "nccl", "refport": "refport"}[args.impl]
    tri = {"auto": None, "on": True, "off": False}
    cfg = preset("cifar_event", algo=algo, model=args.model, backend=backend, device="cuda",
                 dtype=dtype, batch_size=gb, batch_mode="global", epochs=10 ** 6,
                 sync_mode="iter" if algo == "decent" else args.sync_mode,
                 horizon=args.horizon, topk_percent=args.topk,
                 overlap_push=tri[args.overlap] if backend == "p2p" else False,
                 channels_last=False if args.no_channels_last else None, conv_tc=conv_tc,
                 cuda_graph=False if args.no_graph else None,
                 ce_push=args.ce_push, double_buffer=args.double_buffer,
                 train_samples=len(src), test_samples=256, quiet=True, augment=True)
    tr = Trainer(cfg, env, train_source=src)
    cfg = tr.cfg                      # with the auto switches resolved for this device / world size
    dev = env.device
    table = tr.arena.table
    # ---------------- device-timed: inputs resident on the GPU (a rotating pool of batches) -------
    pool = []
    it = iter(tr.loader)
    for _ in range(4):
        x, y = next(it)
        pool.append((x.clone(), y.clone()))
    torch.cuda.synchronize()
    prewarm = max(args.warmup, Trainer.GRAPH_WARMUP_STEPS + 2)   # eager warm-up + graph capture, untimed
    for i in range(prewarm):
        tr.train_step(*pool[i % len(pool)])
    torch.cuda.synchronize()
    barrier(env)
    sampler = NvmlClockSampler(dev.index or 0, 2.0).start() if (env.rank == 0 and sample_clocks) else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(env)
    torch.cuda.synchronize()
    own0 = tr.own_launches_total
    if sampler is not None:
        sampler.mark_begin()
    e0.record()
    for i in range(args.steps):
        tr.train_step(*pool[i % len(pool)])
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler is not None else None
    own_launches = tr.own_launches_total - own0
    barrier(env)
    ms = max_over_ranks(e0.elapsed_time(e1), env)
    tr.backend.check_status() if hasattr(tr.backend, "check_status") else None
    res = {"dtype": dtype, "ms_per_step": ms / args.steps, "value": gb * args.steps / (ms / 1e3),
           "loss": float(tr.last_loss), "clocks": clocks, "gpu_launches": int(own_launches),
           "own_kernels_per_step": dict(tr.own_launches_per_step), "cfg": cfg, "gb": gb, "per_rank": per_rank,
           "table": table, "algo": algo, "backend": backend}
    if dump_dir:
        res["dumped"] = dump_outputs(tr, dump_dir, env.rank, N)

    # ---------------- end to end through the public API: H2D every step + D2H loss every step ----
    if want_e2e:
        it = iter(tr.loader)
        for _ in range(args.warmup):
            x, y = next(it)
            tr.train_step(x, y)
        torch.cuda.synchronize()
        barrier(env)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        d2h = 0
        tl = tt = ti = 0.0
        # the step's result (loss) is read back EVERY step through a pinned host buffer; the read of
        # step k is issued right after its kernels are enqueued and consumed after step k+1 has been
        # launched (standard 1-step-lagged async logging), so the D2H never drains the GPU queue
        host_loss = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        evs = [torch.cuda.Event() for _ in range(2)]
        losses = []
        for i in range(args.steps):
            ta = time.perf_counter()
            try:
                x, y = next(it)
            except StopIteration:
                it = iter(tr.loader)
                x, y = next(it)
            tb = time.perf_counter()
            loss = tr.train_step(x, y)
            host_loss[i & 1].copy_(loss.reshape(1), non_blocking=True)     # D2H of this step's result
            evs[i & 1].record()
            tc = time.perf_counter()
            if i > 0:
                evs[(i - 1) & 1].synchronize()
                losses.append(float(host_loss[(i - 1) & 1][0]))
            td = time.perf_counter()
            tl += tb - ta; tt += tc - tb; ti += td - tc
            d2h += loss.element_size()
        evs[(args.steps - 1) & 1].synchronize()
        losses.append(float(host_loss[(args.steps - 1) & 1][0]))
        assert len(losses) == args.steps
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        barrier(env)
        ms2 = max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3), env)
        c, h, w = src.sample_shape
        res["e2e"] = {"value": gb * args.steps / (ms2 / 1e3), "unit": "images/s",
                      "ms_per_step": ms2 / args.steps,
                      "h2d_bytes_per_step": int(per_rank * (c * h * w + 8) * N),
                      "d2h_bytes_per_step": int(d2h / args.steps * N),
                      "result_read": "every step, async D2H into pinned memory, consumed one step later",
                      "host_ms": {"loader": tl / args.steps * 1e3, "launch": tt / args.steps * 1e3,
                                  "result_wait": ti / args.steps * 1e3},
                      "last_loss": losses[-1]}

    if args.profile and env.rank == 0 and want_e2e:
        from torch.profiler import ProfilerActivity, profile
        it = iter(tr.loader)
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(4):
                x, y = next(it)
                loss = tr.train_step(x, y)
                loss.item()
        os.makedirs(os.path.dirname(os.path.abspath(args.profile)), exist_ok=True)
        with open(args.profile, "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))

    # ---------------- communication accounting ----------------------------------------------------
    be = tr.backend
    total_steps = be.pass_num
    bytes_rank = be.bytes_sent()
    bytes_all = sum_over_ranks(bytes_rank, env)
    events_all = sum_over_ranks(be.num_events(), env)
    dense_msgs = 2 * table.n_tensors * total_steps * N
    res["comm"] = {"bytes_pushed_per_step_per_gpu": bytes_rank / max(1, total_steps),
                   "events_total": events_all, "dense_messages": dense_msgs,
                   "messages_saved": (1.0 - events_all / dense_msgs)
                   if (algo in ("event", "spevent") and dense_msgs and N > 1) else 0.0,
                   "bytes_pushed_total": bytes_all,
                   "wire_dedup_2rank_ring": bool(getattr(be, "wire_dedup", False))}
    res["dbuf"] = bool(getattr(be, "dbuf", False))
    res["nvls"] = bool(getattr(be, "nvls", False))
    tr.close()
    del tr
    torch.cuda.empty_cache()
    return res


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    from eventgrad_b200.data import synthetic_source
    from eventgrad_b200.utils.dist import init_distributed, shutdown

    if not torch.cuda.is_available():
        print(json.dumps({"impl": args.impl, "error": "bench.py needs a CUDA device (run it through gpurun / on the B200 box)"}))
        return 2
    env = init_distributed("cuda")
    N = env.world
    if N != args.gpus and env.rank == 0:
        print(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={N}", file=sys.stderr)
    gb = args.global_batch if args.scaling == "strong" else args.global_batch * N
    n_train = max(max(1, gb // N) * N * 8, 4096)
    src = synthetic_source("cifar10", n_train).pin()
    r = measure(args, env, args.dtype, not args.no_e2e, src, True, args.dump_outputs)
    others = {}
    for dt in [d for d in args.also.split(",") if d and d != args.dtype]:
        if dt == "fp32_cudnn" and (args.dtype != "fp32" or not r["cfg"].conv_tc):
            continue                       # only meaningful next to a tensor-core fp32 headline
        o = measure(args, env, dt, False, src, False)
        others[dt] = {"value": o["value"], "ms_per_step": o["ms_per_step"], "loss": o["loss"],
                      "gpu_launches": o["gpu_launches"], "timing": "device-timed (CUDA events), same config otherwise"}
    cfg, table, algo = r["cfg"], r["table"], r["algo"]
    out = {
        "metric": "images/sec, CIFAR-10 ResNet (reference topology) D-PSGD ring gossip training step",
        "value": r["value"], "unit": "images/s", "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "impl": args.impl,
        "config": {"model": f"{args.model}-ref(12 BasicBlocks, 86 tensors, {table.n_elems} params)"
                            if args.model == "resnet18" else args.model,
                   "global_batch": r["gb"], "per_gpu_batch": r["per_rank"], "seq_len": None, "image": "3x32x32",
                   "parallelism": f"dp{N}-ring-gossip" if algo != "cent" else f"dp{N}-allreduce",
                   "algorithm": args.algo, "backend": r["backend"], "sync_mode": cfg.sync_mode,
                   "precision": {"fp32": ("fp32 storage and fp32 accuracy, TF32 off; eligible 3x3 convolutions on the tcgen05 "
                                          "tensor cores via 3 bf16 planes x 6 MMAs per product with fp32 round-to-nearest "
                                          "accumulation (rms error vs fp64 1e-7, cuDNN's fp32 kernels: 2-4e-7, "
                                          "tests/test_gpu_conv_tc.py); the other convs on cuDNN fp32"
                                          if cfg.conv_tc else "IEEE fp32 forward/backward on cuDNN, TF32 off")
                                         + " (reference precision)",
                                 "tf32": "TF32 tensor-core convolutions / GEMMs", "bf16": "bf16 autocast"}[args.dtype]
                                + "; parameters, exchange, average and SGD are fp32 in every mode",
                   "overlap_push": bool(cfg.overlap_push), "double_buffer": r["dbuf"], "ce_push": bool(cfg.ce_push),
                   "nvls": r["nvls"],
                   "optimizer": "SGD lr=1e-2 momentum=0.9", "cuda_graph": bool(cfg.cuda_graph),
                   "channels_last": bool(cfg.channels_last), "conv_tc": bool(cfg.conv_tc),
                   "defaults": "execution switches are the Trainer's defaults for this device (same as the CLI)"
                               if (args.overlap == "auto" and not args.no_graph and not args.no_channels_last
                                   and args.conv_tc == "auto" and not args.ce_push and args.double_buffer is None) else "overridden by flags",
                   "l2_policy": "per-step working set (theta,grad,mom,2 inboxes = "
                                f"{5 * table.n_padded * 4 / 1e6:.0f} MB + activations) exceeds the 126 MB L2; "
                                "no explicit flush"},
        "gpu_launches": r["gpu_launches"],
        "gpu_launches_how": "counted by the extension's launchers (csrc/api.h eg_count_launch) inside the timed "
                            "region on rank 0; kernels replayed from the step's CUDA graph are counted from the capture",
        "own_kernels_per_step": r["own_kernels_per_step"],
        "comm": r["comm"],
        "loss": r["loss"],
    }
    if r["clocks"] is not None:
        out["clocks"] = r["clocks"]
    if "e2e" in r:
        out["e2e"] = r["e2e"]
    if others:
        out["other_dtypes"] = others
    if "dumped" in r:
        out["outputs_dumped"] = {"dir": args.dump_outputs, "files": r["dumped"],
                                 "of": "the last device-timed step of the headline dtype"}
    if env.rank == 0:
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    shutdown()
    return 0


if __name__ == "__main__":
    sys.exit(main())
