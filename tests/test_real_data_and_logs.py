"""Real-dataset readers (tiny fake files in the on-disk formats the reference consumes) and the
reference debug-file formats (SURVEY.md A.3)."""
import gzip
import json
import os
import struct
import subprocess
import sys

import numpy as np
import torch

from eventgrad_b200.data.sources import cifar10_source, mnist_source
from eventgrad_b200.parallel.base import StepLog
from eventgrad_b200.utils.logfiles import RefLogWriter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _write_idx(path, arr, gz=False):
    op = gzip.open if gz else open
    with op(path, "wb") as f:
        f.write(struct.pack(">I", 0x0800 | arr.ndim))
        f.write(struct.pack(">" + "I" * arr.ndim, *arr.shape))
        f.write(arr.astype(np.uint8).tobytes())


def test_mnist_idx_reader(tmp_path):
    imgs = np.random.randint(0, 256, (50, 28, 28), dtype=np.uint8)
    labs = np.random.randint(0, 10, (50,), dtype=np.uint8)
    _write_idx(tmp_path / "train-images-idx3-ubyte", imgs)
    _write_idx(tmp_path / "train-labels-idx1-ubyte.gz", labs, gz=True)
    src = mnist_source(str(tmp_path), train=True)
    assert src.images.shape == (50, 1, 28, 28) and src.images.dtype == torch.uint8
    assert torch.equal(src.images[:, 0], torch.from_numpy(imgs)) and torch.equal(src.labels, torch.from_numpy(labs).long())
    assert abs(src.scale - 1 / 255) < 1e-9 and (src.mean, src.std) == (0.1307, 0.3081)     # event.cpp:133-136


def test_cifar_binary_and_folder_readers(tmp_path):
    # (c) binary batches
    raw = np.random.randint(0, 256, (20, 3073), dtype=np.uint8)
    raw[:, 0] = np.arange(20) % 10
    b = tmp_path / "bin"
    b.mkdir()
    for i in range(1, 6):
        raw[(i - 1) * 4:i * 4].tofile(b / f"data_batch_{i}.bin")
    src = cifar10_source(str(b), train=True)
    assert src.images.shape == (20, 3, 32, 32) and src.labels.tolist() == (np.arange(20) % 10).tolist()
    assert (src.scale, src.mean, src.std) == (1.0, 0.0, 1.0)                                  # Q7: raw 0..255
    # (a) the reference's image-folder tree train/<class>/<0000>.jpg (custom.hpp:77-118), decoded with cv2
    import cv2
    from eventgrad_b200.data.sources import CIFAR_CLASSES
    f = tmp_path / "folders"
    for ci, cname in enumerate(CIFAR_CLASSES):
        d = f / "train" / cname
        d.mkdir(parents=True)
        for k in range(2):
            im = np.full((40, 36, 3), 20 * ci + k, dtype=np.uint8)      # not 32x32: reader must resize
            cv2.imwrite(str(d / f"{k:04d}.png"), im)
    src2 = cifar10_source(str(f), train=True)
    assert src2.images.shape == (20, 3, 32, 32) and sorted(src2.labels.tolist()) == sorted(list(range(10)) * 2)
    i0 = int((src2.labels == 3).nonzero()[0])
    assert int(src2.images[i0].float().mean().round()) in (60, 61)


def test_reference_log_formats(tmp_path):
    sz = 3
    lg = StepLog(1, torch.tensor([1.5, 0.25, 2.0]), torch.tensor([0.0, 0.125, 1e-3]), torch.tensor([True, False, True]),
                 torch.tensor([1.0, 0.0, 3.0]), torch.tensor([0.5, 0.0, 2.0]),
                 torch.tensor([True, False, True]), torch.tensor([False, False, True]))
    for ds, mnist in (("cifar10", False), ("mnist", True)):
        d = tmp_path / ds
        w = RefLogWriter(str(d), 2, "event", ds, True)
        w.write_steps([lg])
        w.write_train(7, 0.123456789)
        w.close()
        send = open(d / "send2.txt").read()
        assert send == "1.5,  0,  1,  0.25,  0.125,  0,  2,  0.001,  1,  \n"          # "<norm>,  <thres>,  <1|0>,  "
        recv = open(d / "recv2.txt").read()
        if mnist:    # flag only written when a new value arrived (dmnist/event/event.cpp:418-426)
            assert recv == "1,  1,  0.5,  0,  0,  1,  3,  1,  2,  \n"
        else:        # CIFAR writes the 0 as well (dcifar10/event/event.cpp:400-412)
            assert recv == "1,  1,  0,  0.5,  0,  0,  0,  0,  1,  3,  1,  2,  \n"
            assert open(d / "train2.txt").read() == "7, 0.123457\n"                     # iostream default = %g


def _check_reference_line(d):
    assert d["impl"] == "reference"
    assert d["value"] > 0 and d["unit"] == "images/s" and d["dtype"] == "fp32" and d["steps"] == 1
    assert d["config"]["identical_to_reference"] is True and d["gpu_launches"] == 0
    assert d["e2e"]["value"] == d["value"]


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` either times the unmodified reference (baseline/_ref built) and prints the bench
    schema with impl=reference, or says why it cannot -- always one JSON line, exit 0, none of our package loaded.
    tests/golden holds the line the reference's cifar_event printed for these arguments (CPU, 8 cores): it must meet
    the same schema, and a live run must have been built from the same source and start from the same loss (the
    program seeds its weights, sampler and transforms)."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_arm_cifar_event.json")) as f:
        golden = json.load(f)
    _check_reference_line(golden)
    env = dict(os.environ, EGREF_BUDGET_S="240")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference"
    if "unavailable" in d:
        assert isinstance(d["unavailable"], str) and d["unavailable"]
    else:
        _check_reference_line(d)
        for k in ("source_sha256", "program", "model", "global_batch"):
            assert d["config"][k] == golden["config"][k], k
        assert np.allclose(d["loss_first_last"], golden["loss_first_last"], rtol=1e-3, atol=0)
