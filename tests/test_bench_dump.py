"""`bench.py --dump-outputs`: what the last timed step computed, as float32 .npy files of bounded size, sampled the
same way on every run so that two builds can be compared output for output."""
import os
import types

import numpy as np
import torch

import bench
from eventgrad_b200.models import build_model


def _fake_trainer(model):
    return types.SimpleNamespace(model=model, last_loss=torch.tensor(2.302585, dtype=torch.float32))


def test_dump_outputs_files_dtypes_and_size(tmp_path):
    torch.manual_seed(0)
    model = build_model("resnet18")
    n_params = sum(p.numel() for p in model.parameters())
    assert n_params > bench.DUMP_PARAM_SAMPLE                  # the flagship model is sampled, not written whole
    files = bench.dump_outputs(_fake_trainer(model), str(tmp_path), 0, 1)
    assert files == ["bn_running_stats.npy", "loss.npy", "params_sample.npy"]
    total = 0
    for f in files:
        a = np.load(tmp_path / f)
        assert a.dtype == np.float32
        total += os.path.getsize(tmp_path / f)
    assert total <= 64 << 20
    assert np.load(tmp_path / "loss.npy").tolist() == [np.float32(2.302585)]
    sample = np.load(tmp_path / "params_sample.npy")
    assert sample.shape == (bench.DUMP_PARAM_SAMPLE,)
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy()
    assert np.isin(sample, flat).all()
    n_stats = sum(b.numel() for b in model.buffers() if b.is_floating_point())
    assert np.load(tmp_path / "bn_running_stats.npy").shape == (n_stats,)


def test_dump_outputs_sample_is_fixed_and_split_over_ranks(tmp_path):
    torch.manual_seed(0)
    model = build_model("resnet18")
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(_fake_trainer(model), str(a), 0, 1)
    bench.dump_outputs(_fake_trainer(model), str(b), 0, 1)
    assert np.array_equal(np.load(a / "params_sample.npy"), np.load(b / "params_sample.npy"))
    files = bench.dump_outputs(_fake_trainer(model), str(tmp_path / "r"), 3, 8)
    assert "params_sample_rank3.npy" in files
    assert np.load(tmp_path / "r" / "params_sample_rank3.npy").shape == (bench.DUMP_PARAM_SAMPLE // 8,)
