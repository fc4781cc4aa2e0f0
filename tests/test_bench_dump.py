"""`bench.py --dump-outputs`: the loss and the updated weights of the last timed step, fp32 master copies preferred,
sampled at fixed positions so two runs (or two builds) can be compared element for element."""
import numpy as np
import torch
import torch.nn as nn

from colossalai_b200.amp.naive_amp.mixed_precision_optimizer import MixedPrecisionOptimizer
from colossalai_b200.interface import ModelWrapper


def _boosted(seed):
    torch.manual_seed(seed)
    model = nn.Sequential(nn.Linear(64, 48), nn.LayerNorm(48)).to(torch.bfloat16)
    opt = MixedPrecisionOptimizer(torch.optim.SGD(model.parameters(), lr=0.1), model, precision="bf16")
    return ModelWrapper(model), opt


def test_dump_outputs(tmp_path, monkeypatch):
    monkeypatch.setenv("PYTORCH_CUDA_ALLOC_CONF", "")       # importing bench must not change the allocator of this process
    import bench

    monkeypatch.setattr(bench, "DUMP_SAMPLES_PER_TENSOR", 100)
    model, opt = _boosted(0)
    masters = opt.get_working_to_master_map()
    w = model.unwrap()[0].weight
    masters[id(w)].add_(1e-4)                              # an update the bf16 working copy cannot represent
    bench.dump_outputs(str(tmp_path / "a"), 2.5, model, opt)

    loss = np.load(tmp_path / "a" / "loss.npy")
    assert loss.dtype == np.float64 and loss.tolist() == [2.5]
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["loss.npy", "param.0.bias.npy", "param.0.weight.npy", "param.1.bias.npy", "param.1.weight.npy"]
    sample = np.load(tmp_path / "a" / "param.0.weight.npy")
    assert sample.dtype == np.float32 and sample.shape == (100,)
    assert np.isin(sample, masters[id(w)].reshape(-1).numpy()).all()
    assert not np.isin(sample, w.detach().float().reshape(-1).numpy()).all()
    bias = np.load(tmp_path / "a" / "param.0.bias.npy")       # small tensors are written whole
    np.testing.assert_array_equal(bias, masters[id(model.unwrap()[0].bias)].numpy())

    model2, opt2 = _boosted(0)
    opt2.get_working_to_master_map()[id(model2.unwrap()[0].weight)].add_(1e-4)
    bench.dump_outputs(str(tmp_path / "b"), 2.5, model2, opt2)
    for n in names:
        np.testing.assert_array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n))
