"""bench.py --dump-outputs: the files it writes for comparing two builds output for output."""
import numpy as np
import torch

import bench


def _nets():
    torch.manual_seed(0)
    return {"G": torch.nn.Sequential(torch.nn.Linear(200, 100), torch.nn.BatchNorm1d(100)),
            "D": torch.nn.Sequential(torch.nn.Linear(8, 4), torch.nn.BatchNorm1d(4))}


def test_dump_is_complete_typed_and_repeatable(tmp_path):
    nets = _nets()
    losses = torch.arange(9, dtype=torch.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), nets, losses)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["D.buffers.npy", "D.params.npy", "G.buffers.npy", "G.params.npy", "losses.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
    assert np.array_equal(np.load(tmp_path / "a" / "losses.npy"), losses.numpy())
    g = np.load(tmp_path / "a" / "G.params.npy")
    w = nets["G"][0].weight.detach().reshape(-1).numpy()
    # the 20000-value weight is sampled, the small tensors are kept whole
    assert g.shape == (bench.DUMP_SAMPLE + 100 + 100 + 100,)
    assert np.isin(g[:bench.DUMP_SAMPLE], w).all()
    assert np.array_equal(g[bench.DUMP_SAMPLE:bench.DUMP_SAMPLE + 100], nets["G"][0].bias.detach().numpy())
    d = np.load(tmp_path / "a" / "D.params.npy")
    assert np.array_equal(d, torch.cat([p.detach().reshape(-1) for p in nets["D"].parameters()]).numpy())
    buf = np.load(tmp_path / "a" / "G.buffers.npy")
    assert buf.dtype == np.float64 and buf.shape == (100 + 100 + 1,)
