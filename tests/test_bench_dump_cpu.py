"""CPU: bench.py --dump-outputs writes a fixed, seeded sample of the last step's outputs as float32 .npy files (plus the sampled
game indices as float64), within its byte budget and row for row equal to the tensors it was given."""
import os

import numpy as np
import torch

import bench


def _step_out(G, N, seed):
    g = torch.Generator().manual_seed(seed)
    return dict(obs=torch.randint(-1, 2, (G, N, N), dtype=torch.int8, generator=g),
                mask=torch.randint(0, 2, (G, N * N), dtype=torch.uint8, generator=g),
                reward=torch.randn(G, generator=g), done=torch.randint(0, 2, (G,), dtype=torch.uint8, generator=g))


def test_dump_is_a_fixed_sample_within_budget(tmp_path):
    G, N, budget, offset = 5000, 5, 64 << 10, 7000
    out = _step_out(G, N, 1)
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    bench.dump_outputs(a, out, G, offset, max_bytes=budget)
    bench.dump_outputs(b, _step_out(G, N, 2), G, offset, max_bytes=budget)
    names = sorted(os.listdir(a))
    assert names == ["done.npy", "game_index.npy", "mask.npy", "obs.npy", "reward.npy"]
    assert sum(os.path.getsize(os.path.join(a, f)) for f in names) <= budget + 5 * 256   # + the .npy headers
    idx = np.load(os.path.join(a, "game_index.npy"))
    assert idx.dtype == np.float64 and 0 < len(idx) < G
    assert np.array_equal(idx, np.load(os.path.join(b, "game_index.npy")))     # the same games whatever the outputs
    rows = idx.astype(np.int64) - offset
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < G
    for k, t in out.items():
        got = np.load(os.path.join(a, k + ".npy"))
        assert got.dtype == np.float32
        assert np.array_equal(got, t.numpy()[rows].astype(np.float32)), k


def test_dump_keeps_every_game_when_they_fit(tmp_path):
    G, N = 40, 4
    out = _step_out(G, N, 3)
    bench.dump_outputs(str(tmp_path), out, G, 0)
    assert np.array_equal(np.load(str(tmp_path / "game_index.npy")), np.arange(G, dtype=np.float64))
    assert np.array_equal(np.load(str(tmp_path / "obs.npy")), out["obs"].numpy().astype(np.float32))
