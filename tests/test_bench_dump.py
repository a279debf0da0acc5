"""CPU: the output files of bench.py --dump-outputs (format, exactness of the state words, the sample of large batches)."""
import types

import numpy as np
import torch

import bench


def _fake_env(e, w, seed):
    rng = np.random.default_rng(seed)
    words = rng.integers(-2**63, 2**63 - 1, size=(e, w), dtype=np.int64)
    return types.SimpleNamespace(state=torch.from_numpy(words),
                                 reward=torch.from_numpy(rng.normal(size=e).astype(np.float32)),
                                 terminated=torch.from_numpy(rng.integers(0, 2, size=e, dtype=np.uint8)),
                                 truncated=torch.from_numpy(rng.integers(0, 2, size=e, dtype=np.uint8)))


def _words(state_u32):
    halves = state_u32.astype(np.uint64).reshape(state_u32.shape[0], -1, 2)
    return (halves[..., 0] | (halves[..., 1] << np.uint64(32))).view(np.int64)


def test_dump_writes_every_result_exactly(tmp_path):
    env = _fake_env(1000, 2, 1)
    bench.dump_outputs(env, str(tmp_path / "out"))
    got = {p.stem: np.load(p) for p in (tmp_path / "out").glob("*.npy")}
    assert sorted(got) == ["reward", "state_u32", "terminated", "truncated"]
    assert got["state_u32"].dtype == np.float64 and got["state_u32"].shape == (1000, 4)
    assert np.array_equal(_words(got["state_u32"]), env.state.numpy())
    for name in ("reward", "terminated", "truncated"):
        assert got[name].dtype == np.float32
        assert np.array_equal(got[name], getattr(env, name).numpy().astype(np.float32))


def test_dump_samples_a_large_batch_the_same_way_every_time(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 20000)
    env = _fake_env(5000, 1, 2)
    for d in ("a", "b"):
        bench.dump_outputs(env, str(tmp_path / d))
    files = sorted((tmp_path / "a").glob("*.npy"))
    assert sum(np.load(p).nbytes for p in files) <= 20000
    for p in files:
        assert np.array_equal(np.load(p), np.load(tmp_path / "b" / p.name))
    keep = np.load(tmp_path / "a" / "env_index.npy").astype(np.int64)
    assert len(keep) > 0 and np.all(np.diff(keep) > 0)
    assert np.array_equal(_words(np.load(tmp_path / "a" / "state_u32.npy")), env.state.numpy()[keep])
    assert np.array_equal(np.load(tmp_path / "a" / "reward.npy"), env.reward.numpy()[keep])
