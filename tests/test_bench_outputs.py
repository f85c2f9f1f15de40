"""bench.py --dump-outputs: what the last timed env step returned, as float arrays, at most 64 MiB, the same envs on
every run."""
import numpy as np
import torch

import bench


def fake_step(n):
    g = torch.Generator().manual_seed(n)
    return ({"obs": torch.rand(n, 487, generator=g)}, torch.rand(n, generator=g), torch.randint(0, 2, (n,), generator=g),
            {"time_outs": torch.randint(0, 2, (n,), generator=g), "stacked_rewards": torch.rand(n, 15, generator=g),
             "reward_names": ["r"] * 15})


def test_step_outputs_whole_batch():
    out = fake_step(4096)
    got = bench.step_outputs(out)
    assert sorted(got) == ["env_index", "obs", "reset", "rew", "stacked_rewards", "time_outs"]
    assert got["obs"].dtype == np.float32 and got["reset"].dtype == np.float64 and got["env_index"].dtype == np.float64
    assert np.array_equal(got["obs"], out[0]["obs"].numpy()) and np.array_equal(got["reset"], out[2].numpy())
    assert np.array_equal(got["env_index"], np.arange(4096))


def test_step_outputs_sampled_beyond_64_mib(tmp_path):
    out = fake_step(65536)
    got = bench.step_outputs(out)
    idx = got["env_index"].astype(np.int64)
    assert 0 < len(idx) < 65536 and np.all(np.diff(idx) > 0)
    assert np.array_equal(got["obs"], out[0]["obs"].numpy()[idx]) and np.array_equal(got["time_outs"], out[3]["time_outs"].numpy()[idx])
    assert np.array_equal(bench.step_outputs(out)["env_index"], got["env_index"])
    bench.write_outputs(str(tmp_path / "d"), got)
    assert sum(f.stat().st_size for f in (tmp_path / "d").iterdir()) <= 64 << 20
