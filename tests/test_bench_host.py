"""Host-side logic of bench.py that does not need a GPU: the CPU-baseline thread calibration and its per-box cache (the
reference arm and the engine arm's ``cpu_baseline`` leg must time the CPU implementation with the same thread count)."""
import json
import time

import bench


def fake_time_fn(speed_by_threads, calls):
    def time_fn(num_envs, horizon, net_dims, warmup, cycles, threads, batch_size, repeat_times):
        calls.append(threads)
        per_cycle = num_envs * horizon / speed_by_threads[threads]
        # one slow outlier per candidate: the calibration must score the BEST cycle, not the mean
        return {"explore_s": [0.7 * per_cycle] * (cycles - 1) + [7.0 * per_cycle],
                "update_s": [0.3 * per_cycle] * cycles}
    return time_fn


def test_thread_calibration_picks_best_and_is_cached(tmp_path, monkeypatch):
    monkeypatch.setattr(bench.os, "cpu_count", lambda: 128)   # the GPU boxes' host; this container has 8
    cache = str(tmp_path / "threads.json")
    calls = []
    speeds = {8: 5.0e6, 16: 8.0e6, 32: 3.0e6}
    best, scores = bench.calibrate_threads(fake_time_fn(speeds, calls), num_envs=1024, cache=cache)
    assert best == 16 and sorted(calls) == [8, 16, 32]
    assert abs(scores[16] - 8.0e6) / 8.0e6 < 1e-9           # best cycle, not the mean with the outlier
    # a second arm on the same box reuses the choice without timing anything
    calls2 = []
    best2, scores2 = bench.calibrate_threads(fake_time_fn({8: 1.0, 16: 0.5, 32: 0.1}, calls2), num_envs=1024, cache=cache)
    assert best2 == 16 and calls2 == [] and scores2 == scores
    # another workload size, or a stale entry, is calibrated afresh
    calls3 = []
    best3, _ = bench.calibrate_threads(fake_time_fn({8: 9.0e6, 16: 8.0e6, 32: 3.0e6}, calls3), num_envs=2048, cache=cache)
    assert best3 == 8 and sorted(calls3) == [8, 16, 32]
    c = json.load(open(cache))
    c["when"] = time.time() - 7200
    json.dump(c, open(cache, "w"))
    calls4 = []
    best4, _ = bench.calibrate_threads(fake_time_fn({8: 1.0e6, 16: 2.0e6, 32: 3.0e6}, calls4), num_envs=2048, cache=cache)
    assert best4 == 32 and sorted(calls4) == [8, 16, 32]


def test_workload_config_names_the_baseline_configuration():
    cfg = bench.workload_config(1, bench.NUM_ENVS)
    assert "65 536" in cfg["workload"] and cfg["num_envs_total"] == bench.NUM_ENVS
    cfg8 = bench.workload_config(8, 8192)
    assert cfg8["num_envs_per_gpu"] == 8192 and cfg8["num_envs_total"] == 65536 and cfg8["parallelism"] == "env-shard x8"


def test_both_arms_describe_the_same_workload():
    """The reference arm builds its ``config`` from ``workload_config(gpus)``, the engine arm from ``workload_config(world,
    envs_per_gpu)``: for the default (weak-scaling) run they must be the same dict, key for key (the driver compares them)."""
    for n in (1, 2, 4, 8):
        assert bench.workload_config(n) == bench.workload_config(n, bench.NUM_ENVS)
    src = open(bench.__file__).read()
    assert '"config": workload_config(args.gpus)' in src and '"config": workload_config(world, n_envs)' in src


def test_dump_outputs_writes_a_seeded_float32_sample(tmp_path):
    """--dump-outputs: one float32 .npy per output; the same env columns on every call; the full-size buffer stays far below
    64 MB."""
    import numpy as np
    import torch as th
    from elegantrl_b200.agents.nets import ActorPPO, CriticPPO
    h, n = 128, bench.NUM_ENVS
    g = th.Generator().manual_seed(0)
    buffer = [th.rand((h, n, 3), generator=g), th.rand((h, n, 1), generator=g), th.rand((h, n), generator=g),
              th.rand((h, n), generator=g), th.ones((h, n), dtype=th.bool), th.rand((h, n), generator=g) > 0.01]
    agent = type("Agent", (), dict(last_state=th.rand((n, 3), generator=g), act=ActorPPO([64, 64], 3, 1),
                                   cri=CriticPPO([64, 64], 3, 1)))()
    buffer[0][..., 0] = th.arange(n, dtype=th.float32)      # the env index, to see which columns were kept
    losses = th.tensor([0.5, -0.25, 1.4])
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), buffer, losses, agent)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(p.name for p in (tmp_path / "b").iterdir())
    assert {f"{k}.npy" for k in bench.BUFFER_NAMES + ("last_state", "losses", "act.net.0.weight", "cri.net.4.bias")} <= set(files)
    total = 0
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b), f
        total += a.nbytes
    assert total <= 64 << 20
    states = np.load(tmp_path / "a" / "states.npy")
    assert states.shape == (h, bench.DUMP_ENVS, 3)
    cols = states[0, :, 0].astype(np.int64)
    assert len(np.unique(cols)) == bench.DUMP_ENVS and np.array_equal(states, buffer[0].numpy()[:, cols])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "losses.npy"), losses.numpy())
