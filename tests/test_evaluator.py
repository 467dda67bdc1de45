"""SURVEY section 8 row f4 (evaluator rollout): ``elegantrl_b200.train.evaluator`` against the reference's own
``get_cumulative_rewards_and_step_from_vec_env`` (``elegantrl/train/evaluator.py:200-238``): the (return, steps) lists it
produced for the same actor and injected reset noise are stored in ``tests/golden/evaluator_pendulum.npz``
(``oracle/make_golden.py::main_evaluator``)."""
import numpy as np
import pytest
import torch as th

from tests import golden_utils as gu


def _reference_segmentation(returns, dones):
    """The host loop of the reference (evaluator.py:222-237), restated for a [T, N] pair."""
    out = []
    for i in range(returns.shape[1]):
        where = (np.nonzero(dones[:, i])[0] + 1).tolist()
        j0 = 0
        for j1 in where:
            out.append((float(returns[j0:j1, i].sum()), j1 - j0))
            j0 = j1
    return out


@pytest.mark.parametrize("t_len,n,p", [(40, 7, 0.1), (33, 64, 0.03), (12, 5, 0.0), (9, 3, 1.0)])
def test_episode_segmentation_matches_the_reference_loop(t_len, n, p):
    from elegantrl_b200.train.evaluator import episodes_from_returns_dones
    rng = np.random.default_rng(t_len * 100 + n)
    returns = rng.standard_normal((t_len, n)).astype(np.float32)
    dones = rng.random((t_len, n)) < p
    got = episodes_from_returns_dones(th.from_numpy(returns), th.from_numpy(dones))
    want = _reference_segmentation(returns, dones)
    assert [s for _, s in got] == [s for _, s in want]
    np.testing.assert_allclose([r for r, _ in got], [r for r, _ in want], rtol=1e-5, atol=1e-5)


def _reference_result(n, max_step, seed):
    """What the reference function returned on the CPU env with ``n`` envs, ``max_step`` and reset-noise seed ``seed``."""
    g = gu.load("evaluator_pendulum")
    return list(zip(g[f"n{n}_t{max_step}_s{seed}.returns"].tolist(), g[f"n{n}_t{max_step}_s{seed}.steps"].tolist()))


def _actor(device):
    """ActorPPO 2x64 with the parameters the golden was minted with (seeded init, perturbed biases)."""
    from elegantrl_b200.agents.nets import ActorPPO
    g = gu.load("evaluator_pendulum")
    actor = ActorPPO([64, 64], 3, 1)
    actor.load_state_dict({k[len("actor."):]: th.from_numpy(v) for k, v in g.items() if k.startswith("actor.")})
    return actor.to(device)


def test_generic_path_equals_reference_function_on_cpu():
    from elegantrl_b200.envs import PendulumVecEnv
    from elegantrl_b200.train.evaluator import get_cumulative_rewards_and_step_from_vec_env
    actor = _actor("cpu")
    noise = th.rand((64, 24, 2), generator=th.Generator().manual_seed(3))
    env = PendulumVecEnv(num_envs=24, gpu_id=-1, max_step=30)
    env.inject_reset_noise(noise)
    with th.no_grad():
        out = [_reference_result(24, 30, 3), get_cumulative_rewards_and_step_from_vec_env(env, actor)]
    assert [s for _, s in out[0]] == [s for _, s in out[1]] == [30] * 24
    np.testing.assert_allclose([r for r, _ in out[1]], [r for r, _ in out[0]], rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("n,max_step", [(24, 30), (1344, 40)])
def test_fused_evaluation_rollout_equals_reference_function(n, max_step):
    """One deterministic launch of the fused kernel + GPU segmentation == the reference's Python loop over the torch env
    (CPU) with the torch actor, same injected reset noise."""
    from elegantrl_b200.envs import PendulumVecEnv
    from elegantrl_b200.train import evaluator as ev
    actor_gpu = _actor("cuda:0")
    noise = th.rand((max_step + 2, n, 2), generator=th.Generator().manual_seed(11))
    want = _reference_result(n, max_step, 11)
    env_gpu = PendulumVecEnv(num_envs=n, gpu_id=0, max_step=max_step)
    env_gpu.inject_reset_noise(noise)
    assert ev._fused_pendulum_ok(env_gpu, actor_gpu)
    got = ev.get_cumulative_rewards_and_step_from_vec_env(env_gpu, actor_gpu)
    assert len(got) == len(want) == n and [s for _, s in got] == [s for _, s in want]
    np.testing.assert_allclose([r for r, _ in got], [r for r, _ in want], rtol=1e-4, atol=1e-4)


@pytest.mark.gpu
def test_fused_evaluation_at_full_size_is_one_episode_per_env():
    from elegantrl_b200.envs import PendulumVecEnv
    from elegantrl_b200.train import evaluator as ev
    env = PendulumVecEnv(num_envs=65536, gpu_id=0, max_step=200, seed=1)
    got = ev.get_cumulative_rewards_and_step_from_vec_env(env, _actor("cuda:0"))
    assert len(got) == 65536 and all(s == 200 for _, s in got)
    r = np.array([x for x, _ in got])
    assert np.isfinite(r).all() and (r <= 0).all() and r.std() > 1.0   # Pendulum returns are costs; untrained policy: wide spread
