"""The drop-in agent under a training loop (north_star: "drops in behind examples/demo_A2C_PPO.py").

The loop below makes the calls the reference's single-process ``train_agent`` makes on an on-policy agent
(``elegantrl/train/run.py:39-138``), in the same order and with the configuration of ``examples/demo_A2C_PPO.py:57-88``:
agent construction, ``last_state`` from ``env.reset()`` (a ``[1, S]`` tensor for the single env), ``explore_env`` /
``buffer[:] = items`` / ``update_net`` with autograd switched on only around the update, ``agent.explore_rate``, an evaluation
that calls ``actor(state)`` on a separate eval env, ``th.save(actor)`` and ``save_or_load_agent``.  It runs a few cycles on
the B200 and checks what the loop leaves behind."""
import os

import numpy as np
import pytest
import torch as th

pytestmark = pytest.mark.gpu


def _evaluate(env, actor, device):
    """(return, steps) of one episode per sub-env of ``env``: the vec env's fused path, or a step loop for the single env."""
    from elegantrl_b200.train.evaluator import get_cumulative_rewards_and_step_from_vec_env
    if env.num_envs > 1:
        return get_cumulative_rewards_and_step_from_vec_env(env, actor)
    state, _ = env.reset()
    total, steps = 0.0, 0
    for steps in range(1, env.max_step + 1):
        action = actor(th.as_tensor(state, dtype=th.float32, device=device).unsqueeze(0))
        state, reward, terminal, truncate, _ = env.step(action[0].cpu().numpy())
        total += reward
        if terminal or truncate:
            break
    return [(total, steps)]


@pytest.mark.parametrize("num_envs", [512, 1])
def test_training_loop_runs_the_dropin(tmp_path, num_envs):
    from elegantrl_b200 import Config
    from elegantrl_b200.agents import AgentPPO
    from elegantrl_b200.envs import PendulumEnv, PendulumVecEnv

    th.cuda.set_device(0)
    device = th.device("cuda:0")
    horizon_len, cycles = 32, 4
    env_class = PendulumVecEnv if num_envs > 1 else PendulumEnv
    env_args = {'env_name': 'Pendulum-v1', 'num_envs': num_envs, 'max_step': 40, 'state_dim': 3, 'action_dim': 1,
                'if_discrete': False}
    args = Config(agent_class=AgentPPO, env_class=env_class, env_args=env_args)   # demo_A2C_PPO.py:73-88
    args.net_dims = [64, 64]
    args.horizon_len = horizon_len
    args.batch_size, args.repeat_times = (128, 8) if num_envs > 1 else (16, 2)
    args.gamma, args.state_value_tau = 0.97, 0.1
    args.gpu_id, args.random_seed = 0, 0
    cwd = str(tmp_path / "run")
    os.makedirs(cwd)

    th.manual_seed(args.random_seed)
    env = env_class(num_envs=num_envs, gpu_id=0, max_step=40, seed=0)
    eval_env = env_class(num_envs=num_envs, gpu_id=0, max_step=40, seed=1)
    agent = args.agent_class(args.net_dims, args.state_dim, args.action_dim, gpu_id=args.gpu_id, args=args)
    state, _ = env.reset()
    if num_envs == 1:
        assert isinstance(state, np.ndarray) and state.shape == (3,)
        state = th.tensor(state, dtype=th.float32, device=agent.device).unsqueeze(0)
    assert state.shape == (num_envs, 3)
    agent.last_state = state.detach()

    recorder, buffer, total_step = [], [], 0
    th.set_grad_enabled(False)
    try:
        for _ in range(cycles):
            buffer[:] = agent.explore_env(env, horizon_len)
            assert [t.shape[:2] for t in buffer] == [(horizon_len, num_envs)] * 6
            exp_r = buffer[3].mean().item()
            th.set_grad_enabled(True)
            obj_critic, obj_actor, obj_entropy = agent.update_net(buffer)
            explore_rate = agent.explore_rate
            th.set_grad_enabled(False)
            total_step += horizon_len * num_envs
            returns = np.array([r for r, _ in _evaluate(eval_env, agent.act, device)])
            recorder.append((total_step, returns.mean(), returns.std(), exp_r, obj_critic, obj_actor, obj_entropy, explore_rate))
            th.save(agent.act, os.path.join(cwd, f"actor__{total_step:012}_{returns.mean():09.3f}.pt"))
        agent.save_or_load_agent(cwd, if_save=True)
    finally:
        th.set_grad_enabled(True)

    recorder = np.array(recorder)
    assert recorder.shape == (cycles, 8) and np.isfinite(recorder).all()
    assert list(recorder[:, 0]) == sorted(recorder[:, 0]) and recorder[-1, 0] == cycles * horizon_len * num_envs
    assert sum(f.startswith("actor__") and f.endswith(".pt") for f in os.listdir(cwd)) == cycles
    for name in ("act.pth", "cri.pth", "act_optimizer.pth", "cri_optimizer.pth"):             # save_or_load_agent (AgentBase.py:280-297)
        assert os.path.isfile(os.path.join(cwd, name)), name
    actor = th.load(os.path.join(cwd, "act.pth"), map_location="cuda:0", weights_only=False)
    out = actor(th.zeros((5, 3), device="cuda:0"))
    assert out.shape == (5, 1) and bool((out.abs() <= 1).all())
    # a fresh agent resumes from the checkpoint (continue_train, run.py:48-49)
    resumed = args.agent_class(args.net_dims, args.state_dim, args.action_dim, gpu_id=args.gpu_id, args=args)
    resumed.save_or_load_agent(cwd, if_save=False)
    probe = th.randn((7, 3), device="cuda:0")
    with th.no_grad():
        assert th.equal(resumed.act(probe), agent.act(probe)) and th.equal(resumed.cri(probe), agent.cri(probe))
