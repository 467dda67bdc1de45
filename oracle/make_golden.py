"""Mint golden vectors for the on-policy hot path FROM THE IMPORTABLE PYTHON REFERENCE.  Test infrastructure.

Runs only in the build container (needs ``/root/reference``); the GPU box consumes the committed
``tests/golden/*.npz``.  Usage::

    python oracle/make_golden.py            # rewrites tests/golden/*.npz

What is recorded (SURVEY.md section 8(c) checkpoints), all produced by the UNMODIFIED reference classes
``elegantrl.agents.AgentPPO`` (``elegantrl/agents/AgentPPO.py``) on CPU, float32:

1. nets:     (state, action) -> actor mean / tanh action / logprob / entropy, critic value
             (``ActorPPO.forward`` :363, ``get_logprob_entropy`` :378, ``CriticPPO.forward`` :435)
2. gae:      (states, rewards, undones, unmasks, last_state) -> values, advantages, reward_sums, normalised
             advantages, and the in-place mutated rewards / undones (``update_net`` :141-149,
             ``get_advantages`` :207-232), for both scan branches
3. update:   k consecutive ``update_objectives`` calls (:173-205) with the minibatch ids replayed from
             ``th.manual_seed`` -> the three logged scalars per minibatch, post-update parameters and Adam
             moments; plus a full ``update_net`` (:135-171) from the same start
4. rollout:  ``_explore_vec_env`` (:87-129) on ``elegantrl_b200.envs.PendulumVecEnv`` (CPU torch) with the
             policy noise replayed from ``th.manual_seed`` and the env's reset noise injected
5. indices / masks: ids % H, ids // H, ~terminals, ~truncates are part of 2-4 and compared bit-exactly.
"""
import copy
import os
import sys

import numpy as np
import torch as th

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.environ.get("ELEGANTRL_REFERENCE", "/root/reference")
sys.path.insert(0, REFERENCE)
sys.path.insert(0, REPO)

from elegantrl.agents import AgentPPO as RefAgentPPO  # noqa: E402  (the reference)
from elegantrl.train.config import Config as RefConfig  # noqa: E402
from elegantrl_b200.envs import PendulumVecEnv  # noqa: E402

OUT_DIR = os.path.join(REPO, "tests", "golden")


def make_ref_agent(state_dim, action_dim, net_dims, num_envs, seed, **hyper):
    th.manual_seed(seed)
    env_args = {'env_name': 'golden', 'num_envs': num_envs, 'max_step': 200, 'state_dim': state_dim,
                'action_dim': action_dim, 'if_discrete': False}
    args = RefConfig(agent_class=RefAgentPPO, env_class=None, env_args=env_args)
    args.net_dims = list(net_dims)
    for k, v in hyper.items():
        setattr(args, k, v)
    agent = RefAgentPPO(list(net_dims), state_dim, action_dim, gpu_id=-1, args=args)
    return agent


def perturb_nets(agent, seed, std_log=-0.3, norm_stats=False):
    """Move off the init point so that nothing is trivially zero (action_std_log, biases, norm stats)."""
    g = th.Generator().manual_seed(seed)
    with th.no_grad():
        agent.act.action_std_log += std_log + 0.1 * th.randn(agent.act.action_std_log.shape, generator=g)
        for net in (agent.act.net, agent.cri.net):
            for layer in net:
                if hasattr(layer, "bias"):
                    layer.bias += 0.05 * th.randn(layer.bias.shape, generator=g)
        if norm_stats:
            avg = 0.3 * th.randn(agent.act.state_avg.shape, generator=g)
            std = 0.5 + th.rand(agent.act.state_std.shape, generator=g)
            for m in (agent.act, agent.cri):
                m.state_avg[:] = avg
                m.state_std[:] = std


def dump_net(prefix, module, out):
    linears = [m for m in module.net if isinstance(m, th.nn.Linear)]
    out[f"{prefix}.n_layers"] = np.int64(len(linears))
    for i, l in enumerate(linears):
        out[f"{prefix}.W{i}"] = l.weight.detach().numpy().copy()
        out[f"{prefix}.b{i}"] = l.bias.detach().numpy().copy()
    out[f"{prefix}.state_avg"] = module.state_avg.detach().numpy().copy()
    out[f"{prefix}.state_std"] = module.state_std.detach().numpy().copy()
    if hasattr(module, "action_std_log"):
        out[f"{prefix}.action_std_log"] = module.action_std_log.detach().numpy().copy()


def dump_adam(prefix, optimizer, module, out):
    linears = [m for m in module.net if isinstance(m, th.nn.Linear)]
    params = [p for l in linears for p in (l.weight, l.bias)]
    names = [n for i in range(len(linears)) for n in (f"W{i}", f"b{i}")]
    if hasattr(module, "action_std_log"):
        params.append(module.action_std_log)
        names.append("action_std_log")
    for p, n in zip(params, names):
        st = optimizer.state[p]
        if "exp_avg" not in st:  # ActorDiscretePPO.action_std_log never receives a gradient: Adam never creates its state
            continue
        out[f"{prefix}.m.{n}"] = st["exp_avg"].detach().numpy().copy()
        out[f"{prefix}.v.{n}"] = st["exp_avg_sq"].detach().numpy().copy()
        out[f"{prefix}.step"] = np.float64(float(st["step"]))


def synth_buffer(agent, horizon_len, num_envs, seed, p_term=0.08, p_trunc=0.08):
    g = th.Generator().manual_seed(seed)
    s_dim, a_dim = agent.state_dim, agent.action_dim
    states = th.randn((horizon_len, num_envs, s_dim), generator=g)
    actions = 0.7 * th.randn((horizon_len, num_envs, a_dim), generator=g)
    with th.no_grad():
        logprobs = agent.act.get_logprob_entropy(states.reshape(-1, s_dim), actions.reshape(-1, a_dim))[0]
        logprobs = logprobs.reshape(horizon_len, num_envs) + 0.05 * th.randn((horizon_len, num_envs), generator=g)
    rewards = th.randn((horizon_len, num_envs), generator=g)
    terminals = th.rand((horizon_len, num_envs), generator=g) < p_term
    truncates = (th.rand((horizon_len, num_envs), generator=g) < p_trunc) & ~terminals
    last_state = th.randn((num_envs, s_dim), generator=g)
    return states, actions, logprobs, rewards, ~terminals, ~truncates, last_state


def record_nets(agent, out, seed):
    g = th.Generator().manual_seed(seed)
    state = th.randn((37, agent.state_dim), generator=g) * 1.5
    action = th.randn((37, agent.action_dim), generator=g)
    with th.no_grad():
        logprob, entropy = agent.act.get_logprob_entropy(state, action)
        out["nets.state"] = state.numpy()
        out["nets.action"] = action.numpy()
        out["nets.actor_mean"] = agent.act.net(agent.act.state_norm(state)).numpy()
        out["nets.actor_forward"] = agent.act(state).numpy()
        out["nets.logprob"] = logprob.numpy()
        out["nets.entropy"] = entropy.numpy()
        out["nets.value"] = agent.cri(state).squeeze(1).numpy()


def record_gae(agent, buf, out, tag):
    states, actions, logprobs, rewards, undones, unmasks, last_state = [t.clone() for t in buf]
    agent.last_state = last_state
    with th.no_grad():
        values = agent.cri(states).squeeze(-1)
        advantages = agent.get_advantages(states, rewards, undones, unmasks, values)  # mutates rewards/undones
        reward_sums = advantages + values
        adv_norm = (advantages - advantages.mean()) / (advantages[::4, ::4].std() + 1e-5)
    out[f"{tag}.values"] = values.numpy()
    out[f"{tag}.last_value"] = agent.cri(last_state).detach().squeeze(-1).numpy()
    out[f"{tag}.advantages"] = advantages.numpy()
    out[f"{tag}.reward_sums"] = reward_sums.numpy()
    out[f"{tag}.adv_norm"] = adv_norm.numpy()
    out[f"{tag}.adv_mean"] = np.float64(advantages.mean().item())
    out[f"{tag}.adv_std"] = np.float64(advantages[::4, ::4].std().item())
    out[f"{tag}.rewards_after"] = rewards.numpy()
    out[f"{tag}.undones_after"] = undones.numpy()
    return states, actions, unmasks, logprobs, adv_norm, reward_sums


def record_update(agent, train_buffer, out, num_updates, seed):
    """k update_objectives calls with replayed ids, on a deep copy (the caller's agent stays untouched)."""
    agent = copy.deepcopy(agent)
    horizon_len, num_envs = train_buffer[0].shape[:2]
    th.manual_seed(seed)
    ids = th.stack([th.randint(horizon_len * num_envs, size=(agent.batch_size,)) for _ in range(num_updates)])
    out["update.ids"] = ids.numpy()
    out["update.ids0"] = th.fmod(ids, horizon_len).numpy()
    out["update.ids1"] = th.div(ids, horizon_len, rounding_mode='floor').numpy()
    th.manual_seed(seed)
    scalars = []
    with th.enable_grad():
        for update_t in range(num_updates):
            scalars.append(agent.update_objectives(train_buffer, update_t))
            if update_t == 0:
                dump_net("update.after1.actor", agent.act, out)
                dump_net("update.after1.critic", agent.cri, out)
    out["update.scalars"] = np.array(scalars, dtype=np.float64)
    dump_net("update.after.actor", agent.act, out)
    dump_net("update.after.critic", agent.cri, out)
    dump_adam("update.after.actor_adam", agent.act_optimizer, agent.act, out)
    dump_adam("update.after.critic_adam", agent.cri_optimizer, agent.cri, out)


def record_update_net(agent, buf, out, seed):
    """Full update_net from the raw rollout buffer (values + GAE + normalise + all minibatches)."""
    agent = copy.deepcopy(agent)
    states, actions, logprobs, rewards, undones, unmasks, last_state = [t.clone() for t in buf]
    agent.last_state = last_state
    horizon_len, num_envs = states.shape[:2]
    update_times = int(horizon_len * agent.repeat_times / agent.batch_size)
    th.manual_seed(seed)
    ids = th.stack([th.randint(horizon_len * num_envs, size=(agent.batch_size,)) for _ in range(update_times)])
    out["update_net.ids"] = ids.numpy()
    th.manual_seed(seed)
    result = agent.update_net([states, actions, logprobs, rewards, undones, unmasks])
    th.set_grad_enabled(True)
    out["update_net.result"] = np.array(result, dtype=np.float64)
    dump_net("update_net.after.actor", agent.act, out)
    dump_net("update_net.after.critic", agent.cri, out)


def record_hyper(agent, out):
    out["hp.gamma"] = np.float64(agent.gamma)
    out["hp.lambda_gae_adv"] = np.float64(agent.lambda_gae_adv)
    out["hp.ratio_clip"] = np.float64(agent.ratio_clip)
    out["hp.lambda_entropy"] = np.float64(float(agent.lambda_entropy))
    out["hp.clip_grad_norm"] = np.float64(agent.clip_grad_norm)
    out["hp.learning_rate"] = np.float64(agent.learning_rate)
    out["hp.reward_scale"] = np.float64(agent.reward_scale)
    out["hp.batch_size"] = np.int64(agent.batch_size)
    out["hp.repeat_times"] = np.float64(agent.repeat_times)
    out["hp.if_use_v_trace"] = np.int64(int(agent.if_use_v_trace))


def case_synthetic(name, state_dim, action_dim, net_dims, num_envs, horizon_len, seed, num_updates=3,
                   norm_stats=False, **hyper):
    out = {}
    agent = make_ref_agent(state_dim, action_dim, net_dims, num_envs, seed, **hyper)
    perturb_nets(agent, seed + 1, norm_stats=norm_stats)
    record_hyper(agent, out)
    out["dims"] = np.array([state_dim, action_dim, num_envs, horizon_len] + list(net_dims), dtype=np.int64)
    dump_net("actor", agent.act, out)
    dump_net("critic", agent.cri, out)
    record_nets(agent, out, seed + 2)

    buf = synth_buffer(agent, horizon_len, num_envs, seed + 3)
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks", "last_state"), buf):
        out[f"buf.{k}"] = t.numpy().copy()
    train_buffer = record_gae(agent, buf, out, "gae")
    agent.if_use_v_trace = not agent.if_use_v_trace  # the other scan branch (AgentPPO.py:228-231)
    record_gae(agent, buf, out, "gae_alt")
    agent.if_use_v_trace = not agent.if_use_v_trace
    record_update(agent, train_buffer, out, num_updates, seed + 4)
    record_update_net(agent, buf, out, seed + 5)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def case_rollout(name, num_envs, horizon_len, max_step, seed, net_dims=(64, 64), **hyper):
    """Reference _explore_vec_env + update_net on the torch Pendulum vec env (the bench workload, small)."""
    out = {}
    agent = make_ref_agent(3, 1, net_dims, num_envs, seed, **hyper)
    perturb_nets(agent, seed + 1, std_log=-0.5)
    record_hyper(agent, out)
    out["dims"] = np.array([3, 1, num_envs, horizon_len] + list(net_dims), dtype=np.int64)
    out["max_step"] = np.int64(max_step)
    dump_net("actor", agent.act, out)
    dump_net("critic", agent.cri, out)

    env = PendulumVecEnv(num_envs=num_envs, gpu_id=-1, max_step=max_step, seed=seed)
    g = th.Generator().manual_seed(seed + 2)
    reset_noise = th.rand((horizon_len + 1, num_envs, 2), generator=g)
    env.inject_reset_noise(reset_noise)
    state, _ = env.reset()
    # stagger episode phases so truncations land at different t for different envs
    env.cur_step[:] = th.randint(0, max_step, (num_envs,), generator=g, dtype=th.int32)
    out["env.theta0"] = env.theta.numpy().copy()
    out["env.theta_dot0"] = env.theta_dot.numpy().copy()
    out["env.cur_step0"] = env.cur_step.numpy().copy()
    out["env.reset_noise"] = reset_noise[1:].numpy().copy()  # row t is consumed by step t
    out["state0"] = state.numpy().copy()
    agent.last_state = state

    th.manual_seed(seed + 3)
    eps = th.stack([th.randn((num_envs, 1)) for _ in range(horizon_len)])
    out["eps"] = eps.numpy()
    th.manual_seed(seed + 3)
    with th.no_grad():
        states, actions, logprobs, rewards, undones, unmasks = agent.explore_env(env, horizon_len)
    # the replayed noise must be what Normal.sample() consumed
    with th.no_grad():
        mean0 = agent.act.net(agent.act.state_norm(states[0]))
    assert th.equal(actions[0], mean0 + agent.act.action_std_log.exp() * eps[0]), "noise replay mismatch"
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks"),
                    (states, actions, logprobs, rewards, undones, unmasks)):
        out[f"rollout.{k}"] = t.numpy().copy()
    out["rollout.last_state"] = agent.last_state.numpy().copy()
    out["rollout.theta"] = env.theta.numpy().copy()
    out["rollout.theta_dot"] = env.theta_dot.numpy().copy()
    out["rollout.cur_step"] = env.cur_step.numpy().copy()

    buf = (states, actions, logprobs, rewards, undones, unmasks, agent.last_state.clone())
    record_gae(agent, buf, out, "gae")
    record_update_net(agent, buf, out, seed + 5)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main():
    os.makedirs(OUT_DIR, exist_ok=True)
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    # BASELINE config-2 dims (Pendulum, 2x64), small N/H, non-trivial norm stats
    case_synthetic("synth_s3_a1_64x64", 3, 1, (64, 64), num_envs=16, horizon_len=24, seed=11,
                   batch_size=32, repeat_times=4, norm_stats=True)
    # LunarLanderContinuous dims (BASELINE config 5), demo net_dims style
    case_synthetic("synth_s8_a2_128x64", 8, 2, (128, 64), num_envs=12, horizon_len=20, seed=23,
                   batch_size=48, repeat_times=8, gamma=0.97, lambda_entropy=0.04, learning_rate=2e-4,
                   ratio_clip=0.4)
    # three hidden layers, ragged N/H (lattice [::4, ::4] edge), reward_scale != 1
    case_synthetic("synth_s5_a3_64x48x32", 5, 3, (64, 48, 32), num_envs=10, horizon_len=9, seed=37,
                   batch_size=16, repeat_times=4, clip_grad_norm=0.5, lambda_gae_adv=0.9)
    # N == 1 (single env shapes [H, 1, ...]) -- reference _explore_one_env reshapes to this (:78-84)
    case_synthetic("synth_s3_a1_n1", 3, 1, (32, 32), num_envs=1, horizon_len=64, seed=41,
                   batch_size=16, repeat_times=2)
    # the bench workload in miniature: fused rollout + update_net
    case_rollout("rollout_pendulum_n32_h40", num_envs=32, horizon_len=40, max_step=25, seed=53,
                 batch_size=64, repeat_times=8, reward_scale=0.25)
    case_rollout("rollout_pendulum_n8_h16", num_envs=8, horizon_len=16, max_step=200, seed=61,
                 batch_size=16, repeat_times=4)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "elegantrl"):
    main()


def main_large_rollout():
    """One rollout golden that spans a whole persistent CTA of the tcgen05 kernels (448 envs = 3.5 tiles of 128 rows)
    three times over: N = 1 344 = 3 CTAs incl. their half tiles, H = 40 (the horizon of the small golden: Pendulum
    amplifies rounding differences chaotically beyond that), truncations staggered over the envs."""
    os.makedirs(OUT_DIR, exist_ok=True)
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    case_rollout("rollout_pendulum_n1344_h40", num_envs=1344, horizon_len=40, max_step=25, seed=71,
                 batch_size=64, repeat_times=4, reward_scale=0.5)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "large"):
    main_large_rollout()


# --------------------------------------------------------------------------- helloworld variant (BASELINE configs[0])
def import_helloworld():
    """Import the reference's helloworld/helloworld_PPO_single_file.py with a stub `gymnasium` (absent here; the
    file only touches it in its env wrapper and in get_gym_env_args, neither of which the agent arithmetic uses)."""
    import types
    gym = types.ModuleType("gymnasium")
    gym.Wrapper = type("Wrapper", (), {"__init__": lambda self, env=None: setattr(self, "env", env)})
    gym.make = lambda *a, **k: None
    spaces = types.ModuleType("gymnasium.spaces")
    spaces.Discrete, spaces.Box = type("Discrete", (), {}), type("Box", (), {})
    gym.spaces = spaces
    sys.modules.setdefault("gymnasium", gym)
    sys.modules.setdefault("gymnasium.spaces", spaces)
    sys.path.insert(0, os.path.join(REFERENCE, "helloworld"))
    import helloworld_PPO_single_file as hw
    return hw


def dump_plain_net(prefix, module, out):
    linears = [m for m in module.net if isinstance(m, th.nn.Linear)]
    out[f"{prefix}.n_layers"] = np.int64(len(linears))
    for i, l in enumerate(linears):
        out[f"{prefix}.W{i}"] = l.weight.detach().numpy().copy()
        out[f"{prefix}.b{i}"] = l.bias.detach().numpy().copy()
    if hasattr(module, "action_std_log"):
        out[f"{prefix}.action_std_log"] = module.action_std_log.detach().numpy().copy()


def case_helloworld(name, state_dim, action_dim, net_dims, horizon_len, seed, **hyper):
    """helloworld AgentPPO.update_net (helloworld_PPO_single_file.py:283-364) on a synthetic single-env buffer with the
    minibatch indices replayed: ReLU nets, no state_norm, SmoothL1 critic, min/clamp clip, entropy bonus, no grad clip."""
    hw = import_helloworld()
    out = {}
    th.manual_seed(seed)
    args = hw.Config(agent_class=hw.AgentPPO, env_class=None,
                     env_args={'env_name': 'golden', 'state_dim': state_dim, 'action_dim': action_dim, 'if_discrete': False})
    args.net_dims = list(net_dims)
    for k, v in hyper.items():
        setattr(args, k, v)
    agent = hw.AgentPPO(list(net_dims), state_dim, action_dim, gpu_id=-1, args=args)
    g = th.Generator().manual_seed(seed + 1)
    with th.no_grad():
        agent.act.action_std_log += -0.4 + 0.1 * th.randn(agent.act.action_std_log.shape, generator=g)
    out["dims"] = np.array([state_dim, action_dim, 1, horizon_len] + list(net_dims), dtype=np.int64)
    for k in ("gamma", "lambda_gae_adv", "ratio_clip", "learning_rate", "repeat_times"):
        out[f"hp.{k}"] = np.float64(getattr(agent, k))
    out["hp.lambda_entropy"] = np.float64(float(agent.lambda_entropy))
    out["hp.batch_size"] = np.int64(agent.batch_size)
    dump_plain_net("actor", agent.act, out)
    dump_plain_net("critic", agent.cri, out)

    states = th.randn((horizon_len, state_dim), generator=g)
    actions = 0.6 * th.randn((horizon_len, action_dim), generator=g)
    with th.no_grad():
        logprobs = agent.act.get_logprob_entropy(states, actions)[0] + 0.05 * th.randn(horizon_len, generator=g)
    rewards = th.randn((horizon_len, 1), generator=g)
    terminals = th.rand((horizon_len, 1), generator=g) < 0.06
    truncates = (th.rand((horizon_len, 1), generator=g) < 0.06) & ~terminals
    last_state = th.randn(state_dim, generator=g).numpy()
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks"),
                    (states, actions, logprobs, rewards, ~terminals, ~truncates)):
        out[f"buf.{k}"] = t.numpy().copy()
    out["buf.last_state"] = last_state.copy()

    agent.last_state = last_state
    # run the real thing: update_net does values + GAE + normalisation + all minibatches
    update_times = int(horizon_len * agent.repeat_times / agent.batch_size)
    th.manual_seed(seed + 5)
    ids = th.stack([th.randint(horizon_len, size=(agent.batch_size,)) for _ in range(update_times)])
    out["update_net.ids"] = ids.numpy()
    agent2 = copy.deepcopy(agent)
    th.manual_seed(seed + 5)
    buf = (states.clone(), actions.clone(), logprobs.clone(), rewards.clone(), (~terminals).clone(), (~truncates).clone())
    th.set_grad_enabled(False)  # as its train_agent does (helloworld_PPO_single_file.py:491); update_net re-enables it
    result = agent2.update_net(buf)
    th.set_grad_enabled(True)
    out["update_net.result"] = np.array(result, dtype=np.float64)
    out["update_net.rewards_after"] = buf[3].numpy().copy()
    out["update_net.undones_after"] = buf[4].numpy().copy()
    dump_plain_net("update_net.after.actor", agent2.act, out)
    dump_plain_net("update_net.after.critic", agent2.cri, out)
    with th.no_grad():
        out["values"] = agent.cri(states).squeeze(1).numpy()
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main_helloworld():
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    # helloworld Pendulum recipe (helloworld_PPO_single_file.py:535-557): net_dims [64, 32], gamma 0.97, repeat 16
    case_helloworld("helloworld_s3_a1_64x32", 3, 1, (64, 32), horizon_len=96, seed=71, gamma=0.97, repeat_times=4,
                    batch_size=32, learning_rate=3e-4, lambda_entropy=0.01)
    case_helloworld("helloworld_s8_a2_64x64", 8, 2, (64, 64), horizon_len=64, seed=73, repeat_times=2, batch_size=64)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "helloworld"):
    main_helloworld()


# --------------------------------------------------------------------------- discrete PPO (SURVEY 8(f2))
def make_ref_discrete_agent(state_dim, action_dim, net_dims, num_envs, seed, **hyper):
    from elegantrl.agents import AgentDiscretePPO as RefAgentDiscretePPO
    th.manual_seed(seed)
    env_args = {'env_name': 'golden', 'num_envs': num_envs, 'max_step': 200, 'state_dim': state_dim,
                'action_dim': action_dim, 'if_discrete': True}
    args = RefConfig(agent_class=RefAgentDiscretePPO, env_class=None, env_args=env_args)
    args.net_dims = list(net_dims)
    for k, v in hyper.items():
        setattr(args, k, v)
    return RefAgentDiscretePPO(list(net_dims), state_dim, action_dim, gpu_id=-1, args=args)


def replay_exponential(shape, seed):
    """The Exp(1) draw torch.multinomial's one-sample fast path consumes (q = empty_like(probs).exponential_(1))."""
    th.manual_seed(seed)
    return th.empty(shape, dtype=th.float32).exponential_(1)


def case_discrete(name, state_dim, action_dim, net_dims, num_envs, horizon_len, seed, num_updates=3, **hyper):
    """AgentDiscretePPO (AgentPPO.py:252-270) + ActorDiscretePPO (:393-425): nets / sampling with the multinomial noise
    replayed / update_objectives / update_net on a synthetic buffer whose actions are int32 [H, N] (:103-104)."""
    out = {}
    agent = make_ref_discrete_agent(state_dim, action_dim, net_dims, num_envs, seed, **hyper)
    perturb_nets(agent, seed + 1)
    with th.no_grad():
        agent.act.net[-1].weight *= 8.0  # the 0.1-std orthogonal head gives near-uniform probabilities: sharpen them
    record_hyper(agent, out)
    out["dims"] = np.array([state_dim, action_dim, num_envs, horizon_len] + list(net_dims), dtype=np.int64)
    dump_net("actor", agent.act, out)
    dump_net("critic", agent.cri, out)

    g = th.Generator().manual_seed(seed + 2)
    state = th.randn((41, state_dim), generator=g) * 1.5
    action = th.randint(action_dim, (41,), generator=g, dtype=th.int32)
    with th.no_grad():
        logprob, entropy = agent.act.get_logprob_entropy(state, action)
        out["nets.state"], out["nets.action"] = state.numpy(), action.numpy()
        out["nets.logits"] = agent.act.net(agent.act.state_norm(state)).numpy()
        out["nets.actor_forward"] = agent.act(state).numpy()
        out["nets.logprob"], out["nets.entropy"] = logprob.numpy(), entropy.numpy()
        out["nets.value"] = agent.cri(state).squeeze(1).numpy()
        # get_action with the sampler's noise replayed
        expo = replay_exponential((41, action_dim), seed + 6)
        th.manual_seed(seed + 6)
        sampled, sampled_logprob = agent.act.get_action(state)
        probs = th.softmax(agent.act.net(agent.act.state_norm(state)), dim=-1)
        assert th.equal(sampled, (probs / expo).argmax(dim=-1)), "multinomial noise replay mismatch"
        out["sample.expo"], out["sample.action"] = expo.numpy(), sampled.numpy()
        out["sample.logprob"] = sampled_logprob.numpy()

    g = th.Generator().manual_seed(seed + 3)
    states = th.randn((horizon_len, num_envs, state_dim), generator=g)
    actions = th.randint(action_dim, (horizon_len, num_envs), generator=g, dtype=th.int32)
    with th.no_grad():
        logprobs = agent.act.get_logprob_entropy(states.reshape(-1, state_dim), actions.reshape(-1))[0]
        logprobs = logprobs.reshape(horizon_len, num_envs) + 0.05 * th.randn((horizon_len, num_envs), generator=g)
    rewards = th.randn((horizon_len, num_envs), generator=g)
    terminals = th.rand((horizon_len, num_envs), generator=g) < 0.08
    truncates = (th.rand((horizon_len, num_envs), generator=g) < 0.08) & ~terminals
    last_state = th.randn((num_envs, state_dim), generator=g)
    buf = (states, actions, logprobs, rewards, ~terminals, ~truncates, last_state)
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks", "last_state"), buf):
        out[f"buf.{k}"] = t.numpy().copy()
    train_buffer = record_gae(agent, buf, out, "gae")
    record_update(agent, train_buffer, out, num_updates, seed + 4)
    record_update_net(agent, buf, out, seed + 5)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def case_discrete_rollout(name, num_envs, horizon_len, max_step, seed, net_dims=(64, 64), **hyper):
    """Reference _explore_vec_env (:87-129, discrete branch :103-104) + update_net on the torch CartPole vec env: the
    external-env (per-step) path with integer actions and real terminal flags."""
    from elegantrl_b200.envs import CartPoleVecEnv
    out = {}
    agent = make_ref_discrete_agent(4, 2, net_dims, num_envs, seed, **hyper)
    perturb_nets(agent, seed + 1)
    with th.no_grad():
        agent.act.net[-1].weight *= 8.0
    record_hyper(agent, out)
    out["dims"] = np.array([4, 2, num_envs, horizon_len] + list(net_dims), dtype=np.int64)
    out["max_step"] = np.int64(max_step)
    dump_net("actor", agent.act, out)
    dump_net("critic", agent.cri, out)

    env = CartPoleVecEnv(num_envs=num_envs, gpu_id=-1, max_step=max_step, seed=seed)
    g = th.Generator().manual_seed(seed + 2)
    reset_noise = th.rand((horizon_len + 1, num_envs, 4), generator=g)
    env.inject_reset_noise(reset_noise)
    state, _ = env.reset()
    env.cur_step[:] = th.randint(0, max_step, (num_envs,), generator=g, dtype=th.int32)
    out["env.state0"] = env.state.numpy().copy()
    out["env.cur_step0"] = env.cur_step.numpy().copy()
    out["env.reset_noise"] = reset_noise[1:].numpy().copy()
    agent.last_state = state

    th.manual_seed(seed + 3)
    expo = th.stack([th.empty((num_envs, 2), dtype=th.float32).exponential_(1) for _ in range(horizon_len)])
    out["expo"] = expo.numpy()
    th.manual_seed(seed + 3)
    with th.no_grad():
        states, actions, logprobs, rewards, undones, unmasks = agent.explore_env(env, horizon_len)
        probs0 = th.softmax(agent.act.net(agent.act.state_norm(states[0])), dim=-1)
    assert th.equal(actions[0].long(), (probs0 / expo[0]).argmax(dim=-1)), "multinomial noise replay mismatch"
    assert (~undones).any() and (~unmasks).any(), "pick a seed with terminals and truncations"
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks"),
                    (states, actions, logprobs, rewards, undones, unmasks)):
        out[f"rollout.{k}"] = t.numpy().copy()
    out["rollout.last_state"] = agent.last_state.numpy().copy()
    out["rollout.cur_step"] = env.cur_step.numpy().copy()
    buf = (states, actions, logprobs, rewards, undones, unmasks, agent.last_state.clone())
    record_gae(agent, buf, out, "gae")
    record_update_net(agent, buf, out, seed + 5)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main_discrete():
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    # CartPole dims (examples/demo_A2C_PPO_discrete.py), LunarLander-discrete dims (8 states, 4 actions)
    case_discrete("discrete_s4_a2_64x64", 4, 2, (64, 64), num_envs=12, horizon_len=20, seed=83, batch_size=32, repeat_times=4)
    case_discrete("discrete_s8_a4_128x64", 8, 4, (128, 64), num_envs=9, horizon_len=14, seed=89, batch_size=24,
                  repeat_times=4, lambda_entropy=0.05, ratio_clip=0.3, learning_rate=2e-4)
    case_discrete_rollout("cartpole_n16_h48", num_envs=16, horizon_len=48, max_step=30, seed=97,
                          batch_size=32, repeat_times=4)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "discrete"):
    main_discrete()


# --------------------------------------------------------------------------- A2C (SURVEY 8(f2)), single-env buffers
def case_a2c(name, state_dim, action_dim, net_dims, horizon_len, seed, **hyper):
    """AgentA2C (AgentPPO.py:252-311) on a synthetic single-env buffer [H, 1, ...] (the only shape its time-only indexing
    handles): full update_net with the CPU-drawn time indices replayed."""
    from elegantrl.agents import AgentA2C as RefAgentA2C
    out = {}
    th.manual_seed(seed)
    env_args = {'env_name': 'golden', 'num_envs': 1, 'max_step': 200, 'state_dim': state_dim, 'action_dim': action_dim,
                'if_discrete': False}
    args = RefConfig(agent_class=RefAgentA2C, env_class=None, env_args=env_args)
    args.net_dims = list(net_dims)
    for k, v in hyper.items():
        setattr(args, k, v)
    agent = RefAgentA2C(list(net_dims), state_dim, action_dim, gpu_id=-1, args=args)
    perturb_nets(agent, seed + 1, norm_stats=True)
    record_hyper(agent, out)
    out["dims"] = np.array([state_dim, action_dim, 1, horizon_len] + list(net_dims), dtype=np.int64)
    dump_net("actor", agent.act, out)
    dump_net("critic", agent.cri, out)
    buf = synth_buffer(agent, horizon_len, 1, seed + 3)
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks", "last_state"), buf):
        out[f"buf.{k}"] = t.numpy().copy()
    record_gae(agent, buf, out, "gae")
    agent2 = copy.deepcopy(agent)
    states, actions, logprobs, rewards, undones, unmasks, last_state = [t.clone() for t in buf]
    agent2.last_state = last_state
    update_times = int(horizon_len * agent2.repeat_times / agent2.batch_size)
    th.manual_seed(seed + 5)
    ids = th.stack([th.randint(horizon_len, size=(agent2.batch_size,)) for _ in range(update_times)])
    out["update_net.ids"] = ids.numpy()
    th.manual_seed(seed + 5)
    result = agent2.update_net([states, actions, logprobs, rewards, undones, unmasks])
    th.set_grad_enabled(True)
    out["update_net.result"] = np.array([float(x) for x in result], dtype=np.float64)
    dump_net("update_net.after.actor", agent2.act, out)
    dump_net("update_net.after.critic", agent2.cri, out)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main_a2c():
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    case_a2c("a2c_s3_a1_64x64", 3, 1, (64, 64), horizon_len=96, seed=101, batch_size=32, repeat_times=2)
    case_a2c("a2c_s8_a2_64x32", 8, 2, (64, 32), horizon_len=80, seed=103, batch_size=16, repeat_times=1, learning_rate=2e-4,
             clip_grad_norm=0.7)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "a2c"):
    main_a2c()


# --------------------------------------------------------------------------- SAC + ReplayBuffer (SURVEY 8(f3)), oracle groundwork
def dump_layers(prefix, seq, out):
    linears = [m for m in seq if isinstance(m, th.nn.Linear)]
    out[f"{prefix}.n_layers"] = np.int64(len(linears))
    for i, l in enumerate(linears):
        out[f"{prefix}.W{i}"] = l.weight.detach().numpy().copy()
        out[f"{prefix}.b{i}"] = l.bias.detach().numpy().copy()


def dump_sac(prefix, agent, out):
    dump_layers(f"{prefix}.actor.net_s", agent.act.net_s, out)
    dump_layers(f"{prefix}.actor.net_a", agent.act.net_a, out)
    for name, cri in (("critic", agent.cri), ("critic_target", agent.cri_target)):
        dump_layers(f"{prefix}.{name}.encoder", cri.encoder_sa, out)
        for e, dec in enumerate(cri.decoder_qs):
            dump_layers(f"{prefix}.{name}.decoder{e}", dec, out)
    out[f"{prefix}.alpha_log"] = agent.alpha_log.detach().numpy().copy()


def case_sac(name, state_dim, action_dim, net_dims, num_seqs, max_size, seed, num_updates=3, **hyper):
    """ReplayBuffer.update (with wrap-around) / sample and AgentSAC.update_objectives (AgentSAC.py:42-86), minibatch indices
    and both rsample draws replayed from th.manual_seed."""
    from elegantrl.agents import AgentSAC as RefAgentSAC
    from elegantrl.train.replay_buffer import ReplayBuffer as RefReplayBuffer
    out = {}
    th.manual_seed(seed)
    env_args = {'env_name': 'golden', 'num_envs': num_seqs, 'max_step': 200, 'state_dim': state_dim,
                'action_dim': action_dim, 'if_discrete': False}
    args = RefConfig(agent_class=RefAgentSAC, env_class=None, env_args=env_args)
    args.net_dims = list(net_dims)
    for k, v in hyper.items():
        setattr(args, k, v)
    agent = RefAgentSAC(list(net_dims), state_dim, action_dim, gpu_id=-1, args=args)
    g = th.Generator().manual_seed(seed + 1)
    with th.no_grad():  # move off the init point; make the target differ from the online critic
        for p in list(agent.act.parameters()) + list(agent.cri.parameters()):
            p += 0.05 * th.randn(p.shape, generator=g)
        for p in agent.cri_target.parameters():
            p += 0.03 * th.randn(p.shape, generator=g)
    for k in ("gamma", "clip_grad_norm", "learning_rate", "soft_update_tau", "batch_size", "repeat_times", "reward_scale"):
        out[f"hp.{k}"] = np.float64(getattr(agent, k))
    out["hp.target_entropy"] = np.float64(agent.target_entropy)
    out["hp.num_ensembles"] = np.int64(agent.num_ensembles)
    out["dims"] = np.array([state_dim, action_dim, num_seqs, max_size] + list(net_dims), dtype=np.int64)
    dump_sac("init", agent, out)

    # ---- replay buffer: three appends, the last one wraps around
    buffer = RefReplayBuffer(max_size=max_size, state_dim=state_dim, action_dim=action_dim, gpu_id=-1, num_seqs=num_seqs, args=args)
    for i, rows in enumerate((max_size // 2, max_size // 3, max_size // 2)):
        items = (th.randn((rows, num_seqs, state_dim), generator=g), th.rand((rows, num_seqs, action_dim), generator=g) * 2 - 1,
                 th.randn((rows, num_seqs), generator=g), (th.rand((rows, num_seqs), generator=g) > 0.1).float(),
                 (th.rand((rows, num_seqs), generator=g) > 0.1).float())
        for k, t in zip(("states", "actions", "rewards", "undones", "unmasks"), items):
            out[f"append{i}.{k}"] = t.numpy().copy()
        buffer.update(items)
        out[f"append{i}.p"], out[f"append{i}.cur_size"] = np.int64(buffer.p), np.int64(buffer.cur_size)
    for k in ("states", "actions", "rewards", "undones", "unmasks"):
        out[f"buffer.{k}"] = getattr(buffer, k).numpy().copy()

    # ---- k updates; RNG consumption per call: randint (sample :121), normal_ (rsample :51), normal_ (rsample :72)
    b = agent.batch_size
    th.manual_seed(seed + 5)
    ids, eps_next, eps_pg = [], [], []
    for _ in range(num_updates):
        ids.append(th.randint((buffer.cur_size - 1) * num_seqs, size=(b,)))
        eps_next.append(th.empty((b, action_dim)).normal_())
        eps_pg.append(th.empty((b, action_dim)).normal_())
    out["update.ids"], out["update.eps_next"], out["update.eps_pg"] = (th.stack(x).numpy() for x in (ids, eps_next, eps_pg))
    th.manual_seed(seed + 5)
    scalars = []
    th.set_grad_enabled(True)
    for u in range(num_updates):
        scalars.append(agent.update_objectives(buffer, u))
        assert th.equal(buffer.ids0, th.fmod(ids[u], buffer.cur_size - 1)), "index replay mismatch"
        if u == 0:
            dump_sac("after1", agent, out)
    out["update.scalars"] = np.array(scalars, dtype=np.float64)
    dump_sac("after", agent, out)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main_sac():
    th.set_num_threads(1)
    # BipedalWalker dims of BASELINE config 4 (demo_A2C_PPO.py:212-219 style), small; and a 3-layer / 2-critic variant
    case_sac("sac_s24_a4_64x32", 24, 4, (64, 32), num_seqs=6, max_size=40, seed=107, batch_size=48, learning_rate=3e-4,
             soft_update_tau=0.02)
    case_sac("sac_s3_a1_32x32x16", 3, 1, (32, 32, 16), num_seqs=3, max_size=30, seed=109, batch_size=32, num_ensembles=2,
             gamma=0.97, clip_grad_norm=0.5)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "sac"):
    main_sac()


def case_sac_cycle(name, num_envs, horizon_len, max_step, max_size, seed, net_dims=(64, 32), **hyper):
    """One off-policy cycle of the reference: AgentSAC.explore_env (AgentBase.py:130-170) on the torch Pendulum vec env ->
    ReplayBuffer.update -> AgentSAC.update_net (AgentBase.py:172-189), every random draw replayed."""
    from elegantrl.agents import AgentSAC as RefAgentSAC
    from elegantrl.train.replay_buffer import ReplayBuffer as RefReplayBuffer
    out = {}
    th.manual_seed(seed)
    env_args = {'env_name': 'golden', 'num_envs': num_envs, 'max_step': max_step, 'state_dim': 3, 'action_dim': 1, 'if_discrete': False}
    args = RefConfig(agent_class=RefAgentSAC, env_class=None, env_args=env_args)
    args.net_dims = list(net_dims)
    for k, v in hyper.items():
        setattr(args, k, v)
    agent = RefAgentSAC(list(net_dims), 3, 1, gpu_id=-1, args=args)
    for k in ("gamma", "clip_grad_norm", "learning_rate", "soft_update_tau", "batch_size", "repeat_times", "reward_scale"):
        out[f"hp.{k}"] = np.float64(getattr(agent, k))
    out["hp.target_entropy"] = np.float64(agent.target_entropy)
    out["hp.num_ensembles"] = np.int64(agent.num_ensembles)
    out["dims"] = np.array([3, 1, num_envs, max_size] + list(net_dims), dtype=np.int64)
    out["horizon_len"], out["max_step"] = np.int64(horizon_len), np.int64(max_step)
    dump_sac("init", agent, out)

    env = PendulumVecEnv(num_envs=num_envs, gpu_id=-1, max_step=max_step, seed=seed)
    g = th.Generator().manual_seed(seed + 2)
    reset_noise = th.rand((horizon_len + 1, num_envs, 2), generator=g)
    env.inject_reset_noise(reset_noise)
    state, _ = env.reset()
    env.cur_step[:] = th.randint(0, max_step, (num_envs,), generator=g, dtype=th.int32)
    out["env.theta0"], out["env.theta_dot0"], out["env.cur_step0"] = env.theta.numpy().copy(), env.theta_dot.numpy().copy(), env.cur_step.numpy().copy()
    out["env.reset_noise"] = reset_noise[1:].numpy().copy()
    agent.last_state = state
    th.manual_seed(seed + 3)
    eps = th.stack([th.empty((num_envs, 1)).normal_() for _ in range(horizon_len)])
    out["explore.eps"] = eps.numpy()
    th.manual_seed(seed + 3)
    th.set_grad_enabled(False)
    items = agent.explore_env(env, horizon_len)
    for k, t in zip(("states", "actions", "rewards", "undones", "unmasks"), items):
        out[f"explore.{k}"] = t.numpy().copy()
    out["explore.last_state"] = agent.last_state.numpy().copy()
    buffer = RefReplayBuffer(max_size=max_size, state_dim=3, action_dim=1, gpu_id=-1, num_seqs=num_envs, args=args)
    buffer.update(items)
    update_times = int(buffer.cur_size * agent.repeat_times / agent.batch_size)
    b = agent.batch_size
    th.manual_seed(seed + 5)
    ids, eps_next, eps_pg = [], [], []
    for _ in range(update_times):
        ids.append(th.randint((buffer.cur_size - 1) * num_envs, size=(b,)))
        eps_next.append(th.empty((b, 1)).normal_())
        eps_pg.append(th.empty((b, 1)).normal_())
    out["update.ids"], out["update.eps_next"], out["update.eps_pg"] = (th.stack(x).numpy() for x in (ids, eps_next, eps_pg))
    th.manual_seed(seed + 5)
    result = agent.update_net(buffer)
    th.set_grad_enabled(True)
    out["update_net.result"] = np.array([float(x) for x in result], dtype=np.float64)
    dump_sac("after", agent, out)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main_sac_cycle():
    th.set_num_threads(1)
    case_sac_cycle("saccycle_pendulum_n12_h24", num_envs=12, horizon_len=24, max_step=9, max_size=64, seed=113,
                   batch_size=32, repeat_times=4.0, reward_scale=0.5, learning_rate=3e-4)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "saccycle"):
    main_sac_cycle()


# ------------------------------------------------------------------ single-env rollout (SURVEY 8 row a5)
def case_one_env(name, horizon_len, max_step, seed, net_dims=(64, 64), **hyper):
    """Reference AgentPPO._explore_one_env (elegantrl/agents/AgentPPO.py:34-85) with ``num_envs = 1`` on the numpy
    gym-style ``elegantrl_b200.envs.PendulumEnv``: numpy action out / numpy state in per step, ``env.reset()`` by the
    agent after a truncated step, outputs reshaped to [H, 1, ...].  Policy noise replayed from ``th.manual_seed``,
    the env's reset noise injected (the same rows are handed to the env of the drop-in agent in the parity test)."""
    from elegantrl_b200.envs import PendulumEnv
    out = {}
    agent = make_ref_agent(3, 1, net_dims, 1, seed, **hyper)
    assert not agent.if_vec_env
    perturb_nets(agent, seed + 1, std_log=-0.5, norm_stats=True)
    record_hyper(agent, out)
    out["dims"] = np.array([3, 1, 1, horizon_len] + list(net_dims), dtype=np.int64)
    out["max_step"] = np.int64(max_step)
    dump_net("actor", agent.act, out)
    dump_net("critic", agent.cri, out)

    env = PendulumEnv(max_step=max_step, seed=seed)
    g = th.Generator().manual_seed(seed + 2)
    reset_noise = th.rand((2 * horizon_len + 2, 1, 2), generator=g)   # a truncated step consumes two rows (step + reset)
    out["env.reset_noise"] = reset_noise.numpy().copy()
    env.inner.inject_reset_noise(reset_noise)
    state, _ = env.reset()
    out["state0"] = np.asarray(state, dtype=np.float32).copy()
    agent.last_state = th.as_tensor(state, dtype=th.float32).unsqueeze(0)

    th.manual_seed(seed + 3)
    eps = th.stack([th.randn((1, 1)) for _ in range(horizon_len)])
    out["eps"] = eps.numpy()
    th.manual_seed(seed + 3)
    with th.no_grad():
        states, actions, logprobs, rewards, undones, unmasks = agent.explore_env(env, horizon_len)
    with th.no_grad():
        mean0 = agent.act.net(agent.act.state_norm(states[0]))
    assert th.equal(actions[0], mean0 + agent.act.action_std_log.exp() * eps[0]), "noise replay mismatch"
    assert tuple(states.shape) == (horizon_len, 1, 3) and int((~unmasks).sum()) >= 2
    for k, t in zip(("states", "actions", "logprobs", "rewards", "undones", "unmasks"),
                    (states, actions, logprobs, rewards, undones, unmasks)):
        out[f"rollout.{k}"] = t.numpy().copy()
    out["rollout.last_state"] = agent.last_state.numpy().copy()
    buf = (states, actions, logprobs, rewards, undones, unmasks, agent.last_state.clone())
    record_gae(agent, buf, out, "gae")
    record_update_net(agent, buf, out, seed + 5)
    np.savez_compressed(os.path.join(OUT_DIR, f"{name}.npz"), **out)
    print(f"| wrote {name}.npz  ({len(out)} arrays)")


def main_one_env():
    os.makedirs(OUT_DIR, exist_ok=True)
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    case_one_env("oneenv_pendulum_h48", horizon_len=48, max_step=13, seed=83, batch_size=16, repeat_times=2,
                 reward_scale=0.5)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "oneenv"):
    main_one_env()


# ------------------------------------------------ BASELINE configs[2] / [4] state / action dims on the default 64 x 64 net
def main_tc_shapes():
    """Synthetic-buffer goldens for the shapes the tcgen05 update kernel (csrc/update_tc.cu) specialises on beyond Pendulum:
    LunarLanderContinuous dims (S = 8, A = 2: layer-1 K = 24, two K steps more than Pendulum) and Hopper dims (S = 11, A = 3,
    the kernel's largest S), both with non-trivial state_norm statistics and a batch that is not a multiple of 32."""
    os.makedirs(OUT_DIR, exist_ok=True)
    th.set_num_threads(1)
    th.set_grad_enabled(True)
    case_synthetic("synth_s8_a2_64x64", 8, 2, (64, 64), num_envs=14, horizon_len=18, seed=91,
                   batch_size=100, repeat_times=8, norm_stats=True, lambda_entropy=0.02)
    case_synthetic("synth_s11_a3_64x64", 11, 3, (64, 64), num_envs=9, horizon_len=20, seed=97,
                   batch_size=72, repeat_times=6, norm_stats=True, gamma=0.98, clip_grad_norm=1.0)


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "tcshapes"):
    main_tc_shapes()


# --------------------------------------------------------------------------- evaluator rollout (SURVEY section 8 row f4)
# (num_envs, max_step, seed and rows of the injected reset noise)
EVALUATOR_CASES = ((24, 30, 3, 64), (24, 30, 11, 32), (1344, 40, 11, 42))


def evaluator_actor():
    """The actor of tests/test_evaluator.py: ActorPPO 2x64 from th.manual_seed(5), biases perturbed."""
    from elegantrl_b200.agents.nets import ActorPPO
    th.manual_seed(5)
    actor = ActorPPO([64, 64], 3, 1)
    with th.no_grad():
        for layer in actor.net:
            if hasattr(layer, "bias"):
                layer.bias += 0.1 * th.randn_like(layer.bias)
    return actor


def main_evaluator():
    """The reference's ``get_cumulative_rewards_and_step_from_vec_env`` (``elegantrl/train/evaluator.py:200-238``) on the
    CPU torch Pendulum vec env with reset noise of ``th.rand((rows, n, 2))`` from a seeded generator: the (return, steps)
    list of every case, in the reference's order, and the actor's parameters."""
    from elegantrl.train.evaluator import get_cumulative_rewards_and_step_from_vec_env as ref_fn
    os.makedirs(OUT_DIR, exist_ok=True)
    th.set_num_threads(1)
    actor = evaluator_actor()
    out = {f"actor.{k}": v.numpy().copy() for k, v in actor.state_dict().items()}
    for n, max_step, seed, rows in EVALUATOR_CASES:
        env = PendulumVecEnv(num_envs=n, gpu_id=-1, max_step=max_step)
        env.inject_reset_noise(th.rand((rows, n, 2), generator=th.Generator().manual_seed(seed)))
        with th.no_grad():
            got = ref_fn(env, actor)
        out[f"n{n}_t{max_step}_s{seed}.returns"] = np.array([r for r, _ in got], dtype=np.float32)
        out[f"n{n}_t{max_step}_s{seed}.steps"] = np.array([s for _, s in got], dtype=np.int64)
    np.savez_compressed(os.path.join(OUT_DIR, "evaluator_pendulum.npz"), **out)
    print(f"| wrote evaluator_pendulum.npz  ({len(out)} arrays)")


if __name__ == "__main__" and os.environ.get("GOLDEN_ONLY", "") in ("", "evaluator"):
    main_evaluator()
