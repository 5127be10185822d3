"""Batched vary_hp evaluation (BASELINE config 4): many DDQN agents with sampled hyper-parameters trained on ONE fixed
Synthetic Environment and tested on the real env.

Mirrors experiments/syn_env_evaluate_cartpole_vary_hp_2.py:25-48 (`train_test_agents`): the overrides
init_episodes=10, train_episodes=1000, test_episodes=10, early_out_num=10, early_out_virtual_diff=0.01; per agent
`select_agent('DDQN_vary')` -> `agent.train(env=SE)` (no test_env: virtual-env plateau early-out) -> `agent.test(real_env)`;
returns (reward_list, train_steps_needed, episodes_needed).  Here every agent is one lane: agents whose sampled Q-net
fits the register kernel set (hidden_layer <= 1, hidden_size <= 128) run in one launch, the others (two hidden layers
or wider) in a second launch of the general kernel; lr / batch_size / hidden_size / hidden_layer travel per lane.

The transfer evaluations (agent types the SE never saw during its training) run the same way with agent_name="duelingddqn"
(DuelingDDQN_vary agents, all lanes on the general kernel) or agent_name="td3_discrete_vary" (TD3_discrete_vary agents, one
le_td3_run launch per hidden_layer).
"""
import copy

import numpy as np
import torch

from . import config as le_config
from . import ops
from ._abi import ENV_REAL, ENV_SE, Td3Cfg
from .agents import _varied_config, vary_hyperparameters
from .rng import lane_keys

OVERRIDES = dict(print_rate=10, early_out_num=10, train_episodes=1000, init_episodes=10, test_episodes=10,
                 early_out_virtual_diff=0.01)


#: agent_name -> (config section of the agent, section holding its vary_hp flag)
AGENT_SECTIONS = {"ddqn": ("ddqn", "ddqn_vary"), "duelingddqn": ("duelingddqn", "duelingddqn_vary"),
                  "td3_discrete_vary": ("td3_discrete_vary", "td3_discrete_vary")}


def _base(c):
    return c.base if isinstance(c, Td3Cfg) else c


def sample_agent_cfgs(config, agents_num, rng, overrides=None, vary=True, env_slopes=None, agent_name="ddqn"):
    """One lane configuration per agent, `overrides` (default OVERRIDES) applied to the agent's config section.

    agent_name "ddqn": le_lane_cfg with DDQN_vary sampling (agents/DDQN_vary.py:26-59) when `vary`.
    "duelingddqn": le_lane_cfg with DuelingDDQN_vary sampling (agents/DuelingDDQN_vary.py:24-75, feature_dim too) and
    "td3_discrete_vary": Td3Cfg with TD3_discrete_vary sampling, each when `vary` and, as in those constructors, the config's
    duelingddqn_vary / td3_discrete_vary "vary_hp" flag are set.  Draws come from `rng` in agent order."""
    if agent_name not in AGENT_SECTIONS:
        raise ValueError("agent_name must be one of %s" % sorted(AGENT_SECTIONS))
    section, flag = AGENT_SECTIONS[agent_name]
    cfgs = []
    base = copy.deepcopy(config)
    base["agents"][section].update(OVERRIDES if overrides is None else overrides)
    for _ in range(agents_num):
        if agent_name == "ddqn":
            c = copy.deepcopy(base)
            if vary:
                a = vary_hyperparameters(c["agents"]["ddqn"], rng)
                a["hidden_layer"] = max(a["hidden_layer"], 1)
                c["agents"]["ddqn"] = a
            lc = le_config.lane_cfg(c, "ddqn", ENV_SE, use_test_env=False, final_test=True)
        else:
            c = _varied_config(base, section, flag, rng, vary_feature_dim=agent_name == "duelingddqn") if vary else base
            if agent_name == "duelingddqn":
                lc = le_config.lane_cfg(c, section, ENV_SE, use_test_env=False, final_test=True)
            else:
                lc = le_config.td3_lane_cfg(c, ENV_SE, use_test_env=False, final_test=True)
        if env_slopes is not None:
            for i in range(3):
                _base(lc).env_slope[i] = env_slopes[i]
        cfgs.append(lc)
    return cfgs


def _max_cfg(cfgs):
    """The configuration that fixes strides / kernel set / slot sizes for a group: elementwise maxima of the shape fields."""
    m = cfgs[0].copy()
    b, bs = _base(m), [_base(c) for c in cfgs]
    b.q_hidden = max(c.q_hidden for c in bs)
    b.q_layers = max(c.q_layers for c in bs)
    b.batch_size = max(c.batch_size for c in bs)
    b.q_feature_dim = max(c.q_feature_dim for c in bs)
    return m


def launch_groups(cfgs, indices=None):
    """Splits lanes into one launch per kernel family and orders every launch's lane queue longest-first.

    Families: the warp-per-lane register kernel sets by hidden units per thread (U = 2: hidden_size <= 64, U = 4: <= 128,
    U = 6: <= 192, CartPole shapes) — a lane with 40 hidden units should not pay for the 128-unit kernel of its neighbour — and
    the general CTA-per-lane kernel for everything else (two hidden layers, wider nets).  Inside a launch the persistent
    kernel hands out lanes in queue order, so the most expensive lanes (cost ~ batch_size x parameters) go first and the
    cheap ones fill the ragged tail.  TD3 lanes (Td3Cfg) form one launch per hidden_layer, so that the slots sized for a launch's
    maxima stay close to what its lanes use; their cost is batch_size x (actor + two critics).  Returns a list of index arrays
    into `cfgs`."""
    idx_all = np.arange(len(cfgs)) if indices is None else np.asarray(indices)
    td3 = len(cfgs) > 0 and isinstance(cfgs[0], Td3Cfg)
    family = (lambda c: c.base.q_layers) if td3 else (lambda c: c.register_units())
    params = (lambda c: c.param_counts()[0] + 2 * c.param_counts()[1]) if td3 else (lambda c: c.q_params())
    fam = {}
    for i in idx_all:
        fam.setdefault(family(cfgs[i]), []).append(int(i))
    out = []
    for u in sorted(fam, key=(lambda k: k) if td3 else (lambda k: (k == 0, k))):   # register families first, the general kernel last
        idx = np.asarray(fam[u])
        cost = np.array([_base(cfgs[i]).batch_size * params(cfgs[i]) for i in idx], np.float64)
        out.append(idx[np.argsort(-cost, kind="stable")])
    return out


def _run_group(sub, cfg0, theta, env_index, keys, n_env, device):
    """One launch of the fused kernel (le_lane_cfg lanes) or of the TD3 kernel (Td3Cfg lanes) for lanes that share a kernel
    family.  Returns (final test rewards [k, T] f64, training agent steps [k], episodes [k]) as numpy arrays.  (the CPU
    host-logic tests substitute their own launch function.)"""
    th = None if theta is None else torch.as_tensor(theta).to(device).contiguous()
    ei = None if env_index is None else torch.as_tensor(env_index.astype(np.int32)).to(device)
    if isinstance(cfg0, Td3Cfg):
        bufs = ops.Td3Buffers(cfg0, len(sub), max(n_env, 1), device, n_cfg=len(sub))
        ops.td3_run(bufs, sub, th, ei, ops.keys_tensor(keys, device))
    else:
        bufs = ops.InnerLoopBuffers(cfg0, len(sub), max(n_env, 1), device, n_cfg=len(sub))
        ops.inner_loop_run(bufs, sub, th, ei, ops.keys_tensor(keys, device), cfg0=cfg0)
    torch.cuda.current_stream().synchronize()
    out = bufs.results()
    return bufs.test_rewards.cpu().numpy(), out["train_steps"].astype(np.int64), out["n_episodes"].astype(np.int64)


def _rank_world(shard):
    import torch.distributed as dist
    if shard and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def evaluate_agents(config, env_thetas, agents_num=10, seed=0, overrides=None, vary=True, env_slopes=None, device="cuda",
                    env_kind=ENV_SE, n_envs=None, shard=True, agent_name="ddqn"):
    """`agents_num` freshly sampled agents on EACH of the given training environments, all lanes in one launch per
    kernel family (lane = env * agents_num + agent; lanes of one environment share its weight pack).

    env_thetas: [n_env, P] SE parameter vectors (ENV_SE), or None with env_kind=ENV_REAL and n_envs repetitions
    (mode 0 of experiments/syn_env_run_vary_hp.py:48-59: train on the real env itself).
    With an initialised torch.distributed group (one process per GPU) and shard=True the lanes are block-sharded over the
    ranks — every rank samples the same agent configurations from `seed`, runs lanes [n*rank/world, n*(rank+1)/world) and
    the only exchange is ONE all-reduce that assembles the result table on every rank (BASELINE config 4).
    agent_name: "ddqn" (DDQN_vary agents), "duelingddqn" (DuelingDDQN_vary) or "td3_discrete_vary" (sample_agent_cfgs).  For
    every family `overrides` defaults to OVERRIDES, the overrides of the DDQN evaluator
    (experiments/syn_env_evaluate_cartpole_vary_hp_2.py); the reference's evaluator scripts for the other two families are not
    part of this tree, so that choice is not checked against them.
    Returns (rewards [n_env][agents][test_episodes], train_steps [n_env][agents], episodes [n_env][agents], lane_cfgs)."""
    if env_thetas is None:
        n_env = int(n_envs or 1)
        theta = None
    else:
        theta = np.ascontiguousarray(np.asarray(env_thetas, np.float32))
        theta = theta.reshape(1, -1) if theta.ndim == 1 else theta
        n_env = theta.shape[0]
    n = n_env * agents_num
    rng = np.random.RandomState(seed)
    cfgs = sample_agent_cfgs(config, n, rng, overrides, vary, env_slopes, agent_name)
    for c in cfgs:
        _base(c).env_kind = env_kind
    env_of = np.arange(n) // agents_num
    keys = lane_keys(seed, 0, env_of, np.zeros(n, int), np.arange(n) % agents_num)
    rank, world = _rank_world(shard)
    lo, hi = n * rank // world, n * (rank + 1) // world
    T = max(_base(c).test_episodes for c in cfgs)
    table = np.zeros((n, T + 2), np.float64)      # [test rewards | train steps | episodes] per lane; zero outside this rank's block
    for idx in launch_groups(cfgs, np.arange(lo, hi)):
        sub = [cfgs[i] for i in idx]
        env_index = None if theta is None or n_env == 1 else env_of[idx]
        tr, st, ep = _run_group(sub, _max_cfg(sub), theta, env_index, keys[idx], n_env, device)
        for k, i in enumerate(idx):
            c = _base(cfgs[i])
            table[i, :c.test_episodes] = tr[k, :c.test_episodes]
            table[i, T] = int(st[k]) * max(int(c.same_action_num), 1)   # sum(episode_length)
            table[i, T + 1] = int(ep[k])
    if world > 1:
        import torch.distributed as dist
        t = torch.from_numpy(table)
        if dist.get_backend() == "nccl":
            t = t.to(device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)       # blocks are disjoint: the sum is the gather
        table = t.cpu().numpy()
    rewards = [table[i, :_base(cfgs[i]).test_episodes].tolist() for i in range(n)]
    steps = [int(table[i, T]) for i in range(n)]
    episodes = [int(table[i, T + 1]) for i in range(n)]
    nest = lambda v: [v[e * agents_num:(e + 1) * agents_num] for e in range(n_env)]
    return nest(rewards), nest(steps), nest(episodes), cfgs


def train_test_agents(config, se_theta, agents_num=10, seed=0, overrides=None, vary=True, env_slopes=None, device="cuda",
                      agent_name="ddqn"):
    """One SE: returns (reward_list [agents][test_episodes], train_steps_needed [agents], episodes_needed [agents], lane_cfgs)."""
    r, s, e, cfgs = evaluate_agents(config, np.asarray(se_theta, np.float32).reshape(1, -1), agents_num, seed, overrides, vary,
                                    env_slopes, device, agent_name=agent_name)
    return r[0], s[0], e[0], cfgs


def train_test_agents_envs(train_env, test_env, config, agents_num, seed=0, overrides=None, vary=None, agent_name="ddqn"):
    """Drop-in for the evaluator callback `custom_train_test_agents(train_env, test_env, config, agents_num)`
    (experiments/syn_env_evaluate_cartpole_vary_hp_2.py:25-48): same return shape
    (reward_list [[test rewards]...], train_steps_needed [[n]...], episodes_needed [[n]...]), all agents in one launch."""
    kind, theta, fields = train_env.kernel_env()
    if vary is None:
        vary = True      # the evaluator sets config['agents']['ddqn_vary']['vary_hp'] = True (:31)
    slopes = fields.get("env_slope")
    if kind == ENV_SE:
        r, s, e, _ = evaluate_agents(config, theta.numpy().reshape(1, -1), agents_num, seed, overrides, vary, slopes, agent_name=agent_name)
    else:
        if kind != ENV_REAL:
            raise NotImplementedError("vary_hp evaluation trains on a synthetic env or on the real env")
        r, s, e, _ = evaluate_agents(config, None, agents_num, seed, overrides, vary, None, env_kind=ENV_REAL, n_envs=1, agent_name=agent_name)
    return r[0], [[x] for x in s[0]], [[x] for x in e[0]]


def load_envs_and_config(file_name, model_dir, device):
    """experiments/syn_env_evaluate_cartpole_vary_hp_2.py:12-22: checkpoint {'model': state_dict, 'config': config}
    (agents/GTN_master.py:133-139) -> (virtual_env, real_env, config)."""
    import os
    from .envs import EnvFactory
    save_dict = torch.load(os.path.join(model_dir, file_name), weights_only=False)
    config = save_dict['config']
    config['device'] = device
    env_factory = EnvFactory(config=config)
    virtual_env = env_factory.generate_virtual_env()
    virtual_env.load_state_dict(save_dict['model'])
    real_env = env_factory.generate_real_env()
    return virtual_env, real_env, config


def get_all_files(with_vary_hp, model_num, model_dir, custom_load_envs_and_config, env_name, device, filter_models_list=None):
    """experiments/syn_env_run_vary_hp.py:8-29: checkpoints of `env_name` trained with/without vary_hp, in the
    deterministic order of their random 6-character suffix."""
    import os
    file_list = []
    for file_name in os.listdir(model_dir):
        if env_name not in file_name:
            continue
        _, _, config = custom_load_envs_and_config(file_name=file_name, model_dir=model_dir, device=device)
        if config['agents']['ddqn_vary']['vary_hp'] == with_vary_hp:
            file_list.append(file_name)
    file_list = sorted(file_list, key=lambda elem: elem[-9:])
    if len(file_list) < model_num and filter_models_list is None:
        raise ValueError("Not enough saved models")
    if filter_models_list is not None:
        return [f for f in file_list if f in filter_models_list]
    return file_list[:model_num]


def run_vary_hp(mode, experiment_name, model_num, agents_num, model_dir, custom_load_envs_and_config=load_envs_and_config,
                custom_train_test_agents=None, env_name="CartPole", pool=None, device="cuda", filter_models_list=None,
                correlation_exp=False, out_dir=None, seed=0, overrides=None, agent_name="ddqn"):
    """experiments/syn_env_run_vary_hp.py:32-137 with the same modes, result lists and result file
    (utils.save_lists): mode 0 trains on the real env, mode 1 / 2 on the SEs that were trained without / with varied
    hyper-parameters.  `pool` is accepted and ignored: instead of one process per model, ALL models x agents are lanes
    of one launch (custom_train_test_agents=None), or the callback is invoked per model like the reference does.
    agent_name selects the agent family of the one-launch path (evaluate_agents)."""
    from .utils import save_lists
    if mode not in (0, 1, 2):
        raise ValueError("mode must be 0, 1 or 2")
    train_on_venv = mode != 0
    with_vary_hp = mode == 2
    env_reward_overview, reward_list, train_steps_needed, episode_length_needed = {}, [], [], []
    import os
    if not train_on_venv:
        file_name = sorted(os.listdir(model_dir))[0]
        _, real_env, config = custom_load_envs_and_config(file_name=file_name, model_dir=model_dir, device=device)
        names = [real_env.env.env_name + "_" + str(i) for i in range(model_num)]
        if custom_train_test_agents is None:
            r, s, e, _ = evaluate_agents(config, None, agents_num, seed, overrides, True, None, device, env_kind=ENV_REAL, n_envs=model_num,
                                         agent_name=agent_name)
            per_model = [(r[i], [[x] for x in s[i]], [[x] for x in e[i]]) for i in range(model_num)]
        else:
            per_model = [custom_train_test_agents(train_env=real_env, test_env=real_env, config=config, agents_num=agents_num)
                         for _ in range(model_num)]
    else:
        names = get_all_files(with_vary_hp=with_vary_hp, model_num=model_num, model_dir=model_dir,
                              custom_load_envs_and_config=custom_load_envs_and_config, env_name=env_name, device=device,
                              filter_models_list=filter_models_list)
        loaded = [custom_load_envs_and_config(file_name=f, model_dir=model_dir, device=device) for f in names]
        config = loaded[-1][2]
        if custom_train_test_agents is None:
            thetas = np.stack([v.kernel_env()[1].numpy() for v, _, _ in loaded])
            slopes = loaded[0][0].kernel_env()[2].get("env_slope")
            r, s, e, _ = evaluate_agents(config, thetas, agents_num, seed, overrides, True, slopes, device, agent_name=agent_name)
            per_model = [(r[i], [[x] for x in s[i]], [[x] for x in e[i]]) for i in range(len(names))]
        else:
            per_model = [custom_train_test_agents(train_env=v, test_env=r_, config=c, agents_num=agents_num) for v, r_, c in loaded]
    for name, (r_i, s_i, e_i) in zip(names, per_model):
        if correlation_exp and train_on_venv and pool is not None:
            reward_list.append(r_i); train_steps_needed.append(s_i); episode_length_needed.append(e_i)
        else:
            reward_list += r_i; train_steps_needed += s_i; episode_length_needed += e_i
        env_reward_overview[name] = {} if correlation_exp else np.hstack(r_i)
    if _rank_world(True)[0] != 0:      # sharded run: every rank holds the full result table, rank 0 writes it
        return os.path.join(out_dir or os.getcwd(), str(mode) + '_' + (experiment_name or "_experiment_") + '.pt')
    return save_lists(mode=mode, config=config, reward_list=reward_list, train_steps_needed=train_steps_needed,
                      episode_length_needed=episode_length_needed, env_reward_overview=env_reward_overview,
                      experiment_name=experiment_name, out_dir=out_dir)
