"""Maps the reference's nested YAML config (default_config_*.yaml, passed around as a dict) to le_lane_cfg.

Follows what the reference constructors read: agents/base_agent.py:14-26, agents/DDQN.py:20-32,
envs/env_factory.py:45-59 (lists -> float(value[1])), envs/virtual_env.py:11-21, envs/reward_env.py:11-21.
"""
import copy

from ._abi import ACT_IDS, ENV_REAL, ENV_RN, ENV_SE, Q_DQN, Q_DUELING, REAL_ENV_IDS, LaneCfg

ENV_DIMS = {"CartPole-v0": (4, 2), "Acrobot-v1": (6, 3)}


def env_kwargs(config):
    """EnvFactory._get_default_parameters (envs/env_factory.py:45-59) without the gym objects."""
    env_name = config["env_name"]
    kw = {"env_name": env_name, "device": config.get("device", "cpu")}
    for key, value in config["envs"][env_name].items():
        kw[key] = float(value[1]) if isinstance(value, list) else value
    return kw


def lane_cfg(config, agent_name="ddqn", env_kind=ENV_SE, use_test_env=True, final_test=True, step_budget=0, gamma=None):
    """Builds the le_lane_cfg for one (agent, training env) pair.

    env_kind: ENV_SE (VirtualEnv), ENV_RN (RewardEnv) or ENV_REAL (train on the gym env itself).
    use_test_env/final_test: GTN_Worker.calc_score trains with test_env=real_env and then tests
    (agents/GTN_worker.py:187-221); the vary_hp evaluators train with test_env=None.
    """
    env_name = config["env_name"]
    if env_name not in ENV_DIMS:
        raise NotImplementedError("real environment %r has no device kernel (CartPole-v0 / Acrobot-v1 only)" % env_name)
    a = config["agents"][agent_name]
    e = env_kwargs(config)
    c = LaneCfg()
    c.sd, c.ad = ENV_DIMS[env_name]
    c.env_kind = env_kind
    c.real_env = REAL_ENV_IDS[env_name]
    if int(e.get("hidden_layer", 1)) > 1 and env_kind != ENV_REAL:
        raise NotImplementedError("SE/RN nets with hidden_layer > 1 are outside the compiled kernel set")
    if int(a.get("hidden_layer", 1)) > 3:
        raise NotImplementedError("Q-nets with hidden_layer > 3 are outside the compiled kernel set")
    if int(a.get("same_action_num", 1)) < 1:
        raise ValueError("same_action_num must be >= 1")
    c.same_action_num = int(a.get("same_action_num", 1))
    c.env_hidden = int(e.get("hidden_size", 0))
    c.env_act = ACT_IDS[str(e.get("activation_fn", "identity"))]
    slope = 0.25 if c.env_act == ACT_IDS["prelu"] else 0.01
    for i in range(3):
        c.env_slope[i] = slope
    c.rn_type = int(e.get("reward_env_type", 0))
    c.q_hidden = int(a["hidden_size"])
    c.q_kind = Q_DUELING if agent_name.startswith("duelingddqn") else Q_DQN
    c.q_layers = max(int(a.get("hidden_layer", 1)), 1)
    c.q_feature_dim = int(a.get("feature_dim", 0)) if c.q_kind == Q_DUELING else 0
    c.q_act = ACT_IDS[str(a["activation_fn"])]
    if c.q_act not in (ACT_IDS["tanh"], ACT_IDS["relu"], ACT_IDS["leakyrelu"]):
        raise NotImplementedError("Q-net activation %r is outside the compiled kernel set" % a["activation_fn"])
    c.batch_size = int(a["batch_size"])
    c.rb_size = int(a["rb_size"])
    c.train_episodes = int(a["train_episodes"])
    c.test_episodes = int(a["test_episodes"])
    c.init_episodes = int(a["init_episodes"])
    c.max_steps = int(e["max_steps"])
    c.early_out_num = int(a["early_out_num"])
    c.use_test_env = 1 if use_test_env else 0
    c.final_test = 1 if final_test else 0
    c.step_budget = int(step_budget)
    c.gamma = float(a["gamma"] if gamma is None else gamma)
    c.lr = float(a["lr"])
    c.tau = float(a["tau"])
    c.eps_init = float(a["eps_init"])
    c.eps_min = float(a["eps_min"])
    c.eps_decay = float(a["eps_decay"])
    c.early_out_virtual_diff = float(a["early_out_virtual_diff"])
    c.solved_reward = float(e["solved_reward"])
    c.beta1, c.beta2, c.adam_eps = 0.9, 0.999, 1e-8
    return c


def td3_lane_cfg(config, env_kind=ENV_SE, use_test_env=True, final_test=True, max_action=1.0):
    """le_td3_cfg of the config's td3_discrete_vary section (agents/TD3_discrete_vary.py:20-59); max_action of the discrete
    envs is 1 (envs/env_wrapper.py:106-110).  The eps_* fields of the base configuration are unused by TD3 lanes."""
    from ._abi import Td3Cfg
    a = config["agents"]["td3_discrete_vary"]
    cfg = dict(config, agents=dict(config["agents"], td3_discrete_vary=dict(a, eps_init=0.0, eps_min=0.0, eps_decay=0.0)))
    t = Td3Cfg()
    t.base = lane_cfg(cfg, "td3_discrete_vary", env_kind, use_test_env, final_test)
    t.policy_delay, t.gumbel_hard = int(a["policy_delay"]), int(bool(a["gumbel_softmax_hard"]))
    t.action_std, t.policy_std, t.policy_std_clip = float(a["action_std"]), float(a["policy_std"]), float(a["policy_std_clip"])
    t.gumbel_temp, t.max_action = float(a["gumbel_softmax_temp"]), float(max_action)
    return t


def clone_config(config):
    return copy.deepcopy(config)
