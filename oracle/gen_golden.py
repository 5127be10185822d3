"""TEST INFRASTRUCTURE ONLY — generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, imported through oracle/ref_harness.py) on fixed seeds with its RNG sources redirected to
the Philox lane streams.  Run in the build container (the reference cannot travel to the GPU box):

    python -m oracle.gen_golden            # rewrites tests/golden/

The fixtures pin (a) the C restatement oracle/le_oracle.c (tests/test_oracle_vs_golden.py, CPU) and
(b) the CUDA path (tests/test_gpu_*.py, GPU) to the reference's own outputs.
"""
import copy
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ref_harness as rh  # noqa: E402
from learning_environments_b200 import config as le_config  # noqa: E402
from learning_environments_b200._abi import ENV_SE, ENV_RN, ENV_REAL  # noqa: E402


def cfg_bytes(cfg, agent_name, env_kind, **kw):
    """le_lane_cfg bytes: the fixtures must be self-contained (the YAML files do not exist on the GPU box)."""
    c = le_config.lane_cfg(cfg, agent_name=agent_name, env_kind=env_kind, **kw)
    return np.frombuffer(bytes(c), dtype=np.uint8).copy()

GOLDEN = os.path.join(ROOT, "tests", "golden")


def linear_params(module):
    """Concatenate nn.Linear weights/biases in module order (the parameter vector 'theta' of le_b200.h)."""
    import torch.nn as nn
    out = []
    for l in module.modules():
        if isinstance(l, nn.Linear):
            out.append(l.weight.detach().numpy().reshape(-1))
            if l.bias is not None:
                out.append(l.bias.detach().numpy().reshape(-1))
    return np.concatenate(out).astype(np.float32)


def small_config(name, agent_name=None, **agent_overrides):
    cfg = rh.load_reference_yaml(name)
    if agent_name is not None:
        cfg["agents"].setdefault("gtn", {})["agent_name"] = agent_name
    agent = cfg["agents"]["gtn"]["agent_name"].lower()
    cfg["agents"][agent].update(agent_overrides)
    cfg["agents"][agent]["print_rate"] = 10 ** 9
    return cfg, agent


# ------------------------------------------------------------------------------------------------------
def gen_se_step(yaml_name, tag, seed, env_overrides=None):
    import torch
    mods = rh.import_reference()
    cfg = rh.load_reference_yaml(yaml_name)
    if env_overrides:
        cfg["envs"][cfg["env_name"]].update(env_overrides)
    torch.manual_seed(seed)
    fac = mods["envs.env_factory"].EnvFactory(cfg)
    venv = fac.generate_virtual_env()
    sd, ad = venv.get_state_dim(), venv.get_action_dim()
    rng = np.random.RandomState(seed)
    n = 64
    states = rng.uniform(-1.0, 1.0, size=(n, sd)).astype(np.float32)
    actions = rng.randint(0, ad, size=n).astype(np.int32)
    ns = np.zeros((n, sd), np.float32)
    rew = np.zeros(n, np.float32)
    done = np.zeros(n, np.float32)
    with torch.no_grad():
        for i in range(n):
            # the single-agent call of agents/base_agent.py:117: EnvWrapper.step(action) on env.state
            venv.env.state = torch.from_numpy(states[i])
            a = torch.tensor([actions[i]], dtype=torch.float32)
            s2, r, d = venv.step(action=a)
            ns[i], rew[i], done[i] = s2.numpy(), r.item(), d.item()
        # the batched entry (envs/virtual_env.py:45-47, histogram experiment): state passed explicitly
        s2b, rb, db = venv.step(action=torch.from_numpy(actions.astype(np.float32)), state=torch.from_numpy(states))
    assert np.allclose(s2b.numpy(), ns, atol=1e-6)
    np.savez(os.path.join(GOLDEN, "se_step_%s.npz" % tag), theta=linear_params(venv), states=states, actions=actions,
             next_states=ns, rewards=rew, dones=done, yaml=yaml_name,
             cfg=cfg_bytes(cfg, cfg["agents"]["gtn"]["agent_name"].lower(), ENV_SE))


def gen_rn_reward(seed):
    import torch
    mods = rh.import_reference()
    yaml_name = "default_config_cartpole_reward_env.yaml"
    rng = np.random.RandomState(seed)
    n = 32
    s = rng.uniform(-1, 1, size=(n, 4))
    s2 = rng.uniform(-1, 1, size=(n, 4))
    rr = rng.uniform(-1, 2, size=n)
    out = {}
    theta = None
    for t in (0, 1, 2, 5, 6):
        cfg = rh.load_reference_yaml(yaml_name)
        cfg["envs"]["CartPole-v0"]["reward_env_type"] = t
        torch.manual_seed(seed)
        fac = mods["envs.env_factory"].EnvFactory(cfg)
        renv = fac.generate_reward_env()
        renv.set_agent_params(same_action_num=1, gamma=0.99)
        if t != 0:
            th = linear_params(renv)
            if theta is None:
                theta = th
            assert np.array_equal(theta, th)
        res = np.zeros(n, np.float32)
        with torch.no_grad():
            for i in range(n):
                res[i] = np.float32(renv.env._calc_reward(state=s[i], next_state=s2[i], reward=rr[i], info={}))
        out["type%d" % t] = res
    np.savez(os.path.join(GOLDEN, "rn_reward_cartpole.npz"), theta=theta, s=s, s2=s2, real_reward=rr, gamma=0.99,
             yaml=yaml_name, cfg=cfg_bytes(cfg, "ddqn", ENV_RN, gamma=0.99), **out)


def gen_td_update(yaml_name, tag, seed, steps=5, agent=None, **overrides):
    """DDQN.learn / DuelingDDQN.learn (agents/DDQN.py:60-95, agents/DuelingDDQN.py:59-94) `steps` times on explicit minibatches."""
    import torch
    mods = rh.import_reference()
    cfg, agent_name = small_config(yaml_name, agent, **overrides)
    torch.manual_seed(seed)
    fac = mods["envs.env_factory"].EnvFactory(cfg)
    real_env = fac.generate_real_env()
    agent = mods["agents.agent_utils"].select_agent(cfg, cfg["agents"]["gtn"]["agent_name"])
    sd, ad, B = agent.state_dim, agent.action_dim, agent.batch_size
    rng = np.random.RandomState(seed)
    rows = np.zeros((steps, B, 2 * sd + 3), np.float32)
    rows[:, :, :sd] = rng.uniform(-1, 1, size=(steps, B, sd))
    rows[:, :, sd] = rng.randint(0, ad, size=(steps, B))
    rows[:, :, sd + 1:2 * sd + 1] = rng.uniform(-1, 1, size=(steps, B, sd))
    rows[:, :, 2 * sd + 1] = rng.uniform(-1, 1, size=(steps, B))
    rows[:, :, 2 * sd + 2] = (rng.uniform(size=(steps, B)) < 0.1) * 1.0 + rng.uniform(-0.05, 0.05, size=(steps, B))

    class FakeRB(object):
        def __init__(self):
            self.k = 0

        def sample(self, batch_size):
            r = torch.from_numpy(rows[self.k])
            self.k += 1
            return (r[:, :sd], r[:, sd:sd + 1], r[:, sd + 1:2 * sd + 1], r[:, 2 * sd + 1:2 * sd + 2], r[:, 2 * sd + 2:])

    q0 = linear_params(agent.model)
    rb = FakeRB()
    thetas, targets, losses = [], [], []
    for k in range(steps):
        loss = agent.learn(replay_buffer=rb, env=real_env, episode=10)
        losses.append(loss.item())
        thetas.append(linear_params(agent.model))
        targets.append(linear_params(agent.model_target))
    st = agent.optimizer.state_dict()["state"]
    m = np.concatenate([st[i]["exp_avg"].numpy().reshape(-1) for i in range(len(st))])
    v = np.concatenate([st[i]["exp_avg_sq"].numpy().reshape(-1) for i in range(len(st))])
    save_td_update(tag, dict(q_init=q0, rows=rows, losses=np.array(losses, np.float32), yaml=yaml_name,
                             cfg=cfg_bytes(cfg, agent_name, ENV_RN if "reward_env" in yaml_name else ENV_SE)),
                   dict(thetas=np.stack(thetas), targets=np.stack(targets), adam_m=m, adam_v=v))


GOLDEN_FILE_BYTES = 1000000     # no fixture is larger


def save_td_update(tag, inputs, after):
    """Writes td_update_<tag>.npz.  `inputs` (q_init, rows, losses, yaml, cfg) are stored whole.  `after` holds the parameter
    vectors after the steps (thetas, targets [steps, P], adam_m, adam_v [P]); when storing them whole would make the file larger
    than GOLDEN_FILE_BYTES they are kept at the sorted parameter indices `param_idx` instead: every bias and the same seeded
    fraction of every weight matrix, as many as fit."""
    from learning_environments_b200._abi import LaneCfg
    size = sum(np.asarray(a).nbytes for a in list(inputs.values()) + list(after.values())) + 4096     # + npy headers
    if size > GOLDEN_FILE_BYTES:
        dims = LaneCfg.from_buffer_copy(inputs["cfg"].tobytes()).q_layer_dims()
        n_bias, n_weight = sum(o for _, o in dims), sum(i * o for i, o in dims)
        per_index = 4 + sum(a.nbytes // a.shape[-1] for a in after.values())
        room = (GOLDEN_FILE_BYTES - 4096 - sum(np.asarray(a).nbytes for a in inputs.values())) // per_index - n_bias
        rng = np.random.RandomState(0)
        idx, off = [], 0
        for i, o in dims:
            idx += [off + np.sort(rng.choice(i * o, max(1, room * i * o // n_weight), replace=False)), off + i * o + np.arange(o)]
            off += i * o + o
        assert off == inputs["q_init"].size
        param_idx = np.concatenate(idx).astype(np.int32)
        after = dict({k: a[..., param_idx] for k, a in after.items()}, param_idx=param_idx)
    np.savez(os.path.join(GOLDEN, "td_update_%s.npz" % tag), **inputs, **after)


def gen_td3_learn(seed, steps=5, tag="cartpole", yaml_name="default_config_cartpole_syn_env.yaml", **overrides):
    """TD3_discrete_vary.learn (agents/TD3_discrete_vary.py:62-119) `steps` times on explicit minibatches with the random
    draws (policy noise randn_like, the exponential_() of both gumbel_softmax calls) logged: groundwork for SURVEY §8(f) rank 2."""
    import torch
    mods = rh.import_reference()
    kw = dict(hidden_size=24, hidden_layer=2, batch_size=16, policy_delay=2, vary_hp=False)
    kw.update(overrides)
    cfg, agent_name = small_config(yaml_name, "td3_discrete_vary", **kw)
    torch.manual_seed(seed)
    agent = mods["agents.agent_utils"].select_agent(cfg, "td3_discrete_vary")
    sd, ad, B = agent.state_dim, agent.action_dim, agent.batch_size
    rng = np.random.RandomState(seed)
    ROW = 2 * sd + ad + 2
    rows = np.zeros((steps, B, ROW), np.float32)
    rows[:, :, :sd] = rng.uniform(-1, 1, size=(steps, B, sd))
    onehot = np.eye(ad, dtype=np.float32)[rng.randint(0, ad, size=(steps, B))]
    rows[:, :, sd:sd + ad] = onehot + rng.standard_normal((steps, B, ad)).astype(np.float32) * 0.04
    rows[:, :, sd + ad:2 * sd + ad] = rng.uniform(-1, 1, size=(steps, B, sd))
    rows[:, :, 2 * sd + ad] = rng.uniform(-1, 1, size=(steps, B))
    rows[:, :, 2 * sd + ad + 1] = (rng.uniform(size=(steps, B)) < 0.1) * 1.0

    class FakeRB(object):
        k = 0

        def sample(self, batch_size):
            r = torch.from_numpy(rows[FakeRB.k])
            FakeRB.k += 1
            return (r[:, :sd], r[:, sd:sd + ad], r[:, sd + ad:2 * sd + ad], r[:, 2 * sd + ad:2 * sd + ad + 1], r[:, 2 * sd + ad + 1:])

    log = {"randn": [], "expo": []}
    orig_randn_like, orig_expo = torch.randn_like, torch.Tensor.exponential_

    def fake_randn_like(t, **kw):
        v = torch.from_numpy(rng.standard_normal(tuple(t.shape)).astype(np.float32))
        log["randn"].append(v.numpy().copy())
        return v

    def fake_exponential_(self, lambd=1.0, generator=None):
        v = torch.from_numpy(rng.exponential(size=tuple(self.shape)).astype(np.float32))
        log["expo"].append(v.numpy().copy())
        with torch.no_grad():
            self.copy_(v)
        return self

    nets = ("actor", "actor_target", "critic_1", "critic_target_1", "critic_2", "critic_target_2")
    init = {n: linear_params(getattr(agent, n)) for n in nets}
    per_step = {n: [] for n in nets}
    temps, updated, n_expo = [], [], []
    torch.randn_like, torch.Tensor.exponential_ = fake_randn_like, fake_exponential_
    try:
        rb = FakeRB()
        for k in range(steps):
            before = len(log["expo"])
            agent.learn(replay_buffer=rb, env=None, episode=10)
            temps.append(float(agent.gumbel_temp_annealed))
            n_expo.append(len(log["expo"]) - before)
            updated.append(int(agent.total_it % agent.policy_delay == 0))
            for n in nets:
                per_step[n].append(linear_params(getattr(agent, n)))
    finally:
        torch.randn_like, torch.Tensor.exponential_ = orig_randn_like, orig_expo
    assert n_expo == [1 + u for u in updated], n_expo
    expo_target, expo_actor, i = [], [], 0
    for u in updated:
        expo_target.append(log["expo"][i]); i += 1
        expo_actor.append(log["expo"][i] if u else np.zeros((B, ad), np.float32)); i += u
    a = cfg["agents"]["td3_discrete_vary"]
    np.savez(os.path.join(GOLDEN, "td3_learn_%s.npz" % tag), sd=sd, ad=ad, hidden=a["hidden_size"], layers=a["hidden_layer"],
             act=le_config.ACT_IDS[str(a["activation_fn"])],
             gamma=a["gamma"], tau=a["tau"], lr=a["lr"], policy_delay=a["policy_delay"], policy_std=a["policy_std"],
             policy_std_clip=a["policy_std_clip"], gumbel_hard=int(a["gumbel_softmax_hard"]), max_action=float(agent.max_action),
             temps=np.array(temps, np.float64), updated=np.array(updated, np.int32), rows=rows, policy_noise=np.stack(log["randn"]),
             expo_target=np.stack(expo_target), expo_actor=np.stack(expo_actor),
             **{"init_" + n: init[n] for n in nets}, **{"after_" + n: np.stack(per_step[n]) for n in nets})
    print("td3_learn: steps", steps, "policy updates", updated, "temps", temps[:2])


class _RingRestatement(object):
    """utils.ReplayBuffer.add / get_all restated (utils.py:24-32: write row ptr, ptr = (ptr + 1) % max_size,
    size = min(size + 1, max_size); every field stored as float32 rows).  Used only where the reference tree is absent."""

    def __init__(self, dims, max_size):
        self.rows = [np.zeros((max_size, d), np.float32) for d in dims]
        self.ptr = self.size = 0
        self.max_size = max_size

    def add(self, *values):
        for r, x in zip(self.rows, values):
            r[self.ptr] = np.asarray(x, np.float32).reshape(-1)
        self.ptr = (self.ptr + 1) % self.max_size
        self.size = min(self.size + 1, self.max_size)

    def get_all(self):
        return [r[:self.size] for r in self.rows]


class _MeterRestatement(object):
    """utils.AverageMeter.get_mean / get_mean_last restated (utils.py:75-105): the mean of the last `num` values, or of the `num`
    before them, as sum / (count + 1e-9) over however many exist.  Used only where the reference tree is absent."""

    def __init__(self):
        self.vals = []

    def update(self, v, print_rate=10):
        self.vals.append(v)

    def _mean(self, num, skip):
        hi = max(len(self.vals) - skip, 0)
        w = self.vals[max(hi - num, 0):hi]
        return sum(w) / (len(w) + 1e-9)

    def get_mean(self, num=10):
        return self._mean(num, 0)

    def get_mean_last(self, num=10):
        return self._mean(num, num)


def gen_utils_semantics(seed=0, adds=9, max_size=4, updates=25):
    """utils.ReplayBuffer (ptr / size after every add, get_all()) and utils.AverageMeter (get_mean(10), get_mean_last(10) after
    every update) on seeded inputs, which are stored with the results.  The reference's own classes where its tree is present;
    elsewhere the restatements above, and `source` says which."""
    rng = np.random.RandomState(seed)
    rb_in = np.zeros((adds, 9), np.float32)          # state[3] action[1] next_state[3] reward[1] done[1]
    for i in range(adds):
        rb_in[i] = np.concatenate([rng.rand(3), [i % 2], rng.rand(3), [i], [i % 3 == 0]]).astype(np.float32)
    meter_in = rng.rand(updates)
    if rh.reference_available():
        import torch
        ref = rh.import_reference()["utils"]
        rb, meter, source = ref.ReplayBuffer(3, 1, "cpu", max_size=max_size), ref.AverageMeter(""), "reference"
        cols = [(0, 3), (3, 4), (4, 7), (7, 8)]
        add = lambda r: rb.add(*[torch.from_numpy(r[a:b].copy()) for a, b in cols], torch.tensor(float(r[8])))
    else:
        rb, meter, source = _RingRestatement((3, 1, 3, 1, 1), max_size), _MeterRestatement(), "restatement"
        add = lambda r: rb.add(r[0:3], r[3:4], r[4:7], r[7:8], r[8:9])
    ptr_size = []
    for r in rb_in:
        add(r)
        ptr_size.append((rb.ptr, rb.size))
    out = {"rb_" + k: np.asarray(x, np.float32) for k, x in zip(("state", "action", "next_state", "reward", "done"), rb.get_all())}
    means = []
    for v in meter_in:
        meter.update(v, print_rate=10 ** 9)
        means.append((meter.get_mean(10), meter.get_mean_last(10)))
    np.savez(os.path.join(GOLDEN, "utils_semantics.npz"), rb_inputs=rb_in, rb_max_size=max_size, ptr_size=np.array(ptr_size, np.int64),
             meter_inputs=meter_in, means=np.array(means, np.float64), source=source, **out)


def gen_real_env(seed):
    """Trajectories of the gym stand-in (oracle/stubs/gym) — pins the C/CUDA dynamics to the restated equations."""
    import gym
    rng = np.random.RandomState(seed)
    for name, tag, nact in (("CartPole-v0", "cartpole", 2), ("Acrobot-v1", "acrobot", 3)):
        env = gym.make(name)
        eps = []
        for ep in range(4):
            st0 = rng.uniform(-0.05, 0.05, size=4) if tag == "cartpole" else rng.uniform(-0.1, 0.1, size=4)
            env.unwrapped.reset_hook = lambda e, s=st0: s
            obs0 = env.reset()
            T = 60 if tag == "cartpole" else 120
            acts = rng.randint(0, nact, size=T)
            states, obs, rew, done = [np.array(env.unwrapped.state, np.float64)], [obs0], [], []
            for a in acts:
                o, r, d, _ = env.step(int(a))
                states.append(np.array(env.unwrapped.state, np.float64))
                obs.append(o)
                rew.append(r)
                done.append(d)
                if d:
                    break
            eps.append(dict(actions=acts[:len(rew)], states=np.stack(states), obs=np.stack(obs), rewards=np.array(rew),
                            dones=np.array(done)))
        flat = {}
        for i, e in enumerate(eps):
            for k, v in e.items():
                flat["ep%d_%s" % (i, k)] = v
        np.savez(os.path.join(GOLDEN, "real_env_%s.npz" % tag), n_episodes=len(eps), **flat)


def gen_trajectory(yaml_name, tag, seed, key, env_kind, overrides, trace_cap, use_test_env=True, agent=None, env_overrides=None):
    """Full BaseAgent.train(+test) of the reference under RNG injection; per-step trace of the first steps."""
    import torch
    mods = rh.import_reference()
    cfg, agent_name = small_config(yaml_name, agent, **overrides)
    if env_overrides:
        cfg["envs"][cfg["env_name"]].update(env_overrides)
    torch.manual_seed(seed)
    fac = mods["envs.env_factory"].EnvFactory(cfg)
    real_env = fac.generate_real_env()
    if env_kind == "se":
        train_env = fac.generate_virtual_env()
        env_theta = linear_params(train_env)
        reset_envs = [train_env.env.reset_env.env.unwrapped, real_env.env.unwrapped]
        spaces = [train_env.env.action_space]
    elif env_kind == "rn":
        train_env = fac.generate_reward_env()
        env_theta = linear_params(train_env)
        reset_envs = [train_env.env.real_env.unwrapped, real_env.env.unwrapped]
        spaces = [train_env.env.action_space]
    else:
        train_env = fac.generate_real_env()
        env_theta = np.zeros(1, np.float32)
        reset_envs = [train_env.env.unwrapped, real_env.env.unwrapped]
        spaces = [train_env.env.action_space]
    agent = mods["agents.agent_utils"].select_agent(cfg, cfg["agents"]["gtn"]["agent_name"])
    q_init = linear_params(agent.model)
    sd, ad = agent.state_dim, agent.action_dim
    inj = rh.LaneRngInjector(key, ad, "cartpole" if "CartPole" in cfg["env_name"] else "acrobot")

    tr = dict(action=[], explore=[], next_state=[], reward=[], done=[], loss=[])
    orig_learn, orig_select, orig_step = agent.learn, agent.select_train_action, train_env.step
    state_now = {"explore": 0}

    def learn(replay_buffer, env, episode):
        loss = orig_learn(replay_buffer=replay_buffer, env=env, episode=episode)
        tr["loss"][-1] = float(loss.item())
        return loss

    def select(state, env, episode):
        before = inj.train_steps
        a = orig_select(state=state, env=env, episode=episode)
        assert inj.train_steps == before + 1
        u = float(inj._act_words[0] >> 8) / 16777216.0
        tr["explore"].append(1 if u < agent.eps else 0)
        return a

    def step(action, state=None):
        s2, r, d = orig_step(action=action) if state is None else orig_step(action=action, state=state)
        tr["action"].append(int(action.reshape(-1)[0].item()))
        tr["next_state"].append(s2.detach().numpy().astype(np.float32).copy())
        tr["reward"].append(float(r))
        tr["done"].append(float(d))
        tr["loss"].append(float("nan"))
        return s2, r, d

    agent.learn, agent.select_train_action, train_env.step = learn, select, step
    with rh.injected_rng(inj, reset_envs=reset_envs, action_spaces=spaces):
        rewards, lengths, _ = agent.train(env=train_env, test_env=real_env if use_test_env else None)
        test_rewards, _, _ = agent.test(env=real_env)
    n = min(trace_cap, len(tr["action"]))
    kind_id = {"se": ENV_SE, "rn": ENV_RN, "real": ENV_REAL}[env_kind]
    np.savez(os.path.join(GOLDEN, "trajectory_%s.npz" % tag), yaml=yaml_name, env_kind=env_kind, key=np.array(key, np.uint32),
             cfg=cfg_bytes(cfg, agent_name, kind_id, use_test_env=use_test_env, final_test=True),
             overrides_keys=np.array(list(overrides.keys())), overrides_vals=np.array([float(v) for v in overrides.values()]),
             use_test_env=int(use_test_env), env_theta=env_theta, q_init=q_init, q_final=linear_params(agent.model),
             rewards=np.array(rewards, np.float64), lengths=np.array(lengths, np.int32),
             test_rewards=np.array(test_rewards, np.float64), train_steps=len(tr["action"]), learn_iters=inj.learn_iters,
             action=np.array(tr["action"][:n], np.int32), explore=np.array(tr["explore"][:n], np.int32),
             next_state=np.stack(tr["next_state"][:n]), reward=np.array(tr["reward"][:n], np.float32),
             done=np.array(tr["done"][:n], np.float32), loss=np.array(tr["loss"][:n], np.float32),
             sample0=inj.sample_log[0] if inj.sample_log else np.zeros(0, np.int32))
    print("trajectory", tag, "episodes", len(rewards), "steps", len(tr["action"]), "learn", inj.learn_iters, "rewards",
          rewards[:4], "test", test_rewards[:3])


def gen_trajectory_td3(tag, seed, key, overrides, trace_cap, yaml_name="default_config_cartpole_syn_env.yaml", env_kind="se"):
    """BaseAgent.train (+ per-episode test) and test of the reference's TD3_discrete_vary on a CartPole SE under RNG injection
    (oracle/ref_harness.py Td3RngInjector): groundwork for SURVEY §8(f) rank 2."""
    import torch
    mods = rh.import_reference()
    cfg, agent_name = small_config(yaml_name, "td3_discrete_vary", **overrides)
    torch.manual_seed(seed)
    fac = mods["envs.env_factory"].EnvFactory(cfg)
    real_env = fac.generate_real_env()
    if env_kind == "se":
        train_env = fac.generate_virtual_env()
        env_theta = linear_params(train_env)
        reset_envs = [train_env.env.reset_env.env.unwrapped, real_env.env.unwrapped]
    else:
        train_env = fac.generate_real_env()
        env_theta = np.zeros(1, np.float32)
        reset_envs = [train_env.env.unwrapped, real_env.env.unwrapped]
    agent = mods["agents.agent_utils"].select_agent(cfg, "td3_discrete_vary")
    init = {n: linear_params(getattr(agent, n)) for n in ("actor", "critic_1", "critic_2")}
    inj = rh.Td3RngInjector(key, agent.action_dim, "cartpole" if "CartPole" in cfg["env_name"] else "acrobot")
    tr = dict(action=[], next_state=[], reward=[], done=[])
    orig_step = train_env.step

    def step(action, state=None):
        s2, r, d = orig_step(action=action) if state is None else orig_step(action=action, state=state)
        tr["action"].append(int(action.reshape(-1)[0].item()))
        tr["next_state"].append(s2.detach().numpy().astype(np.float32).copy())
        tr["reward"].append(float(r))
        tr["done"].append(float(d))
        return s2, r, d

    train_env.step = step
    with rh.injected_rng_td3(inj, agent, reset_envs=reset_envs, action_spaces=[train_env.env.action_space]):
        rewards, lengths, _ = agent.train(env=train_env, test_env=real_env)
        test_rewards, _, _ = agent.test(env=real_env)
    n = min(trace_cap, len(tr["action"]))
    a = cfg["agents"]["td3_discrete_vary"]
    np.savez(os.path.join(GOLDEN, "trajectory_td3_%s.npz" % tag), key=np.array(key, np.uint32),
             cfg=cfg_bytes_td3(cfg, ENV_SE if env_kind == "se" else ENV_REAL), agent_cfg_json=np.array(__import__("json").dumps(a)), max_action=float(agent.max_action),
             env_theta=env_theta, init_actor=init["actor"], init_critic_1=init["critic_1"], init_critic_2=init["critic_2"],
             actor_final=linear_params(agent.actor), rewards=np.array(rewards, np.float64), lengths=np.array(lengths, np.int32),
             test_rewards=np.array(test_rewards, np.float64), train_steps=len(tr["action"]), learn_iters=inj.learn_iters,
             action=np.array(tr["action"][:n], np.int32), next_state=np.stack(tr["next_state"][:n]),
             reward=np.array(tr["reward"][:n], np.float32), done=np.array(tr["done"][:n], np.float32))
    print("trajectory_td3", tag, "episodes", len(rewards), "steps", len(tr["action"]), "learn", inj.learn_iters, "rewards", rewards[:4],
          "test", test_rewards[:3])


def cfg_bytes_td3(cfg, env_kind=ENV_SE):
    """le_lane_cfg bytes for a TD3 lane: env / loop fields from the ddqn-style mapping, MLP shape from the td3 section."""
    d = copy.deepcopy(cfg)
    a = d["agents"]["td3_discrete_vary"]
    ddqn_like = dict(d["agents"]["ddqn"])
    for k in ("train_episodes", "test_episodes", "init_episodes", "batch_size", "gamma", "lr", "tau", "rb_size", "same_action_num",
              "activation_fn", "hidden_size", "hidden_layer", "early_out_num", "early_out_virtual_diff"):
        ddqn_like[k] = a[k]
    d["agents"]["ddqn"] = ddqn_like
    c = le_config.lane_cfg(d, agent_name="ddqn", env_kind=env_kind, use_test_env=True, final_test=True)
    return np.frombuffer(bytes(c), dtype=np.uint8).copy()


def gen_nes(seed):
    """GTN_Master.score_transform (agents/GTN_master.py:197-265) for all 8 types, and update_env (:267-298)."""
    import torch
    mods = rh.import_reference()
    cfg = rh.load_reference_yaml("default_config_cartpole_syn_env.yaml")
    cfg["agents"]["gtn"]["num_workers"] = 8
    rng = np.random.RandomState(seed)
    score_lists = [
        [10, 200, 35.5, 9.4, 150, 200, 60, 12],                 # SURVEY Appendix C (tie between members 1 and 5)
        list(rng.uniform(0, 200, size=8)),
        [50.0] * 8,                                             # all equal
        [-500.0, -100.0, -480.0, -90.0, -500.0, -250.0, -100.0, -499.0],        # Acrobot-like negative scores with ties
    ]
    orig_lists = [[50] * 8, list(rng.uniform(0, 200, size=8)), [50.0] * 8, [-300.0] * 8]
    out = {}
    with rh.in_tmp_cwd():
        torch.manual_seed(seed)
        master = mods["agents.GTN_master"].GTN_Master(cfg, bohb_id=-1)
        for li, (sl, ol) in enumerate(zip(score_lists, orig_lists)):
            out["scores%d" % li] = np.array(sl, np.float64)
            out["scores_orig%d" % li] = np.array(ol, np.float64)
            for t in range(8):
                master.score_transform_type = t
                master.score_list = list(sl)
                master.score_orig_list = list(ol)
                with np.errstate(all="ignore"):
                    master.score_transform()
                out["transform%d_type%d" % (li, t)] = np.array(master.score_transform_list, np.float64)
        # update_env with explicit eps: theta, eps_i, weights -> theta'
        theta0 = linear_params(master.synthetic_env_orig)
        P = theta0.size
        eps = (rng.standard_normal(size=(8, P)) * 0.0124).astype(np.float32)
        import torch.nn as nn
        for i in range(8):
            off = 0
            for l in master.eps_list[i].modules():
                if isinstance(l, nn.Linear):
                    nw = l.weight.numel()
                    l.weight = nn.Parameter(torch.from_numpy(eps[i, off:off + nw].reshape(l.weight.shape).copy()))
                    off += nw
                    nb = l.bias.numel()
                    l.bias = nn.Parameter(torch.from_numpy(eps[i, off:off + nb].copy()))
                    off += nb
            assert off == P
        for wd, tag in ((0.0, "nowd"), (0.01, "wd")):
            fresh = mods["agents.GTN_master"].GTN_Master(cfg, bohb_id=-1)
            fresh.synthetic_env_orig.load_state_dict(master.synthetic_env_orig.state_dict())
            fresh.eps_list = master.eps_list
            fresh.weight_decay = wd
            fresh.score_transform_list = list(out["transform0_type3"])
            fresh.update_env()
            out["theta_after_%s" % tag] = linear_params(fresh.synthetic_env_orig)
    np.savez(os.path.join(GOLDEN, "nes_cartpole.npz"), theta0=theta0, eps=eps, step_size=float(cfg["agents"]["gtn"]["step_size"]),
             n_lists=len(score_lists), **out)


def main():
    """python oracle/gen_golden.py [name ...] — regenerates all fixtures, or only those whose name contains an argument."""
    os.makedirs(GOLDEN, exist_ok=True)
    import torch
    torch.set_num_threads(1)
    CP, AC, RN = "default_config_cartpole_syn_env.yaml", "default_config_acrobot_syn_env.yaml", "default_config_cartpole_reward_env.yaml"
    jobs = [
        ("se_step_cartpole", lambda: gen_se_step(CP, "cartpole", 1)),
        ("se_step_acrobot", lambda: gen_se_step(AC, "acrobot", 2)),
        # the other activation functions of models/model_utils.py:9-19 and other hidden widths for the SE
        ("se_step_cartpole_tanh", lambda: gen_se_step(CP, "cartpole_tanh", 31, dict(activation_fn="tanh", hidden_size=96))),
        ("se_step_cartpole_relu", lambda: gen_se_step(CP, "cartpole_relu", 32, dict(activation_fn="relu", hidden_size=32))),
        ("se_step_acrobot_identity", lambda: gen_se_step(AC, "acrobot_identity", 33, dict(activation_fn="identity", hidden_size=40))),
        ("se_step_acrobot_leaky", lambda: gen_se_step(AC, "acrobot_leaky", 34, dict(activation_fn="leakyrelu", hidden_size=300))),
        ("rn_reward_cartpole", lambda: gen_rn_reward(3)),
        ("td_update_cartpole", lambda: gen_td_update(CP, "cartpole", 4)),
        ("td_update_acrobot", lambda: gen_td_update(AC, "acrobot", 5)),
        ("td_update_cartpole_rn", lambda: gen_td_update(RN, "cartpole_rn", 6)),
        ("td_update_cartpole_dueling", lambda: gen_td_update(CP, "cartpole_dueling", 8, agent="DuelingDDQN")),
        ("td_update_acrobot_dueling", lambda: gen_td_update("default_config_acrobot.yaml", "acrobot_dueling", 9, steps=3, agent="DuelingDDQN")),
        ("td_update_cartpole_ddqn_l2", lambda: gen_td_update(CP, "cartpole_ddqn_l2", 10, steps=3, agent="DDQN", hidden_layer=2, hidden_size=150)),
        # three hidden layers: DuelingDDQN_vary samples hidden_layer in {L-1, L, L+1} = {1, 2, 3} from default_config_acrobot.yaml
        # (agents/DuelingDDQN_vary.py:52-57); DDQN_vary does the same around the CartPole yaml
        ("td_update_acrobot_dueling_l3", lambda: gen_td_update("default_config_acrobot.yaml", "acrobot_dueling_l3", 47, steps=3, agent="DuelingDDQN",
                                                               hidden_layer=3, hidden_size=96, batch_size=100)),
        ("td_update_cartpole_ddqn_l3", lambda: gen_td_update(CP, "cartpole_ddqn_l3", 48, steps=3, agent="DDQN", hidden_layer=3, hidden_size=40)),
        ("td3_learn_cartpole", lambda: gen_td3_learn(41)),
        # soft Gumbel-softmax, relu nets, one hidden layer, policy update on every call; Acrobot shapes (sd 6, ad 3) with leakyrelu
        ("td3_learn_cartpole_soft", lambda: gen_td3_learn(43, tag="cartpole_soft", gumbel_softmax_hard=False, activation_fn="relu",
                                                          hidden_layer=1, policy_delay=1)),
        ("td3_learn_acrobot", lambda: gen_td3_learn(44, tag="acrobot", yaml_name="default_config_acrobot_syn_env.yaml",
                                                    activation_fn="leakyrelu", policy_delay=3, steps=7)),
        ("trajectory_td3_cartpole_se", lambda: gen_trajectory_td3("cartpole_se", 42, (0x81, 0x82),
                                                                  dict(train_episodes=4, test_episodes=2, init_episodes=1, hidden_size=24,
                                                                       hidden_layer=2, batch_size=16, policy_delay=2, vary_hp=False),
                                                                  trace_cap=400)),
        ("trajectory_td3_acrobot_se", lambda: gen_trajectory_td3("acrobot_se", 45, (0x83, 0x84),
                                                                 dict(train_episodes=2, test_episodes=1, init_episodes=1, hidden_size=20,
                                                                      hidden_layer=1, batch_size=12, policy_delay=1, vary_hp=False,
                                                                      activation_fn="relu"), trace_cap=700,
                                                                 yaml_name="default_config_acrobot_syn_env.yaml")),
        ("trajectory_td3_cartpole_real", lambda: gen_trajectory_td3("cartpole_real", 46, (0x85, 0x86),
                                                                    dict(train_episodes=12, test_episodes=2, init_episodes=2, hidden_size=24,
                                                                         hidden_layer=2, batch_size=16, policy_delay=2, vary_hp=False,
                                                                         same_action_num=2), trace_cap=300, env_kind="real")),
        ("real_env", lambda: gen_real_env(7)),
        ("utils_semantics", gen_utils_semantics),
        ("trajectory_cartpole_se", lambda: gen_trajectory(CP, "cartpole_se", 11, (0x1234, 0xABCD), "se",
                                                          dict(train_episodes=5, test_episodes=3, init_episodes=1), trace_cap=400)),
        ("trajectory_acrobot_se", lambda: gen_trajectory(AC, "acrobot_se", 12, (0x77, 0x99), "se",
                                                         dict(train_episodes=4, test_episodes=2, init_episodes=1), trace_cap=800)),
        ("trajectory_cartpole_rn", lambda: gen_trajectory(RN, "cartpole_rn", 13, (0x5, 0x6), "rn",
                                                          dict(train_episodes=12, test_episodes=1, init_episodes=2), trace_cap=300)),
        ("trajectory_cartpole_se_notest", lambda: gen_trajectory(CP, "cartpole_se_notest", 14, (0x42, 0x43), "se",
                                                                 dict(train_episodes=8, test_episodes=3, init_episodes=2, early_out_num=2),
                                                                 trace_cap=200, use_test_env=False)),
        ("trajectory_cartpole_se_dueling", lambda: gen_trajectory(CP, "cartpole_se_dueling", 15, (0x51, 0x52), "se",
                                                                  dict(train_episodes=3, test_episodes=2, init_episodes=1), trace_cap=300,
                                                                  agent="DuelingDDQN")),
        # same_action_num > 1 (envs/env_wrapper.py:24-61; agents/base_agent.py:104,123) on all three env branches, and
        # training directly on the real env (experiments/syn_env_run_vary_hp.py mode 0)
        ("trajectory_cartpole_se_k2", lambda: gen_trajectory(CP, "cartpole_se_k2", 16, (0x61, 0x62), "se",
                                                             dict(train_episodes=5, test_episodes=3, init_episodes=1, same_action_num=2),
                                                             trace_cap=300)),
        ("trajectory_cartpole_rn_k3", lambda: gen_trajectory(RN, "cartpole_rn_k3", 17, (0x63, 0x64), "rn",
                                                             dict(train_episodes=12, test_episodes=2, init_episodes=2, same_action_num=3),
                                                             trace_cap=300)),
        ("trajectory_cartpole_real_k2", lambda: gen_trajectory(CP, "cartpole_real_k2", 18, (0x65, 0x66), "real",
                                                               dict(train_episodes=10, test_episodes=2, init_episodes=2, same_action_num=2),
                                                               trace_cap=300)),
        ("trajectory_acrobot_real", lambda: gen_trajectory(AC, "acrobot_real", 19, (0x67, 0x68), "real",
                                                           dict(train_episodes=2, test_episodes=1, init_episodes=1), trace_cap=700)),
        # general-kernel lanes end to end: Acrobot yaml DuelingDDQN (2 x 128 relu, feature_dim 128), 2-hidden-layer DDQN
        ("trajectory_acrobot_se_dueling", lambda: gen_trajectory("default_config_acrobot.yaml", "acrobot_se_dueling", 22, (0x71, 0x72), "se",
                                                                 dict(train_episodes=2, test_episodes=1, init_episodes=1), trace_cap=500,
                                                                 agent="DuelingDDQN")),
        ("trajectory_cartpole_se_ddqn_l2", lambda: gen_trajectory(CP, "cartpole_se_ddqn_l2", 23, (0x73, 0x74), "se",
                                                                  dict(train_episodes=3, test_episodes=2, init_episodes=1, hidden_layer=2,
                                                                       hidden_size=150), trace_cap=300)),
        ("trajectory_cartpole_se_ddqn_l3", lambda: gen_trajectory(CP, "cartpole_se_ddqn_l3", 49, (0x8A, 0x8B), "se",
                                                                  dict(train_episodes=3, test_episodes=2, init_episodes=1, hidden_layer=3,
                                                                       hidden_size=40), trace_cap=300)),
        # hidden_layer = 0 builds the same net as 1 (models/model_utils.py:34); reward types 1 / 5 / 6 through the whole loop;
        # the real-env early-out rule (agents/base_agent.py:49-62) firing
        ("trajectory_cartpole_se_h0", lambda: gen_trajectory(CP, "cartpole_se_h0", 24, (0x75, 0x76), "se",
                                                             dict(train_episodes=3, test_episodes=2, init_episodes=1, hidden_layer=0),
                                                             trace_cap=300)),
        ("trajectory_cartpole_rn_t1", lambda: gen_trajectory(RN, "cartpole_rn_t1", 25, (0x77, 0x78), "rn",
                                                             dict(train_episodes=8, test_episodes=1, init_episodes=2), trace_cap=200,
                                                             env_overrides=dict(reward_env_type=1))),
        ("trajectory_cartpole_rn_t5", lambda: gen_trajectory(RN, "cartpole_rn_t5", 26, (0x79, 0x7A), "rn",
                                                             dict(train_episodes=8, test_episodes=1, init_episodes=2), trace_cap=200,
                                                             env_overrides=dict(reward_env_type=5))),
        ("trajectory_cartpole_rn_t6", lambda: gen_trajectory(RN, "cartpole_rn_t6", 27, (0x7B, 0x7C), "rn",
                                                             dict(train_episodes=8, test_episodes=1, init_episodes=2), trace_cap=200,
                                                             env_overrides=dict(reward_env_type=6))),
        ("trajectory_cartpole_real_solved", lambda: gen_trajectory(CP, "cartpole_real_solved", 28, (0x7D, 0x7E), "real",
                                                                   dict(train_episodes=12, test_episodes=2, init_episodes=1, early_out_num=2),
                                                                   trace_cap=300, env_overrides=dict(solved_reward=9.9))),
        ("nes_cartpole", lambda: gen_nes(21)),
    ]
    want = sys.argv[1:]
    for name, fn in jobs:
        if not want or any(w in name for w in want):
            fn()
    print("golden fixtures written to", GOLDEN)


if __name__ == "__main__":
    main()
