"""CPU tests of the batched transfer evaluations (DuelingDDQN_vary and TD3_discrete_vary agents in vary_hp): the le_td3_run /
le_td3_workspace_bytes argument checks, the P_TD3_INIT restatement, the sampled configurations, the launch grouping and the
result file, with a stub in place of the GPU launch."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from learning_environments_b200 import _abi, config as le_config, default_configs, envs, vary_hp
from learning_environments_b200._abi import ENV_REAL, ENV_RN, ENV_SE, LaneCfg, LaneOut, Td3Cfg
from oracle import philox
from tests import td3_init_stream


def _lib():
    return _abi.load_library()


def _td3_cfg(env_kind=ENV_SE):
    return le_config.td3_lane_cfg(default_configs.get("cartpole_syn_env"), env_kind)


def _run(tcfg, n_cfg=1, n_lanes=2, null_out=False):
    """le_td3_run with non-null dummy host pointers: every check must fire before anything touches them."""
    lib = _lib()
    dummy = C.c_void_p(16)
    ws = C.c_int64(1 << 20)
    rc = lib.le_td3_run(C.byref(tcfg), C.c_int(n_cfg), C.byref(tcfg), dummy, C.c_int(1), None, dummy, None, None, None, C.c_int(0), None,
                        C.c_int(n_lanes), None if null_out else dummy, dummy, dummy, dummy, dummy, ws, None, C.c_int(0), None)
    return rc, lib.le_last_error().decode()


def test_td3_entry_points_are_exported_and_reject_bad_arguments():
    lib = _lib()
    for name in ("le_td3_workspace_bytes", "le_td3_run"):
        assert name in _abi.EXPORTED_SYMBOLS and hasattr(lib, name)
    t = _td3_cfg()
    rc, msg = _run(t, n_cfg=3, n_lanes=2)
    assert rc == -1 and "n_cfg" in msg
    rc, msg = _run(t, null_out=True)
    assert rc == -1 and "NULL" in msg
    rn = _td3_cfg(ENV_RN)
    rc, msg = _run(rn)
    assert rc == -3 and "reward-network" in msg
    assert lib.le_td3_workspace_bytes(C.byref(rn), C.c_int(4), C.c_int(1)) == -3 and b"reward-network" in lib.le_last_error()
    assert lib.le_td3_workspace_bytes(None, C.c_int(4), C.c_int(1)) == -1
    # the host-buffer entry reports the same code and message
    keys = np.zeros((1, 2), np.uint32)
    out, rew, ln, tr = LaneOut(), np.zeros(8), np.zeros(8, np.int32), np.zeros(8)
    w = np.zeros(1 << 16, np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib.le_td3_run_host(C.byref(rn), None, C.c_int(0), None, p(keys), p(w), p(w), p(w), C.c_int(1), None, C.c_int(1), C.byref(out),
                             p(rew), p(ln), p(tr), None, C.c_int(0), C.c_int(0))
    assert rc == -3 and b"reward-network" in lib.le_last_error()


def test_td3_init_stream_restatement():
    key = philox.lane_key(3, 0, 1, 0, 2)
    a, c1, c2 = td3_init_stream.td3_init(key, 6, 3, 40, 2)
    t = _td3_cfg()
    t.base.sd, t.base.ad, t.base.q_hidden, t.base.q_layers = 6, 3, 40, 2
    assert (a.size, c1.size) == t.param_counts()
    pa = C.c_int()
    pc = C.c_int()
    assert _lib().le_td3_param_counts(C.byref(t), C.byref(pa), C.byref(pc)) == 0 and (pa.value, pc.value) == t.param_counts()
    # word p & 3 of block p >> 2 on counter (block, net, P_TD3_INIT, 0), scaled by the layer's 1/sqrt(fan_in)
    for net, v, fan_in in ((0, a, 6), (1, c1, 9), (2, c2, 9)):
        for p_ in (0, 5, 6 * 40 + 39):
            w = philox.philox4x32(p_ >> 2, net, td3_init_stream.P_TD3_INIT, 0, key[0], key[1])[p_ & 3]
            want = np.float32((2.0 * ((w + 0.5) / 4294967296.0) - 1.0) / math.sqrt(fan_in))
            assert v[p_] == want
        assert np.abs(v).max() <= 1.0 / math.sqrt(fan_in)
    hidden_w = a[6 * 40 + 40:6 * 40 + 40 + 1600]
    assert np.abs(hidden_w).max() <= 1.0 / math.sqrt(40) and np.abs(hidden_w).max() > 0.9 / math.sqrt(40)
    assert not np.array_equal(c1, c2) and not np.array_equal(a[:100], philox.qnet_init(key, 100, np.full(100, 1 / math.sqrt(6))))


def _vary_config(name="acrobot_syn_env"):
    cfg = default_configs.get(name)
    cfg["agents"]["td3_discrete_vary"]["vary_hp"] = True
    return cfg


def test_sampled_transfer_configurations_have_the_constructors_ranges():
    cfg = _vary_config()
    du = cfg["agents"]["duelingddqn"]
    cfgs = vary_hp.sample_agent_cfgs(cfg, 300, np.random.RandomState(0), agent_name="duelingddqn")
    assert all(isinstance(c, LaneCfg) and c.q_kind == _abi.Q_DUELING for c in cfgs)
    assert all(du["lr"] / 3 <= c.lr <= du["lr"] * 3 for c in cfgs)
    assert all(int(du["batch_size"] / 3) <= c.batch_size <= int(du["batch_size"] * 3) for c in cfgs)
    assert all(int(du["hidden_size"] / 3) <= c.q_hidden <= int(du["hidden_size"] * 3) for c in cfgs)
    fds = [c.q_feature_dim for c in cfgs]
    assert min(fds) >= int(du["feature_dim"] / 3) and max(fds) <= int(du["feature_dim"] * 3) and len(set(fds)) > 50
    assert {c.q_layers for c in cfgs} == {1, 2, 3}
    assert all(c.train_episodes == 1000 and c.init_episodes == 10 and c.early_out_num == 10 for c in cfgs)   # OVERRIDES
    # the same draws as the DuelingDDQN_vary constructor's config sampling
    rng = np.random.RandomState(0)
    from learning_environments_b200.agents import _varied_config
    base = default_configs.get("acrobot_syn_env")
    base["agents"]["duelingddqn"].update(vary_hp.OVERRIDES)
    for c in cfgs[:5]:
        a = _varied_config(base, "duelingddqn", "duelingddqn_vary", rng, vary_feature_dim=True)["agents"]["duelingddqn"]
        assert (c.q_hidden, c.q_layers, c.batch_size, c.q_feature_dim, c.lr) == (a["hidden_size"], a["hidden_layer"], a["batch_size"],
                                                                                 a["feature_dim"], a["lr"])

    td = cfg["agents"]["td3_discrete_vary"]
    tcfgs = vary_hp.sample_agent_cfgs(cfg, 300, np.random.RandomState(1), agent_name="td3_discrete_vary")
    assert all(isinstance(t, Td3Cfg) for t in tcfgs)
    assert all(td["lr"] / 3 <= t.base.lr <= td["lr"] * 3 for t in tcfgs)
    assert all(int(td["hidden_size"] / 3) <= t.base.q_hidden <= int(td["hidden_size"] * 3) for t in tcfgs)
    assert all(int(td["batch_size"] / 3) <= t.base.batch_size <= int(td["batch_size"] * 3) for t in tcfgs)
    assert {t.base.q_layers for t in tcfgs} == {1, 2, 3}
    assert all(t.policy_delay == td["policy_delay"] and t.gumbel_temp == td["gumbel_softmax_temp"] and t.max_action == 1.0 for t in tcfgs)
    # gated by the vary_hp flags like the constructors: the yaml's td3_discrete_vary.vary_hp = False samples nothing
    fixed = vary_hp.sample_agent_cfgs(default_configs.get("acrobot_syn_env"), 4, np.random.RandomState(1), agent_name="td3_discrete_vary")
    assert {(t.base.q_hidden, t.base.q_layers, t.base.batch_size) for t in fixed} == {(td["hidden_size"], td["hidden_layer"], td["batch_size"])}
    with pytest.raises(ValueError, match="agent_name"):
        vary_hp.sample_agent_cfgs(cfg, 1, np.random.RandomState(0), agent_name="ppo")


def test_max_cfg_covers_feature_dim_and_td3_shapes():
    cfgs = vary_hp.sample_agent_cfgs(_vary_config(), 40, np.random.RandomState(2), agent_name="duelingddqn")
    m = vary_hp._max_cfg(cfgs)
    assert m.q_feature_dim == max(c.q_feature_dim for c in cfgs) > min(c.q_feature_dim for c in cfgs)
    assert (m.q_hidden, m.q_layers, m.batch_size) == tuple(max(getattr(c, f) for c in cfgs) for f in ("q_hidden", "q_layers", "batch_size"))
    assert m.q_params() >= max(c.q_params() for c in cfgs)
    tcfgs = vary_hp.sample_agent_cfgs(_vary_config(), 40, np.random.RandomState(3), agent_name="td3_discrete_vary")
    tm = vary_hp._max_cfg(tcfgs)
    assert isinstance(tm, Td3Cfg) and tm.base.q_hidden == max(t.base.q_hidden for t in tcfgs)
    assert tm.base.batch_size == max(t.base.batch_size for t in tcfgs) and tm.base.q_layers == max(t.base.q_layers for t in tcfgs)
    assert tm.param_counts()[0] >= max(t.param_counts()[0] for t in tcfgs)


def _stub(calls):
    def run_group(sub, cfg0, theta, env_index, keys, n_env, device):
        calls.append(dict(sub=list(sub), cfg0=cfg0, env_index=None if env_index is None else np.asarray(env_index), keys=np.asarray(keys)))
        k = len(sub)
        T = vary_hp._base(cfg0).test_episodes
        steps = np.array([vary_hp._base(c).batch_size for c in sub], np.int64)
        return np.tile(np.arange(T, dtype=np.float64), (k, 1)), steps, np.full(k, 3, np.int64)
    return run_group


@pytest.mark.parametrize("agent_name", ["duelingddqn", "td3_discrete_vary"])
def test_evaluate_agents_groups_and_orders_transfer_lanes(monkeypatch, agent_name):
    calls = []
    monkeypatch.setattr(vary_hp, "_run_group", _stub(calls))
    cfg = _vary_config()
    n_env, agents_num, seed = 2, 12, 5
    thetas = np.random.RandomState(0).standard_normal((n_env, LaneCfg.mlp_params(9, 167, 6) + 2 * LaneCfg.mlp_params(9, 167, 1))).astype(np.float32)
    r, s, e, cfgs = vary_hp.evaluate_agents(cfg, thetas, agents_num, seed, device="cpu", agent_name=agent_name)
    n = n_env * agents_num
    td3 = agent_name == "td3_discrete_vary"
    base = [vary_hp._base(c) for c in cfgs]
    if td3:       # one launch per hidden_layer, in increasing order
        assert [vary_hp._base(c["cfg0"]).q_layers for c in calls] == sorted({b.q_layers for b in base})
        for c in calls:
            assert len({vary_hp._base(x).q_layers for x in c["sub"]}) == 1
    else:         # every dueling lane runs on the general kernel: one launch
        assert len(calls) == 1
    seen = []
    for c in calls:
        sub = c["sub"]
        cost = [vary_hp._base(x).batch_size * (x.param_counts()[0] + 2 * x.param_counts()[1] if td3 else x.q_params()) for x in sub]
        assert cost == sorted(cost, reverse=True)                                   # longest first
        idx = [next(i for i in range(n) if cfgs[i] is x or bytes(cfgs[i]) == bytes(x)) for x in sub]
        seen += idx
        assert np.array_equal(c["env_index"], np.asarray(idx) // agents_num)      # SE per lane as on the DDQN path
        want_keys = np.array([philox.lane_key(seed, 0, i // agents_num, 0, i % agents_num) for i in idx], np.uint32)
        assert np.array_equal(c["keys"].astype(np.uint32), want_keys)
        m = vary_hp._base(c["cfg0"])
        assert m.q_hidden == max(vary_hp._base(x).q_hidden for x in sub) and m.batch_size == max(vary_hp._base(x).batch_size for x in sub)
        if not td3:
            assert m.q_feature_dim == max(x.q_feature_dim for x in sub)
    assert sorted(seen) == list(range(n))
    assert len(r) == n_env and all(len(x) == agents_num for x in r) and r[0][0] == list(np.arange(10, dtype=np.float64))
    assert [x for row in s for x in row] == [b.batch_size for b in base] and e == [[3] * agents_num] * n_env
    # mode 0: the real env for both families
    calls.clear()
    vary_hp.evaluate_agents(cfg, None, 3, seed, device="cpu", env_kind=ENV_REAL, n_envs=2, agent_name=agent_name)
    assert all(vary_hp._base(x).env_kind == ENV_REAL for c in calls for x in c["sub"]) and all(c["env_index"] is None for c in calls)


def test_ddqn_default_is_unchanged_by_the_agent_name_keyword(monkeypatch):
    calls = []
    monkeypatch.setattr(vary_hp, "_run_group", _stub(calls))
    cfg = default_configs.get("cartpole_syn_env")
    theta = np.zeros(LaneCfg.mlp_params(6, 83, 4) + 2 * LaneCfg.mlp_params(6, 83, 1), np.float32)
    a = vary_hp.evaluate_agents(cfg, theta, 9, 4, device="cpu")
    calls_a = [[bytes(x) for x in c["sub"]] for c in calls]
    calls.clear()
    b = vary_hp.evaluate_agents(cfg, theta, 9, 4, device="cpu", agent_name="ddqn")
    assert a[:3] == b[:3] and calls_a == [[bytes(x) for x in c["sub"]] for c in calls]


@pytest.mark.parametrize("agent_name", ["duelingddqn", "td3_discrete_vary"])
def test_run_vary_hp_transfer_result_file_keeps_the_save_lists_format(monkeypatch, tmp_path, agent_name):
    calls = []
    monkeypatch.setattr(vary_hp, "_run_group", _stub(calls))
    model_dir = tmp_path / "models"
    model_dir.mkdir()
    for i, suffix in enumerate(("AAAAAA", "BBBBBB")):
        cfg = _vary_config("cartpole_syn_env")
        torch.manual_seed(i)
        venv = envs.EnvFactory(cfg).generate_virtual_env()
        torch.save({"model": venv.state_dict(), "config": cfg}, str(model_dir / ("CartPole-v0_%s.pt" % suffix)))
    f = vary_hp.run_vary_hp(mode=2, experiment_name="t", model_num=2, agents_num=3, model_dir=str(model_dir), env_name="CartPole",
                            device="cpu", out_dir=str(tmp_path), agent_name=agent_name)
    d = torch.load(f, weights_only=False)
    assert set(d) == {"config", "reward_list", "train_steps_needed", "episode_length_needed", "env_reward_overview"}
    assert len(d["reward_list"]) == 6 and len(d["train_steps_needed"]) == 6 and d["episode_length_needed"] == [[3]] * 6
    assert all(len(x) == 1 for x in d["train_steps_needed"]) and d["env_reward_overview"].shape == (2, 30)
    assert all(isinstance(x, Td3Cfg) == (agent_name == "td3_discrete_vary") for c in calls for x in c["sub"])
