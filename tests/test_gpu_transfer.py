"""GPU tests of the batched transfer evaluations: heterogeneous vary_hp batches of DuelingDDQN_vary lanes (general CTA-per-lane
kernel) and TD3_discrete_vary lanes (le_td3_run) — each lane bit-identical to the same lane run alone, each lane against the CPU
restatement, and run_vary_hp end to end."""
import concurrent.futures as cf
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import c_oracle
from tests import td3_init_stream
from tests.helpers import assert_divergence_is_near_tie, first_divergence, rel_err, sync_prefix

pytestmark = pytest.mark.gpu

OVER = dict(print_rate=10, early_out_num=10, train_episodes=3, init_episodes=1, test_episodes=2, early_out_virtual_diff=0.01)
# smaller base shapes than the yaml (the sampled ranges are x1/3 .. x3 of these) keep the CPU restatement fast
SMALL = {"duelingddqn": dict(hidden_size=32, batch_size=32, feature_dim=24),
         "td3_discrete_vary": dict(hidden_size=48, batch_size=32, vary_hp=True)}
FAMILIES = ["duelingddqn", "td3_discrete_vary"]


def _ses(cfg, n_env=2):
    from learning_environments_b200 import envs
    thetas = []
    for i in range(n_env):
        torch.manual_seed(100 + i)
        _, th, fields = envs.EnvFactory(cfg).generate_virtual_env().kernel_env()
        thetas.append(th.numpy())
    return np.stack(thetas).astype(np.float32), fields.get("env_slope")


def _batch(agent_name, agents_num=8, seed=21, **over):
    from learning_environments_b200 import default_configs, vary_hp
    from learning_environments_b200.rng import lane_keys
    cfg = default_configs.get("cartpole_syn_env")
    thetas, slopes = _ses(cfg)
    n = 2 * agents_num
    cfgs = vary_hp.sample_agent_cfgs(cfg, n, np.random.RandomState(seed), dict(OVER, **SMALL[agent_name], **over), True, slopes, agent_name)
    env_of = np.arange(n) // agents_num
    keys = lane_keys(seed, 0, env_of, np.zeros(n, int), np.arange(n) % agents_num)
    return cfgs, thetas, env_of.astype(np.int32), keys


def _base(c):
    return c.base if hasattr(c, "base") else c


def _shape(c):
    b = _base(c)
    return (b.q_hidden, b.q_layers, b.batch_size, b.q_feature_dim)


def _run(agent_name, cfgs, thetas, env_index, keys, trace_cap=0, inits=None):
    from learning_environments_b200 import ops, vary_hp
    cfg0 = vary_hp._max_cfg(cfgs)
    n = len(cfgs)
    th, ei, k = torch.from_numpy(thetas).cuda(), torch.from_numpy(np.asarray(env_index, np.int32)).cuda(), ops.keys_tensor(keys, "cuda")
    if agent_name == "td3_discrete_vary":
        bufs = ops.Td3Buffers(cfg0, n, thetas.shape[0], "cuda", n_cfg=n, trace_cap=trace_cap, want_actor_final=True)
        ops.td3_run(bufs, cfgs, th, ei, k, inits=inits)
        final = bufs.actor_final
    else:
        bufs = ops.InnerLoopBuffers(cfg0, n, thetas.shape[0], "cuda", n_cfg=n, trace_cap=trace_cap, want_q_final=True)
        ops.inner_loop_run(bufs, cfgs, th, ei, k, cfg0=cfg0)
        final = bufs.q_final
    torch.cuda.synchronize()
    res = dict(out=bufs.results(), rewards=bufs.rewards.cpu().numpy(), lengths=bufs.lengths.cpu().numpy(),
               test_rewards=bufs.test_rewards.cpu().numpy(), final=final.cpu().numpy())
    if trace_cap:
        res["trace"] = {name: v.cpu().numpy() for name, v in bufs.trace.items() if name != "cap"}
    return res


def _alone(agent_name, cfgs, thetas, env_index, keys, i, trace_cap=0):
    return _run(agent_name, [cfgs[i]], thetas[int(env_index[i])][None], np.zeros(1, np.int32), keys[i:i + 1], trace_cap=trace_cap)


def _n_params(c):
    return c.param_counts()[0] if hasattr(c, "base") else c.q_params()


@pytest.mark.parametrize("agent_name", FAMILIES)
def test_transfer_batch_lanes_match_the_same_lane_alone(agent_name):
    cfgs, thetas, env_index, keys = _batch(agent_name)
    assert len({_shape(c) for c in cfgs}) >= 8 and len(set(env_index)) == 2
    res = _run(agent_name, cfgs, thetas, env_index, keys)
    for i in range(len(cfgs)):
        one = _alone(agent_name, cfgs, thetas, env_index, keys, i)
        for f in ("n_episodes", "train_steps", "learn_iters", "test_steps", "score"):
            assert res["out"][f][i] == one["out"][f][0], (i, f)
        n = int(one["out"]["n_episodes"][0])
        assert np.array_equal(res["rewards"][i, :n], one["rewards"][0, :n]) and np.array_equal(res["lengths"][i, :n], one["lengths"][0, :n])
        assert np.array_equal(res["test_rewards"][i], one["test_rewards"][0])
        P = _n_params(cfgs[i])
        assert np.array_equal(res["final"][i, :P], one["final"][0, :P]), "lane %d: trained parameters differ" % i


def _oracle_td3_cfg(t):
    o = c_oracle.Td3Cfg()
    C.memmove(C.byref(o), C.byref(t), C.sizeof(o))
    return o


def _td3_inits(t, key):
    b = t.base
    return td3_init_stream.td3_init(key, b.sd, b.ad, b.q_hidden, b.q_layers)


def _oracle(agent_name, c, theta, key, trace_cap=0):
    key = tuple(int(k) for k in key)
    if agent_name == "td3_discrete_vary":
        return c_oracle.run_lane_td3(_oracle_td3_cfg(c), theta, key, *_td3_inits(c, key), trace_cap=trace_cap)
    return c_oracle.run_lane(c, theta, key, trace_cap=trace_cap)


@pytest.mark.parametrize("agent_name", FAMILIES)
def test_transfer_batch_lanes_vs_cpu_restatement(agent_name):
    cfgs, thetas, env_index, keys = _batch(agent_name)
    res = _run(agent_name, cfgs, thetas, env_index, keys)
    n = len(cfgs)
    with cf.ThreadPoolExecutor(8) as ex:
        want = list(ex.map(lambda i: _oracle(agent_name, cfgs[i], thetas[env_index[i]], keys[i]), range(n)))
    ws = np.array([w["train_steps"] for w in want])
    we = np.array([w["n_episodes"] for w in want])
    same = (res["out"]["train_steps"] == ws) & (res["out"]["n_episodes"] == we)
    assert same.mean() >= 0.7, (res["out"]["train_steps"], ws)
    assert np.array_equal(res["lengths"][:, 0], np.array([w["lengths"][0] for w in want]))     # the random first episode: exact
    assert np.array_equal(res["out"]["learn_iters"][same], np.array([w["learn_iters"] for w in want])[same])
    for i in np.nonzero(~same)[0][:4]:          # a lane may leave the restatement only at a near-tie
        cap = int(max(res["out"]["train_steps"][i], ws[i]))
        got = _alone(agent_name, cfgs, thetas, env_index, keys, i, trace_cap=cap)["trace"]
        ref = _oracle(agent_name, cfgs[i], thetas[env_index[i]], keys[i], trace_cap=cap)["trace"]
        m = int(min(res["out"]["train_steps"][i], ws[i]))
        t = first_divergence(ref, got, m)
        if t < m:
            assert_divergence_is_near_tie(ref, got, t, "lane %d" % i)
        else:
            k = ~np.isnan(ref.loss[:m]) & ~np.isnan(got["loss"][:m])
            assert np.allclose(ref.loss[:m][k], got["loss"][:m][k], rtol=1e-3, atol=1e-6)


def test_td3_traced_lane_losses_vs_cpu_restatement():
    cfgs, thetas, env_index, keys = _batch("td3_discrete_vary")
    i = int(np.argmax([_base(c).batch_size for c in cfgs]))
    cap = 600
    got = _alone("td3_discrete_vary", cfgs, thetas, env_index, keys, i, trace_cap=cap)["trace"]
    ref = _oracle("td3_discrete_vary", cfgs[i], thetas[env_index[i]], keys[i], trace_cap=cap)["trace"]
    n = sync_prefix(ref.action, got["action"])
    k = np.nonzero(~np.isnan(ref.loss[:n]))[0]
    assert len(k) >= 20 and np.array_equal(np.isnan(got["loss"][:n]), np.isnan(ref.loss[:n]))
    assert rel_err(got["loss"][k[:20]], ref.loss[k[:20]]) < 1e-5


def test_td3_device_init_is_the_restated_stream():
    """No learn() call (train_episodes <= init_episodes): every lane returns its initial actor, which is the numpy restatement of
    P_TD3_INIT bit for bit; and a heterogeneous batch fed those weights as init arrays (rows of the maxima's stride) reproduces
    the device-initialised batch exactly."""
    cfgs, thetas, env_index, keys = _batch("td3_discrete_vary", agents_num=4, train_episodes=1)
    res = _run("td3_discrete_vary", cfgs, thetas, env_index, keys)
    assert (res["out"]["learn_iters"] == 0).all()
    inits = [_td3_inits(c, tuple(int(x) for x in keys[i])) for i, c in enumerate(cfgs)]
    for i, c in enumerate(cfgs):
        assert np.array_equal(res["final"][i, :c.param_counts()[0]], inits[i][0]), "lane %d" % i
    cfgs3, _, _, _ = _batch("td3_discrete_vary", agents_num=4)
    from learning_environments_b200 import vary_hp
    pa, pc = vary_hp._max_cfg(cfgs3).param_counts()
    rows = [np.zeros((len(cfgs3), p), np.float32) for p in (pa, pc, pc)]
    for i, c in enumerate(cfgs3):
        for r, v in zip(rows, _td3_inits(c, tuple(int(x) for x in keys[i]))):
            r[i, :v.size] = v
    dev = _run("td3_discrete_vary", cfgs3, thetas, env_index, keys)
    host = _run("td3_discrete_vary", cfgs3, thetas, env_index, keys, inits=tuple(torch.from_numpy(r).cuda() for r in rows))
    for f in ("n_episodes", "train_steps", "learn_iters", "score"):
        assert np.array_equal(dev["out"][f], host["out"][f]), f
    assert np.array_equal(dev["final"], host["final"]) and np.array_equal(dev["rewards"], host["rewards"])


@pytest.mark.parametrize("agent_name", FAMILIES)
def test_run_vary_hp_transfer_end_to_end(tmp_path, agent_name):
    from learning_environments_b200 import default_configs, envs, vary_hp
    model_dir = tmp_path / "models"
    model_dir.mkdir()
    for i, suffix in enumerate(("AAAAAA", "BBBBBB")):
        cfg = default_configs.get("cartpole_syn_env")
        cfg["agents"]["td3_discrete_vary"]["vary_hp"] = True
        torch.manual_seed(i)
        venv = envs.EnvFactory(cfg).generate_virtual_env()
        torch.save({"model": venv.state_dict(), "config": cfg}, str(model_dir / ("CartPole-v0_%s.pt" % suffix)))
    f = vary_hp.run_vary_hp(mode=2, experiment_name="tr", model_num=2, agents_num=3, model_dir=str(model_dir), env_name="CartPole",
                            out_dir=str(tmp_path), overrides=dict(OVER, **SMALL[agent_name]), agent_name=agent_name)
    d = torch.load(f, weights_only=False)
    assert set(d) == {"config", "reward_list", "train_steps_needed", "episode_length_needed", "env_reward_overview"}
    assert len(d["reward_list"]) == len(d["train_steps_needed"]) == len(d["episode_length_needed"]) == 6
    assert all(len(r) == 2 and all(1.0 <= x <= 200.0 for x in r) for r in d["reward_list"])
    assert all(s[0] > 0 for s in d["train_steps_needed"]) and all(1 <= e[0] <= 3 for e in d["episode_length_needed"])
