"""Pins the CPU restatement (oracle/le_oracle.c) to golden vectors produced by the UNMODIFIED reference
(oracle/gen_golden.py).  Tolerances: fp32 outputs 1e-5 relative (BASELINE.json north_star); actions / replay
indices / explore flags bit-exact while the two trajectories are in sync (argmax near-ties excepted)."""
import numpy as np
import pytest

from oracle import c_oracle, philox
from tests.helpers import assert_params_close, cfg_from_bytes, load_golden, param_index, rel_err, sync_prefix

RTOL = 1e-5


@pytest.mark.parametrize("tag", ["cartpole", "acrobot", "cartpole_tanh", "cartpole_relu", "acrobot_identity", "acrobot_leaky"])
def test_se_step(tag):
    g = load_golden("se_step_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    assert g["theta"].size == cfg.se_params()
    for i in range(len(g["actions"])):
        ns, r, d = c_oracle.se_step(cfg, g["theta"], g["states"][i], g["actions"][i])
        # 1e-5 relative; floor 1e-2 = scale of the summands (outputs that cancel to ~1e-4 keep ~1e-8 abs error)
        assert rel_err(ns, g["next_states"][i], 1e-2) < RTOL
        assert rel_err(r, g["rewards"][i], 1e-2) < RTOL
        assert rel_err(d, g["dones"][i], 1e-2) < RTOL


def test_rn_reward_types():
    g = load_golden("rn_reward_cartpole.npz")
    cfg = cfg_from_bytes(g["cfg"])
    assert g["theta"].size == cfg.rn_params()
    for t in (0, 1, 2, 5, 6):
        cfg.rn_type = t
        for i in range(len(g["real_reward"])):
            s = g["s"][i].astype(np.float32)
            s2 = g["s2"][i].astype(np.float32)
            r = c_oracle.rn_reward(cfg, g["theta"], s, s2, np.float32(g["real_reward"][i]))
            assert rel_err(r, g["type%d" % t][i], 1e-2) < RTOL
    for t in (3, 4, 7, 8, 101, 102):   # info-vector types: the reference raises for CartPole (envs/reward_env.py:92)
        cfg.rn_type = t
        with pytest.raises(ValueError):
            c_oracle.rn_reward(cfg, g["theta"], g["s"][0], g["s2"][0], 1.0)


@pytest.mark.parametrize("tag", ["cartpole", "acrobot", "cartpole_rn", "cartpole_dueling", "acrobot_dueling", "cartpole_ddqn_l2",
                                 "acrobot_dueling_l3", "cartpole_ddqn_l3"])
def test_td_update(tag):
    g = load_golden("td_update_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    th = g["q_init"].copy()
    assert th.size == cfg.q_params()
    thT = th.copy()
    m = np.zeros_like(th)
    v = np.zeros_like(th)
    t = 0
    idx = param_index(g)
    for k in range(g["rows"].shape[0]):
        loss, t = c_oracle.td_update(cfg, th, thT, m, v, t, g["rows"][k])
        assert rel_err(loss, g["losses"][k]) < RTOL
        # parameters: 1e-5 relative to the parameter scale (Adam's m/sqrt(v) amplifies ulp noise of tiny gradients)
        assert_params_close(th[idx], g["thetas"][k], cfg.lr, "theta")
        assert_params_close(thT[idx], g["targets"][k], cfg.lr, "target")
    assert np.max(np.abs(m[idx] - g["adam_m"])) < 1e-5 * max(1.0, np.abs(g["adam_m"]).max())
    assert np.max(np.abs(v[idx] - g["adam_v"])) < 1e-5 * max(1.0, np.abs(g["adam_v"]).max())


@pytest.mark.parametrize("tag,stepfn", [("cartpole", 0), ("acrobot", 1)])
def test_real_env_dynamics(tag, stepfn):
    g = load_golden("real_env_%s.npz" % tag)
    sd = 4 if tag == "cartpole" else 6
    max_steps = 200 if tag == "cartpole" else 500
    for ep in range(int(g["n_episodes"])):
        st = g["ep%d_states" % ep][0].copy()
        el = 0
        for t, a in enumerate(g["ep%d_actions" % ep]):
            st, el, obs, r, d = c_oracle.real_step(stepfn, max_steps, st, el, a, sd)
            # same equations, same libm (glibc) as the python stand-in: bit-exact in float64
            assert np.array_equal(st, g["ep%d_states" % ep][t + 1]), (tag, ep, t)
            assert np.array_equal(obs, g["ep%d_obs" % ep][t + 1].astype(np.float32))
            assert r == np.float32(g["ep%d_rewards" % ep][t]) and bool(d) == bool(g["ep%d_dones" % ep][t])


@pytest.mark.parametrize("tag", ["cartpole_se", "acrobot_se", "cartpole_rn", "cartpole_se_notest", "cartpole_se_dueling", "cartpole_se_k2",
                                 "cartpole_rn_k3", "cartpole_real_k2", "acrobot_real", "acrobot_se_dueling", "cartpole_se_ddqn_l2", "cartpole_se_ddqn_l3",
                                 "cartpole_se_h0", "cartpole_rn_t1", "cartpole_rn_t5", "cartpole_rn_t6", "cartpole_real_solved"])
def test_trajectory_lockstep(tag):
    g = load_golden("trajectory_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    key = tuple(int(k) for k in g["key"])
    cap = len(g["action"])
    res = c_oracle.run_lane(cfg, g["env_theta"], key, q_init_w=g["q_init"], trace_cap=cap)
    tr = res["trace"]
    # first replay sample: integer-exact
    if g["sample0"].size and np.any(~np.isnan(g["loss"])):
        first_learn = int(np.nonzero(~np.isnan(g["loss"]))[0][0])
        size_then = first_learn + 1
        assert np.array_equal(philox.sample_indices(key, 0, cfg.batch_size, size_then), g["sample0"])
    n_sync = sync_prefix(g["action"], tr.action)
    # trajectories are chaotic: demand lock-step for a long prefix, exactness inside it
    assert n_sync >= min(cap, 150), "oracle left the reference trajectory after %d steps" % n_sync
    n = n_sync
    assert np.array_equal(tr.explore[:n], g["explore"][:n])
    assert rel_err(tr.next_state[:n], g["next_state"][:n], 1e-3) < 2e-4
    assert rel_err(tr.reward[:n], g["reward"][:n], 1e-3) < 2e-4
    assert np.array_equal(np.isnan(tr.loss[:n]), np.isnan(g["loss"][:n]))
    k = ~np.isnan(g["loss"][:n])
    # early losses (before fp32 drift is amplified by training) within 1e-5
    early = np.nonzero(k)[0][:20]
    assert rel_err(tr.loss[early], g["loss"][early]) < RTOL
    assert rel_err(tr.loss[:n][k], g["loss"][:n][k]) < 5e-3
    if n_sync == int(g["train_steps"]) == res["train_steps"]:   # whole run traced and in lock-step
        assert np.array_equal(res["lengths"], g["lengths"])
        assert np.allclose(res["rewards"], g["rewards"], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("tag", ["cartpole", "cartpole_soft", "acrobot"])
def test_td3_discrete_learn_restatement_vs_reference_golden(tag):
    """SURVEY §8(f) rank 2: TD3_discrete_vary.learn (agents/TD3_discrete_vary.py:62-119: Gumbel-softmax actor, twin critics,
    delayed policy update) restated in C and held to learn() calls of the unmodified reference — hard and soft Gumbel-softmax,
    tanh / relu / leakyrelu nets, one and two hidden layers, policy_delay 1 / 2 / 3, CartPole and Acrobot shapes."""
    g = load_golden("td3_learn_%s.npz" % tag)
    names = ("actor", "actor_target", "critic_1", "critic_target_1", "critic_2", "critic_target_2")
    nets = {n: g["init_" + n].astype(np.float32).copy() for n in names}
    Pa, Pc = nets["actor"].size, nets["critic_1"].size
    adam = dict(m_a=np.zeros(Pa, np.float32), v_a=np.zeros(Pa, np.float32), m_c1=np.zeros(Pc, np.float32), v_c1=np.zeros(Pc, np.float32),
                m_c2=np.zeros(Pc, np.float32), v_c2=np.zeros(Pc, np.float32))
    hyper = dict(gamma=float(g["gamma"]), tau=float(g["tau"]), lr=float(g["lr"]), policy_delay=int(g["policy_delay"]),
                 max_action=float(g["max_action"]), policy_std=float(g["policy_std"]), policy_std_clip=float(g["policy_std_clip"]),
                 gumbel_hard=int(g["gumbel_hard"]))
    dims = (int(g["sd"]), int(g["ad"]), int(g["hidden"]), int(g["layers"]), int(g["act"]))
    counters = [0, 0]
    for k in range(len(g["temps"])):
        closs, aloss = c_oracle.td3_learn(dims, hyper, nets, adam, counters, k + 1, g["rows"][k], g["policy_noise"][k],
                                          g["expo_target"][k], g["expo_actor"][k], float(g["temps"][k]))
        assert np.isfinite(closs) and (np.isfinite(aloss) == bool(g["updated"][k]))
        for n in names:
            err = np.abs(nets[n] - g["after_" + n][k]).max()      # weights move by ~lr = 1.7e-3 per step; observed error ~1 ulp
            assert err < 1e-6, (tag, k, n, err)
    assert counters == [int(g["updated"].sum()), len(g["temps"])]


@pytest.mark.parametrize("tag", ["cartpole_se", "acrobot_se", "cartpole_real"])
def test_td3_discrete_trajectory_lockstep_vs_reference_golden(tag):
    """SURVEY §8(f) rank 2: the whole TD3_discrete_vary lane (BaseAgent.train with per-episode test() + final test(),
    Gumbel-softmax acting, learn()) restated in C, in lock-step with the unmodified reference under RNG injection:
    CartPole SE (tanh, 2 hidden layers), Acrobot SE (relu, 1 hidden layer, policy_delay 1), training on the real CartPole
    with same_action_num 2."""
    import json
    g = load_golden("trajectory_td3_%s.npz" % tag)
    base = cfg_from_bytes(g["cfg"])
    tcfg = c_oracle.td3_cfg(base, json.loads(str(g["agent_cfg_json"])), float(g["max_action"]))
    key = tuple(int(k) for k in g["key"])
    cap = len(g["action"])
    res = c_oracle.run_lane_td3(tcfg, g["env_theta"] if base.env_kind == 0 else None, key, g["init_actor"], g["init_critic_1"],
                                g["init_critic_2"], trace_cap=cap)
    tr = res["trace"]
    n = sync_prefix(g["action"], tr.action)
    assert n >= min(cap, 300), "restatement left the reference trajectory after %d steps" % n
    assert rel_err(tr.next_state[:n], g["next_state"][:n], 1e-3) < 2e-4
    assert rel_err(tr.reward[:n], g["reward"][:n], 1e-3) < 2e-4
    assert np.array_equal(tr.done[:n] > 0.5, g["done"][:n] > 0.5)
    if n == int(g["train_steps"]) == res["train_steps"]:
        assert np.array_equal(res["lengths"], g["lengths"])
        assert np.allclose(res["rewards"], g["rewards"]) and np.allclose(res["test_rewards"], g["test_rewards"])
        assert res["learn_iters"] == int(g["learn_iters"])
        assert np.abs(res["actor_final"] - g["actor_final"]).max() < 1e-4      # observed <= 1e-5 after up to 600 learn() calls
