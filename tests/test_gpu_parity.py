"""GPU parity tests: the CUDA path (through the C ABI) against (a) golden vectors produced by the UNMODIFIED
reference (tests/golden, oracle/gen_golden.py) and (b) the CPU restatement (oracle/le_oracle.c) on seeded inputs.

Tolerances (BASELINE.json north_star): SE/RN outputs and TD losses 1e-5 relative in fp32; replay indices,
Philox words and argmax actions bit-exact away from near-ties.
"""
import numpy as np
import pytest
import torch

from oracle import c_oracle, nes, philox
from tests.helpers import (assert_divergence_is_near_tie, assert_params_close, cfg_from_bytes, first_divergence, load_golden, param_index,
                           rel_err, sync_prefix)

pytestmark = pytest.mark.gpu
RTOL = 1e-5


@pytest.fixture(scope="module")
def ops():
    from learning_environments_b200 import ops as _ops
    assert _ops.version() == 100
    return _ops


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


@pytest.mark.parametrize("tag", ["cartpole", "acrobot", "cartpole_tanh", "cartpole_relu", "acrobot_identity", "acrobot_leaky"])
def test_se_forward_vs_reference_golden(ops, tag):
    g = load_golden("se_step_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    ns, r, d = ops.se_forward(cfg, dev(g["theta"])[None], dev(g["states"]), dev(g["actions"], torch.int32))
    assert rel_err(ns.cpu().numpy(), g["next_states"], 1e-2) < RTOL
    assert rel_err(r.cpu().numpy(), g["rewards"], 1e-2) < RTOL
    assert rel_err(d.cpu().numpy(), g["dones"], 1e-2) < RTOL


def test_se_forward_population_batched_vs_oracle(ops):
    """pop members x lanes: row r uses member r // lanes (the batched surface of SURVEY §8b)."""
    g = load_golden("se_step_cartpole.npz")
    cfg = cfg_from_bytes(g["cfg"])
    rng = np.random.RandomState(0)
    pop, lanes = 5, 7
    thetas = (g["theta"][None] + rng.standard_normal((pop, g["theta"].size)).astype(np.float32) * 0.05).astype(np.float32)
    states = rng.uniform(-1, 1, size=(pop * lanes, 4)).astype(np.float32)
    actions = rng.randint(0, 2, size=pop * lanes).astype(np.int32)
    ns, r, d = ops.se_forward(cfg, dev(thetas), dev(states), dev(actions), lanes_per_member=lanes)
    ns, r, d = ns.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()
    for i in range(pop * lanes):
        ons, orr, od = c_oracle.se_step(cfg, thetas[i // lanes], states[i], actions[i])
        assert rel_err(ns[i], ons, 1e-2) < RTOL and rel_err(r[i], orr, 1e-2) < RTOL and rel_err(d[i], od, 1e-2) < RTOL


def test_rn_reward_types_vs_reference_golden(ops):
    g = load_golden("rn_reward_cartpole.npz")
    cfg = cfg_from_bytes(g["cfg"])
    s, s2 = dev(g["s"], torch.float32), dev(g["s2"], torch.float32)
    rr = dev(g["real_reward"], torch.float32)
    for t in (0, 1, 2, 5, 6):
        cfg.rn_type = t
        out = ops.rn_reward(cfg, dev(g["theta"])[None], s, s2, rr)
        assert rel_err(out.cpu().numpy(), g["type%d" % t], 1e-2) < RTOL, t
    for t in (3, 4, 7, 8, 101, 102):
        cfg.rn_type = t
        with pytest.raises(ValueError):
            ops.rn_reward(cfg, dev(g["theta"])[None], s, s2, rr)


@pytest.mark.parametrize("tag", ["cartpole", "acrobot", "cartpole_rn", "cartpole_dueling", "acrobot_dueling", "cartpole_ddqn_l2",
                                 "acrobot_dueling_l3", "cartpole_ddqn_l3"])
def test_qnet_forward_argmax_vs_oracle(ops, tag):
    g = load_golden("td_update_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    rng = np.random.RandomState(1)
    n = 257 if cfg.q_is_register_resident() else 24
    P = cfg.q_params()
    thetas = (g["q_init"][None] + rng.standard_normal((n, P)).astype(np.float32) * 0.1).astype(np.float32)
    states = rng.uniform(-2, 2, size=(n, cfg.sd)).astype(np.float32)
    q, am = ops.qnet_forward(cfg, dev(thetas), dev(states))
    q, am = q.cpu().numpy(), am.cpu().numpy()
    for i in range(n):
        oq, oa = c_oracle.q_forward(cfg, thetas[i], states[i])
        assert rel_err(q[i], oq, 5e-2) < RTOL      # floor = scale of the summed terms (q values cancel to ~1e-2)
        srt = np.sort(oq)
        if srt[-1] - srt[-2] > 1e-5 * max(1.0, abs(srt[-1])):   # away from near-ties: bit-exact argmax
            assert am[i] == oa


@pytest.mark.parametrize("tag,kind", [("cartpole", 0), ("acrobot", 1)])
def test_real_env_step_vs_golden(ops, tag, kind):
    g = load_golden("real_env_%s.npz" % tag)
    sd = 4 if kind == 0 else 6
    max_steps = 200 if kind == 0 else 500
    for ep in range(int(g["n_episodes"])):
        states = g["ep%d_states" % ep]
        st = dev(states[:1].copy())
        el = torch.zeros(1, dtype=torch.int32, device="cuda")
        for t, a in enumerate(g["ep%d_actions" % ep]):
            obs, r, d = ops.real_env_step(kind, max_steps, st, el, dev(np.array([a], np.int32)), sd)
            got = st.cpu().numpy()[0]
            # fp64 dynamics: identical op order, only sin/cos implementations differ (<= 2 ulp each)
            assert np.allclose(got, states[t + 1], rtol=1e-12, atol=1e-13), (tag, ep, t)
            assert np.allclose(obs.cpu().numpy()[0], g["ep%d_obs" % ep][t + 1].astype(np.float32), rtol=2e-7, atol=1e-7)
            assert float(r) == np.float32(g["ep%d_rewards" % ep][t]) and bool(d.item()) == bool(g["ep%d_dones" % ep][t])
        assert int(el.item()) == len(g["ep%d_actions" % ep])


@pytest.mark.parametrize("tag", ["cartpole", "acrobot", "cartpole_rn", "cartpole_dueling", "acrobot_dueling", "cartpole_ddqn_l2",
                                 "acrobot_dueling_l3", "cartpole_ddqn_l3"])
def test_td_update_vs_reference_golden(ops, tag):
    g = load_golden("td_update_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    n = 3  # three identical lanes: also checks lane indexing
    th = dev(np.repeat(g["q_init"][None], n, 0))
    thT = th.clone()
    m = torch.zeros_like(th)
    v = torch.zeros_like(th)
    t = torch.zeros(n, dtype=torch.int32, device="cuda")
    idx = param_index(g)
    for k in range(g["rows"].shape[0]):
        rows = dev(np.repeat(g["rows"][k][None], n, 0))
        loss = ops.td_update(cfg, th, thT, m, v, t, rows).cpu().numpy()
        assert rel_err(loss, np.repeat(g["losses"][k], n)) < RTOL, (k, loss, g["losses"][k])
        for lane in range(n):
            assert_params_close(th[lane].cpu().numpy()[idx], g["thetas"][k], cfg.lr, "theta")
            assert_params_close(thT[lane].cpu().numpy()[idx], g["targets"][k], cfg.lr, "target")
    assert t.cpu().tolist() == [g["rows"].shape[0]] * n
    assert np.max(np.abs(m[0].cpu().numpy()[idx] - g["adam_m"])) < 1e-5 * max(1.0, np.abs(g["adam_m"]).max())
    assert np.max(np.abs(v[0].cpu().numpy()[idx] - g["adam_v"])) < 1e-5 * max(1.0, np.abs(g["adam_v"]).max())


def _run_fused(ops, cfg, env_theta, keys, q_init, trace_cap=0, n_env=1, env_index=None):
    n = len(keys)
    bufs = ops.InnerLoopBuffers(cfg, n, n_env, "cuda", trace_cap=trace_cap, want_q_final=True)
    th = None if env_theta is None else dev(np.asarray(env_theta, np.float32).reshape(n_env, -1))
    ei = None if env_index is None else dev(np.asarray(env_index, np.int32))
    ops.inner_loop_run(bufs, cfg, th, ei, ops.keys_tensor(keys, "cuda"), q_init=None if q_init is None else dev(q_init))
    torch.cuda.synchronize()
    return bufs


@pytest.mark.parametrize("tag", ["cartpole_se", "acrobot_se", "cartpole_rn", "cartpole_se_notest", "cartpole_se_dueling", "cartpole_se_k2",
                                 "cartpole_rn_k3", "cartpole_real_k2", "acrobot_real", "acrobot_se_dueling", "cartpole_se_ddqn_l2", "cartpole_se_ddqn_l3",
                                 "cartpole_se_h0", "cartpole_rn_t1", "cartpole_rn_t5", "cartpole_rn_t6", "cartpole_real_solved"])
@pytest.mark.parametrize("mw", ["0", "1"])
def test_fused_trajectory_lockstep_vs_reference_golden(ops, tag, mw, monkeypatch):
    """The fused persistent kernel, one lane, against the reference's own BaseAgent.train trace — on the warp-per-lane kernel
    (LE_MW=0) and on the multi-warp lane kernel a single lane would get by default (LE_MW=1; same kernel for the lanes of the
    general CTA-per-lane family, which has no multi-warp variant)."""
    monkeypatch.setenv("LE_MW", mw)
    g = load_golden("trajectory_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    key = [tuple(int(k) for k in g["key"])]
    cap = len(g["action"])
    bufs = _run_fused(ops, cfg, g["env_theta"], key, g["q_init"][None], trace_cap=cap)
    tr = {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in bufs.trace.items()}
    res = bufs.results()[0]
    n_sync = sync_prefix(g["action"], tr["action"])
    assert n_sync >= min(cap, 150), "kernel left the reference trajectory after %d steps" % n_sync
    if n_sync < min(cap, int(g["train_steps"]), int(res["train_steps"])):
        # the kernel may leave the reference's own trajectory only at a greedy near-tie (bound derived from this lane's drift)
        assert_divergence_is_near_tie({k: g[k] for k in ("action", "explore", "loss", "next_state", "done")}, tr, n_sync, tag)
    n = n_sync
    assert np.array_equal(tr["explore"][:n], g["explore"][:n])
    assert rel_err(tr["next_state"][:n], g["next_state"][:n], 1e-2) < 2e-4
    assert rel_err(tr["reward"][:n], g["reward"][:n], 1e-2) < 2e-4
    assert np.array_equal(np.isnan(tr["loss"][:n]), np.isnan(g["loss"][:n]))
    k = np.nonzero(~np.isnan(g["loss"][:n]))[0]
    assert rel_err(tr["loss"][k[:20]], g["loss"][k[:20]]) < RTOL      # TD losses: 1e-5 before drift is amplified
    assert rel_err(tr["loss"][k], g["loss"][k]) < 5e-3
    if n_sync == int(g["train_steps"]) == int(res["train_steps"]):
        assert int(res["n_episodes"]) == len(g["rewards"])
        assert np.array_equal(bufs.lengths.cpu().numpy()[0, :len(g["lengths"])], g["lengths"])
        assert np.allclose(bufs.rewards.cpu().numpy()[0, :len(g["rewards"])], g["rewards"], rtol=1e-4, atol=1e-4)
        assert np.allclose(bufs.test_rewards.cpu().numpy()[0], g["test_rewards"])


def test_multi_warp_lanes_deterministic_and_independent_of_scheduling(ops, monkeypatch):
    """Multi-warp lanes (one lane per CTA, the minibatch of every learn() split over the CTA's warps; selected when there are
    fewer lanes than SMs, forced here with LE_MW=1 so that 200 lanes queue on the CTAs): bit-identical across launches and
    independent of the lane queue; against the warp-per-lane kernel the integer bookkeeping of lanes that stay off near-ties
    agrees and the final Q-nets agree to fp32 reassociation."""
    g = load_golden("trajectory_cartpole_se.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 4, 5, 1
    n_env, n = 4, 200
    rng = np.random.RandomState(11)
    thetas = (g["env_theta"][None] + rng.standard_normal((n_env, g["env_theta"].size)).astype(np.float32) * 0.02).astype(np.float32)
    keys = [philox.lane_key(41, 1, i, i % 3, 0) for i in range(n)]
    env_index = (np.arange(n) % n_env).astype(np.int32)
    monkeypatch.setenv("LE_MW", "1")
    monkeypatch.setenv("LE_MWC", "0")      # one kernel family for the 200-lane run and its 37-lane subset (cluster lanes: below)
    r1, rew1, q1 = _full_size_run(ops, cfg, thetas, keys, env_index, n_env)
    r2, rew2, q2 = _full_size_run(ops, cfg, thetas, keys, env_index, n_env)
    sub = rng.permutation(n)[:37]
    r3, rew3, q3 = _full_size_run(ops, cfg, thetas, [keys[i] for i in sub], env_index[sub], n_env)
    for f in ("n_episodes", "train_steps", "learn_iters", "test_steps", "score"):
        assert np.array_equal(r1[f], r2[f]), f
        assert np.array_equal(r3[f], r1[f][sub]), f
    assert np.array_equal(rew1, rew2) and np.array_equal(q1, q2)
    assert np.array_equal(rew3, rew1[sub]) and np.array_equal(q3, q1[sub])
    # cluster lanes (one lane per thread-block cluster of two CTAs; at most 74 lanes): deterministic, independent of the lane set, and
    # against the single-CTA multi-warp lanes equal up to the order in which the participants' gradient sums are added
    monkeypatch.setenv("LE_MWC", "1")
    c1, crew1, cq1 = _full_size_run(ops, cfg, thetas, [keys[i] for i in sub], env_index[sub], n_env)
    c2, crew2, cq2 = _full_size_run(ops, cfg, thetas, [keys[i] for i in sub], env_index[sub], n_env)
    sub2 = np.arange(0, 37, 3)
    c3, crew3, cq3 = _full_size_run(ops, cfg, thetas, [keys[sub[i]] for i in sub2], env_index[sub][sub2], n_env)
    for f in ("n_episodes", "train_steps", "learn_iters", "test_steps", "score"):
        assert np.array_equal(c1[f], c2[f]), f
        assert np.array_equal(c3[f], c1[f][sub2]), f
    assert np.array_equal(cq1, cq2) and np.array_equal(cq3, cq1[sub2])
    csame = (c1["train_steps"] == r3["train_steps"]) & (c1["n_episodes"] == r3["n_episodes"])
    assert csame.mean() >= 0.8 and rel_err(cq1[csame], q3[csame]) < 5e-2
    monkeypatch.setenv("LE_MW", "0")
    r0, rew0, q0 = _full_size_run(ops, cfg, thetas, keys, env_index, n_env)
    same = (r0["train_steps"] == r1["train_steps"]) & (r0["n_episodes"] == r1["n_episodes"])
    assert same.mean() >= 0.8, same
    assert np.array_equal(r0["learn_iters"][same], r1["learn_iters"][same])
    assert rel_err(q1[same], q0[same]) < 5e-2      # four episodes of training amplify the last-bit differences of the gradient sums


def _assert_divergent_lanes_left_at_near_ties(ops, cfg, thetas, env_index, keys, res, oracle, limit=4):
    """Every lane whose bookkeeping differs from the CPU restatement is re-run ALONE with a full trace on both sides (a lane's
    result does not depend on its neighbours: test_full_size_population_is_deterministic...) and must have left the oracle at a
    near-tie (tests/helpers.assert_divergence_is_near_tie).  Returns the number of divergent lanes."""
    bad = np.nonzero((res["train_steps"] != oracle["train_steps"]) | (res["n_episodes"] != oracle["n_episodes"]))[0]
    thetas = None if thetas is None else np.asarray(thetas, np.float32).reshape(-1, cfg.env_params() if cfg.env_params() else 1)
    for i in bad[:limit]:
        th = None if thetas is None else thetas[0 if env_index is None else int(env_index[i])]
        cap = int(max(res["train_steps"][i], oracle["train_steps"][i]))
        b1 = _run_fused(ops, cfg, th, [keys[i]], None, trace_cap=cap)
        got = {k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in b1.trace.items()}
        assert int(b1.results()["train_steps"][0]) == int(res["train_steps"][i])        # alone == inside the population
        ref = c_oracle.run_lane(cfg, th, tuple(int(k) for k in keys[i]), trace_cap=cap)["trace"]
        n = int(min(res["train_steps"][i], oracle["train_steps"][i]))
        t = first_divergence(ref, got, n)
        if t < n:
            assert_divergence_is_near_tie(ref, got, t, "lane %d" % i)
        else:   # identical steps over the common length: the difference is in the episode bookkeeping after the last step
            assert np.allclose(np.asarray(ref.loss[:n])[~np.isnan(ref.loss[:n])], got["loss"][:n][~np.isnan(got["loss"][:n])], rtol=1e-3, atol=1e-6)
    return len(bad)


def test_fused_many_lanes_vs_oracle(ops):
    """64 lanes (8 SE members x 8 keys) through the lane queue; every lane vs the CPU restatement."""
    g = load_golden("trajectory_cartpole_se.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 3, 2, 1
    rng = np.random.RandomState(3)
    n_env, per = 8, 8
    thetas = (g["env_theta"][None] + rng.standard_normal((n_env, g["env_theta"].size)).astype(np.float32) * 0.02).astype(np.float32)
    keys = [philox.lane_key(7, 0, i // per, 0, i % per) for i in range(n_env * per)]
    env_index = np.arange(n_env * per, dtype=np.int32) // per
    bufs = _run_fused(ops, cfg, thetas, keys, None, n_env=n_env, env_index=env_index)
    res = bufs.results()
    oracle = c_oracle.run_lanes(cfg, thetas, env_index, np.array(keys, np.uint32), n_threads=8)
    # integer bookkeeping is exact while trajectories agree; a lane may leave the oracle only at a greedy near-tie
    same_steps = (res["train_steps"] == oracle["train_steps"])
    assert same_steps.mean() >= 0.8, same_steps
    _assert_divergent_lanes_left_at_near_ties(ops, cfg, thetas, env_index, keys, res, oracle)
    ok = same_steps & (res["n_episodes"] == oracle["n_episodes"])
    assert np.array_equal(res["learn_iters"][ok], oracle["learn_iters"][ok])
    assert np.allclose(res["score"][ok], oracle["score"][ok], atol=1e-9) or (np.isclose(res["score"][ok], oracle["score"][ok]).mean() > 0.8)
    # Philox-initialised Q-nets: first-episode (pre-learning) lengths depend only on init + SE + RNG -> exact
    assert np.array_equal(bufs.lengths.cpu().numpy()[:, 0], oracle["lengths"][:, 0])


def test_host_buffer_entry_matches_device_entry(ops):
    g = load_golden("trajectory_cartpole_se.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.train_episodes, cfg.test_episodes = 3, 2
    keys = [(11, 12), (13, 14), (15, 16), (17, 18), (19, 20)]
    bufs = _run_fused(ops, cfg, g["env_theta"], keys, None)
    dres = bufs.results()
    h = ops.inner_loop_run_host(cfg, g["env_theta"], None, keys, want_q_final=True)
    for f in ("n_episodes", "train_steps", "learn_iters", "test_steps", "score"):
        assert np.array_equal(h["out"][f], dres[f]), f
    assert np.array_equal(h["rewards"], bufs.rewards.cpu().numpy())
    assert np.array_equal(h["q_final"], bufs.q_final.cpu().numpy())     # same kernel, same order: bit-exact


def test_nes_noise_perturb_update(ops):
    P, pop, seed, gen, std = 2247, 16, 1234, 5, 0.0124
    eps = ops.nes_noise(P, 0, pop, seed, gen, std, "cuda").cpu().numpy()
    want = np.stack([nes.noise(seed, gen, i, P, std) for i in range(pop)])
    # Philox words are exact; Box-Muller runs in fp64 on both sides, libm log/sincos differ by <= 2 ulp(fp64):
    # after rounding to fp32 the normals agree to 1 ulp (almost always exactly)
    assert np.max(np.abs(eps - want) / np.maximum(np.abs(want), 1e-6)) < 2.5e-7
    assert (eps == want).mean() > 0.999
    sub = ops.nes_noise(P, 5, 3, seed, gen, std, "cuda").cpu().numpy()
    assert np.array_equal(sub, eps[5:8])                                  # member offset = sharding over ranks
    rng = np.random.RandomState(0)
    theta = rng.standard_normal(P).astype(np.float32) * 0.1
    pert = ops.nes_perturb(dev(theta), pop, 4, 6, seed, gen, std).cpu().numpy().reshape(6, 3, P)
    assert np.array_equal(pert[:, 0], np.repeat(theta[None], 6, 0))
    assert np.array_equal(pert[:, 1], theta[None] + eps[4:10]) and np.array_equal(pert[:, 2], theta[None] - eps[4:10])
    # update_env: device update with regenerated noise == numpy restatement fed the device's eps, bit-exact
    scores = rng.uniform(0, 200, size=pop)
    w = nes.score_transform(scores, scores * 0.5, 3)
    sign = np.where(rng.uniform(size=pop) < 0.5, -1.0, 1.0).astype(np.float32)
    for wd in (0.0, 0.01):
        coef = np.array([np.float32(0.148 * wi) for wi in w], np.float32)
        th = dev(theta.copy())
        ops.nes_update(th, pop, seed, gen, std, wd, dev(coef), dev(sign))
        want_th = nes.update_env(theta, eps * sign[:, None], w, 0.148, weight_decay=wd)
        assert np.array_equal(th.cpu().numpy(), want_th)
    # sharded partial sums (allreduce path) add up to the same update within fp32 reassociation
    parts = [ops.nes_partial_update(P, lo, lo + 4, seed, gen, std, dev(coef), dev(sign)).cpu().numpy() for lo in range(0, pop, 4)]
    full = nes.update_env(theta, eps * sign[:, None], w, 0.148) - theta
    assert np.allclose(sum(parts), full, rtol=1e-4, atol=1e-7)


def test_general_kernel_many_lanes_vs_oracle(ops):
    """DuelingDDQN lanes through the CTA-per-lane kernel and its lane queue, each vs the CPU restatement."""
    g = load_golden("trajectory_cartpole_se_dueling.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 2, 2, 1
    rng = np.random.RandomState(4)
    n_env, per = 3, 2
    thetas = (g["env_theta"][None] + rng.standard_normal((n_env, g["env_theta"].size)).astype(np.float32) * 0.02).astype(np.float32)
    keys = [philox.lane_key(9, 0, i // per, 0, i % per) for i in range(n_env * per)]
    env_index = np.arange(n_env * per, dtype=np.int32) // per
    bufs = _run_fused(ops, cfg, thetas, keys, None, n_env=n_env, env_index=env_index)
    res = bufs.results()
    oracle = c_oracle.run_lanes(cfg, thetas, env_index, np.array(keys, np.uint32), n_threads=6)
    assert np.array_equal(bufs.lengths.cpu().numpy()[:, 0], oracle["lengths"][:, 0])       # pre-learning episode: exact
    same = res["train_steps"] == oracle["train_steps"]
    assert same.mean() >= 0.6, (res["train_steps"], oracle["train_steps"])
    _assert_divergent_lanes_left_at_near_ties(ops, cfg, thetas, env_index, keys, res, oracle, limit=2)
    assert np.array_equal(res["learn_iters"][same], oracle["learn_iters"][same])


def test_wide_synthetic_env_h1024_scaling_sweep_shape(ops):
    """BASELINE config 5 shape: SE hidden width 1024 (27 654 parameters), many lanes per member."""
    g = load_golden("trajectory_cartpole_se.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.env_hidden = 1024
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 2, 2, 1
    P = cfg.se_params()
    assert P == 27654
    rng = np.random.RandomState(8)
    pop, lanes = 2, 6
    thetas = (rng.uniform(-1, 1, size=(pop, P)) * 0.05).astype(np.float32)
    states = rng.uniform(-1, 1, size=(pop * lanes, 4)).astype(np.float32)
    actions = rng.randint(0, 2, size=pop * lanes).astype(np.int32)
    ns, r, d = ops.se_forward(cfg, dev(thetas), dev(states), dev(actions), lanes_per_member=lanes)
    ns, r, d = ns.cpu().numpy(), r.cpu().numpy(), d.cpu().numpy()
    for i in range(pop * lanes):
        ons, orr, od = c_oracle.se_step(cfg, thetas[i // lanes], states[i], actions[i])
        assert rel_err(ns[i], ons, 1e-2) < RTOL and rel_err(r[i], orr, 1e-2) < RTOL and rel_err(d[i], od, 1e-2) < RTOL
    keys = [philox.lane_key(2, 0, i // lanes, 0, i % lanes) for i in range(pop * lanes)]
    env_index = np.arange(pop * lanes, dtype=np.int32) // lanes
    bufs = _run_fused(ops, cfg, thetas, keys, None, n_env=pop, env_index=env_index)
    res = bufs.results()
    oracle = c_oracle.run_lanes(cfg, thetas, env_index, np.array(keys, np.uint32), n_threads=6)
    assert np.array_equal(bufs.lengths.cpu().numpy()[:, 0], oracle["lengths"][:, 0])
    assert (res["train_steps"] == oracle["train_steps"]).mean() >= 0.75


def _edge_cfg(**over):
    g = load_golden("trajectory_cartpole_se.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 4, 3, 1
    for k, v in over.items():
        setattr(cfg, k, v)
    return cfg, g["env_theta"]


@pytest.mark.parametrize("name,over", [
    ("ring_wraps", dict(rb_size=37)),                         # replay ring smaller than the run: ptr wraps, size saturates
    ("tiny_batch", dict(batch_size=1)),                       # B = 1 (a chunk with 7 padded rows)
    ("odd_batch", dict(batch_size=67)),                       # B not a multiple of the 8-row chunk or the 64-row round
    ("big_batch", dict(batch_size=597)),                      # upper end of DDQN_vary's batch range: 10 gather rounds
    ("narrow_net", dict(q_hidden=19)),                        # fewer hidden units than lanes (masked units stay zero)
    ("relu", dict(q_act=1)),                                  # nn.ReLU Q-net
    ("leaky", dict(q_act=2)),
    ("many_test_episodes", dict(test_episodes=40)),           # more test episodes than threads in a warp: two passes
    ("step_budget", dict(step_budget=150)),                   # time_is_up analog: stops before an episode starts
    ("no_test_env", dict(use_test_env=0, early_out_num=1)),   # virtual-env plateau early-out rule
    ("init_only", dict(init_episodes=9)),                     # never learns: pure acting / replay filling
    ("solved_early_out", dict(solved_reward=5.0)),            # real-env early-out fires after the first learning episode
    ("same_action_3", dict(same_action_num=3)),               # EnvWrapper.step repeats the action (SE: chained steps, summed reward)
    ("same_action_odd", dict(same_action_num=7, max_steps=200)),   # max_steps not a multiple of same_action_num
])
def test_fused_edge_cases_vs_oracle(ops, name, over):
    cfg, theta = _edge_cfg(**over)
    keys = [philox.lane_key(21, 0, i, 0, 0) for i in range(6)]
    bufs = _run_fused(ops, cfg, theta, keys, None)
    res = bufs.results()
    oracle = c_oracle.run_lanes(cfg, theta, None, np.array(keys, np.uint32), n_threads=6)
    assert np.array_equal(bufs.lengths.cpu().numpy()[:, 0], oracle["lengths"][:, 0]), name       # pre-learning episode: exact
    same = (res["train_steps"] == oracle["train_steps"]) & (res["n_episodes"] == oracle["n_episodes"])
    assert same.mean() >= 0.66, (name, res["train_steps"], oracle["train_steps"])
    _assert_divergent_lanes_left_at_near_ties(ops, cfg, theta, None, keys, res, oracle, limit=2)
    assert np.array_equal(res["learn_iters"][same], oracle["learn_iters"][same]), name
    assert np.array_equal(res["timed_out"][same], oracle["timed_out"][same]), name
    assert np.array_equal(res["test_steps"][same], oracle["test_steps"][same]) or np.isclose(res["score"][same], oracle["score"][same]).mean() >= 0.6, name
    if name in ("step_budget", "init_only", "solved_early_out"):
        assert same.all(), name        # no learning-driven chaos before the stop: bookkeeping must be exact
        assert np.allclose(res["score"], oracle["score"]) or name == "step_budget"
    if name == "step_budget":
        assert res["timed_out"].all() and (res["train_steps"] >= 150).all()
    if name == "solved_early_out":
        assert (res["n_episodes"] == 2).all()


def test_general_kernel_edge_cases_vs_oracle(ops):
    g = load_golden("trajectory_cartpole_se_dueling.npz")
    for over in (dict(rb_size=41, batch_size=70), dict(test_episodes=70, train_episodes=2), dict(step_budget=120),
                 dict(q_kind=0, q_layers=2, q_hidden=150, q_feature_dim=0, q_act=1), dict(same_action_num=2)):
        cfg = cfg_from_bytes(g["cfg"])
        cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 3, 2, 1
        for k, v in over.items():
            setattr(cfg, k, v)
        keys = [philox.lane_key(22, 0, i, 0, 0) for i in range(3)]
        bufs = _run_fused(ops, cfg, g["env_theta"], keys, None)
        res = bufs.results()
        oracle = c_oracle.run_lanes(cfg, g["env_theta"], None, np.array(keys, np.uint32), n_threads=3)
        assert np.array_equal(bufs.lengths.cpu().numpy()[:, 0], oracle["lengths"][:, 0]), over
        same = res["train_steps"] == oracle["train_steps"]
        assert same.mean() >= 0.66, (over, res["train_steps"], oracle["train_steps"])
        assert np.array_equal(res["timed_out"], oracle["timed_out"]), over


# ---- BASELINE-size runs: properties that do not need the (slow) CPU restatement ---------------------------------------
def _full_size_run(ops, cfg, theta, keys, env_index=None, n_env=1):
    bufs = _run_fused(ops, cfg, theta, keys, None, n_env=n_env, env_index=env_index)
    res = bufs.results()
    return res, bufs.rewards.cpu().numpy(), bufs.q_final.cpu().numpy()


@pytest.mark.parametrize("tag", ["cartpole_se", "cartpole_se_dueling"])
def test_full_size_population_is_deterministic_and_independent_of_scheduling(ops, tag, monkeypatch):
    """bench.py's lane count (one full residency wave + a ragged second one) at the yaml batch size.  (1) the same launch
    twice is bit-identical; (2) a lane's result does not depend on which slot runs it, how many lanes share the GPU or
    the order of the lane queue (run a permuted subset alone); (3) every lane made progress and the bookkeeping is
    consistent (learn_iters = steps after the init episodes, episode lengths sum to train_steps).
    LE_MW=0 keeps the 53-lane subset on the warp-per-lane kernel of the full population (fewer lanes than SMs would otherwise
    select the multi-warp lanes, whose gradient summation order differs in the last bit); the multi-warp family has its own
    run of the same property below."""
    monkeypatch.setenv("LE_MW", "0")
    g = load_golden("trajectory_%s.npz" % tag)
    cfg = cfg_from_bytes(g["cfg"])
    dueling = tag.endswith("dueling")
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = (2, 3, 1) if dueling else (6, 10, 1)
    n_env = 8
    n = 148 * 2 + 37 if dueling else 148 * 8 * 2 + 101
    rng = np.random.RandomState(5)
    thetas = (g["env_theta"][None] + rng.standard_normal((n_env, g["env_theta"].size)).astype(np.float32) * 0.02).astype(np.float32)
    keys = [philox.lane_key(31, 2, i, i % 3, 0) for i in range(n)]
    env_index = (np.arange(n) % n_env).astype(np.int32)
    r1, rew1, q1 = _full_size_run(ops, cfg, thetas, keys, env_index, n_env)
    r2, rew2, q2 = _full_size_run(ops, cfg, thetas, keys, env_index, n_env)
    for f in ("n_episodes", "train_steps", "learn_iters", "test_steps", "score"):
        assert np.array_equal(r1[f], r2[f]), f
    assert np.array_equal(rew1, rew2) and np.array_equal(q1, q2)
    sub = rng.permutation(n)[:53]
    r3, rew3, q3 = _full_size_run(ops, cfg, thetas, [keys[i] for i in sub], env_index[sub], n_env)
    for f in ("n_episodes", "train_steps", "learn_iters", "test_steps", "score"):
        assert np.array_equal(r3[f], r1[f][sub]), f
    assert np.array_equal(rew3, rew1[sub]) and np.array_equal(q3, q1[sub])
    assert (r1["n_episodes"] >= 1).all() and (r1["train_steps"] >= r1["n_episodes"]).all()
    lengths = _run_fused(ops, cfg, thetas, [keys[i] for i in sub], None, n_env=n_env, env_index=env_index[sub]).lengths.cpu().numpy()
    assert np.array_equal(lengths.sum(1), r3["train_steps"])
    first = lengths[:, 0]
    assert np.array_equal(r3["learn_iters"], r3["train_steps"] - first)         # init_episodes = 1: every later step learns
    assert np.isfinite(q1).all() and np.isfinite(r1["score"]).all()


def test_full_size_mirrored_lanes_with_zero_noise_agree(ops):
    """NES mirrored sampling at sigma = 0: theta+eps and theta-eps are the same environment, so lanes that share a
    lane key must return the same score through different env slots (encode -> perturb -> evaluate round trip)."""
    g = load_golden("trajectory_cartpole_se.npz")
    cfg = cfg_from_bytes(g["cfg"])
    cfg.train_episodes, cfg.test_episodes, cfg.init_episodes = 4, 5, 1
    pop = 64
    theta = torch.from_numpy(g["env_theta"]).cuda()
    thetas = ops.nes_perturb(theta, pop, 0, pop, 77, 3, 0.0).reshape(pop, 3, -1)          # rows (theta, +eps, -eps), sigma = 0
    assert torch.equal(thetas[:, 0], thetas[:, 1]) and torch.equal(thetas[:, 0], thetas[:, 2])
    keys = [philox.lane_key(77, 3, m, 0, 0) for m in range(pop) for _ in range(3)]
    env_index = np.arange(pop * 3, dtype=np.int32)
    bufs = ops.InnerLoopBuffers(cfg, pop * 3, pop * 3, "cuda")
    ops.inner_loop_run(bufs, cfg, thetas.reshape(pop * 3, -1).contiguous(), dev(env_index), ops.keys_tensor(keys, "cuda"))
    torch.cuda.synchronize()
    sc = bufs.results()["score"].reshape(pop, 3)
    assert np.array_equal(sc[:, 0], sc[:, 1]) and np.array_equal(sc[:, 0], sc[:, 2])
    assert len(np.unique(sc[:, 0])) > 4           # different members (keys) do differ
