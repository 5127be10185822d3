"""Host-side logic of the drop-in API on CPU (no CUDA calls): config mapping, helpers, error behaviour,
GTN_Master with an oracle-backed evaluator, and the world_size-2 path over gloo."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from learning_environments_b200 import agents, config as le_config, default_configs, envs, gtn, nes, utils
from learning_environments_b200._abi import ENV_RN, ENV_SE, LaneCfg
from tests.helpers import cfg_from_bytes, load_golden
from tests.oracle_backend import OracleEvaluator, patch_master_for_cpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_default_configs_map_to_the_reference_lane_cfg():
    """default_configs + config.lane_cfg reproduce the le_lane_cfg generated from the reference's YAML files."""
    for tag, name, kind, over in (("cartpole_se", "cartpole_syn_env", ENV_SE, dict(train_episodes=5, test_episodes=3, init_episodes=1)),
                                  ("acrobot_se", "acrobot_syn_env", ENV_SE, dict(train_episodes=4, test_episodes=2, init_episodes=1)),
                                  ("cartpole_rn", "cartpole_reward_env", ENV_RN, dict(train_episodes=12, test_episodes=1, init_episodes=2))):
        g = load_golden("trajectory_%s.npz" % tag)
        want = cfg_from_bytes(g["cfg"])
        d = default_configs.get(name)
        d["agents"]["ddqn"].update(over)
        got = le_config.lane_cfg(d, "ddqn", kind, use_test_env=True, final_test=True)
        assert bytes(got) == bytes(want), tag


def test_lane_cfg_rejects_shapes_outside_the_kernel_set():
    d = default_configs.get("cartpole_syn_env")
    d["agents"]["ddqn"]["hidden_layer"] = 4          # DDQN_vary samples at most yaml hidden_layer + 1 = 3
    with pytest.raises(NotImplementedError):
        le_config.lane_cfg(d, "ddqn", ENV_SE)
    d["agents"]["ddqn"]["hidden_layer"] = 3
    assert le_config.lane_cfg(d, "ddqn", ENV_SE).q_layers == 3
    d["agents"]["ddqn"]["hidden_layer"] = 2          # two hidden layers: general (CTA-per-lane) kernel
    c2 = le_config.lane_cfg(d, "ddqn", ENV_SE)
    assert c2.q_layers == 2 and not c2.q_is_register_resident() and c2.q_params() == 57 * 5 + 57 * 58 + 2 * 58
    d = default_configs.get("cartpole_syn_env")
    d["env_name"] = "Pendulum-v0"
    d["envs"]["Pendulum-v0"] = d["envs"]["CartPole-v0"]
    with pytest.raises(NotImplementedError):
        le_config.lane_cfg(d, "ddqn", ENV_SE)


def test_env_factory_state_dict_keys_and_theta_roundtrip():
    f = envs.EnvFactory(default_configs.get("cartpole_syn_env"))
    v = f.generate_virtual_env()
    assert v.is_virtual_env() and v.get_state_dim() == 4 and v.get_action_dim() == 2 and v.max_episode_steps() == 200
    keys = sorted(v.state_dict().keys())
    assert keys == sorted("env.%s.%d.%s" % (n, i, p) for n in ("state_net", "reward_net", "done_net") for i in (0, 2)
                          for p in ("weight", "bias"))
    th = v.env.theta()
    assert th.numel() == 2247
    envs.set_linear_theta(v.env, th * 2)
    assert torch.equal(v.env.theta(), th * 2)
    r = envs.EnvFactory(default_configs.get("cartpole_reward_env")).generate_reward_env()
    assert not r.is_virtual_env() and r.env.theta().numel() == 385 and "env.reward_net.1.weight" in r.state_dict()
    a = envs.EnvFactory(default_configs.get("acrobot_syn_env")).generate_virtual_env()
    assert a.env.theta().numel() == 6354 and a.get_solved_reward() == -100.0
    for t in (3, 9):
        c = default_configs.get("cartpole_reward_env")
        c["envs"]["CartPole-v0"]["reward_env_type"] = t
        if t == 9:
            with pytest.raises(NotImplementedError):
                envs.EnvFactory(c).generate_reward_env()


def test_average_meter_and_one_hot_match_reference_semantics():
    m = utils.AverageMeter("x")
    for v in (1.0, 2.0, 3.0, 10.0):
        m.update(v, print_rate=10 ** 9)
    assert abs(m.get_mean(2) - 6.5 / (1 + 1e-9 / 2)) < 1e-6 and abs(m.get_mean_last(2) - 1.5) < 1e-6
    assert m.get_mean(10) == sum([1.0, 2.0, 3.0, 10.0]) / (4 + 1e-9)
    assert utils.to_one_hot_encoding(torch.tensor([1.0]), 3).tolist() == [0, 1, 0]
    assert utils.to_one_hot_encoding(torch.tensor([0.0, 2.0]), 3).tolist() == [[1, 0, 0], [0, 0, 1]]
    assert utils.from_one_hot_encoding(torch.tensor([0.0, 0.0, 1.0])).tolist() == [2]


def test_replay_buffer_ring_semantics():
    rb = utils.ReplayBuffer(state_dim=2, action_dim=1, device="cpu", max_size=5)
    for i in range(7):
        rb.add(torch.tensor([i, i], dtype=torch.float32), torch.tensor([i % 2]), torch.tensor([i + 1.0, i + 1.0]),
               torch.tensor(float(i)), torch.tensor(0.0))
    assert rb.size == 5 and rb.ptr == 2
    assert rb.state[:5, 0].tolist() == [5.0, 6.0, 2.0, 3.0, 4.0]      # rows 0,1 overwritten by transitions 5,6
    s, a, s2, r, d = rb.sample(64)
    assert s.shape == (64, 2) and set(r.reshape(-1).tolist()) <= {2.0, 3.0, 4.0, 5.0, 6.0}
    assert rb.get_all()[0].shape == (5, 2)


def test_replay_buffer_and_average_meter_against_the_reference_classes(golden_dir):
    """utils.ReplayBuffer and utils.AverageMeter against what the reference's classes return on the same seeded inputs
    (tests/golden/utils_semantics.npz, oracle/gen_golden.py): ptr / size after every add, get_all(), and get_mean(10) /
    get_mean_last(10) after every update, all exact."""
    g = np.load(os.path.join(golden_dir, "utils_semantics.npz"))
    a = utils.ReplayBuffer(3, 1, "cpu", max_size=int(g["rb_max_size"]))
    for r, want in zip(g["rb_inputs"], g["ptr_size"]):
        a.add(torch.from_numpy(r[0:3].copy()), torch.tensor([r[3]]), torch.from_numpy(r[4:7].copy()), torch.tensor([r[7]]),
              torch.tensor(r[8]))
        assert [a.ptr, a.size] == want.tolist()
    for x, k in zip(a.get_all(), ("state", "action", "next_state", "reward", "done")):
        assert torch.equal(x, torch.from_numpy(g["rb_" + k])), k
    m = utils.AverageMeter("")
    for v, want in zip(g["meter_inputs"], g["means"]):
        m.update(v, print_rate=10 ** 9)
        assert m.get_mean(10) == want[0] and m.get_mean_last(10) == want[1]


def test_vary_hyperparameters_ranges():
    base = default_configs.get("cartpole_syn_env")["agents"]["ddqn"]
    rng = np.random.RandomState(0)
    seen_layers = set()
    for _ in range(300):
        v = agents.vary_hyperparameters(base, rng)
        assert base["lr"] / 3 <= v["lr"] <= base["lr"] * 3
        assert int(199 / 3) <= v["batch_size"] <= 597 and int(57 / 3) <= v["hidden_size"] <= 171
        seen_layers.add(v["hidden_layer"])
    assert seen_layers == {0, 1, 2}


def test_select_agent_error_behaviour_without_gpu():
    cfg = default_configs.get("cartpole_syn_env")
    with pytest.raises(NotImplementedError, match="Unknownn RL agent"):
        agents.select_agent(cfg, "nonsense")
    with pytest.raises(NotImplementedError, match="outside the B200 hot path"):
        agents.select_agent(cfg, "TD3")
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA device is required"):      # fails loudly: no CPU fallback
            agents.select_agent(cfg, "DDQN")


def _small_gtn_config(workers=4, iters=2):
    cfg = default_configs.get("cartpole_syn_env")
    cfg["agents"]["gtn"].update(num_workers=workers, max_iterations=iters)
    cfg["agents"]["ddqn"].update(train_episodes=2, test_episodes=2, init_episodes=1)
    return cfg


def test_run_vary_hp_file_selection_and_result_format(tmp_path):
    """experiments/syn_env_run_vary_hp.py: checkpoint filtering by vary_hp flag, suffix ordering, save_lists result dict
    (per-model callback path; the one-launch path is covered on the GPU)."""
    import torch
    from learning_environments_b200 import vary_hp
    model_dir = tmp_path / "models"
    model_dir.mkdir()
    for i, (suffix, flag, env) in enumerate([("ZZZAAA", True, "CartPole-v0"), ("AAAZZZ", True, "CartPole-v0"), ("BBBBBB", False, "CartPole-v0"),
                                             ("CCCCCC", True, "Acrobot-v1")]):
        cfg = default_configs.get("cartpole_syn_env" if env == "CartPole-v0" else "acrobot_syn_env")
        cfg["agents"]["ddqn_vary"]["vary_hp"] = flag
        torch.manual_seed(i)
        venv = envs.EnvFactory(cfg).generate_virtual_env()
        torch.save({"model": venv.state_dict(), "config": cfg}, str(model_dir / ("%s_%s.pt" % (env, suffix))))
    calls = []

    def stub(train_env, test_env, config, agents_num):
        calls.append((train_env.is_virtual_env(), test_env.is_virtual_env(), float(train_env.env.theta().abs().sum()) if train_env.is_virtual_env() else 0.0))
        return [[1.0, 2.0]] * agents_num, [[10]] * agents_num, [[3]] * agents_num

    files = vary_hp.get_all_files(True, 2, str(model_dir), vary_hp.load_envs_and_config, "CartPole", "cpu")
    assert files == ["CartPole-v0_AAAZZZ.pt", "CartPole-v0_ZZZAAA.pt"]
    with pytest.raises(ValueError, match="Not enough saved models"):
        vary_hp.get_all_files(False, 2, str(model_dir), vary_hp.load_envs_and_config, "CartPole", "cpu")
    f = vary_hp.run_vary_hp(mode=2, experiment_name="x", model_num=2, agents_num=3, model_dir=str(model_dir),
                            custom_train_test_agents=stub, env_name="CartPole", device="cpu", out_dir=str(tmp_path))
    d = torch.load(f, weights_only=False)
    assert os.path.basename(f) == "2_x.pt" and set(d) == {"config", "reward_list", "train_steps_needed", "episode_length_needed",
                                                          "env_reward_overview"}
    assert len(d["reward_list"]) == 6 and d["train_steps_needed"] == [[10]] * 6 and d["episode_length_needed"] == [[3]] * 6
    assert list(d["env_reward_overview"].index) == files and d["env_reward_overview"].shape == (2, 6)
    assert [c[:2] for c in calls] == [(True, False)] * 2 and calls[0][2] != calls[1][2]     # the two checkpoints' own weights
    f1 = vary_hp.run_vary_hp(mode=1, experiment_name="x", model_num=1, agents_num=1, model_dir=str(model_dir),
                             custom_train_test_agents=stub, env_name="CartPole", device="cpu", out_dir=str(tmp_path))
    assert list(torch.load(f1, weights_only=False)["env_reward_overview"].index) == ["CartPole-v0_BBBBBB.pt"]
    f0 = vary_hp.run_vary_hp(mode=0, experiment_name="x", model_num=2, agents_num=1, model_dir=str(model_dir),
                             custom_train_test_agents=stub, env_name="CartPole", device="cpu", out_dir=str(tmp_path))
    d0 = torch.load(f0, weights_only=False)
    assert len(d0["reward_list"]) == 2 and calls[-1][:2] == (False, False)


def test_gtn_master_generation_logic_with_oracle_backend(monkeypatch, tmp_path):
    from oracle import nes as onese
    patch_master_for_cpu(monkeypatch)
    monkeypatch.chdir(tmp_path)
    torch.manual_seed(0)
    cfg = _small_gtn_config()
    m = gtn.GTN_Master(cfg, seed=77, evaluator_cls=OracleEvaluator, verbose=False)
    theta0 = m.theta.clone()
    mean_score, mean_list, model_name = m.run()                       # 3-tuple, as agents/GTN_master.py:114
    assert len(mean_list) == 2 and model_name.endswith(".pt") and np.isfinite(mean_score)
    assert not torch.equal(m.theta, theta0)
    assert torch.equal(envs.linear_theta(m.synthetic_env_orig.env), m.theta)     # the env object carries the new theta
    # replay generation 1's update by hand from the recorded scores
    w = onese.score_transform(m.score_list, m.score_orig_list, 3)
    assert np.array_equal(np.asarray(m.score_transform_list), w)
    assert all(s in (-1.0, 1.0) for s in m.sign_list)
    # checkpoint rule: SE models are saved only above solved_reward (195) -> nothing saved for random SEs
    assert not os.path.exists(model_name)
    m.best_score = -1e9
    m.real_env.env.solved_reward = -1e9
    assert m.save_good_model(10.0) is True and os.path.exists(model_name)
    ck = torch.load(model_name, weights_only=False)
    assert set(ck.keys()) == {"model", "config"} and "env.state_net.0.weight" in ck["model"]
    # a second run() continues the Philox generation counter (fresh perturbations and lane keys, not a replay of generations 0, 1)
    seen = []
    orig = m.evaluator.evaluate
    m.evaluator.evaluate = lambda theta, generation: (seen.append(generation), orig(theta, generation))[1]
    m.run()
    assert seen == [2, 3] and m.generation == 3


def test_gtn_master_unknown_options_raise_like_the_reference(monkeypatch, tmp_path):
    patch_master_for_cpu(monkeypatch)
    monkeypatch.chdir(tmp_path)
    cfg = _small_gtn_config()
    cfg["agents"]["gtn"]["synthetic_env_type"] = 2
    with pytest.raises(NotImplementedError, match="Unknown synthetic_env_type"):
        gtn.GTN_Master(cfg, evaluator_cls=OracleEvaluator, verbose=False)
    cfg = _small_gtn_config()
    cfg["agents"]["gtn"]["score_transform_type"] = 11
    m = gtn.GTN_Master(cfg, seed=1, evaluator_cls=OracleEvaluator, verbose=False)
    m.score_list, m.score_orig_list = [1.0, 2.0, 3.0, 4.0], [1.0] * 4
    with pytest.raises(ValueError, match="Unknown rank transform type"):
        m.score_transform()
    cfg = _small_gtn_config()
    cfg["agents"]["gtn"]["agent_name"] = "TD3_discrete_vary"
    with pytest.raises(NotImplementedError, match="outside the B200 hot path"):
        gtn.GTN_Master(cfg, evaluator_cls=OracleEvaluator, verbose=False)


@pytest.mark.parametrize("mode", ["replicated", "allreduce"])
def test_gtn_master_two_ranks_gloo_matches_single_rank(tmp_path, mode):
    """world_size 2 over gloo: block-sharded members, all-gather of scores, identical theta on both ranks and
    equal (replicated: bit-exact; allreduce: fp32 reassociation) to the single-process result."""
    script = os.path.join(ROOT, "tests", "gloo_gtn_worker.py")
    env = dict(os.environ, PYTHONPATH=ROOT)
    out1 = tmp_path / "single.npy"
    subprocess.check_call([sys.executable, script, "--mode", mode, "--out", str(out1)], env=env, cwd=str(tmp_path))
    out2 = tmp_path / "dist"
    port = 29000 + os.getpid() % 2000
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                           "127.0.0.1", "--master-port", str(port), script, "--mode", mode, "--out", str(out2)], env=env,
                          cwd=str(tmp_path), timeout=600)
    single = np.load(out1)
    r0, r1 = np.load(str(out2) + ".rank0.npy"), np.load(str(out2) + ".rank1.npy")
    assert np.array_equal(r0, r1)
    if mode == "replicated":
        assert np.array_equal(r0, single)
    else:
        assert np.allclose(r0, single, rtol=1e-5, atol=1e-7)


def test_vary_hp_two_ranks_gloo_matches_single_rank(tmp_path):
    """BASELINE config 4 sharding: world_size 2 over gloo, agents block-sharded (3 + 3 lanes), one all-reduce assembles
    the result table: both ranks return the single-process result, each having run only its own block."""
    import json
    script = os.path.join(ROOT, "tests", "gloo_vary_hp_worker.py")
    env = dict(os.environ, PYTHONPATH=ROOT)
    out1 = tmp_path / "single.json"
    subprocess.check_call([sys.executable, script, "--out", str(out1)], env=env, cwd=str(tmp_path))
    out2 = tmp_path / "dist"
    port = 31000 + os.getpid() % 2000
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                           "127.0.0.1", "--master-port", str(port), script, "--out", str(out2)], env=env, cwd=str(tmp_path),
                          timeout=600)
    single = json.load(open(out1))
    r0, r1 = json.load(open(str(out2) + ".rank0.json")), json.load(open(str(out2) + ".rank1.json"))
    assert single["lanes_run_here"] == 6 and r0["lanes_run_here"] == 3 and r1["lanes_run_here"] == 3
    for k in ("rewards", "steps", "episodes", "hidden"):
        assert r0[k] == single[k] and r1[k] == single[k], k
    assert len(single["rewards"]) == 2 and len(single["rewards"][0]) == 3 and len(single["rewards"][0][0]) == 2
    assert len(set(single["hidden"])) > 2          # per-lane hyper-parameters really vary


def test_bohb_level_sweep_space_mapping_and_objective(tmp_path, monkeypatch):
    """SURVEY §8(f) rank 3: the reference's third optimisation level (experiments/GTNC_evaluate_cartpole_params.py:16-118) on top
    of GTN_Master — configuration space bounds / defaults, the mapping onto the yaml config, the objective (total generations of
    the GTN runs; a failing configuration scores +inf with the traceback recorded) and one successive-halving bracket.
    GTN_Master runs on the oracle-backed evaluator (CPU) with tiny budgets."""
    from learning_environments_b200 import bohb_sweep as bs
    patch_master_for_cpu(monkeypatch)
    monkeypatch.chdir(tmp_path)
    ew = bs.ExperimentWrapper()
    assert ew.get_bohb_parameters() == {"min_budget": 1, "max_budget": 3, "eta": 3, "random_fraction": 0.3, "iterations": 10000}
    names = [s[0] for s in ew.get_configspace()]
    assert len(names) == 18 and names[0] == "gtn_score_transform_type" and names[-1] == "cartpole_hidden_layer"
    rng = np.random.RandomState(3)
    for _ in range(200):           # samples respect bounds and types
        c = bs.sample_configuration(rng)
        for name, kind, lo, hi, log, default in bs.SPACE:
            if kind == "cat":
                assert c[name] in lo
            else:
                assert lo <= c[name] <= hi and (kind != "int" or isinstance(c[name], int))
    d = bs.default_configuration()
    cfg = ew.get_specific_config(d, bs.default_cartpole_config(), 1)
    assert cfg["agents"]["ddqn"]["gamma"] == 1 - 0.01 and cfg["agents"]["ddqn"]["eps_decay"] == 1 - 0.1          # :64, :69
    assert cfg["agents"]["gtn"]["score_transform_type"] == 7 and cfg["envs"]["CartPole-v0"]["hidden_size"] == 128
    # tiny evaluation budget: 2 generations of 3 members, 2 training episodes per agent
    base = bs.default_cartpole_config()
    base["agents"]["gtn"].update(num_workers=3, max_iterations=2, quit_when_solved=False)
    base["agents"]["ddqn"].update(train_episodes=2, test_episodes=1)
    kw = dict(default_config=base, master_cls=gtn.GTN_Master, master_kwargs=dict(evaluator_cls=OracleEvaluator, verbose=False, seed=5))
    ok = dict(d, ddqn_hidden_layer=1, ddqn_hidden_size=48, ddqn_batch_size=64, cartpole_hidden_size=48, ddqn_init_episodes=1)
    r = ew.compute(str(tmp_path), 0, 0, ok, budget=3, **kw)
    assert r["loss"] == 3 * 2 and r["info"]["error"] == ""                # three GTN runs x max_iterations generations (:91-95)
    bad = dict(ok, cartpole_hidden_layer=2)                               # SE with two hidden layers: outside the kernel set
    r = ew.compute(str(tmp_path), 0, 1, bad, budget=1, **kw)
    assert r["loss"] == float("inf") and "NotImplementedError" in r["info"]["error"]
    res = bs.run_sweep(n_configs=3, seed=1, working_dir=str(tmp_path), default_config=base, master_cls=gtn.GTN_Master,
                       master_kwargs=kw["master_kwargs"])
    assert res[0]["budget"] >= res[-1]["budget"] and len(res) >= 3
    assert all(np.isfinite(x["loss"]) or x["info"]["error"] for x in res)
