"""Transfer-evaluation throughput: N agents of one family trained on ONE fixed SE in one batched call
(vary_hp.evaluate_agents(agent_name=...)) against the per-agent route select_agent -> train -> test.

    python tools/bench_transfer.py [--agents 296] [--seq-agents 3] [--train-episodes 3] [--init-episodes 1]

Prints one JSON line per (agent family, yaml): DuelingDDQN_vary on cartpole_syn_env and acrobot_syn_env, TD3_discrete_vary on
cartpole_syn_env.  The SE is seeded (torch.manual_seed(0)); agents use the yaml section with vary_hp.OVERRIDES, sampled
hyper-parameters (the vary_hp flags set), --train-episodes and --init-episodes (OVERRIDES' 10 random
episodes would leave a short run without any learn() call).  Batched: env steps / s over device time (CUDA events around
the whole call) and wall time per agent.  Per-agent route: wall time per agent (train on the SE, test on the real env).
The card's name and power limit are read in the same run.  Writes nothing.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from learning_environments_b200 import agents, default_configs, envs, vary_hp  # noqa: E402

CASES = [("duelingddqn", "cartpole_syn_env", "duelingddqn_vary"), ("duelingddqn", "acrobot_syn_env", "duelingddqn_vary"),
         ("td3_discrete_vary", "cartpole_syn_env", "td3_discrete_vary")]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.splitlines()[torch.cuda.current_device()].split(",")]
    return name, power


def setup(yaml, agent_name, train_episodes, init_episodes):
    cfg = default_configs.get(yaml)
    cfg["device"] = "cuda"
    cfg["agents"]["td3_discrete_vary"]["vary_hp"] = True
    torch.manual_seed(0)
    venv = envs.EnvFactory(cfg).generate_virtual_env()
    _, theta, fields = venv.kernel_env()
    over = dict(vary_hp.OVERRIDES, train_episodes=train_episodes, init_episodes=init_episodes)
    return cfg, venv, theta.numpy()[None], fields.get("env_slope"), over


def batched(cfg, theta, slopes, over, agent_name, n):
    vary_hp.evaluate_agents(cfg, theta, min(n, 8), seed=1, overrides=over, env_slopes=slopes, agent_name=agent_name)   # warm-up
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    _, steps, _, _ = vary_hp.evaluate_agents(cfg, theta, n, seed=0, overrides=over, env_slopes=slopes, agent_name=agent_name)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return sum(steps[0]) / (e0.elapsed_time(e1) * 1e-3), wall / n, e0.elapsed_time(e1) * 1e-3


def sequential(cfg, venv, over, agent_name, vary_name, n):
    c = dict(cfg, agents=dict(cfg["agents"]))
    c["agents"][agent_name] = dict(cfg["agents"][agent_name], **over)
    real = envs.EnvFactory(c).generate_real_env()
    walls = []
    for _ in range(n):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):      # the *_vary constructors print their sampled config
            agent = agents.select_agent(c, vary_name)
        agent.train(env=venv)
        agent.test(env=real)
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    return float(np.mean(walls))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=296)
    ap.add_argument("--seq-agents", type=int, default=3)
    ap.add_argument("--train-episodes", type=int, default=3)
    ap.add_argument("--init-episodes", type=int, default=1)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_transfer.py measures on a CUDA device"
    name, power = card()
    for agent_name, yaml, vary_name in CASES:
        cfg, venv, theta, slopes, over = setup(yaml, agent_name, args.train_episodes, args.init_episodes)
        sps, wall_b, dev_s = batched(cfg, theta, slopes, over, agent_name, args.agents)
        wall_s = sequential(cfg, venv, over, agent_name, vary_name, args.seq_agents)
        print(json.dumps(dict(family=vary_name, yaml=yaml, agents=args.agents, train_episodes=args.train_episodes, init_episodes=args.init_episodes,
                              batched_env_steps_per_s=round(sps, 1), batched_device_s=round(dev_s, 3),
                              batched_wall_s_per_agent=round(wall_b, 5), seq_agents=args.seq_agents,
                              sequential_wall_s_per_agent=round(wall_s, 4), speedup_per_agent=round(wall_s / wall_b, 1),
                              card=name, power_limit=power)), flush=True)


if __name__ == "__main__":
    main()
