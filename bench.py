#!/usr/bin/env python
"""bench.py — SE env-steps/s of the NES inner loop (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--extras all|none]
                    [--scaling weak|strong] [--population P] [--dump-outputs DIR]

One "step" = one NES generation's population evaluation over one batch of synthetic input: every member's SE is
perturbed from the Philox stream (theta, theta+eps, theta-eps) and every resulting lane runs a complete, bounded
calc_score (agents/GTN_worker.py:187-221: DDQN train() with per-episode test() on the real env, then the final
test()) inside the persistent fused kernel; with N > 1 ranks members are sharded (weak scaling, no data-path
collective) and the generation ends with the all-gather of fitness scores + the NES update on every rank.

value  = training env-steps of all lanes of all ranks / device time (CUDA events, max over ranks), inputs resident in HBM
e2e    = the same through PopulationEvaluator.evaluate() with HOST theta: H2D of theta/keys and D2H of lane results inside
roofline.achieved = F_step (SURVEY.md §8d algorithmic flop per inner-loop step) x steps / fused-kernel time
with_update       = the same generation timed on the device INCLUDING the score all-gather (NCCL) + score transform + NES update
workloads         = (default run, headline workload) every other named workload timed for 2-3 steps in the same process:
                    acrobot_se, cartpole_rn, both DuelingDDQN workloads, sweep_h1024, vary_hp, the full-size-ring regime
strong_scaling    = (default run) a FIXED population of 8 x 1184 members split over the ranks (scaling: strong)
cpu_baseline      = the UNMODIFIED reference (oracle/_ref/pyref, staged by oracle/make_ref.py; kind "reference") on all host
                    cores, one single-thread worker process per core; the C restatement (kind "port") is kept as a 2nd figure
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# workload name -> (default_configs name, env kind, members per GPU, bounded train_episodes)
WORKLOADS = {
    "cartpole_se": dict(cfg="cartpole_syn_env", kind="se", members_per_gpu=1184, train_episodes=10),
    "acrobot_se": dict(cfg="acrobot_syn_env", kind="se", members_per_gpu=1184, train_episodes=3, init_episodes=1),
    "cartpole_rn": dict(cfg="cartpole_reward_env", kind="rn", members_per_gpu=1184, train_episodes=40),
    # BASELINE config 5 (scaling sweep): SE hidden width 1024, 257 lanes per member (theta + 128 x (+eps, -eps) evaluations);
    # 64 members per GPU = population 512 x 256 envs on 8 GPUs
    "sweep_h1024": dict(cfg="cartpole_syn_env", kind="se", members_per_gpu=64, train_episodes=2, env_hidden=1024, grad_evals=128),
    # DuelingDDQN inner loops (general CTA-per-lane kernel): CartPole yaml section, Acrobot section of default_config_acrobot.yaml
    "cartpole_se_dueling": dict(cfg="cartpole_syn_env", kind="se", agent="duelingddqn", members_per_gpu=296, train_episodes=3),
    # 197 members x 3 lanes = 591 lanes = two full waves of the 296 resident CTAs
    "acrobot_se_dueling": dict(cfg="acrobot_syn_env", kind="se", agent="duelingddqn", members_per_gpu=197, train_episodes=2, init_episodes=1),
    # the same with the dense hidden x hidden layers on the tcgen05 tensor cores (LE_TC=1: 3xTF32, TMEM accumulators, one CTA per SM)
    "acrobot_se_dueling_tc": dict(cfg="acrobot_syn_env", kind="se", agent="duelingddqn", members_per_gpu=197, train_episodes=2, init_episodes=1, tc=True),
    # BASELINE config 4 (vary_hp evaluation): 4096 DDQN agents per GPU with per-lane lr / batch_size / hidden_size / hidden_layer
    # on ONE fixed CartPole SE, init_episodes=10, plateau early-out; train_episodes bounded (the evaluator's cap is 1000)
    "vary_hp": dict(cfg="cartpole_syn_env", kind="se", members_per_gpu=4096, train_episodes=30),
    # the yaml's replay regime: rb_size 100 000 and a step budget large enough that the rings of all resident slots total > 4 GB
    # (50 200 rows x 48 B x 1776 slots): the random 48-byte gathers come from HBM, not from the 126 MB L2
    "cartpole_se_fullring": dict(cfg="cartpole_syn_env", kind="se", members_per_gpu=1184, train_episodes=500, step_budget=50000),
    # BASELINE config 1 as the reference runs it: the yaml's population of 16 members (48 lanes on 1184+ resident warp slots):
    # latency of ONE small generation, directly comparable with cpu_baseline.nes_generations_per_hour_pop16
    "cartpole_se_pop16": dict(cfg="cartpole_syn_env", kind="se", members_per_gpu=16, train_episodes=10),
}
# (f)2: TD3_discrete_vary lanes (le_td3.cu, CTA-per-lane) on the CartPole SE with the yaml's td3_discrete_vary section; host-buffer entry
TD3_WORKLOAD = dict(cfg="cartpole_syn_env", lanes_per_gpu=296, train_episodes=3, init_episodes=1)
EXTRA_WORKLOADS = ["acrobot_se", "cartpole_rn", "cartpole_se_dueling", "acrobot_se_dueling", "acrobot_se_dueling_tc", "sweep_h1024",
                   "cartpole_se_fullring", "cartpole_se_pop16", "vary_hp"]
STRONG_POPULATION = 8 * 1184


def build_lane_cfg(workload):
    from learning_environments_b200 import config, default_configs
    from learning_environments_b200._abi import ENV_RN, ENV_SE
    w = WORKLOADS[workload]
    d = default_configs.get(w["cfg"])
    name = w.get("agent", "ddqn")
    agent = d["agents"][name]
    agent["train_episodes"] = w["train_episodes"]
    if "init_episodes" in w:
        agent["init_episodes"] = w["init_episodes"]
    if "env_hidden" in w:
        d["envs"][d["env_name"]]["hidden_size"] = w["env_hidden"]
    if "grad_evals" in w:
        d["agents"]["gtn"]["num_grad_evals"] = w["grad_evals"]
    cfg = config.lane_cfg(d, name, ENV_SE if w["kind"] == "se" else ENV_RN, use_test_env=True, final_test=True)
    if "step_budget" in w:
        cfg.step_budget = w["step_budget"]
    return d, cfg


def f_parts(cfg):
    """(flop per env step without learning, flop per TD update): F_env + F_q and 5*B*F_q (SURVEY.md §8d)."""
    from learning_environments_b200._abi import ENV_SE, ENV_RN
    fq = 2 * sum(i * o for i, o in cfg.q_layer_dims())
    if cfg.env_kind == ENV_SE:
        i, h = cfg.sd + cfg.ad, cfg.env_hidden
        fenv = 2 * (3 * i * h + h * (cfg.sd + 2))
    elif cfg.env_kind == ENV_RN:
        fenv = 2 * 2 * (cfg.sd * cfg.env_hidden + cfg.env_hidden)
    else:
        fenv = 0
    return fenv + fq, 5 * cfg.batch_size * fq


def f_step(cfg):
    """Algorithmic flop per inner-loop step (SURVEY.md §8d): F_env + F_q + 5*B*F_q, F_mlp = sum 2*in*out."""
    from learning_environments_b200._abi import ENV_SE, ENV_RN
    fq = 2 * sum(i * o for i, o in cfg.q_layer_dims())
    if cfg.env_kind == ENV_SE:
        i, h = cfg.sd + cfg.ad, cfg.env_hidden
        fenv = 2 * (3 * i * h + h * (cfg.sd + 2))
    elif cfg.env_kind == ENV_RN:
        fenv = 2 * 2 * (cfg.sd * cfg.env_hidden + cfg.env_hidden)
    else:
        fenv = 0
    return fenv + fq + 5 * cfg.batch_size * fq


def synthetic_theta(cfg, seed=0):
    """torch-default-init-like parameter vector of the SE / RN (U(+-1/sqrt(fan_in)) per layer), seeded."""
    from learning_environments_b200._abi import ENV_SE
    rng = np.random.RandomState(seed)
    parts = []
    if cfg.env_kind == ENV_SE:
        i, h = cfg.sd + cfg.ad, cfg.env_hidden
        for out in (cfg.sd, 1, 1):
            parts += [rng.uniform(-1, 1, h * i) / np.sqrt(i), rng.uniform(-1, 1, h) / np.sqrt(i),
                      rng.uniform(-1, 1, out * h) / np.sqrt(h), rng.uniform(-1, 1, out) / np.sqrt(h)]
    else:
        i, h = cfg.sd, cfg.env_hidden
        parts += [rng.uniform(-1, 1, h * i) / np.sqrt(i), rng.uniform(-1, 1, h) / np.sqrt(i),
                  rng.uniform(-1, 1, h) / np.sqrt(h), rng.uniform(-1, 1, 1) / np.sqrt(h)]
    return np.concatenate(parts).astype(np.float32)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU during the timed region (pynvml)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        while self.nv is not None and not self._halt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_port_baseline(cfg, theta, target_seconds, n_threads):
    """Times the C restatement (oracle/) on a bounded sample of the same workload: `n` lanes on n_threads threads."""
    from oracle import c_oracle, philox
    c_oracle.build()
    keys1 = np.array([philox.lane_key(99, 0, 0, 0, 0)], np.uint32)
    t0 = time.perf_counter()
    r1 = c_oracle.run_lanes(cfg, theta, None, keys1, n_threads=1)
    t1 = max(time.perf_counter() - t0, 1e-4)
    n = int(max(n_threads, min(4096, n_threads * target_seconds / t1)))
    keys = np.array([philox.lane_key(99, 0, i, 0, 0) for i in range(n)], np.uint32)
    t0 = time.perf_counter()
    r = c_oracle.run_lanes(cfg, theta, None, keys, n_threads=n_threads)
    dt = time.perf_counter() - t0
    steps = int(r["train_steps"].sum())
    return steps / dt, dict(lanes=n, steps=steps, seconds=dt, single_lane_seconds=t1, single_lane_steps=int(r1["train_steps"][0]))


def reference_spec(workload):
    """What oracle/ref_bench.py needs to run the UNMODIFIED reference on the lane configuration of `workload`."""
    w = WORKLOADS[workload]
    yaml_name = {"cartpole_syn_env": "default_config_cartpole_syn_env.yaml", "acrobot_syn_env": "default_config_acrobot_syn_env.yaml",
                 "cartpole_reward_env": "default_config_cartpole_reward_env.yaml"}[w["cfg"]]
    over = {"train_episodes": w["train_episodes"]}
    if "init_episodes" in w:
        over["init_episodes"] = w["init_episodes"]
    env_over = {"hidden_size": w["env_hidden"]} if "env_hidden" in w else {}
    return dict(yaml=yaml_name, agent=w.get("agent", "ddqn"), kind=w["kind"], agent_overrides=over, env_overrides=env_over)


def cpu_reference_baseline(workload, cfg, theta, target_seconds, cores):
    """The reference's own torch CPU path (unmodified, oracle/_ref/pyref or /root/reference) on `cores` single-thread worker
    processes: one calc_score (fresh agent, train on the SE/RN with per-episode test(), final test()) per task.
    Returns (env-steps/s aggregate, info) or None when the reference tree is not staged."""
    from oracle import ref_harness
    if not ref_harness.reference_available():
        return None
    from oracle import ref_bench
    spec = reference_spec(workload)
    n_tasks = max(cores, 16 * 3)                    # at least one NES generation of population 16 (3 calc_scores per member)
    r = ref_bench.run(spec, theta, n_tasks, n_workers=cores, budget_s=target_seconds)
    ts = np.array(r["task_seconds"])
    value = r["steps"] / r["seconds"]
    # one generation of the yaml's population (16 members x 3 calc_scores) on this machine, one worker per core:
    # ceil(48 / workers) waves of the mean task time
    gen_s = float(np.ceil(48.0 / r["workers"]) * ts.mean())
    return value, dict(tasks=r["tasks"], steps=r["steps"], seconds=r["seconds"], workers=r["workers"], task_seconds_mean=float(ts.mean()),
                       steps_per_s_per_core=value / r["workers"], nes_generations_per_hour_pop16=3600.0 / gen_s)


def cpu_baseline_block(workload, cfg, target_seconds):
    """cpu_baseline object of the JSON line: the unmodified reference when staged (kind "reference"), else the C port."""
    cores = os.cpu_count() or 1
    theta = synthetic_theta(cfg)
    ref = cpu_reference_baseline(workload, cfg, theta, target_seconds, cores)
    pv, pinfo = cpu_port_baseline(cfg, theta, target_seconds=min(target_seconds, 8.0), n_threads=cores)
    port = {"value": pv, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": "%d lanes, %d steps in %.1f s on %d pthreads (C restatement oracle/le_oracle.c)" % (pinfo["lanes"], pinfo["steps"], pinfo["seconds"], cores)}
    if ref is None:
        return port, None
    v, info = ref
    blk = {"value": v, "unit": "env-steps/s", "cores": info["workers"], "kind": "reference",
           "sample": "%d calc_scores (fresh %s agent: train on the synthetic env with per-episode test(), final test()) of the UNMODIFIED "
                     "reference, %d env steps in %.1f s on %d single-thread worker processes (torch %s CPU)" % (
                         info["tasks"], reference_spec(workload)["agent"], info["steps"], info["seconds"], info["workers"], _torch_version()),
           "steps_per_s_per_core": info["steps_per_s_per_core"], "nes_generations_per_hour_pop16": info["nes_generations_per_hour_pop16"],
           "port": port}
    return blk, info


def _torch_version():
    import torch
    return torch.__version__


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on all host threads.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    d, cfg = build_lane_cfg(args.workload)
    cores = os.cpu_count() or 1
    theta = synthetic_theta(cfg)
    total = max(args.steps + args.warmup, 1)
    per_step_s = max(6.0, min(40.0, 150.0 / total))      # the whole --steps K --warmup W run ends within a few minutes
    tot_steps = tot_s = 0.0
    infos = []
    kind = "reference"
    for i in range(total):
        ref = cpu_reference_baseline(args.workload, cfg, theta, per_step_s, cores)
        if ref is None:
            kind = "port"
            v, info = cpu_port_baseline(cfg, theta, target_seconds=3.0, n_threads=cores)
            info = dict(info, tasks=info["lanes"], workers=cores, nes_generations_per_hour_pop16=None, steps_per_s_per_core=v / cores)
        else:
            v, info = ref
        if i >= args.warmup:
            tot_steps += info["steps"]
            tot_s += info["seconds"]
            infos.append(info)
    value = tot_steps / tot_s
    gph = [i["nes_generations_per_hour_pop16"] for i in infos if i.get("nes_generations_per_hour_pop16")]
    sample = ("%d calc_scores per step of the same lane config on %d single-thread worker processes, UNMODIFIED reference (oracle/_ref/pyref)"
              % (infos[-1]["tasks"], infos[-1]["workers"])) if kind == "reference" else \
             ("%d lanes/step of the same lane config, C restatement oracle/le_oracle.c, %d pthreads" % (infos[-1]["tasks"], cores))
    line = {
        "impl": "reference", "metric": "se_env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, cfg, 0, None),
        "nes_generations_per_hour": float(np.mean(gph)) if gph else None, "nes_population": 16,
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": infos[-1]["workers"], "kind": kind, "sample": sample,
                         "steps_per_s_per_core": value / infos[-1]["workers"]},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if kind == "reference":
        pv, pinfo = cpu_port_baseline(cfg, theta, target_seconds=3.0, n_threads=cores)
        line["cpu_baseline"]["port"] = {"value": pv, "unit": "env-steps/s", "cores": cores, "kind": "port"}
    print(json.dumps(line))
    return 0


def workload_config(name, cfg, members_per_gpu, plan):
    w = WORKLOADS[name]
    c = {"workload": "%s: NES generation, %s, %s inner loop (B=%d, Q %d->%d->%d), per lane %d train episodes x <=%d steps "
                     "+ per-episode test() of %d real-env episodes + final test()" % (
                         name, w["cfg"], "DuelingDDQN" if cfg.q_kind else "DDQN", cfg.batch_size, cfg.sd, cfg.q_hidden, cfg.ad,
                         cfg.train_episodes, cfg.max_steps,
                         cfg.test_episodes),
         "members_per_gpu": members_per_gpu, "lanes_per_member": 1 + 2 * w.get("grad_evals", 1), "env_hidden": cfg.env_hidden,
         "l2": "256 MiB buffer written between timed steps (L2 flush)"}
    if cfg.step_budget:
        c["step_budget_per_lane"] = int(cfg.step_budget)
    if plan:
        c.update({"resident_warp_slots": plan["slots"], "replay_ring_rows": plan["ring_cap"], "units_per_thread": plan["units"],
                  "replay_rings_bytes": int(plan["slots"]) * int(plan["ring_cap"]) * (2 * cfg.sd + 4) * 4})
    return c


class Dist(object):
    """torch.distributed plumbing of one bench process (one rank per GPU)."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise RuntimeError("bench.py --impl ours needs a CUDA device: the hot path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_sum(self, values):
        """(max over ranks, sum over ranks) of a list of floats."""
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return t.tolist(), t.tolist()
        a, b = t.clone(), t.clone()
        self.dist.all_reduce(a, op=self.dist.ReduceOp.MAX)
        self.dist.all_reduce(b, op=self.dist.ReduceOp.SUM)
        return a.tolist(), b.tolist()

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


DUMP_BYTES = 64 << 20          # all files of one --dump-outputs directory together


def lane_fields(res, order=None):
    """The fields of a lane-result structured array (ops.lane_out_dtype) as separate arrays, optionally re-ordered."""
    return {"lane_" + k: res[k] if order is None else res[k][order] for k in res.dtype.names}


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy: float32 stays float32, every other dtype becomes float64.  The files share
    DUMP_BYTES: arrays are taken smallest first, each may use an equal share of what is left, and one that does not fit keeps
    a sample of its rows (elements for 1-D arrays) drawn from a fixed seed, with the row indices in <name>_rows.npy, so that
    two builds run with the same arguments are compared on the same elements."""
    header = 128                                                   # bytes of one .npy header
    arrays = {k: np.asarray(a) for k, a in arrays.items()}
    arrays = {k: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    for n, name in enumerate(sorted(arrays, key=lambda k: (arrays[k].nbytes, k))):
        a = arrays[name]
        share = left // (len(arrays) - n) - header
        if a.nbytes > share:
            k = max((share - header) // (a.nbytes // a.shape[0] + 8), 1)
            rows = np.sort(np.random.RandomState(0).choice(a.shape[0], k, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            left -= rows.nbytes + header
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes + header


def measure_vary_hp(D, steps, warmup, members_per_gpu=0, ffma_peak=None, outputs=None):
    """BASELINE config 4.  One step = every agent of this rank trained on the SE (virtual-env plateau rule) and tested on
    the real env: one launch per kernel family (register kernel sets by hidden width, general kernel for the rest), per-lane
    le_lane_cfg; the lane queue of every launch is ordered longest-first.  `outputs` (a dict) receives the lane results of
    the last timed step in agent order."""
    import torch
    from learning_environments_b200 import default_configs, ops, vary_hp
    from learning_environments_b200.rng import lane_keys
    dev, rank, world = D.dev, D.rank, D.world
    w = WORKLOADS["vary_hp"]
    d = default_configs.get(w["cfg"])
    n = members_per_gpu or w["members_per_gpu"]
    over = dict(vary_hp.OVERRIDES, train_episodes=w["train_episodes"])
    cfgs = vary_hp.sample_agent_cfgs(d, n, np.random.RandomState(1000 + rank), over, True, None)
    theta_host = synthetic_theta(cfgs[0])
    theta_dev = torch.from_numpy(theta_host).to(dev).reshape(1, -1)
    groups = []
    for idx in vary_hp.launch_groups(cfgs):
        sub = [cfgs[i] for i in idx]
        cfg0 = vary_hp._max_cfg(sub)
        groups.append(dict(idx=idx, idx_dev=torch.from_numpy(idx).to(dev), sub=sub, cfg0=cfg0,
                           bufs=ops.InnerLoopBuffers(cfg0, len(idx), 1, dev, n_cfg=len(idx))))
    total = warmup + steps
    keys = [torch.from_numpy(lane_keys(4321, g, rank * n + np.arange(n), np.zeros(n, int), np.zeros(n, int)).view(np.int32).copy()).to(dev)
            for g in range(total)]
    ffma_peak = ffma_peak or ops.bench_ffma()

    def step(g):
        for gr in groups:
            ops.inner_loop_run(gr["bufs"], gr["sub"], theta_dev, None, keys[g][gr["idx_dev"]].contiguous(), cfg0=gr["cfg0"])

    for g in range(warmup):
        step(g)
    D.barrier()
    sampler = ClockSampler(D.local_rank)
    sampler.start()
    dev_ms, steps_done, flop = 0.0, 0, 0.0
    for k in range(steps):
        D.flush.fill_(k & 0xFF)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(warmup + k)
        e1.record()
        torch.cuda.synchronize()
        dev_ms += e0.elapsed_time(e1)
        for gr in groups:
            res = gr["bufs"].results()
            steps_done += int(res["train_steps"].sum())
            for c, st, li in zip(gr["sub"], res["train_steps"], res["learn_iters"]):
                a, b = f_parts(c)
                flop += float(st) * a + float(li) * b
    D.barrier()
    clocks = sampler.stop()
    if outputs is not None:
        res = np.concatenate([gr["bufs"].results() for gr in groups])
        outputs.update(lane_fields(res, np.argsort(np.concatenate([gr["idx"] for gr in groups]))))
    mx, sm = D.max_sum([dev_ms, float(steps_done), flop])
    dev_ms, steps_all, flop_all = mx[0], sm[1], sm[2]
    # end to end through the public API: sampling, H2D of theta / keys / per-lane cfgs, all launches, D2H of the results
    D.barrier()
    t0 = time.perf_counter()
    e2e_steps = 0
    for k in range(steps):
        _, st, _, _ = vary_hp.evaluate_agents(d, theta_host.reshape(1, -1), n, seed=1000 + rank, overrides=over, device=dev, shard=False)
        e2e_steps += sum(st[0])
    D.barrier()
    e2e_s = time.perf_counter() - t0
    mx, sm = D.max_sum([e2e_s, float(e2e_steps)])
    e2e_s, e2e_steps = mx[0], sm[1]
    achieved = flop_all / world / (dev_ms * 1e-3) / 1e12
    n_gen = sum(len(g["idx"]) for g in groups if not g["cfg0"].q_is_register_resident())
    return {
        "metric": "se_env_steps_per_s", "value": steps_all / (dev_ms * 1e-3), "unit": "env-steps/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": dev_ms / max(steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "vary_hp: %d DDQN_vary agents per GPU on one CartPole SE (lr, batch_size in [66,597], hidden_size in "
                               "[19,171], hidden_layer in {1,2} per lane), init_episodes=10, <=%d train episodes, plateau early-out, "
                               "final test() of 10 real-env episodes" % (n, w["train_episodes"]),
                   "agents_per_gpu": n, "general_kernel_lanes": n_gen, "launches_per_step": len(groups),
                   "l2": "256 MiB buffer written between timed steps (L2 flush)"},
        "seconds_per_evaluation": dev_ms * 1e-3 / max(steps, 1),
        "e2e": {"value": e2e_steps / e2e_s, "unit": "env-steps/s",
                "h2d_bytes_per_step": int(theta_host.nbytes + n * 8 + n * 200), "d2h_bytes_per_step": int(n * (40 + 10 * 8))},
        "gpu_launches": (1 + len(groups)) * steps, "clocks": clocks,
        "roofline": {"bound": "fp32_ffma", "achieved": achieved, "peak": ffma_peak, "unit": "TFLOP/s",
                     "frac": achieved / ffma_peak if ffma_peak else None, "traffic": None,
                     "peak_source": "le_bench_ffma microbenchmark in this run"},
    }


def measure_td3(D, steps, warmup, lanes_per_gpu=0, ffma_peak=None, outputs=None):
    """TD3_discrete_vary lanes through le_td3_run_host (HOST buffers in and out: the timed region holds the H2D of the SE / initial
    nets / keys, the persistent kernel and the D2H of the lane results), wall clock around the call, max over ranks.
    `outputs` (a dict) receives the arrays le_td3_run_host returned in the last timed step."""
    import copy
    import torch
    from learning_environments_b200 import agents as A, default_configs, ops
    from learning_environments_b200.envs import EnvFactory
    from learning_environments_b200.rng import lane_keys
    w = TD3_WORKLOAD
    d = copy.deepcopy(default_configs.get(w["cfg"]))
    a = d["agents"]["td3_discrete_vary"]
    w = dict(w, train_episodes=int(os.environ.get("LE_TD3_TRAIN_EPISODES", w["train_episodes"])))   # profiling aid (ncu replays the kernel)
    a.update(vary_hp=False, train_episodes=w["train_episodes"], init_episodes=w["init_episodes"])
    n = lanes_per_gpu or w["lanes_per_gpu"]
    torch.manual_seed(7)
    fac = EnvFactory(d)
    env, real = fac.generate_virtual_env(), fac.generate_real_env()
    agent = A.TD3_discrete_vary(env=real, min_action=real.get_min_action(), max_action=real.get_max_action(), config=d)
    env.set_agent_params(same_action_num=agent.same_action_num, gamma=agent.gamma)
    t, theta, nets = agent._td3_cfg(env, real, w["train_episodes"], True, 1e9)
    pa, pc = ops.td3_param_counts(t)
    sd, ad, H, L, B = t.base.sd, t.base.ad, t.base.q_hidden, max(t.base.q_layers, 1), t.base.batch_size
    f_a = 2 * (sd * H + (L - 1) * H * H + H * ad)
    f_c = 2 * ((sd + ad) * H + (L - 1) * H * H + H)
    f_env = 2 * (3 * t.base.env_hidden * (sd + ad) + t.base.env_hidden * (sd + 2))
    f_learn = B * (f_a + 8 * f_c + (3 * f_a + 2 * f_c) / max(t.policy_delay, 1))
    nets_n = [np.repeat(x[None], 1, 0) for x in nets]

    def step(g):
        keys = lane_keys(977, g, D.rank * n + np.arange(n), np.zeros(n, int), np.zeros(n, int))
        return ops.td3_run_host(t, theta, None, keys, nets_n[0], nets_n[1], nets_n[2], device=torch.cuda.current_device())

    for g in range(warmup):
        step(g)
    D.barrier()
    sampler = ClockSampler(D.local_rank)
    sampler.start()
    t0 = time.perf_counter()
    steps_done, learns = 0, 0
    for k in range(steps):
        res = step(warmup + k)
        steps_done += int(res["out"]["train_steps"].sum())
        learns += int(res["out"]["learn_iters"].sum())
    D.barrier()
    sec = time.perf_counter() - t0
    clocks = sampler.stop()
    if outputs is not None:
        outputs.update(lane_fields(res["out"]))
        outputs.update({k: res[k] for k in ("rewards", "lengths", "test_rewards", "actor_final")})
    mx, sm = D.max_sum([sec, float(steps_done), float(learns)])
    sec, steps_all, learns_all = mx[0], sm[1], sm[2]
    achieved = (steps_all * (f_env + f_a) + learns_all * f_learn) / D.world / sec / 1e12
    ffma_peak = ffma_peak or ops.bench_ffma()
    val = steps_all / sec
    return {
        "metric": "se_env_steps_per_s", "value": val, "unit": "env-steps/s", "n_gpus": D.world, "steps": steps, "warmup": warmup,
        "ms_per_step": 1e3 * sec / max(steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "td3_discrete: %d TD3_discrete_vary lanes per GPU on one CartPole SE (actor %d / critic %d parameters, %d hidden "
                               "layers of %d, B=%d, policy_delay %d), %d train episodes + per-episode test() + final test(), host-buffer entry"
                               % (n, pa, pc, L, H, B, t.policy_delay, w["train_episodes"]),
                   "lanes_per_gpu": n, "timing": "wall clock around le_td3_run_host (H2D + kernel + D2H), max over ranks"},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": int((0 if theta is None else theta.nbytes) + sum(x.nbytes for x in nets_n) + n * 8),
                "d2h_bytes_per_step": int(n * (40 + pa * 4))},
        "gpu_launches": 2 * steps, "clocks": clocks,
        "roofline": {"bound": "fp32_ffma", "achieved": achieved, "peak": ffma_peak, "unit": "TFLOP/s",
                     "frac": achieved / ffma_peak if ffma_peak else None, "traffic": None,
                     "peak_source": "le_bench_ffma microbenchmark in this run"},
    }


def measure_nes(D, workload, steps, warmup, members_per_gpu=0, population=0, lane_override=(), ffma_peak=None, with_e2e=True,
                outputs=None):
    """One NES-generation workload on this process group: device-timed `value`, the generation including the score exchange
    and the NES update (`with_update`), and (with_e2e) the end-to-end figure through the host API.  Returns the JSON fields.
    `outputs` (a dict) receives what the last step of the device-timed population evaluation computed: the lane results, the
    per-episode train and test rings and the perturbed SE / RN parameters the lanes ran on."""
    import torch
    from learning_environments_b200 import ops
    from learning_environments_b200.engine import PopulationEvaluator
    from learning_environments_b200.nes import score_transform
    from learning_environments_b200.rng import lane_keys
    dist, dev, world, rank = D.dist, D.dev, D.world, D.rank
    d, cfg = build_lane_cfg(workload)
    os.environ["LE_TC"] = "1" if WORKLOADS[workload].get("tc") else "0"     # read by the library at plan / launch time
    for ov in lane_override:
        k, v = ov.split("=")
        setattr(cfg, k, type(getattr(cfg, k))(float(v)))
    gtn = d["agents"]["gtn"]
    if population:                                   # strong scaling: a fixed population split over the ranks
        mpg = (population + world - 1) // world
        pop = mpg * world
    else:
        mpg = members_per_gpu or WORKLOADS[workload]["members_per_gpu"]
        pop = mpg * world
    ev = PopulationEvaluator(cfg, pop, member_lo=rank * mpg, member_hi=(rank + 1) * mpg, num_grad_evals=gtn["num_grad_evals"],
                             seed=1234, noise_std=gtn["noise_std"], device=dev)
    plan = ops.inner_loop_plan(cfg, ev.n_lanes, ev.n_env)
    theta_host = torch.from_numpy(synthetic_theta(cfg)).pin_memory()
    theta_dev = theta_host.to(dev)
    theta_work = theta_dev.clone()
    scores_all = torch.zeros((world, mpg, 2), dtype=torch.float64, device=dev)
    scores_host = torch.zeros((world, mpg, 2), dtype=torch.float64).pin_memory()
    coef_host = torch.zeros(pop, dtype=torch.float32).pin_memory()
    coef_dev = torch.zeros(pop, dtype=torch.float32, device=dev)
    sign_dev = torch.ones(pop, dtype=torch.float32, device=dev)
    ffma_peak = ffma_peak or ops.bench_ffma()
    total = warmup + steps
    # lane keys are precomputed (host-side key derivation is not the timed work of the device-resident figures)
    key_cache = {}

    def keys_for(gen):
        if gen not in key_cache:
            k = lane_keys(ev.seed, gen, ev.lane_member, ev.lane_variant, ev.lane_eval)
            key_cache[gen] = torch.from_numpy(k.view(np.int32).copy()).to(dev)
        return key_cache[gen]
    for g in range(3 * total + 3):
        keys_for(g)

    def launch_resident(gen):
        ev._theta_dev.copy_(theta_dev)
        ev._keys_dev.copy_(keys_for(gen))
        thetas = ops.nes_perturb(ev._theta_dev, ev.pop, ev.member_lo, ev.n_members, ev.seed, gen, ev.noise_std)
        ops.inner_loop_run(ev.bufs, cfg, thetas, ev.env_index, ev._keys_dev)
        ev._thetas = thetas

    def exchange_and_update(out, gen):
        """score all-gather over the ranks (NCCL), identical score transform on every rank, NES update of theta."""
        orig, add, sub = ev.member_scores(out)
        local = torch.from_numpy(np.stack([np.maximum(add, sub), orig], 1)).to(dev, non_blocking=True)
        if world > 1:
            dist.all_gather_into_tensor(scores_all.view(-1), local.view(-1))
            scores_host.copy_(scores_all, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            sc = scores_host.numpy().reshape(pop, 2)
        else:
            sc = np.stack([np.maximum(add, sub), orig], 1)
        wgt = score_transform(sc[:, 0], sc[:, 1], gtn["score_transform_type"])
        coef_host.copy_(torch.from_numpy((gtn["step_size"] * wgt).astype(np.float32)))
        coef_dev.copy_(coef_host, non_blocking=True)
        theta_work.copy_(theta_dev)
        # every rank regenerates all eps_i and applies them in member order: bit-identical theta on all ranks
        ops.nes_update(theta_work, pop, ev.seed, gen, ev.noise_std, gtn["weight_decay"], coef_dev, sign_dev)

    def timed(fn, first_gen):
        for g in range(warmup):
            fn(first_gen + g)
        D.barrier()
        sampler = ClockSampler(D.local_rank)
        sampler.start()
        ms, st, li = 0.0, 0, 0
        for k in range(steps):
            D.flush.fill_(k & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(first_gen + warmup + k)
            e1.record()
            torch.cuda.synchronize()
            ms += e0.elapsed_time(e1)
            res = ev.bufs.results()
            st += int(res["train_steps"].sum())
            li += int(res["learn_iters"].sum())
        D.barrier()
        clocks = sampler.stop()
        mx, sm = D.max_sum([ms, float(st), float(li)])
        return mx[0], sm[1], sm[2], clocks

    # ---------------- device-resident: population evaluation only (value) ----------------
    dev_ms, steps_all, learn_all, clocks = timed(launch_resident, 0)
    value = steps_all / (dev_ms * 1e-3)
    if outputs is not None:
        b = ev.bufs
        outputs.update(lane_fields(b.results()))
        outputs.update(episode_rewards=b.rewards.cpu().numpy(), episode_lengths=b.lengths.cpu().numpy(),
                       test_rewards=b.test_rewards.cpu().numpy(), test_lengths=b.test_lengths.cpu().numpy(),
                       env_theta=ev._thetas.cpu().numpy())

    # ---------------- device-resident generation INCLUDING the collective and the NES update ----------------
    def generation_with_update(gen):
        launch_resident(gen)
        exchange_and_update(ev.collect(), gen)
    upd_ms, upd_steps, _, _ = timed(generation_with_update, total)
    f_env_q, f_td = f_parts(cfg)
    # per-GPU TFLOP/s of algorithmic work: every env step costs F_env + F_q, every TD update 5*B*F_q (steps of the
    # init_episodes do not learn); the fused kernel is >= 95% of the timed region (profiles/)
    achieved = (steps_all * f_env_q + learn_all * f_td) / world / (dev_ms * 1e-3) / 1e12
    res = {
        "metric": "se_env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": dev_ms / max(steps, 1), "higher_is_better": True, "scaling": "strong" if population else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(workload, cfg, mpg, plan), **({"overrides": list(lane_override)} if lane_override else {})),
        "nes_population": pop,
        "with_update": {"value": upd_steps / (upd_ms * 1e-3), "unit": "env-steps/s", "ms_per_step": upd_ms / max(steps, 1),
                        "what": "device-timed generation incl. D2H of lane results, score all-gather (NCCL), score transform, NES update kernel"},
        "gpu_launches": 3 * steps,
        "clocks": clocks,
        "roofline": {"bound": "fp32_ffma", "achieved": achieved, "peak": ffma_peak, "unit": "TFLOP/s",
                     "frac": achieved / ffma_peak if ffma_peak else None,
                     "traffic": _ncu_traffic(workload, steps_all / world / max(steps, 1)),
                     "flop_per_env_step": f_step(cfg), "td_updates_per_env_step": learn_all / max(steps_all, 1.0),
                     "peak_source": "le_bench_ffma microbenchmark in this run (FP32 FFMA; MEASURED_PEAKS.json has no FP32 figure)",
                     "hbm": {"algorithmic_bytes_per_env_step": (cfg.batch_size + 1) * (2 * cfg.sd + 3) * 4,
                             "achieved_gbs": value / world * (cfg.batch_size + 1) * (2 * cfg.sd + 3) * 4 / 1e9,
                             "peak_gbs": _measured_hbm()}},
    }
    if with_e2e:
        # ---------------- end-to-end through the host API (e2e): HOST theta in, lane results out, every generation -------------
        base = 2 * total
        for g in range(warmup):
            ev.evaluate(theta_host, base + g)
        D.barrier()
        t0 = time.perf_counter()
        e2e_steps = 0
        for k in range(steps):
            gen = base + warmup + k
            out = ev.evaluate(theta_host, gen)          # H2D theta/keys, kernels, D2H lane results
            e2e_steps += int(out["train_steps"].sum())
            exchange_and_update(out, gen)
        D.barrier()
        e2e_s = time.perf_counter() - t0
        mx, sm = D.max_sum([e2e_s, float(e2e_steps)])
        res["e2e"] = {"value": sm[1] / mx[0], "unit": "env-steps/s", "h2d_bytes_per_step": ev.h2d_bytes, "d2h_bytes_per_step": ev.d2h_bytes}
        res["nes_generations_per_hour"] = 3600.0 / (mx[0] / max(steps, 1))
    del ev
    torch.cuda.empty_cache()
    os.environ["LE_TC"] = "0"
    return res, cfg


def compact(r):
    """Sub-workload entry of the headline line's `workloads` object."""
    out = {"value": r["value"], "unit": r["unit"], "ms_per_step": r["ms_per_step"], "steps": r["steps"], "warmup": r["warmup"],
           "frac": r["roofline"]["frac"], "achieved_tflops": r["roofline"]["achieved"], "clocks": r["clocks"], "config": r["config"]}
    for k in ("with_update", "e2e", "seconds_per_evaluation", "nes_population"):
        if k in r:
            out[k] = r[k]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cartpole_se", choices=sorted(WORKLOADS) + ["td3_discrete"])
    ap.add_argument("--members-per-gpu", type=int, default=0)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: --population members split over the ranks")
    ap.add_argument("--population", type=int, default=0, help="total NES population for --scaling strong (default 8 x 1184)")
    ap.add_argument("--extras", default="auto", choices=["auto", "all", "none"],
                    help="auto: the default headline run also times every other workload + the strong-scaling point")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lane-override", action="append", default=[], metavar="FIELD=VALUE",
                    help="profiling aid: override an le_lane_cfg field (e.g. max_steps=100); recorded in config.overrides")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path of --workload computed in its last timed step as DIR/<name>.npy "
                         "(rank 0's lanes; at most 64 MB, larger arrays as a seeded row sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of --impl ours")
        return run_reference_arm(args)
    D = Dist()
    from learning_environments_b200 import ops
    ffma_peak = ops.bench_ffma()
    plain = args.workload == "cartpole_se" and not args.lane_override and not args.members_per_gpu and args.scaling == "weak"
    extras = args.extras == "all" or (args.extras == "auto" and plain and not args.no_cpu_baseline)
    outputs = {} if args.dump_outputs else None
    if args.workload == "vary_hp":
        line = measure_vary_hp(D, args.steps, args.warmup, args.members_per_gpu, ffma_peak, outputs)
        cfg = None
    elif args.workload == "td3_discrete":
        line = measure_td3(D, args.steps, args.warmup, args.members_per_gpu, ffma_peak, outputs)
        cfg = None
    else:
        pop = (args.population or STRONG_POPULATION) if args.scaling == "strong" else 0
        line, cfg = measure_nes(D, args.workload, args.steps, args.warmup, args.members_per_gpu, pop, args.lane_override, ffma_peak,
                                outputs=outputs)
    if outputs is not None and D.rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    if extras:
        wl = {}
        for name in EXTRA_WORKLOADS:
            try:
                if name == "vary_hp":
                    wl[name] = compact(measure_vary_hp(D, 1, 1, 0, ffma_peak))
                else:
                    heavy = name == "cartpole_se_fullring"
                    small = name == "cartpole_se_pop16"
                    r, _ = measure_nes(D, name, 1 if heavy else (5 if small else 2), 1, 0, 0, (), ffma_peak, with_e2e=small)
                    wl[name] = compact(r)
                    if small:   # one generation of the yaml's population through the host API: wall time and lane latency
                        wl[name]["nes_generations_per_hour"] = r["nes_generations_per_hour"]
                        wl[name]["us_per_env_step_per_lane"] = 1e3 * r["ms_per_step"] / max(r["value"] * r["ms_per_step"] * 1e-3 / (3 * 16 * D.world), 1.0)
            except Exception as e:   # a failing side workload must not lose the headline line
                wl[name] = {"error": "%s: %s" % (type(e).__name__, e)}
        try:
            wl["td3_discrete"] = compact(measure_td3(D, 1, 1, 0, ffma_peak))
        except Exception as e:
            wl["td3_discrete"] = {"error": "%s: %s" % (type(e).__name__, e)}
        line["workloads"] = wl
        try:
            r, _ = measure_nes(D, args.workload, 2, 1, 0, STRONG_POPULATION, (), ffma_peak, with_e2e=False)
            line["strong_scaling"] = dict(compact(r), population=STRONG_POPULATION, scaling="strong",
                                          note="fixed population split over the ranks: efficiency(N) = value(N) / (N * value(1))")
        except Exception as e:
            line["strong_scaling"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if D.rank == 0:
        if not args.no_cpu_baseline and cfg is not None:
            blk, _ = cpu_baseline_block(args.workload, cfg, target_seconds=20.0)
            line["cpu_baseline"] = blk
        print(json.dumps(line))
    D.barrier()
    D.close()
    return 0


def _ncu_traffic(workload, env_steps_per_launch):
    """DRAM bytes per launch of the fused kernel from the committed `ncu` capture of THIS workload (profiles/r*_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum of one launch, divided by its env steps), scaled to this run's env steps
    per launch; None if no capture of the workload is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    if not files:
        return None
    try:
        with open(files[-1]) as f:
            t = json.load(f)
        t = t.get("workloads", {}).get(workload, t if workload == "cartpole_se" else None)
        return t["dram_bytes_per_env_step"] * env_steps_per_launch if t else None
    except Exception:
        return None


def _measured_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"]
    except Exception:
        return 6650.0


if __name__ == "__main__":
    sys.exit(main())
