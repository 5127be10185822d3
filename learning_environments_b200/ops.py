"""Thin torch/ctypes front end of the C ABI (include/le_b200.h).

Every function takes CUDA tensors (device memory, current stream) and forwards raw pointers; nothing here
computes on the host.  ``inner_loop_run_host`` is the reference-facing call on HOST (numpy) buffers.
"""
import ctypes as C

import numpy as np
import torch

from . import _abi
from ._abi import LaneCfg, LaneOut, Td3Cfg, Trace, check

_F32, _I32, _F64 = torch.float32, torch.int32, torch.float64


def _lib():
    return _abi.load_library()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _on(object):
    """Makes the device that owns `t` current for the duration of a library call (the C ABI launches on the CURRENT device)
    and yields that device's current stream: a GTN_Master / PopulationEvaluator built with device='cuda:1' works while
    cuda:0 is the process's current device."""

    def __init__(self, t):
        self.dev = t.device if torch.is_tensor(t) else torch.device(t)
        self.ctx = torch.cuda.device(self.dev)

    def __enter__(self):
        self.ctx.__enter__()
        return C.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)

    def __exit__(self, *exc):
        return self.ctx.__exit__(*exc)


def _dev(t, dtype):
    assert t.is_cuda and t.dtype == dtype and t.is_contiguous(), "expected a contiguous CUDA %s tensor" % dtype
    return t


def version():
    return _lib().le_version()


def device_info(device=0):
    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    name = C.create_string_buffer(128)
    check(_lib().le_device_info(C.c_int(device), C.byref(sm), C.byref(ma), C.byref(mi), name, C.c_int(128)), "le_device_info")
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), name=name.value.decode())


def bench_ffma(iters=4096, reps=5):
    """Measured FP32 FFMA peak of the current device in TFLOP/s (roofline denominator of the fused kernel)."""
    out = C.c_double()
    check(_lib().le_bench_ffma(C.c_int(iters), C.c_int(reps), C.byref(out), _stream()), "le_bench_ffma")
    return out.value


# ---------------------------------------------------------------------------------------------------------
def se_forward(cfg, theta, state, action, lanes_per_member=None):
    """VirtualEnv.step (envs/virtual_env.py:43-54). theta [pop, P_se]; state [n, sd]; action [n] int32."""
    theta = _dev(theta.reshape(-1, cfg.se_params()), _F32)
    pop = theta.shape[0]
    n = state.shape[0]
    lpm = lanes_per_member or n // pop
    assert pop * lpm == n
    ns = torch.empty((n, cfg.sd), dtype=_F32, device=state.device)
    r = torch.empty(n, dtype=_F32, device=state.device)
    d = torch.empty(n, dtype=_F32, device=state.device)
    check(_lib().le_se_forward(C.byref(cfg), _ptr(theta), C.c_int(pop), C.c_int(lpm), _ptr(_dev(state, _F32)),
                               _ptr(_dev(action, _I32)), _ptr(ns), _ptr(r), _ptr(d), _stream()), "le_se_forward")
    return ns, r, d


def rn_reward(cfg, theta, state, next_state, real_reward, lanes_per_member=None):
    """RewardEnv._calc_reward (envs/reward_env.py:68-133), reward types 0,1,2,5,6."""
    theta = _dev(theta.reshape(-1, cfg.rn_params()), _F32)
    pop = theta.shape[0]
    n = state.shape[0]
    lpm = lanes_per_member or n // pop
    out = torch.empty(n, dtype=_F32, device=state.device)
    rc = _lib().le_rn_reward(C.byref(cfg), _ptr(theta), C.c_int(pop), C.c_int(lpm), _ptr(_dev(state, _F32)),
                             _ptr(_dev(next_state, _F32)), _ptr(_dev(real_reward, _F32)), _ptr(out), _stream())
    if rc == -3:
        # the reference raises ValueError('No info dict provided by environment') for info-vector types on
        # CartPole / Acrobot (envs/reward_env.py:91-92)
        raise ValueError("No info dict provided by environment")
    check(rc, "le_rn_reward")
    return out


def qnet_forward(cfg, q_theta, state):
    """Critic_DQN.forward + argmax (models/actor_critic.py:84-91, agents/DDQN.py:106-110), one net per row."""
    n = state.shape[0]
    q = torch.empty((n, cfg.ad), dtype=_F32, device=state.device)
    am = torch.empty(n, dtype=_I32, device=state.device)
    check(_lib().le_qnet_forward(C.byref(cfg), _ptr(_dev(q_theta, _F32)), C.c_int(n), _ptr(_dev(state, _F32)), _ptr(q), _ptr(am),
                                 _stream()), "le_qnet_forward")
    return q, am


def real_env_step(real_env, max_steps, state64, elapsed, action, sd):
    """gym CartPole/Acrobot step + TimeLimit, in place on state64 [n,4] (float64) and elapsed [n] (int32)."""
    n = state64.shape[0]
    obs = torch.empty((n, sd), dtype=_F32, device=state64.device)
    r = torch.empty(n, dtype=_F32, device=state64.device)
    d = torch.empty(n, dtype=_F32, device=state64.device)
    check(_lib().le_real_env_step(C.c_int(real_env), C.c_int(max_steps), _ptr(_dev(state64, _F64)), _ptr(_dev(elapsed, _I32)),
                                  _ptr(_dev(action, _I32)), _ptr(obs), _ptr(r), _ptr(d), C.c_int(n), _stream()), "le_real_env_step")
    return obs, r, d


def td_update(cfg, q_theta, q_target, adam_m, adam_v, adam_t, rows):
    """DDQN.learn (agents/DDQN.py:60-95) in place; rows [n, B, 2*sd+3] = [s a s' r d]. Returns loss [n]."""
    n = q_theta.shape[0]
    assert rows.shape[1] == cfg.batch_size and rows.shape[2] == 2 * cfg.sd + 3
    loss = torch.empty(n, dtype=_F32, device=q_theta.device)
    check(_lib().le_td_update(C.byref(cfg), _ptr(_dev(q_theta, _F32)), _ptr(_dev(q_target, _F32)), _ptr(_dev(adam_m, _F32)),
                              _ptr(_dev(adam_v, _F32)), _ptr(_dev(adam_t, _I32)), C.c_int(n), _ptr(_dev(rows, _F32)), _ptr(loss),
                              _stream()), "le_td_update")
    return loss


def tc_gemm(A, B, C_out, form, I, J, L, bias=None, act=0, slope=0.0, accumulate=False):
    """One dense-layer GEMM on the tcgen05 tensor cores (3xTF32): `form` names the nn.Linear contraction
         "nt": C[I,J] = A[I,L] @ B[J,L]^T   (forward  Y = X W^T, + bias, activation)
         "nn": C[I,J] = A[I,L] @ B[L,J]     (input gradient  dX = dZ W)
         "tn": C[I,J] = A[L,I]^T @ B[L,J]   (weight gradient dW = dZ^T X)
    on row-major contiguous CUDA tensors; C_out is written (or accumulated into) in place."""
    a_si, a_sl = (A.shape[1], 1) if form in ("nt", "nn") else (1, A.shape[1])
    b_sl, b_sj = (1, B.shape[1]) if form == "nt" else (B.shape[1], 1)
    check(_lib().le_tc_gemm(_ptr(_dev(A, _F32)), C.c_int(a_si), C.c_int(a_sl), _ptr(_dev(B, _F32)), C.c_int(b_sl), C.c_int(b_sj),
                            _ptr(_dev(C_out, _F32)), C.c_int(C_out.shape[1]), C.c_int(1), C.c_int(I), C.c_int(J), C.c_int(L),
                            _ptr(bias) if bias is not None else None, C.c_int(act), C.c_float(slope), C.c_int(1 if accumulate else 0), _stream()),
          "le_tc_gemm")
    return C_out


# ---------------------------------------------------------------------------------------------------------
def inner_loop_plan(cfg, n_lanes, n_env=1):
    g, s, r, u, o = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_int64()
    check(_lib().le_inner_loop_plan(C.byref(cfg), C.c_int(n_lanes), C.c_int(n_env), C.byref(g), C.byref(s), C.byref(r), C.byref(u),
                                    C.byref(o)), "le_inner_loop_plan")
    return dict(grid=g.value, slots=s.value, ring_cap=r.value, units=u.value, ring_offset_bytes=o.value)


def ring_offset_bytes(cfg, n_lanes, n_env=1):
    return inner_loop_plan(cfg, n_lanes, n_env)["ring_offset_bytes"]


def lane_out_dtype():
    return np.dtype([("n_episodes", np.int32), ("timed_out", np.int32), ("train_steps", np.int64), ("learn_iters", np.int64),
                     ("test_steps", np.int64), ("score", np.float64)])


class InnerLoopBuffers(object):
    """Device buffers of one le_inner_loop_run call (allocated once, reusable across generations)."""

    def __init__(self, cfg, n_lanes, n_env, device, n_cfg=1, trace_cap=0, want_q_final=False):
        self.cfg, self.n_lanes, self.n_env, self.device = cfg, n_lanes, n_env, device
        ws = _lib().le_inner_loop_workspace_bytes(C.byref(cfg), C.c_int(n_lanes), C.c_int(n_env))
        if ws < 0:
            check(int(ws), "le_inner_loop_workspace_bytes")
        self.workspace = torch.empty(int(ws), dtype=torch.uint8, device=device)
        rs = max(cfg.train_episodes, 1)
        self.out = torch.zeros((n_lanes, C.sizeof(LaneOut)), dtype=torch.uint8, device=device)
        self.rewards = torch.zeros((n_lanes, rs), dtype=_F64, device=device)
        self.lengths = torch.zeros((n_lanes, rs), dtype=_I32, device=device)
        self.test_rewards = torch.zeros((n_lanes, cfg.test_episodes), dtype=_F64, device=device)
        self.test_lengths = torch.zeros((n_lanes, cfg.test_episodes), dtype=_I32, device=device)
        self.q_final = torch.zeros((n_lanes, cfg.q_params()), dtype=_F32, device=device) if want_q_final else None
        self.cfg_dev = torch.zeros((n_cfg, C.sizeof(LaneCfg)), dtype=torch.uint8, device=device)
        self.trace = None
        if trace_cap > 0:
            self.trace = dict(cap=trace_cap,
                              action=torch.full((trace_cap,), -1, dtype=_I32, device=device),
                              explore=torch.zeros(trace_cap, dtype=_I32, device=device),
                              next_state=torch.zeros((trace_cap, cfg.sd), dtype=_F32, device=device),
                              reward=torch.zeros(trace_cap, dtype=_F32, device=device),
                              done=torch.zeros(trace_cap, dtype=_F32, device=device),
                              loss=torch.full((trace_cap,), float("nan"), dtype=_F32, device=device),
                              qgap=torch.full((trace_cap,), float("nan"), dtype=_F32, device=device))

    def results(self):
        """One D2H read of the per-lane results."""
        o = np.frombuffer(self.out.cpu().numpy().tobytes(), dtype=lane_out_dtype())
        return o


def inner_loop_run(bufs, cfgs, env_theta, env_index, keys, q_init=None, trace_lane=0, cfg0=None):
    """The fused persistent kernel (le_inner_loop_run): n_lanes complete calc_scores on the current stream.

    cfgs: one LaneCfg or a list of n_lanes LaneCfg (per-lane hyper-parameters); env_theta [n_env, P_env] CUDA f32
    (None for ENV_REAL); env_index [n_lanes] int32 or None; keys [n_lanes, 2] (uint32 values in an int64/int32 tensor).
    """
    cfg0 = bufs.cfg if cfg0 is None else cfg0     # shapes / strides / kernel set: the maxima under per-lane configurations
    if isinstance(cfgs, LaneCfg):
        cfgs = [cfgs]
    n_cfg = len(cfgs)
    assert n_cfg in (1, bufs.n_lanes) and bufs.cfg_dev.shape[0] == n_cfg
    raw = b"".join(bytes(c) for c in cfgs)
    if getattr(bufs, "_cfg_raw", None) != raw:      # lane configurations rarely change between generations: upload once
        bufs.cfg_dev.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8).reshape(n_cfg, -1), non_blocking=False)
        bufs._cfg_raw = raw
    keys = _dev(keys, _I32)
    assert keys.numel() == 2 * bufs.n_lanes
    tr = None
    if bufs.trace is not None:
        tr = Trace()
        tr.cap = bufs.trace["cap"]
        for n in ("action", "explore", "next_state", "reward", "done", "loss", "qgap"):
            setattr(tr, n, bufs.trace[n].data_ptr())
    n_env = 0 if env_theta is None else env_theta.reshape(-1, max(cfg0.env_params(), 1)).shape[0]
    with _on(bufs.workspace) as stream:
        check(_lib().le_inner_loop_run(
            _ptr(bufs.cfg_dev), C.c_int(n_cfg), C.byref(cfg0), _ptr(env_theta) if env_theta is not None else None, C.c_int(n_env),
            _ptr(env_index) if env_index is not None else None, _ptr(keys), _ptr(q_init) if q_init is not None else None,
            _ptr(bufs.q_final) if bufs.q_final is not None else None, C.c_int(bufs.n_lanes), _ptr(bufs.out), _ptr(bufs.rewards),
            _ptr(bufs.lengths), _ptr(bufs.test_rewards), _ptr(bufs.test_lengths), _ptr(bufs.workspace), C.c_int64(bufs.workspace.numel()),
            C.byref(tr) if tr is not None else None, C.c_int(trace_lane), stream), "le_inner_loop_run")


def keys_tensor(keys, device):
    """[n,2] uint32 values -> int32 CUDA tensor with the same bits."""
    k = np.ascontiguousarray(np.asarray(keys, dtype=np.uint32).reshape(-1, 2))
    return torch.from_numpy(k.view(np.int32).copy()).to(device)


def inner_loop_run_host(cfgs, env_theta, env_index, keys, q_init=None, want_q_final=False, device=0):
    """le_inner_loop_run_host: everything in HOST numpy buffers, H2D/D2H inside the call. Returns dict of arrays."""
    if isinstance(cfgs, LaneCfg):
        cfgs = [cfgs]
    c0 = cfgs[0]
    n_cfg = len(cfgs)
    arr = (LaneCfg * n_cfg)(*cfgs)
    keys = np.ascontiguousarray(np.asarray(keys, dtype=np.uint32).reshape(-1, 2))
    n = keys.shape[0]
    n_env = 0
    th = None
    if env_theta is not None:
        th = np.ascontiguousarray(env_theta, np.float32).reshape(-1, c0.env_params())
        n_env = th.shape[0]
    ei = None if env_index is None else np.ascontiguousarray(env_index, np.int32)
    qi = None if q_init is None else np.ascontiguousarray(q_init, np.float32)
    qf = np.zeros((n, c0.q_params()), np.float32) if want_q_final else None
    out = np.zeros(n, dtype=lane_out_dtype())
    rs = max(c0.train_episodes, 1)
    rewards = np.zeros((n, rs), np.float64)
    lengths = np.zeros((n, rs), np.int32)
    test_rewards = np.zeros((n, c0.test_episodes), np.float64)

    def p(a):
        return a.ctypes.data_as(C.c_void_p) if a is not None else None
    check(_lib().le_inner_loop_run_host(arr, C.c_int(n_cfg), p(th), C.c_int(n_env), p(ei), p(keys), p(qi), p(qf), C.c_int(n), p(out),
                                        p(rewards), p(lengths), p(test_rewards), C.c_int(device)), "le_inner_loop_run_host")
    return dict(out=out, rewards=rewards, lengths=lengths, test_rewards=test_rewards, q_final=qf)


# ---------------------------------------------------------------------------------------------------------
def nes_perturb(theta, pop, member_offset, n_members, seed, generation, noise_std):
    """[n_members*3, P]: rows (theta, theta+eps_i, theta-eps_i) for members member_offset.. (agents/GTN_worker.py:156-178)."""
    P = theta.numel()
    out = torch.empty((n_members * 3, P), dtype=_F32, device=theta.device)
    with _on(theta) as stream:
        check(_lib().le_nes_perturb(_ptr(_dev(theta, _F32)), C.c_int(P), C.c_int(pop), C.c_int(member_offset), C.c_int(n_members),
                                    C.c_uint32(seed), C.c_uint32(generation), C.c_float(noise_std), _ptr(out), stream), "le_nes_perturb")
    return out


def nes_noise(P, member_offset, n_members, seed, generation, noise_std, device):
    eps = torch.empty((n_members, P), dtype=_F32, device=device)
    with _on(eps) as stream:
        check(_lib().le_nes_noise(C.c_int(P), C.c_int(member_offset), C.c_int(n_members), C.c_uint32(seed), C.c_uint32(generation),
                                  C.c_float(noise_std), _ptr(eps), stream), "le_nes_noise")
    return eps


def nes_update(theta, pop, seed, generation, noise_std, weight_decay, coef, sign):
    """update_env (agents/GTN_master.py:267-298) in place on theta; coef/sign [pop] f32 CUDA."""
    assert coef.device == theta.device and sign.device == theta.device, "theta, coef and sign must live on the same GPU"
    with _on(theta) as stream:
        check(_lib().le_nes_update(_ptr(_dev(theta, _F32)), C.c_int(theta.numel()), C.c_int(pop), C.c_uint32(seed), C.c_uint32(generation),
                                   C.c_float(noise_std), C.c_double(weight_decay), _ptr(_dev(coef, _F32)), _ptr(_dev(sign, _F32)), stream),
              "le_nes_update")


def nes_partial_update(P, member_lo, member_hi, seed, generation, noise_std, coef, sign):
    delta = torch.empty(P, dtype=_F32, device=coef.device)
    with _on(coef) as stream:
        check(_lib().le_nes_partial_update(_ptr(delta), C.c_int(P), C.c_int(member_lo), C.c_int(member_hi), C.c_uint32(seed),
                                           C.c_uint32(generation), C.c_float(noise_std), _ptr(_dev(coef, _F32)), _ptr(_dev(sign, _F32)),
                                           stream), "le_nes_partial_update")
    return delta


# ---------------------------------------------------------------------------------------------------------
def td3_param_counts(tcfg):
    a, c = C.c_int(), C.c_int()
    check(_lib().le_td3_param_counts(C.byref(tcfg), C.byref(a), C.byref(c)), "le_td3_param_counts")
    return a.value, c.value


class Td3Buffers(object):
    """Device buffers of one le_td3_run call, sized for `tcfg0` (the maxima configuration of the launch); the counterpart of
    InnerLoopBuffers for TD3_discrete_vary lanes."""

    def __init__(self, tcfg0, n_lanes, n_env, device, n_cfg=1, trace_cap=0, want_actor_final=False):
        assert isinstance(tcfg0, Td3Cfg)
        self.cfg, self.n_lanes, self.n_env, self.device = tcfg0, n_lanes, n_env, device
        c = tcfg0.base
        ws = _lib().le_td3_workspace_bytes(C.byref(tcfg0), C.c_int(n_lanes), C.c_int(n_env))
        if ws < 0:
            check(int(ws), "le_td3_workspace_bytes")
        self.workspace = torch.empty(int(ws), dtype=torch.uint8, device=device)
        self.p_actor, self.p_critic = td3_param_counts(tcfg0)
        rs = max(c.train_episodes, 1)
        self.out = torch.zeros((n_lanes, C.sizeof(LaneOut)), dtype=torch.uint8, device=device)
        self.rewards = torch.zeros((n_lanes, rs), dtype=_F64, device=device)
        self.lengths = torch.zeros((n_lanes, rs), dtype=_I32, device=device)
        self.test_rewards = torch.zeros((n_lanes, c.test_episodes), dtype=_F64, device=device)
        self.actor_final = torch.zeros((n_lanes, self.p_actor), dtype=_F32, device=device) if want_actor_final else None
        self.cfg_dev = torch.zeros((n_cfg, C.sizeof(Td3Cfg)), dtype=torch.uint8, device=device)
        self.trace = None
        if trace_cap > 0:
            self.trace = dict(cap=trace_cap,
                              action=torch.full((trace_cap,), -1, dtype=_I32, device=device),
                              explore=torch.zeros(trace_cap, dtype=_I32, device=device),
                              next_state=torch.zeros((trace_cap, c.sd), dtype=_F32, device=device),
                              reward=torch.zeros(trace_cap, dtype=_F32, device=device),
                              done=torch.zeros(trace_cap, dtype=_F32, device=device),
                              loss=torch.full((trace_cap,), float("nan"), dtype=_F32, device=device),
                              qgap=torch.full((trace_cap,), float("nan"), dtype=_F32, device=device))

    def results(self):
        return np.frombuffer(self.out.cpu().numpy().tobytes(), dtype=lane_out_dtype())


def td3_run(bufs, tcfgs, env_theta, env_index, keys, inits=None, trace_lane=0):
    """le_td3_run on the current stream: n_lanes TD3_discrete_vary lanes, lane i with tcfgs[i] (or one Td3Cfg for all).

    Every configuration must fit the maxima `bufs.cfg` (q_hidden, q_layers, batch_size).  env_theta [n_env, P_se] CUDA f32 (None
    for ENV_REAL); env_index [n_lanes] int32 or None; keys [n_lanes, 2] int32 CUDA (keys_tensor).  inits: None (device init from
    the P_TD3_INIT stream) or (actor, critic_1, critic_2) CUDA f32 [1 or n_lanes, P of bufs.cfg] with each lane's own vector first
    in its row."""
    if isinstance(tcfgs, Td3Cfg):
        tcfgs = [tcfgs]
    n_cfg = len(tcfgs)
    assert n_cfg in (1, bufs.n_lanes) and bufs.cfg_dev.shape[0] == n_cfg
    m = bufs.cfg.base
    for t in tcfgs:
        if t.base.q_hidden > m.q_hidden or t.base.q_layers > m.q_layers or t.base.batch_size > m.batch_size:
            raise ValueError("a lane configuration exceeds the maxima the buffers were sized for")
    raw = b"".join(bytes(t) for t in tcfgs)
    if getattr(bufs, "_cfg_raw", None) != raw:
        bufs.cfg_dev.copy_(torch.frombuffer(bytearray(raw), dtype=torch.uint8).reshape(n_cfg, -1), non_blocking=False)
        bufs._cfg_raw = raw
    keys = _dev(keys, _I32)
    assert keys.numel() == 2 * bufs.n_lanes
    a0 = q1 = q2 = None
    n_init = 0
    if inits is not None:
        a0, q1, q2 = inits
        n_init = a0.shape[0]
        assert a0.shape == (n_init, bufs.p_actor) and q1.shape == q2.shape == (n_init, bufs.p_critic) and n_init in (1, bufs.n_lanes)
        a0, q1, q2 = (_dev(x, _F32) for x in (a0, q1, q2))
    tr = None
    if bufs.trace is not None:
        tr = Trace()
        tr.cap = bufs.trace["cap"]
        for n in ("action", "explore", "next_state", "reward", "done", "loss", "qgap"):
            setattr(tr, n, bufs.trace[n].data_ptr())
    n_env = 0 if env_theta is None else env_theta.reshape(-1, max(m.env_params(), 1)).shape[0]
    with _on(bufs.workspace) as stream:
        check(_lib().le_td3_run(
            _ptr(bufs.cfg_dev), C.c_int(n_cfg), C.byref(bufs.cfg), _ptr(env_theta), C.c_int(n_env), _ptr(env_index), _ptr(keys),
            _ptr(a0), _ptr(q1), _ptr(q2), C.c_int(n_init), _ptr(bufs.actor_final), C.c_int(bufs.n_lanes), _ptr(bufs.out),
            _ptr(bufs.rewards), _ptr(bufs.lengths), _ptr(bufs.test_rewards), _ptr(bufs.workspace), C.c_int64(bufs.workspace.numel()),
            C.byref(tr) if tr is not None else None, C.c_int(trace_lane), stream), "le_td3_run")


def td3_run_host(tcfg, env_theta, env_index, keys, actor_init, critic1_init, critic2_init, trace_cap=0, trace_lane=0, device=0):
    """le_td3_run_host: n TD3_discrete_vary lanes (train with per-episode test + final test), HOST numpy buffers in and out.
    actor_init [1 or n, P_actor], critic*_init [1 or n, P_critic].  Returns a dict of arrays (+ 'trace' when trace_cap > 0)."""
    assert isinstance(tcfg, Td3Cfg)
    c = tcfg.base
    keys = np.ascontiguousarray(np.asarray(keys, dtype=np.uint32).reshape(-1, 2))
    n = keys.shape[0]
    Pa, Pc = td3_param_counts(tcfg)
    a0 = np.ascontiguousarray(actor_init, np.float32).reshape(-1, Pa)
    q1 = np.ascontiguousarray(critic1_init, np.float32).reshape(-1, Pc)
    q2 = np.ascontiguousarray(critic2_init, np.float32).reshape(-1, Pc)
    assert a0.shape[0] == q1.shape[0] == q2.shape[0] and a0.shape[0] in (1, n)
    th, n_env = None, 0
    if env_theta is not None:
        th = np.ascontiguousarray(env_theta, np.float32).reshape(-1, c.env_params())
        n_env = th.shape[0]
    ei = None if env_index is None else np.ascontiguousarray(env_index, np.int32)
    af = np.zeros((n, Pa), np.float32)
    out = np.zeros(n, dtype=lane_out_dtype())
    rs = max(c.train_episodes, 1)
    rewards, lengths = np.zeros((n, rs), np.float64), np.zeros((n, rs), np.int32)
    test_rewards = np.zeros((n, c.test_episodes), np.float64)
    tr, trace = None, None
    if trace_cap > 0:
        trace = dict(action=np.zeros(trace_cap, np.int32), explore=np.zeros(trace_cap, np.int32), next_state=np.zeros((trace_cap, c.sd), np.float32),
                     reward=np.zeros(trace_cap, np.float32), done=np.zeros(trace_cap, np.float32), loss=np.zeros(trace_cap, np.float32))
        tr = Trace()
        tr.cap = trace_cap
        for k, v in trace.items():
            setattr(tr, k, v.ctypes.data)

    def p(a):
        return a.ctypes.data_as(C.c_void_p) if a is not None else None
    check(_lib().le_td3_run_host(C.byref(tcfg), p(th), C.c_int(n_env), p(ei), p(keys), p(a0), p(q1), p(q2), C.c_int(a0.shape[0]), p(af),
                                 C.c_int(n), p(out), p(rewards), p(lengths), p(test_rewards), C.byref(tr) if tr is not None else None,
                                 C.c_int(trace_lane), C.c_int(device)), "le_td3_run_host")
    return dict(out=out, rewards=rewards, lengths=lengths, test_rewards=test_rewards, actor_final=af, trace=trace)
