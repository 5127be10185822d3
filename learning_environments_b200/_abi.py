"""ctypes view of include/le_b200.h: the structs and the loader of the CUDA shared library.

The product path fails loudly when ``csrc/lible_b200.so`` is missing: there is no CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", os.environ.get("LE_LIB_NAME", "lible_b200.so"))

ACT_IDS = {"tanh": 0, "relu": 1, "leakyrelu": 2, "prelu": 3, "identity": 4}
ENV_SE, ENV_RN, ENV_REAL = 0, 1, 2
Q_DQN, Q_DUELING = 0, 1
REAL_CARTPOLE, REAL_ACROBOT = 0, 1
REAL_ENV_IDS = {"CartPole-v0": REAL_CARTPOLE, "Acrobot-v1": REAL_ACROBOT}


class LaneCfg(C.Structure):
    """struct le_lane_cfg (include/le_b200.h)."""
    _fields_ = [
        ("sd", C.c_int32), ("ad", C.c_int32),
        ("env_kind", C.c_int32), ("real_env", C.c_int32),
        ("env_hidden", C.c_int32), ("env_act", C.c_int32),
        ("env_slope", C.c_float * 3),
        ("rn_type", C.c_int32),
        ("q_hidden", C.c_int32), ("q_act", C.c_int32),
        ("batch_size", C.c_int32), ("rb_size", C.c_int32),
        ("train_episodes", C.c_int32), ("test_episodes", C.c_int32), ("init_episodes", C.c_int32),
        ("max_steps", C.c_int32), ("early_out_num", C.c_int32),
        ("use_test_env", C.c_int32), ("final_test", C.c_int32),
        ("step_budget", C.c_int64),
        ("gamma", C.c_double), ("lr", C.c_double), ("tau", C.c_double),
        ("eps_init", C.c_double), ("eps_min", C.c_double), ("eps_decay", C.c_double),
        ("early_out_virtual_diff", C.c_double), ("solved_reward", C.c_double),
        ("beta1", C.c_double), ("beta2", C.c_double), ("adam_eps", C.c_double),
        ("q_kind", C.c_int32), ("q_layers", C.c_int32), ("q_feature_dim", C.c_int32), ("same_action_num", C.c_int32),
    ]

    def copy(self):
        o = LaneCfg()
        C.memmove(C.byref(o), C.byref(self), C.sizeof(LaneCfg))
        return o

    # parameter-vector sizes (include/le_b200.h "parameter vectors")
    @staticmethod
    def mlp_params(inp, hidden, out):
        return hidden * inp + hidden + out * hidden + out

    def se_params(self):
        i = self.sd + self.ad
        return self.mlp_params(i, self.env_hidden, self.sd) + 2 * self.mlp_params(i, self.env_hidden, 1)

    def rn_params(self):
        return self.mlp_params(self.sd, self.env_hidden, 1)

    def env_params(self):
        if self.env_kind == ENV_SE:
            return self.se_params()
        if self.env_kind == ENV_RN:
            return self.rn_params()
        return 0

    def q_layer_dims(self):
        """[(in, out), ...] of every nn.Linear of the Q-net in state_dict order."""
        L = max(int(self.q_layers), 1)
        H = self.q_hidden
        if self.q_kind == Q_DQN:
            return [(self.sd, H)] + [(H, H)] * (L - 1) + [(H, self.ad)]
        fd = self.q_feature_dim
        return [(self.sd, H)] + [(H, H)] * (L - 1) + [(H, fd), (fd, fd), (fd, 1), (fd, fd), (fd, self.ad)]

    def q_params(self):
        return sum(i * o + o for i, o in self.q_layer_dims())

    def q_is_register_resident(self):
        """True when the warp-per-lane register kernel set covers this Q-net (else the general CTA-per-lane kernel)."""
        return self.q_kind == Q_DQN and self.q_layers <= 1 and self.q_hidden <= self.max_register_hidden()

    def max_register_hidden(self):
        """Widest single-hidden-layer Critic_DQN of the compiled warp-per-lane kernel sets (32 hidden units per thread-unit U;
        U in {2,4}, plus U = 6 for the CartPole shapes: DDQN_vary samples hidden_size in [19,171])."""
        return 192 if (self.sd == 4 and self.ad == 2) else 128

    def register_units(self):
        """Hidden units per thread (U) of the kernel set that runs this lane, or 0 for the general kernel."""
        if not self.q_is_register_resident():
            return 0
        return 2 if self.q_hidden <= 64 else (4 if self.q_hidden <= 128 else 6)


class Td3Cfg(C.Structure):
    """struct le_td3_cfg (include/le_b200.h): TD3_discrete_vary lanes."""
    _fields_ = [("base", LaneCfg), ("policy_delay", C.c_int32), ("gumbel_hard", C.c_int32), ("action_std", C.c_double),
                ("policy_std", C.c_double), ("policy_std_clip", C.c_double), ("gumbel_temp", C.c_double), ("max_action", C.c_double)]

    def copy(self):
        o = Td3Cfg()
        C.memmove(C.byref(o), C.byref(self), C.sizeof(Td3Cfg))
        return o

    def param_counts(self):
        """(P_actor, P_critic) as le_td3_param_counts: actor sd -> H (x L) -> ad, critics sd+ad -> H (x L) -> 1."""
        b = self.base
        L, H = max(int(b.q_layers), 1), b.q_hidden
        hidden = (L - 1) * (H * H + H)
        return b.sd * H + H + hidden + H * b.ad + b.ad, (b.sd + b.ad) * H + H + hidden + H + 1


class LaneOut(C.Structure):
    """struct le_lane_out."""
    _fields_ = [
        ("n_episodes", C.c_int32), ("timed_out", C.c_int32),
        ("train_steps", C.c_int64), ("learn_iters", C.c_int64), ("test_steps", C.c_int64),
        ("score", C.c_double),
    ]


class Trace(C.Structure):
    """struct le_trace."""
    _fields_ = [
        ("cap", C.c_int32),
        ("action", C.c_void_p), ("explore", C.c_void_p), ("next_state", C.c_void_p),
        ("reward", C.c_void_p), ("done", C.c_void_p), ("loss", C.c_void_p), ("qgap", C.c_void_p),
    ]


_lib = None


def load_library():
    """Loads csrc/lible_b200.so (built by __graft_entry__.build() / csrc/build.py). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            "learning_environments_b200: CUDA extension %s is missing — run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (there is no CPU fallback on this path)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    lib.le_last_error.restype = C.c_char_p
    lib.le_version.restype = C.c_int
    lib.le_inner_loop_workspace_bytes.restype = C.c_int64
    lib.le_td3_workspace_bytes.restype = C.c_int64
    lib.le_td3_learn.argtypes = [C.c_void_p] + [C.c_void_p] * 13 + [C.c_int] + [C.c_void_p] * 6
    lib.le_td3_learn.restype = C.c_int
    _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "le_version", "le_last_error", "le_sizeof_lane_cfg", "le_device_info", "le_bench_ffma",
    "le_se_forward", "le_rn_reward", "le_qnet_forward", "le_real_env_step", "le_td_update", "le_tc_gemm",
    "le_inner_loop_workspace_bytes", "le_inner_loop_plan", "le_inner_loop_run", "le_inner_loop_run_host",
    "le_nes_perturb", "le_nes_noise", "le_nes_update", "le_nes_partial_update",
    "le_td3_param_counts", "le_td3_workspace_bytes", "le_td3_run", "le_td3_run_host", "le_td3_learn",
]


def check(rc, what=""):
    if rc != 0:
        lib = load_library()
        msg = lib.le_last_error()
        raise RuntimeError("%s failed (%d): %s" % (what or "le_b200 call", rc, msg.decode() if msg else ""))
