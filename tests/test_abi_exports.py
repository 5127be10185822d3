"""The C-ABI library builds, loads without a GPU and exports every symbol include/le_b200.h declares."""
import ctypes as C
import os
import re

from learning_environments_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "le_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(le_[a-z0-9_]+)\s*\(", src)))


def test_library_loads_and_exports_all_declared_symbols():
    from learning_environments_b200.csrc import build as le_build
    le_build.build()
    lib = _abi.load_library()
    declared = _declared_symbols()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), "symbol %s declared in include/le_b200.h is not exported" % name
    assert sorted(_abi.EXPORTED_SYMBOLS) == declared
    assert lib.le_version() == 100
    assert lib.le_sizeof_lane_cfg() == C.sizeof(_abi.LaneCfg)


def test_bad_arguments_report_errors_without_gpu():
    lib = _abi.load_library()
    cfg = _abi.LaneCfg()
    cfg.sd, cfg.ad, cfg.real_env, cfg.env_kind = 5, 2, 0, 0      # no kernel set for state_dim 5
    rc = lib.le_inner_loop_workspace_bytes(C.byref(cfg), C.c_int(4), C.c_int(1))
    assert rc < 0 and b"real_env" in lib.le_last_error()
    cfg.sd, cfg.env_kind, cfg.rn_type = 4, 1, 3                   # info-vector reward type
    rc = lib.le_rn_reward(C.byref(cfg), None, C.c_int(1), C.c_int(1), None, None, None, None, None)
    assert rc == -3 and b"info vector" in lib.le_last_error()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "learning_environments_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("oracle/philox.py", "").replace("oracle/le_oracle.c", ""), \
                    "%s mentions the oracle" % os.path.join(dirpath, f)


def test_td3_cfg_layout_is_shared_by_the_binding_and_the_restatement():
    """struct le_td3_cfg (include/le_b200.h) == learning_environments_b200._abi.Td3Cfg == oracle.c_oracle.Td3Cfg field by field,
    and le_td3_param_counts (no GPU needed) agrees with the restatement's parameter counts."""
    from oracle import c_oracle
    a, b = _abi.Td3Cfg, c_oracle.Td3Cfg
    assert C.sizeof(a) == C.sizeof(b) == C.sizeof(_abi.LaneCfg) + 48
    assert [(n, getattr(a, n).offset) for n, _ in a._fields_] == [(n, getattr(b, n).offset) for n, _ in b._fields_]
    lib = _abi.load_library()
    t = _abi.Td3Cfg()
    t.base.sd, t.base.ad, t.base.q_hidden, t.base.q_layers = 6, 3, 20, 1
    pa, pc = C.c_int(), C.c_int()
    assert lib.le_td3_param_counts(C.byref(t), C.byref(pa), C.byref(pc)) == 0
    oa, oc = C.c_int(), C.c_int()
    c_oracle.lib().le_oracle_td3_params(C.c_int(6), C.c_int(3), C.c_int(20), C.c_int(1), C.byref(oa), C.byref(oc))
    assert (pa.value, pc.value) == (oa.value, oc.value) == (6 * 20 + 20 + 20 * 3 + 3, 9 * 20 + 20 + 20 + 1)


def test_td3_entry_rejects_bad_arguments_without_gpu():
    lib = _abi.load_library()
    t = _abi.Td3Cfg()
    assert lib.le_td3_run_host(C.byref(t), None, 0, None, None, None, None, None, 1, None, 1, None, None, None, None, None, 0, 0) == -1
    assert b"bad arguments" in lib.le_last_error()
    import numpy as np
    t.base.sd, t.base.ad, t.base.real_env, t.base.env_kind, t.base.rn_type = 4, 2, 0, 1, 2      # reward-network training env
    t.base.env_hidden, t.base.q_hidden, t.base.q_layers, t.base.batch_size = 8, 8, 1, 4
    t.base.train_episodes, t.base.test_episodes, t.base.max_steps, t.base.rb_size = 1, 1, 10, 100
    t.policy_delay, t.gumbel_temp = 1, 1.0
    keys = np.zeros((1, 2), np.uint32)
    buf = np.zeros(4096, np.float64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib.le_td3_run_host(C.byref(t), p(buf), 1, None, p(keys), p(buf), p(buf), p(buf), 1, None, 1, p(buf), p(buf), p(buf), p(buf), None, 0, 0)
    assert rc == -3 and b"reward-network" in lib.le_last_error()


def test_td3_learn_rejects_bad_arguments_without_gpu():
    """le_td3_learn: LE_EINVAL (-1) for NULL pointers, n < 1 and batch_size < 1; LE_EUNSUPPORTED (-3) for configurations outside the
    compiled set — every check runs before any CUDA call.  The environment fields are not checked: a learn step has none."""
    import numpy as np
    lib = _abi.load_library()
    buf = np.zeros(64, np.float32)
    p = buf.ctypes.data

    def good():
        t = _abi.Td3Cfg()
        t.base.sd, t.base.ad, t.base.q_hidden, t.base.q_layers, t.base.batch_size = 4, 2, 8, 2, 4
        t.base.env_kind, t.base.rn_type, t.base.test_episodes = 1, 3, 0          # would be rejected by the lane entry points
        t.policy_delay, t.gumbel_temp = 2, 1.0
        return t

    def call(t, n=1, null_at=None):
        ptrs = [p] * 18
        if null_at is not None:
            ptrs[null_at] = None
        return lib.le_td3_learn(C.byref(t) if t is not None else None, *ptrs[:13], n, *ptrs[13:], None)

    assert call(None) == -1
    for i in range(18):
        assert call(good(), null_at=i) == -1, "NULL argument %d accepted" % i
        assert b"bad arguments" in lib.le_last_error()
    assert call(good(), n=0) == -1
    t = good()
    t.base.batch_size = 0
    assert call(t) == -1
    for field, value in [("ad", 5), ("q_layers", 4), ("policy_delay", 0), ("gumbel_temp", 0.0), ("gumbel_temp", float("nan")),
                         ("q_act", 9), ("sd", 5), ("q_hidden", 0)]:
        t = good()
        setattr(t if field in ("policy_delay", "gumbel_temp") else t.base, field, value)
        assert call(t) == -3, (field, value)
