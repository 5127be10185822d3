"""GPU tests of the TD3_discrete_vary learn() step (le_td3_learn, the device function the TD3 lanes run after
replay_buffer.sample): every learn() call of the unmodified reference (tests/golden/td3_learn_*.npz), the yaml and vary_hp shapes
against the CPU restatement (c_oracle.td3_learn, pinned to the reference at 1 ulp by the same goldens), and the Gumbel temperature
schedule around its clamp.  All six nets are compared after every call, at the shapes the dense layers take their tiled GEMM path
(> 16 rows); the Adam moments carry each call's gradients and are compared norm-wise."""
import concurrent.futures as cf

import numpy as np
import pytest
import torch

from oracle import c_oracle
from tests.helpers import assert_params_close, load_golden, rel_err

pytestmark = pytest.mark.gpu

NETS = ("actor", "actor_target", "critic_1", "critic_target_1", "critic_2", "critic_target_2")
ADAM = ("m_a", "v_a", "m_c1", "v_c1", "m_c2", "v_c2")
TANH, RELU, LEAKY = 0, 1, 2
# default_config_{cartpole,acrobot}_syn_env.yaml, td3_discrete_vary
YAML = dict(gamma=0.9989, lr=0.0017496, tau=0.0724303, policy_std=0.2225286, policy_std_clip=0.5, max_action=1.0, T0=2.3076235)
LOSS_RTOL = 1e-5
MOMENT_RTOL = 1e-4


def _tcfg(sd, ad, H, L, act, B, policy_delay, hard, gamma, lr, tau, policy_std, policy_std_clip, max_action, T0):
    from learning_environments_b200._abi import Td3Cfg
    t = Td3Cfg()
    b = t.base
    b.sd, b.ad, b.q_hidden, b.q_layers, b.q_act, b.batch_size = sd, ad, H, L, act, B
    b.gamma, b.lr, b.tau = gamma, lr, tau
    b.beta1, b.beta2, b.adam_eps = 0.9, 0.999, 1e-8            # torch.optim.Adam defaults
    t.policy_delay, t.gumbel_hard = policy_delay, int(hard)
    t.policy_std, t.policy_std_clip, t.gumbel_temp, t.max_action = policy_std, policy_std_clip, T0, max_action
    return t


def _hyper(t):
    b = t.base
    return dict(gamma=b.gamma, tau=b.tau, lr=b.lr, policy_delay=t.policy_delay, max_action=t.max_action, policy_std=t.policy_std,
                policy_std_clip=t.policy_std_clip, gumbel_hard=t.gumbel_hard)


def _dims(t):
    b = t.base
    return (b.sd, b.ad, b.q_hidden, b.q_layers, b.q_act)


def _layers(sd, ad, H, L):
    """(in, out) of every nn.Linear of the actor and of a critic, state_dict order."""
    hid = [(H, H)] * (max(L, 1) - 1)
    return [(sd, H)] + hid + [(H, ad)], [(sd + ad, H)] + hid + [(H, 1)]


def _temp(T0, total_it):
    """self.gumbel_temp_annealed of the learn() call that starts at self.total_it = total_it."""
    return float(np.float32(np.linspace(T0, T0 / 20, 2000)[min(total_it, 1999)]))


def _mlp64(theta, dims, act, x):
    """float64 forward of the state_dict-ordered parameter vector `theta` on rows x."""
    p, h = 0, np.asarray(x, np.float64)
    for i, (n_in, n_out) in enumerate(dims):
        W = theta[p:p + n_in * n_out].astype(np.float64).reshape(n_out, n_in)
        p += n_in * n_out
        h = h @ W.T + theta[p:p + n_out]
        p += n_out
        if i < len(dims) - 1:
            h = np.tanh(h) if act == TANH else np.maximum(h, (0.01 if act == LEAKY else 0.0) * h)
    return h


def _argmax_margin(theta, dims, act, x, expo, temp, max_action):
    """Smallest relative top-two gap (y1 - y2) / y1 over the rows of the hard Gumbel-softmax argmax (float64)."""
    z = (_mlp64(theta, dims, act, x) * max_action - np.log(np.asarray(expo, np.float64))) / temp
    y = np.exp(z - z.max(axis=1, keepdims=True))
    y = np.sort(y / y.sum(axis=1, keepdims=True), axis=1)
    return float(np.min((y[:, -1] - y[:, -2]) / y[:, -1]))


def _assert_no_near_tie(t, nets, rows, expo_target, expo_actor, temp, updates, what):
    """A hard Gumbel argmax whose top two are closer than fp32 rounding could flip between two correct implementations and change a
    whole row of the update: the inputs must keep every such margin >= 1e-5 so that a failure points at the kernel, not at a draw."""
    if not t.gumbel_hard:
        return
    sd, ad, H, L, act = _dims(t)
    da, _ = _layers(sd, ad, H, L)
    m = _argmax_margin(nets["actor_target"], da, act, rows[:, sd + ad:2 * sd + ad], expo_target, temp, t.max_action)
    if updates:
        m = min(m, _argmax_margin(nets["actor"], da, act, rows[:, :sd], expo_actor, temp, t.max_action))
    assert m >= 1e-5, "%s: a hard Gumbel argmax is a near-tie (relative margin %.3g): pick another seed" % (what, m)


class DeviceLanes(object):
    """n lanes of one Td3Cfg held in CUDA tensors between le_td3_learn calls."""

    def __init__(self, t, nets, adam, counters):
        self.t = t
        cuda = lambda a: torch.from_numpy(np.ascontiguousarray(np.stack(a))).cuda()
        self.nets = {k: cuda([n[k] for n in nets]) for k in NETS}
        self.adam = {k: cuda([a[k] for a in adam]) for k in ADAM}
        self.counters = torch.tensor(np.asarray(counters, np.int32).reshape(-1, 3)).cuda()

    def learn(self, rows, noise, expo_target, expo_actor):
        from learning_environments_b200 import ops
        cuda = lambda a: torch.from_numpy(np.ascontiguousarray(np.stack(a), np.float32)).cuda()
        loss = ops.td3_learn(self.t, self.nets, self.adam, self.counters, cuda(rows), cuda(noise), cuda(expo_target), cuda(expo_actor))
        torch.cuda.synchronize()
        return (loss.cpu().numpy(), {k: v.cpu().numpy() for k, v in self.nets.items()}, {k: v.cpu().numpy() for k, v in self.adam.items()},
                self.counters.cpu().numpy())


def _moment_err(got, want):
    """Norm-wise relative difference of two Adam moment vectors (0 when both are zero)."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


def _adam_slack(t, m_got, v_got, m_want, v_want, steps):
    """How far apart the Adam steps lr m / (bc1 (sqrt(v / bc2) + eps)) of the two moment pairs are.  A gradient that is a
    near-cancelling sum of B row terms keeps an fp32 rounding error of ~eps32 x the sum of |terms| whatever the summation order;
    where |g| is comparable to Adam's eps (first steps from zero moments: step = lr g / (|g| + eps)) that error is a visible
    fraction of lr.  The moments themselves are held norm-wise to MOMENT_RTOL."""
    b = t.base
    bc1, bc2 = 1.0 - b.beta1 ** steps, 1.0 - b.beta2 ** steps
    step = lambda m, v: b.lr * np.asarray(m, np.float64) / (bc1 * (np.sqrt(np.asarray(v, np.float64) / bc2) + b.adam_eps))
    return np.abs(step(m_got, v_got) - step(m_want, v_want))


def _compare(t, i, k, loss, nets, adam, ref_loss, ref_nets, ref_adam, what, worst, loss_rtol=LOSS_RTOL, slack=None, counters=None,
             updated=True):
    """Critic loss to loss_rtol; every net as helpers.assert_params_close, where a parameter may in addition differ by the Adam
    slack (_adam_slack) its moments accumulated over the calls so far (`slack`: per-lane dict, carried between calls; a target
    net inherits tau x its net's slack at every Polyak update); the six Adam moment vectors to MOMENT_RTOL norm-wise."""
    e = rel_err(loss[i], ref_loss)
    worst["loss"] = max(worst.get("loss", 0.0), e)
    assert e < loss_rtol, "%s call %d: critic loss %r vs %r" % (what, k, float(loss[i]), ref_loss)
    if adam is not None:
        b = t.base
        # a ReLU-family unit whose pre-activation lies within rounding of the kink takes the other slope (1 vs 0 / 0.01) for
        # that row in one of the two implementations: its fan-in gradient then differs by one row's term, ~1/sqrt(B H) of the
        # gradient norm; admit two such (row, unit) pairs per call
        mrtol = MOMENT_RTOL if b.q_act == TANH else MOMENT_RTOL + 2.0 / np.sqrt(b.batch_size * b.q_hidden)
        for n in ADAM:
            e = _moment_err(adam[n][i], ref_adam[n])
            worst["moment"] = max(worst.get("moment", 0.0), e)
            assert e < mrtol, "%s call %d: Adam %s differs by %.3g (norm-wise)" % (what, k, n, e)
    if slack is not None:
        tau = t.base.tau
        for net, online, target, steps in (("a", "actor", "actor_target", counters[0]), ("c1", "critic_1", "critic_target_1", counters[1]),
                                           ("c2", "critic_2", "critic_target_2", counters[1])):
            if net != "a" or updated:
                slack[online] = slack.get(online, 0.0) + _adam_slack(t, adam["m_" + net][i], adam["v_" + net][i], ref_adam["m_" + net],
                                                                       ref_adam["v_" + net], steps)
            if updated:
                slack[target] = (1 - tau) * slack.get(target, 0.0) + tau * slack.get(online, 0.0)
    for n in NETS:
        d = np.abs(nets[n][i].astype(np.float64) - ref_nets[n])
        worst["param/lr"] = max(worst.get("param/lr", 0.0), float(d.max() / t.base.lr))
        want, got = ref_nets[n], nets[n][i]
        if slack is not None and n in slack:
            excess = d - slack[n]
            worst["param-slack/lr"] = max(worst.get("param-slack/lr", 0.0), float(excess.max() / t.base.lr))
            assert excess.max() <= 0.02 * t.base.lr, "%s call %d %s: |diff| exceeds 2%% of lr + the Adam slack by %.3g" % (
                what, k, n, excess.max())
            rel = np.maximum(excess, 0.0) / np.maximum(np.abs(want), 1e-2)
            assert (rel < 5e-5).mean() >= 0.99, "%s call %d %s: only %.2f%% of the parameters within 5e-5" % (what, k, n, 100 * (rel < 5e-5).mean())
        else:
            assert_params_close(got, want, t.base.lr, "%s call %d %s" % (what, k, n))


# ---- 1. the reference's own learn() calls ------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["cartpole", "cartpole_soft", "acrobot"])
def test_td3_learn_replays_the_reference_learn_calls(tag):
    """Every learn() call of td3_learn_<tag>.npz (hard / soft Gumbel-softmax, tanh / relu / leakyrelu, 1 and 2 hidden layers,
    policy_delay 1 / 2 / 3, CartPole and Acrobot) through le_td3_learn on two identical lanes: the lanes agree bit for bit, the
    six nets match the reference after every call, the policy is updated on exactly the reference's calls, and the critic loss
    (not stored by the reference) matches the restatement's."""
    g = load_golden("td3_learn_%s.npz" % tag)
    sd, ad = int(g["sd"]), int(g["ad"])
    steps, B = g["rows"].shape[:2]
    t = _tcfg(sd, ad, int(g["hidden"]), int(g["layers"]), int(g["act"]), B, int(g["policy_delay"]), int(g["gumbel_hard"]),
              float(g["gamma"]), float(g["lr"]), float(g["tau"]), float(g["policy_std"]), float(g["policy_std_clip"]),
              float(g["max_action"]), float(g["temps"][0]))
    ref = {n: g["init_" + n].astype(np.float32).copy() for n in NETS}
    ref_adam = {n: np.zeros_like(ref["actor" if n.endswith("_a") else "critic_1"]) for n in ADAM}
    lanes = DeviceLanes(t, [ref, ref], [ref_adam, ref_adam], np.zeros((2, 3)))
    ref_cnt = [0, 0]
    worst = {}
    for k in range(steps):
        assert _temp(t.gumbel_temp, k) == float(np.float32(g["temps"][k]))
        _assert_no_near_tie(t, ref, g["rows"][k], g["expo_target"][k], g["expo_actor"][k], float(g["temps"][k]), bool(g["updated"][k]),
                            "%s call %d" % (tag, k))
        loss, nets, adam, cnt = lanes.learn([g["rows"][k]] * 2, [g["policy_noise"][k]] * 2, [g["expo_target"][k]] * 2,
                                            [g["expo_actor"][k]] * 2)
        ref_loss, _ = c_oracle.td3_learn(_dims(t), _hyper(t), ref, ref_adam, ref_cnt, k + 1, g["rows"][k], g["policy_noise"][k],
                                         g["expo_target"][k], g["expo_actor"][k], float(g["temps"][k]))
        assert loss[0] == loss[1] and all(np.array_equal(v[0], v[1]) for d in (nets, adam) for v in d.values()), "lanes differ"
        assert cnt[0, 0] == int(g["updated"][:k + 1].sum()) and cnt[0, 1] == k + 1 and cnt[0, 2] == k + 1, (k, cnt[0])
        want = {n: g["after_" + n][k] for n in NETS}
        _compare(t, 0, k, loss, nets, None, ref_loss, want, None, tag, worst)
    print(tag, "max errors", worst)


# ---- 2. the yaml and vary_hp shapes against the restatement ----------------------------------------------------------------
def _random_lane(t, rng, counters=(0, 0, 0), warm_adam=False):
    """Seeded nets (torch's default nn.Linear init distribution; targets a little apart from their nets so that every Polyak
    update is visible), optionally a warm Adam state of `counters` earlier steps."""
    sd, ad, H, L, _ = _dims(t)
    dims_a, dims_c = _layers(sd, ad, H, L)

    def init(dims):
        parts = []
        for n_in, n_out in dims:
            bnd = 1.0 / np.sqrt(n_in)
            parts += [rng.uniform(-bnd, bnd, n_out * n_in), rng.uniform(-bnd, bnd, n_out)]
        return np.concatenate(parts).astype(np.float32)

    nets = {}
    for n in ("actor", "critic_1", "critic_2"):
        th = init(dims_a if n == "actor" else dims_c)
        nets[n] = th
        nets[n.replace("critic", "critic_target") if n != "actor" else "actor_target"] = (th * (1 + 0.05 * rng.standard_normal(th.size))).astype(np.float32)
    adam = {}
    for net, steps in (("a", counters[0]), ("c1", counters[1]), ("c2", counters[1])):
        P = nets["actor" if net == "a" else "critic_1"].size
        g = 1e-3 * rng.standard_normal(P)                       # moments of earlier gradients of this scale: |m| <= sqrt(v)
        warm = warm_adam and steps > 0
        adam["m_" + net] = (0.5 * g * rng.uniform(-1, 1, P) if warm else np.zeros(P)).astype(np.float32)
        adam["v_" + net] = (g * g * rng.uniform(1, 2, P) if warm else np.zeros(P)).astype(np.float32)
    return nets, adam, list(counters)


def _random_batch(t, rng):
    """One minibatch in the replay rows' layout: states in [-1, 1], noisy one-hot action vectors, rewards in [-1, 1], 10 % dones;
    the policy noise and both Gumbel draws."""
    b = t.base
    sd, ad, B = b.sd, b.ad, b.batch_size
    rows = np.zeros((B, 2 * sd + ad + 2), np.float32)
    rows[:, :sd] = rng.uniform(-1, 1, (B, sd))
    rows[:, sd:sd + ad] = np.eye(ad)[rng.randint(0, ad, B)] + 0.04 * rng.standard_normal((B, ad))
    rows[:, sd + ad:2 * sd + ad] = rng.uniform(-1, 1, (B, sd))
    rows[:, 2 * sd + ad] = rng.uniform(-1, 1, B)
    rows[:, 2 * sd + ad + 1] = rng.uniform(size=B) < 0.1
    draws = [rng.standard_normal((B, ad)), rng.exponential(size=(B, ad)), rng.exponential(size=(B, ad))]
    return [rows] + [np.maximum(d, 1e-30).astype(np.float32) if i else d.astype(np.float32) for i, d in enumerate(draws)]


def _run_vs_restatement(t, calls, seed, starts=((0, 0, 0),) * 3, warm_adam=False, loss_rtol=LOSS_RTOL):
    """len(starts) lanes with their own seeded nets, rows and draws, `calls` consecutive le_td3_learn launches; after every call
    each lane is held to its own restatement (run on a thread pool).  Returns the largest errors seen."""
    rng = np.random.RandomState(seed)
    refs = [_random_lane(t, rng, s, warm_adam) for s in starts]
    lanes = DeviceLanes(t, [r[0] for r in refs], [r[1] for r in refs], [r[2] for r in refs])
    worst, slacks = {}, [dict() for _ in refs]
    T0, delay = t.gumbel_temp, t.policy_delay
    with cf.ThreadPoolExecutor(len(refs)) as ex:
        for k in range(calls):
            batches = [_random_batch(t, rng) for _ in refs]
            for i, (nets, _, cnt) in enumerate(refs):
                _assert_no_near_tie(t, nets, batches[i][0], batches[i][2], batches[i][3], _temp(T0, cnt[2]), (cnt[2] + 1) % delay == 0,
                                    "seed %d lane %d call %d" % (seed, i, k))
            loss, nets, adam, cnt = lanes.learn(*[[bt[j] for bt in batches] for j in range(4)])

            def ref_call(i):
                r_nets, r_adam, r_cnt = refs[i]
                rows, noise, expo_t, expo_a = batches[i]
                it = r_cnt[2]
                tc = r_cnt[:2]
                closs, _ = c_oracle.td3_learn(_dims(t), _hyper(t), r_nets, r_adam, tc, it + 1, rows, noise, expo_t, expo_a, _temp(T0, it))
                r_cnt[:] = tc + [it + 1]
                return closs

            updated = [(r[2][2] + 1) % delay == 0 for r in refs]
            ref_losses = list(ex.map(ref_call, range(len(refs))))
            for i, (r_nets, r_adam, r_cnt) in enumerate(refs):
                assert list(cnt[i]) == r_cnt, (i, k, cnt[i], r_cnt)
                _compare(t, i, k, loss, nets, adam, ref_losses[i], r_nets, r_adam, "seed %d lane %d" % (seed, i), worst, loss_rtol,
                         slack=slacks[i], counters=r_cnt, updated=updated[i])
    return worst


SHAPES = {
    # name: (sd, ad, hidden, hidden_layer, batch, activation, hard, policy_delay, calls)
    "yaml_cartpole": (4, 2, 510, 2, 122, TANH, True, 1, 6),
    "yaml_acrobot": (6, 3, 510, 2, 122, TANH, True, 1, 6),
    "vary_min": (4, 2, 170, 1, 40, TANH, True, 2, 6),
    "vary_max": (6, 3, 1530, 3, 366, TANH, True, 2, 2),
    "ragged_B300": (4, 2, 200, 2, 300, TANH, True, 2, 6),     # not a multiple of the 128-row tile; threads own two rows
    "B17": (6, 3, 96, 2, 17, TANH, True, 2, 6),               # one row above the thin path
    "B1": (4, 2, 64, 1, 1, TANH, True, 1, 6),
    "soft_relu_delay3": (6, 3, 256, 2, 96, RELU, False, 3, 6),
    "leaky": (4, 2, 320, 3, 64, LEAKY, True, 2, 6),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_td3_learn_vs_restatement_at_the_yaml_and_vary_hp_shapes(name):
    """Three lanes per launch, each with its own seeded nets, rows and draws, against the C restatement after every call: the
    critic loss to 1e-5 relative, the six nets as helpers.assert_params_close beyond the Adam slack of _adam_slack, the six Adam
    moment vectors to 1e-4 norm-wise (ReLU-family nets: + the kink allowance of _compare).
    Measured on one NVIDIA B200 (power limit 1000 W), largest over lanes and calls, tanh nets: critic loss 6.8e-7 relative (B1;
    6.3e-7 at 510 x 2, 5.5e-7 at 1530 x 3); moments 4.2e-5 norm-wise (510 x 2 Acrobot; 4.3e-6 at 1530 x 3); parameters 0.094 lr at
    1530 x 3, 0.061 lr at 510 x 2, <= 0.012 lr elsewhere, of which at most 5.3e-5 lr beyond the Adam slack.  Leaky (320 x 3, B 64):
    one kink flip moved the critic-2 moments by 3.5e-3 norm-wise (allowance 1.4e-2), a parameter by 0.6 lr (5.1e-5 lr beyond the
    Adam slack) and the loss by 1.8e-6."""
    sd, ad, H, L, B, act, hard, delay, calls = SHAPES[name]
    t = _tcfg(sd, ad, H, L, act, B, delay, hard, YAML["gamma"], YAML["lr"], YAML["tau"], YAML["policy_std"], YAML["policy_std_clip"],
              YAML["max_action"], YAML["T0"])
    worst = _run_vs_restatement(t, calls, seed=1000 + sorted(SHAPES).index(name))
    print(name, "max errors", worst)


# ---- 3. the Gumbel temperature schedule -----------------------------------------------------------------------------------
@pytest.mark.parametrize("hard", [True, False])
def test_td3_learn_temperature_schedule_and_clamp(hard):
    """Lanes that start at self.total_it = 0, 1998, 1999 and 2500 (warm Adam state): the temperature is
    np.linspace(T0, T0/20, 2000)[min(total_it, 1999)] in float32 — at the end of the schedule one step of it is ~1 % — and the
    delayed policy update follows total_it across the clamp."""
    t = _tcfg(4, 2, 128, 2, TANH, 64, 2, hard, YAML["gamma"], YAML["lr"], YAML["tau"], YAML["policy_std"], YAML["policy_std_clip"],
              YAML["max_action"], YAML["T0"])
    starts = [(it // 2, it, it) for it in (0, 1998, 1999, 2500)]
    worst = _run_vs_restatement(t, 3, seed=7 + int(hard), starts=starts, warm_adam=True)
    print("hard" if hard else "soft", "max errors", worst)
