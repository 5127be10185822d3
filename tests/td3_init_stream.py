"""TEST INFRASTRUCTURE ONLY — numpy restatement of the Philox stream the TD3 lanes draw their initial weights from when
le_td3_run gets no init arrays (csrc/le_td3.cu td3_init_net).  It extends the stream table of oracle/philox.py:

  P_TD3_INIT    (block, net)           net 0 actor, 1 critic_1, 2 critic_2; parameter p (state_dict order) takes word p & 3 of
                                       block p >> 2 (counter (p >> 2, net, P_TD3_INIT, 0), the lane key) and becomes
                                       (2 u - 1) / sqrt(fan_in), u = (w + 0.5) * 2^-32, in float64 rounded to float32: torch's
                                       default nn.Linear init U(-1/sqrt(fan_in), +1/sqrt(fan_in)) for W and b, as P_QINIT

The stream id and counter layout keep the draws apart from the DDQN Q-net init (P_QINIT = 5: counter (block, 0, 5, 0)).
"""
import numpy as np

from oracle.philox import philox4x32_np

P_TD3_INIT = 10


def td3_net_init(key, net, layer_dims):
    """Initial parameters (float32, state_dict order) of TD3 net `net` (0 actor, 1 critic_1, 2 critic_2);
    layer_dims: [(fan_in, fan_out), ...] of its nn.Linear layers."""
    bounds = np.concatenate([np.full(i * o + o, 1.0 / np.sqrt(float(i))) for i, o in layer_dims])
    n = bounds.size
    nblk = (n + 3) // 4
    w = philox4x32_np(np.arange(nblk, dtype=np.uint64), np.uint64(net), P_TD3_INIT, 0, key[0], key[1]).reshape(-1)[:n]
    u = (w.astype(np.float64) + 0.5) * (1.0 / 4294967296.0)
    return ((2.0 * u - 1.0) * bounds).astype(np.float32)


def td3_init(key, sd, ad, hidden, layers):
    """(actor, critic_1, critic_2) initial parameters of a TD3_discrete_vary lane with key `key`."""
    L = max(int(layers), 1)
    actor = [(sd, hidden)] + [(hidden, hidden)] * (L - 1) + [(hidden, ad)]
    critic = [(sd + ad, hidden)] + [(hidden, hidden)] * (L - 1) + [(hidden, 1)]
    return td3_net_init(key, 0, actor), td3_net_init(key, 1, critic), td3_net_init(key, 2, critic)
