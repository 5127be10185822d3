// le_td3.cu — TD3_discrete_vary lanes (agents/TD3_discrete_vary.py, models/actor_critic.py:22-36,69-76) on the CTA-per-lane
// machinery of le_general.cuh: one 256-thread CTA owns one agent — actor, two critics, three target nets, Adam state, the
// replay ring and the minibatch activations live in the lane slot's HBM workspace; every dense layer goes through the
// strided GEMM / thin paths of le_general.cuh.  td3_loop_kernel runs the agent loop shared with general_loop_kernel
// (cta_lane_loop, le_cta_lane.cuh: BaseAgent.train / test, agents/base_agent.py:64-227); this file holds the TD3 hooks:
//   select_train_action / select_test_action (:155-166): actor -> * max_action -> F.gumbel_softmax(tau, hard) + N(0,1)*action_std,
//       the environment receives argmax (agents/base_agent.py:111-114), the replay ring the action VECTOR;
//   learn (:62-119): target policy smoothing, twin target critics (min), two Adam optimizers, delayed policy update through
//       critic_1 with the straight-through Gumbel-softmax gradient, Polyak on the three targets — td3_learn_step, which
//       td3_learn_kernel (le_td3_learn: explicit minibatches and draws) runs as well.
// Every lane copies its own le_td3_cfg into shared memory and builds its actor / critic GNets there (vary_hp: per-lane
// q_hidden, q_layers, batch_size, lr, ...); the slot workspace is sized for the maxima configuration of the launch.
// Random draws: Philox streams P_TD3_EXPO / P_TD3_NORMAL (documented with the CPU restatement's stream table) and P_TD3_INIT
// (device init of the nets; restated in numpy by tests/td3_init_stream.py).
#include "le_general.cuh"
#include "le_td3_api.h"

namespace le {

constexpr uint32_t LE_P_TD3_EXPO = 8u, LE_P_TD3_NORMAL = 9u, LE_P_TD3_INIT = 10u;

// Exp(1) draw i of (phase, c0, sub): -ln((w + 0.5) * 2^-32) in fp64, rounded to fp32
__device__ __forceinline__ float td3_expo(uint32_t k0, uint32_t k1, uint32_t phase, uint32_t c0, uint32_t sub, int i) {
    const u32x4 w = philox4x32_10(c0, phase, LE_P_TD3_EXPO, (uint32_t)(i >> 2) + (sub << 16), k0, k1);
    return (float)(-log(((double)pick(w, i & 3) + 0.5) * (1.0 / 4294967296.0)));
}
// N(0,1) draw i: Box-Muller in fp64 on the word pair (2h, 2h+1) of its block (same transform as the NES noise)
__device__ __forceinline__ float td3_normal(uint32_t k0, uint32_t k1, uint32_t phase, uint32_t c0, uint32_t sub, int i) {
    const u32x4 w = philox4x32_10(c0, phase, LE_P_TD3_NORMAL, (uint32_t)(i >> 2) + (sub << 16), k0, k1);
    const int h = (i & 3) >> 1;
    const double u1 = ((double)pick(w, 2 * h) + 1.0) * (1.0 / 4294967296.0), u2 = (double)pick(w, 2 * h + 1) * (1.0 / 4294967296.0);
    const double r = sqrt(-2.0 * log(u1)), t = (2.0 * 3.14159265358979323846) * u2;
    return (float)((i & 1) ? r * sin(t) : r * cos(t));
}

// F.gumbel_softmax for one row (AD <= 4): ret = hard ? (onehot(argmax y) - y) + y : y
template <int AD>
__device__ __forceinline__ void gumbel_softmax_row(const float (&logits)[AD], const float (&expo)[AD], float tau, int hard,
                                                   float (&y)[AD], float (&ret)[AD]) {
    float z[AD], mx = -INFINITY, sum = 0.f;
#pragma unroll
    for (int k = 0; k < AD; ++k) { z[k] = __fdiv_rn(logits[k] + (-logf(expo[k])), tau); mx = fmaxf(mx, z[k]); }
#pragma unroll
    for (int k = 0; k < AD; ++k) { y[k] = expf(z[k] - mx); sum += y[k]; }
#pragma unroll
    for (int k = 0; k < AD; ++k) y[k] = __fdiv_rn(y[k], sum);
    int idx = 0;
#pragma unroll
    for (int k = 1; k < AD; ++k) if (y[k] > y[idx]) idx = k;
#pragma unroll
    for (int k = 0; k < AD; ++k) ret[k] = hard ? ((k == idx ? 1.f : 0.f) - y[k]) + y[k] : y[k];
}

// an MLP in -> H (x L) -> out as a GNet with feature layers only (torch state_dict order)
__host__ __device__ inline void tnet_build(GNet* n, int in, int H, int L, int out, int q_act) {
    int p = 0, y = 0;
    const int act = q_act == LE_ACT_TANH ? 1 : 2;
    n->kind = LE_Q_DQN; n->sd = in; n->ad = out; n->nfeat = 0;
    n->slope = q_act == LE_ACT_LEAKYRELU ? 0.01f : 0.f;
    gnet_add(&n->feat[n->nfeat++], in, H, act, &p, &y);
    for (int i = 1; i < (L > 1 ? L : 1); ++i) gnet_add(&n->feat[n->nfeat++], H, H, act, &p, &y);
    gnet_add(&n->feat[n->nfeat++], H, out, 0, &p, &y);
    n->P = p; n->sum_out = y;
}

// torch's default nn.Linear init, U(-1/sqrt(fan_in), +1/sqrt(fan_in)) for W and b (as g_init_layer), of TD3 net `net_id`
// (0 actor, 1 critic 1, 2 critic 2) from the P_TD3_INIT stream: parameter p takes word p & 3 of counter (p >> 2, net_id, P_TD3_INIT, 0)
static __device__ void td3_init_net(const GNet& n, float* th, uint32_t net_id, uint32_t k0, uint32_t k1) {
    for (int i = 0; i < n.nfeat; ++i) {
        const GLayer& l = n.feat[i];
        const double bnd = 1.0 / sqrt((double)l.in);
        for (int p = l.w_off + threadIdx.x; p < l.b_off + l.out; p += kGThreads) {
            const u32x4 w = philox4x32_10((uint32_t)(p >> 2), net_id, LE_P_TD3_INIT, 0u, k0, k1);
            th[p] = (float)((2.0 * (((double)pick(w, p & 3) + 0.5) * (1.0 / 4294967296.0)) - 1.0) * bnd);
        }
    }
}

// backward of all layers for B rows: dact holds dL/d(output layer) at its y_off (everything else is overwritten);
// grad <- parameter gradients; dX (may be null) <- dL/d(input rows), row stride dxs
static __device__ void t_net_backward(const GNet& n, const float* th, float* grad, const float* X, int xs, const float* acts, float* dact, int B,
                               float* dX, int dxs, float* sm) {
    const int S = n.sum_out;
    for (int i = n.nfeat - 1; i >= 0; --i) {
        const GLayer& l = n.feat[i];
        g_layer_bwd(l, th, grad, i > 0 ? acts + n.feat[i - 1].y_off : X, i > 0 ? S : xs, acts, dact, S, B,
                    i > 0 ? dact + n.feat[i - 1].y_off : dX, i > 0 ? S : dxs, false, n.slope, sm);
    }
}

struct TSlot {
    float *ring, *actor, *actorT, *m_a, *v_a, *g_a, *c1, *c1T, *m_c1, *v_c1, *c2, *c2T, *m_c2, *v_c2, *g_c, *X, *X2, *Xpi, *S2, *misc, *Y, *DX,
        *Aa, *A1, *D, *obs;
};

struct TRunParams {
    RunParams rp;
    const le_td3_cfg* cfg; int n_cfg;   // lane i runs cfg[n_cfg == 1 ? 0 : i] (device memory)
    GNet na_max, nc_max;                // nets of the maxima configuration: they fix the slot layout
    float* slots; int64_t slot_stride;
    int bmax, rowf;
    const float *actor_init, *c1_init, *c2_init;   // null: device init; else row lane_id * init_stride (stride 0: one row for all lanes)
    int init_stride_a, init_stride_c;
    float* actor_final; int final_stride;
};

// self.gumbel_temp_annealed of the learn() call that starts at self.total_it = total_it: np.linspace(T0, T0/20, 2000)[total_it],
// clamped at the last entry
__device__ __forceinline__ float td3_anneal_temp(double T0, int total_it) {
    const double Tstep = (T0 / 20.0 - T0) / 1999.0;
    return (float)(total_it >= 1999 ? T0 / 20.0 : (double)total_it * Tstep + T0);
}

// The three families of random draws of one learn() call, draw k of minibatch row b: the Exp(1) samples of the target
// policy's gumbel_softmax, the randn_like policy noise, the Exp(1) samples of the actor's gumbel_softmax.
// Lanes: the P_TD3_EXPO / P_TD3_NORMAL streams at phase 2 (target) / 3 (actor), counter learn_iters.
template <int AD>
struct Td3PhiloxDraws {
    uint32_t k0, k1, c0;
    __device__ __forceinline__ float expo_target(int b, int k) const { return td3_expo(k0, k1, 2u, c0, 0u, b * AD + k); }
    __device__ __forceinline__ float policy_noise(int b, int k) const { return td3_normal(k0, k1, 2u, c0, 0u, b * AD + k); }
    __device__ __forceinline__ float expo_actor(int b, int k) const { return td3_expo(k0, k1, 3u, c0, 0u, b * AD + k); }
};
// td3_learn_kernel: caller-given [B][AD] arrays
template <int AD>
struct Td3ArrayDraws {
    const float *expo_t, *noise, *expo_a;
    __device__ __forceinline__ float expo_target(int b, int k) const { return expo_t[b * AD + k]; }
    __device__ __forceinline__ float policy_noise(int b, int k) const { return noise[b * AD + k]; }
    __device__ __forceinline__ float expo_actor(int b, int k) const { return expo_a[b * AD + k]; }
};

// learn (agents/TD3_discrete_vary.py:62-119) after replay_buffer.sample, on the B rows staged in w.X ([s | action vector]),
// w.S2 (s') and w.misc ([r, d, -, -]): target policy smoothing, twin target critics (min), the critic loss and the one Adam step
// of both critics, the delayed policy update through critic_1 with the straight-through Gumbel-softmax gradient (when
// total_it, self.total_it after its increment, is a multiple of policy_delay), Polyak on the three targets.  b1pow_* / b2pow_*: beta^t of the two optimizers, advanced here.  Returns the
// critic loss.  The lane kernel and td3_learn_kernel both run this function.
template <int SD, int AD, typename Draws>
__device__ __forceinline__ float td3_learn_step(const GNet& na, const GNet& nc, const TSlot& w, const le_td3_cfg& tc, const LearnScalars& ls,
                                                float temp, int total_it, const Draws& dr, double& b1pow_a, double& b2pow_a,
                                                double& b1pow_c, double& b2pow_c, float* sm, float* red) {
    constexpr int XI = SD + AD;
    const int tid = threadIdx.x;
    const int Sa = na.sum_out, Sc = nc.sum_out, yo_a = na.feat[na.nfeat - 1].y_off, yo_c = nc.feat[nc.nfeat - 1].y_off;
    const float max_action = (float)tc.max_action, policy_std = (float)tc.policy_std, policy_clip = (float)tc.policy_std_clip;
    const int hard = tc.gumbel_hard;
    const int B = ls.batch;
    // target policy smoothing: a' = gumbel_softmax(actor_target(s')) + clip(N * policy_std)
    g_net_forward(na, w.actorT, w.S2, SD, B, w.Aa, sm);
    for (int b = tid; b < B; b += kGThreads) {
        float logits[AD], expo[AD], y[AD], ret[AD];
#pragma unroll
        for (int k = 0; k < AD; ++k) {
            logits[k] = __ldcg(w.Aa + (int64_t)b * Sa + yo_a + k) * max_action;
            expo[k] = dr.expo_target(b, k);
        }
        gumbel_softmax_row<AD>(logits, expo, temp, hard, y, ret);
#pragma unroll
        for (int i = 0; i < SD; ++i) w.X2[b * XI + i] = w.S2[b * SD + i];
#pragma unroll
        for (int k = 0; k < AD; ++k) {
            float nz = dr.policy_noise(b, k) * policy_std;
            nz = nz < -policy_clip ? -policy_clip : (nz > policy_clip ? policy_clip : nz);
            w.X2[b * XI + SD + k] = ret[k] + nz;
        }
    }
    __syncthreads();
    // target_Q = r + (1 - d) * gamma * min(Q1', Q2')
    g_net_forward(nc, w.c1T, w.X2, XI, B, w.A1, sm);
    for (int b = tid; b < B; b += kGThreads) w.misc[4 * b + 2] = __ldcg(w.A1 + (int64_t)b * Sc + yo_c);
    __syncthreads();
    g_net_forward(nc, w.c2T, w.X2, XI, B, w.A1, sm);
    for (int b = tid; b < B; b += kGThreads) {
        const float q1 = w.misc[4 * b + 2], q2 = __ldcg(w.A1 + (int64_t)b * Sc + yo_c);
        w.misc[4 * b + 2] = w.misc[4 * b] + ((1.f - w.misc[4 * b + 1]) * ls.gamma) * fminf(q1, q2);
    }
    __syncthreads();
    // critic loss and the two critic steps (one optimizer: shared step count)
    b1pow_c *= ls.beta1; b2pow_c *= ls.beta2d;
    float lsum = 0.f;
    for (int which = 0; which < 2; ++which) {
        float* cth = which ? w.c2 : w.c1;
        g_net_forward(nc, cth, w.X, XI, B, w.A1, sm);
        float lpart = 0.f;
        for (int b = tid; b < B; b += kGThreads) {
            const float e = __ldcg(w.A1 + (int64_t)b * Sc + yo_c) - w.misc[4 * b + 2];
            lpart = fmaf(e, e, lpart);
            __stcg(w.D + (int64_t)b * Sc + yo_c, ls.norm * e);
        }
        lsum += g_block_sum(lpart, red) / (float)B;
        __syncthreads();
        t_net_backward(nc, cth, w.g_c, w.X, XI, w.A1, w.D, B, nullptr, 0, sm);
        g_adam(cth, nullptr, which ? w.m_c2 : w.m_c1, which ? w.v_c2 : w.v_c1, w.g_c, nc.P, ls, b1pow_c, b2pow_c);
    }
    if (total_it % tc.policy_delay == 0) {
        // actor loss = -mean(critic_1(s, actor(s))) through the (updated) critic and the straight-through Gumbel-softmax
        g_net_forward(na, w.actor, w.X, XI, B, w.Aa, sm);
        for (int b = tid; b < B; b += kGThreads) {
            float logits[AD], expo[AD], y[AD], ret[AD];
#pragma unroll
            for (int k = 0; k < AD; ++k) {
                logits[k] = __ldcg(w.Aa + (int64_t)b * Sa + yo_a + k) * max_action;
                expo[k] = dr.expo_actor(b, k);
            }
            gumbel_softmax_row<AD>(logits, expo, temp, hard, y, ret);
#pragma unroll
            for (int i = 0; i < SD; ++i) w.Xpi[b * XI + i] = w.X[b * XI + i];
#pragma unroll
            for (int k = 0; k < AD; ++k) { w.Xpi[b * XI + SD + k] = ret[k]; w.Y[4 * b + k] = y[k]; }
        }
        __syncthreads();
        g_net_forward(nc, w.c1, w.Xpi, XI, B, w.A1, sm);
        for (int b = tid; b < B; b += kGThreads) __stcg(w.D + (int64_t)b * Sc + yo_c, -1.f / (float)B);
        __syncthreads();
        t_net_backward(nc, w.c1, w.g_c, w.Xpi, XI, w.A1, w.D, B, w.DX, XI, sm);     // only dL/d(action) is used
        for (int b = tid; b < B; b += kGThreads) {
            float dot = 0.f;
#pragma unroll
            for (int k = 0; k < AD; ++k) dot += w.Y[4 * b + k] * __ldcg(w.DX + (int64_t)b * XI + SD + k);
#pragma unroll
            for (int k = 0; k < AD; ++k)
                __stcg(w.D + (int64_t)b * Sa + yo_a + k,
                       __fdiv_rn(w.Y[4 * b + k] * (__ldcg(w.DX + (int64_t)b * XI + SD + k) - dot), temp) * max_action);
        }
        __syncthreads();
        t_net_backward(na, w.actor, w.g_a, w.X, XI, w.Aa, w.D, B, nullptr, 0, sm);
        b1pow_a *= ls.beta1; b2pow_a *= ls.beta2d;
        g_adam(w.actor, nullptr, w.m_a, w.v_a, w.g_a, na.P, ls, b1pow_a, b2pow_a);
        // Polyak on the three targets, after all three updates
        for (int p = tid; p < nc.P; p += kGThreads) {
            __stcg(w.c1T + p, ls.tau * __ldcg(w.c1 + p) + ls.one_minus_tau * __ldcg(w.c1T + p));
            __stcg(w.c2T + p, ls.tau * __ldcg(w.c2 + p) + ls.one_minus_tau * __ldcg(w.c2T + p));
        }
        for (int p = tid; p < na.P; p += kGThreads) __stcg(w.actorT + p, ls.tau * __ldcg(w.actor + p) + ls.one_minus_tau * __ldcg(w.actorT + p));
        __syncthreads();
    }
    return lsum;
}

__host__ __device__ inline int64_t tslot_floats(const GNet& na, const GNet& nc, int sd, int ad, int ring_cap, int rowf, int bmax, int64_t* offs /* [26] */) {
    const int Pa = (na.P + 3) / 4 * 4, Pc = (nc.P + 3) / 4 * 4, XI = sd + ad;
    const int SM = na.sum_out > nc.sum_out ? na.sum_out : nc.sum_out;
    int64_t o = 0;
    int k = 0;
    auto take = [&](int64_t nfl) { offs[k++] = o; o += (nfl + 3) / 4 * 4; };
    take((int64_t)ring_cap * rowf);                                     // 0 ring
    take(Pa); take(Pa); take(Pa); take(Pa); take(Pa);                   // 1..5 actor, actorT, m, v, grad
    take(Pc); take(Pc); take(Pc); take(Pc);                             // 6..9 c1, c1T, m, v
    take(Pc); take(Pc); take(Pc); take(Pc); take(Pc);                   // 10..14 c2, c2T, m, v, grad (shared critic gradient buffer)
    take((int64_t)bmax * XI); take((int64_t)bmax * XI); take((int64_t)bmax * XI);   // 15 X, 16 X2, 17 Xpi
    take((int64_t)bmax * sd); take((int64_t)bmax * 4); take((int64_t)bmax * 4); take((int64_t)bmax * XI);   // 18 S2, 19 misc, 20 Y, 21 DX
    take((int64_t)bmax * na.sum_out); take((int64_t)bmax * nc.sum_out); take((int64_t)bmax * SM);          // 22 Aa, 23 A1, 24 D
    take((int64_t)64 * sd);                                             // 25 obs (test rollouts)
    return o;
}

__device__ inline TSlot tslot_view(float* base, const GNet& na, const GNet& nc, int sd, int ad, int ring_cap, int rowf, int bmax) {
    int64_t offs[26];
    tslot_floats(na, nc, sd, ad, ring_cap, rowf, bmax, offs);
    TSlot w;
    w.ring = base + offs[0]; w.actor = base + offs[1]; w.actorT = base + offs[2]; w.m_a = base + offs[3]; w.v_a = base + offs[4];
    w.g_a = base + offs[5]; w.c1 = base + offs[6]; w.c1T = base + offs[7]; w.m_c1 = base + offs[8]; w.v_c1 = base + offs[9];
    w.c2 = base + offs[10]; w.c2T = base + offs[11]; w.m_c2 = base + offs[12]; w.v_c2 = base + offs[13]; w.g_c = base + offs[14];
    w.X = base + offs[15]; w.X2 = base + offs[16]; w.Xpi = base + offs[17]; w.S2 = base + offs[18]; w.misc = base + offs[19];
    w.Y = base + offs[20]; w.DX = base + offs[21]; w.Aa = base + offs[22]; w.A1 = base + offs[23]; w.D = base + offs[24];
    w.obs = base + offs[25];
    return w;
}

// TD3_discrete_vary agent as the hooks of cta_lane_loop
template <int SD, int AD>
struct Td3Agent {
    static constexpr int XI = SD + AD;
    const TRunParams& G;
    const TSlot w;     // sized for the maxima
    le_td3_cfg& tc;    // this lane's configuration and nets, in shared memory
    GNet& na;
    GNet& nc;
    float* sm;
    float* red;
    uint32_t k0, k1;
    LearnScalars ls;
    double b1pow_a, b2pow_a, b1pow_c, b2pow_c;
    float temp;        // self.gumbel_temp_annealed
    int total_it;
    float avec[AD];    // action vector of the current train step (its replay row)

    __device__ __forceinline__ const le_lane_cfg& begin_lane(int lane_id, uint32_t key0, uint32_t key1) {
        const int tid = threadIdx.x;
        k0 = key0; k1 = key1;
        {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(G.cfg + (G.n_cfg == 1 ? 0 : lane_id));
            uint32_t* dst = reinterpret_cast<uint32_t*>(&tc);
            for (int i = tid; i < (int)(sizeof(le_td3_cfg) / 4); i += kGThreads) dst[i] = src[i];
        }
        __syncthreads();
        if (tid == 0) {
            const le_lane_cfg& c = tc.base;
            tnet_build(&na, c.sd, c.q_hidden, c.q_layers, c.ad, c.q_act);
            tnet_build(&nc, c.sd + c.ad, c.q_hidden, c.q_layers, 1, c.q_act);
        }
        __syncthreads();
        if (G.actor_init) {
            for (int p = tid; p < na.P; p += kGThreads) w.actor[p] = G.actor_init[(int64_t)lane_id * G.init_stride_a + p];
            for (int p = tid; p < nc.P; p += kGThreads) {
                w.c1[p] = G.c1_init[(int64_t)lane_id * G.init_stride_c + p];
                w.c2[p] = G.c2_init[(int64_t)lane_id * G.init_stride_c + p];
            }
        } else {
            td3_init_net(na, w.actor, 0u, k0, k1);
            td3_init_net(nc, w.c1, 1u, k0, k1);
            td3_init_net(nc, w.c2, 2u, k0, k1);
        }
        __syncthreads();
        // targets = copies, Adam state zero (agents/TD3_discrete_vary.py:41-52)
        for (int p = tid; p < na.P; p += kGThreads) { w.actorT[p] = w.actor[p]; w.m_a[p] = 0.f; w.v_a[p] = 0.f; }
        for (int p = tid; p < nc.P; p += kGThreads) {
            w.c1T[p] = w.c1[p]; w.m_c1[p] = 0.f; w.v_c1[p] = 0.f;
            w.c2T[p] = w.c2[p]; w.m_c2[p] = 0.f; w.v_c2[p] = 0.f;
        }
        __syncthreads();
        fill_learn_scalars(ls, tc.base);
        b1pow_a = 1.0; b2pow_a = 1.0; b1pow_c = 1.0; b2pow_c = 1.0;
        temp = (float)tc.gumbel_temp;
        total_it = 0;
        return tc.base;
    }

    __device__ __forceinline__ void begin_episode(int) {}

    // actor(rows) + Gumbel-softmax + action noise for M rows held in `Xrows` (row stride xs): thread m < M handles row m.
    // Returns this thread's argmax; av <- the action vector.
    __device__ __forceinline__ int act_rows(const float* Xrows, int xs, int M, uint32_t phase, uint32_t c0, uint32_t sub_of_thread, bool active,
                                            float (&av)[AD]) {
        const int Sa = na.sum_out, yo_a = na.feat[na.nfeat - 1].y_off;
        g_net_forward(na, w.actor, Xrows, xs, M, w.Aa, sm);
        int best = 0;
        if (active) {
            float logits[AD], expo[AD], y[AD], ret[AD];
#pragma unroll
            for (int k = 0; k < AD; ++k) {
                logits[k] = __ldcg(w.Aa + (int64_t)threadIdx.x * Sa + yo_a + k) * (float)tc.max_action;
                expo[k] = td3_expo(k0, k1, phase, c0, sub_of_thread, k);
            }
            gumbel_softmax_row<AD>(logits, expo, temp, tc.gumbel_hard, y, ret);
#pragma unroll
            for (int k = 0; k < AD; ++k) {
                av[k] = ret[k] + td3_normal(k0, k1, phase, c0, sub_of_thread, k) * (float)tc.action_std;
                if (av[k] > av[best]) best = k;
            }
        }
        return best;
    }

    // select_train_action (:155-162): random before init_episodes, then the actor on row 0; `box` broadcasts the action vector
    __device__ __forceinline__ int train_action(const float (&state)[SD], int episode, int64_t train_steps, bool tracing, bool& explore,
                                                float& qgap, float* box) {
        explore = episode < tc.base.init_episodes;
        if (explore) {
            const u32x4 wa = philox4x32_10((uint32_t)train_steps, 0u, LE_P_ACT, 0u, k0, k1);
            const int action = (int)__umulhi(wa.y, (uint32_t)AD);
#pragma unroll
            for (int k = 0; k < AD; ++k) avec[k] = k == action ? 1.f : 0.f;
            return action;
        }
        const int tid = threadIdx.x;
        __syncthreads();
        if (tid < SD) __stcg(w.X + tid, state[tid]);      // row 0 of the staging area (free between learn() calls)
        __syncthreads();
        float av0[AD];
        act_rows(w.X, XI, 1, 0u, (uint32_t)train_steps, 0u, tid == 0, av0);
        if (tid == 0) {
#pragma unroll
            for (int k = 0; k < AD; ++k) box[k] = av0[k];
        }
        __syncthreads();
        int action = 0;
#pragma unroll
        for (int k = 0; k < AD; ++k) { avec[k] = box[k]; if (avec[k] > avec[action]) action = k; }
        if (tracing) qgap = relative_q_gap<AD>(avec, action);   // near-tie marker of the noisy action vector's argmax
        __syncthreads();
        return action;
    }

    // ring row: [s(SD) | a(AD) | s'(SD) | r | d | pad], with the action VECTOR
    __device__ __forceinline__ void store_row(int rb_ptr, const float (&state)[SD], int, const float (&ns)[SD], float r, float d) {
        if (threadIdx.x == 0) {
            float* row = w.ring + (int64_t)rb_ptr * G.rowf;
#pragma unroll
            for (int i = 0; i < SD; ++i) { __stcg(row + i, state[i]); __stcg(row + SD + AD + i, ns[i]); }
#pragma unroll
            for (int k = 0; k < AD; ++k) __stcg(row + SD + k, avec[k]);
            __stcg(row + 2 * SD + AD, r);
            __stcg(row + 2 * SD + AD + 1, d);
        }
    }

    // learn (:62-119): replay_buffer.sample, then the step shared with td3_learn_kernel
    __device__ __forceinline__ float learn(int64_t learn_iters, int rb_size) {
        const int tid = threadIdx.x;
        __syncthreads();
        temp = td3_anneal_temp(tc.gumbel_temp, total_it);
        total_it += 1;
        const int B = ls.batch;
        for (int b = tid; b < B; b += kGThreads) {     // replay_buffer.sample on the P_SAMPLE stream
            const u32x4 wv = philox4x32_10((uint32_t)learn_iters, (uint32_t)(b >> 2), LE_P_SAMPLE, 0u, k0, k1);
            const float* src = w.ring + (int64_t)__umulhi(pick(wv, b & 3), (uint32_t)rb_size) * G.rowf;
#pragma unroll
            for (int i = 0; i < XI; ++i) w.X[b * XI + i] = __ldcg(src + i);
#pragma unroll
            for (int i = 0; i < SD; ++i) w.S2[b * SD + i] = __ldcg(src + XI + i);
            w.misc[4 * b] = __ldcg(src + 2 * SD + AD);
            w.misc[4 * b + 1] = __ldcg(src + 2 * SD + AD + 1);
        }
        __syncthreads();
        const Td3PhiloxDraws<AD> dr{k0, k1, (uint32_t)learn_iters};
        return td3_learn_step<SD, AD>(na, nc, w, tc, ls, temp, total_it, dr, b1pow_a, b2pow_a, b1pow_c, b2pow_c, sm, red);
    }

    __device__ __forceinline__ float* test_obs() { return w.obs; }

    // select_test_action (:163-166) of test row threadIdx.x: actor + Gumbel-softmax + noise on the P_TD3 phase-1 draws
    __device__ __forceinline__ int test_action(int M, int test_call, int step, int ep0, bool running) {
        float av[AD];
        return act_rows(w.obs, SD, M, 1u, ((uint32_t)test_call << 16) | (uint32_t)step, (uint32_t)(ep0 + threadIdx.x), running, av);
    }

    __device__ __forceinline__ void end_lane(int lane_id) {
        if (G.actor_final) for (int p = threadIdx.x; p < na.P; p += kGThreads) G.actor_final[(int64_t)lane_id * G.final_stride + p] = w.actor[p];
    }
};

template <int SD, int AD>
__global__ void __launch_bounds__(kGThreads, 2) td3_loop_kernel(const TRunParams G) {
    static_assert(AD <= 4, "action vectors are handled as register arrays");
    __shared__ __align__(16) float sm[kGSmemFloats];
    __shared__ float red[32];
    __shared__ le_td3_cfg cfg_sm;
    __shared__ GNet na_sm, nc_sm;
    Td3Agent<SD, AD> ag{G, tslot_view(G.slots + (int64_t)blockIdx.x * G.slot_stride, G.na_max, G.nc_max, SD, AD, G.rp.ring_cap, G.rowf, G.bmax),
                        cfg_sm, na_sm, nc_sm, sm, red};
    cta_lane_loop<SD, AD>(G.rp, ag);
}

// le_td3_learn: one learn() call per CTA on caller-owned nets / Adam state (row blockIdx.x of each [n][P] array), explicit
// minibatch rows and draws; the activations live in the CTA's scratch slot (tslot_floats with no ring)
struct Td3LearnParams {
    le_td3_cfg tc;
    GNet na, nc;
    float *actor, *actorT, *c1, *c1T, *c2, *c2T, *m_a, *v_a, *m_c1, *v_c1, *m_c2, *v_c2;
    int32_t* counters;                                   // [n][3]: actor Adam steps, critic Adam steps, total_it
    const float *rows, *policy_noise, *expo_target, *expo_actor;
    float* loss;
    float* scratch; int64_t scratch_stride;
};

template <int SD, int AD>
__global__ void __launch_bounds__(kGThreads, 2) td3_learn_kernel(const Td3LearnParams Q) {
    static_assert(AD <= 4, "action vectors are handled as register arrays");
    __shared__ __align__(16) float sm[kGSmemFloats];
    __shared__ float red[32];
    constexpr int XI = SD + AD, ROW = 2 * SD + AD + 2;
    const int id = blockIdx.x, tid = threadIdx.x;
    const le_lane_cfg& c = Q.tc.base;
    const int B = c.batch_size;
    const int64_t pa = (int64_t)id * Q.na.P, pc = (int64_t)id * Q.nc.P;
    TSlot w = tslot_view(Q.scratch + (int64_t)id * Q.scratch_stride, Q.na, Q.nc, SD, AD, 0, 0, B);
    w.actor = Q.actor + pa; w.actorT = Q.actorT + pa; w.m_a = Q.m_a + pa; w.v_a = Q.v_a + pa;
    w.c1 = Q.c1 + pc; w.c1T = Q.c1T + pc; w.m_c1 = Q.m_c1 + pc; w.v_c1 = Q.v_c1 + pc;
    w.c2 = Q.c2 + pc; w.c2T = Q.c2T + pc; w.m_c2 = Q.m_c2 + pc; w.v_c2 = Q.v_c2 + pc;
    const float* my_rows = Q.rows + (int64_t)id * B * ROW;
    for (int b = tid; b < B; b += kGThreads) {      // the staging of the lane's replay_buffer.sample
        const float* src = my_rows + (int64_t)b * ROW;
#pragma unroll
        for (int i = 0; i < XI; ++i) w.X[b * XI + i] = src[i];
#pragma unroll
        for (int i = 0; i < SD; ++i) w.S2[b * SD + i] = src[XI + i];
        w.misc[4 * b] = src[2 * SD + AD];
        w.misc[4 * b + 1] = src[2 * SD + AD + 1];
    }
    __syncthreads();
    LearnScalars ls;
    fill_learn_scalars(ls, c);
    int32_t* cnt = Q.counters + 3 * id;
    const int t_a = cnt[0], t_c = cnt[1], it = cnt[2];
    double b1pow_a = pow(c.beta1, (double)t_a), b2pow_a = pow(c.beta2, (double)t_a);
    double b1pow_c = pow(c.beta1, (double)t_c), b2pow_c = pow(c.beta2, (double)t_c);
    const float temp = td3_anneal_temp(Q.tc.gumbel_temp, it);
    const bool update_policy = (it + 1) % Q.tc.policy_delay == 0;
    const int64_t dro = (int64_t)id * B * AD;
    const Td3ArrayDraws<AD> dr{Q.expo_target + dro, Q.policy_noise + dro, Q.expo_actor + dro};
    const float loss = td3_learn_step<SD, AD>(Q.na, Q.nc, w, Q.tc, ls, temp, it + 1, dr, b1pow_a, b2pow_a, b1pow_c, b2pow_c, sm, red);
    if (tid == 0) {
        Q.loss[id] = loss;
        cnt[0] = t_a + (update_policy ? 1 : 0); cnt[1] = t_c + 1; cnt[2] = it + 1;
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------
int td3_plan(const le_td3_cfg* tc, int n_lanes, int ring_cap, int sms, Td3Plan* tp) {
    const le_lane_cfg* c = &tc->base;
    GNet na, nc;
    tnet_build(&na, c->sd, c->q_hidden, c->q_layers, c->ad, c->q_act);
    tnet_build(&nc, c->sd + c->ad, c->q_hidden, c->q_layers, 1, c->q_act);
    int occ = 0;
    if (c->sd == 4) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, td3_loop_kernel<4, 2>, kGThreads, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, td3_loop_kernel<6, 3>, kGThreads, 0);
    if (occ < 1) occ = 1;
    tp->grid = n_lanes < sms * occ ? n_lanes : sms * occ;
    tp->bmax = c->batch_size > 64 ? c->batch_size : 64;
    tp->rowf = (2 * c->sd + c->ad + 2 + 3) / 4 * 4;
    int64_t offs[26];
    tp->slot_floats = tslot_floats(na, nc, c->sd, c->ad, ring_cap, tp->rowf, tp->bmax, offs);
    tp->p_actor = na.P;
    tp->p_critic = nc.P;
    return LE_OK;
}

cudaError_t td3_launch(const le_td3_cfg* cfg_dev, int n_cfg, const le_td3_cfg* cfg_host0, const RunParams& rp, float* slots, const Td3Plan& tp,
                       const float* actor_init, const float* c1_init, const float* c2_init, int per_lane_init, float* actor_final, cudaStream_t st) {
    TRunParams G;
    G.rp = rp;
    G.cfg = cfg_dev; G.n_cfg = n_cfg;
    const le_lane_cfg* c = &cfg_host0->base;
    tnet_build(&G.na_max, c->sd, c->q_hidden, c->q_layers, c->ad, c->q_act);
    tnet_build(&G.nc_max, c->sd + c->ad, c->q_hidden, c->q_layers, 1, c->q_act);
    G.slots = slots; G.slot_stride = tp.slot_floats; G.bmax = tp.bmax; G.rowf = tp.rowf;
    G.actor_init = actor_init; G.c1_init = c1_init; G.c2_init = c2_init;
    G.init_stride_a = per_lane_init ? tp.p_actor : 0;
    G.init_stride_c = per_lane_init ? tp.p_critic : 0;
    G.actor_final = actor_final; G.final_stride = tp.p_actor;
    if (c->sd == 4) td3_loop_kernel<4, 2><<<tp.grid, kGThreads, 0, st>>>(G);
    else td3_loop_kernel<6, 3><<<tp.grid, kGThreads, 0, st>>>(G);
    return cudaGetLastError();
}

int td3_learn(const le_td3_cfg* tc, float* const nets[6], float* const adam[6], int32_t* counters, int n, const float* rows,
              const float* policy_noise, const float* expo_target, const float* expo_actor, float* loss, cudaStream_t st) {
    Td3LearnParams Q;
    Q.tc = *tc;
    const le_lane_cfg* c = &tc->base;
    tnet_build(&Q.na, c->sd, c->q_hidden, c->q_layers, c->ad, c->q_act);
    tnet_build(&Q.nc, c->sd + c->ad, c->q_hidden, c->q_layers, 1, c->q_act);
    Q.actor = nets[0]; Q.actorT = nets[1]; Q.c1 = nets[2]; Q.c1T = nets[3]; Q.c2 = nets[4]; Q.c2T = nets[5];
    Q.m_a = adam[0]; Q.v_a = adam[1]; Q.m_c1 = adam[2]; Q.v_c1 = adam[3]; Q.m_c2 = adam[4]; Q.v_c2 = adam[5];
    Q.counters = counters; Q.rows = rows; Q.policy_noise = policy_noise; Q.expo_target = expo_target; Q.expo_actor = expo_actor;
    Q.loss = loss;
    int64_t offs[26];
    Q.scratch_stride = tslot_floats(Q.na, Q.nc, c->sd, c->ad, 0, 0, c->batch_size, offs);
    LE_CUDA_CHECK(cudaMallocAsync((void**)&Q.scratch, (size_t)Q.scratch_stride * 4 * n, st));
    if (c->sd == 4) td3_learn_kernel<4, 2><<<n, kGThreads, 0, st>>>(Q);
    else td3_learn_kernel<6, 3><<<n, kGThreads, 0, st>>>(Q);
    LE_CUDA_CHECK(cudaGetLastError());
    LE_CUDA_CHECK(cudaFreeAsync(Q.scratch, st));
    return LE_OK;
}

}  // namespace le
