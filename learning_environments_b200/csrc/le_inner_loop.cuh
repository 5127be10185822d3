// le_inner_loop.cuh — the persistent fused kernel: one warp runs one lane's complete calc_score
// (agents/GTN_worker.py:187-221): BaseAgent.train (agents/base_agent.py:64-153) with eps-greedy acting
// (agents/DDQN.py:97-104), SE / RN / real env step, replay append (utils.py:24-32), DDQN.learn
// (agents/DDQN.py:60-95), per-episode greedy test() on the real env (agents/base_agent.py:155-227), the
// early-out rule (agents/base_agent.py:49-62) and the final test().  Warps pull lanes from a global queue.
#pragma once
#include <cooperative_groups.h>
#include "le_envpack.cuh"
#include "le_lane.cuh"

namespace le {

struct RunParams {
    const le_lane_cfg* cfg; int n_cfg;
    const float4* env_pack; int64_t env_pack_stride;  // in float4
    const int32_t* env_index;
    const uint32_t* keys;
    const float* q_init; float* q_final; int q_stride;
    int n_lanes;
    le_lane_out* out;
    double* rewards; int32_t* lengths; double* test_rewards; int32_t* test_lengths;
    int rew_stride, test_stride;
    float* rings; int64_t ring_stride; int ring_cap;  // one replay ring per resident warp slot
    int* work_counter;
    int mw_pack_f4;   // multi-warp lanes: float4s of ONE env pack to stage in shared memory per lane (0: read it from global memory)
    le_trace trace; int trace_lane;
};

constexpr int kWarpsPerCta = 4;
// Fused kernel: U <= 2 -> 2 CTAs x 4 warps per SM (<= 255 registers each); U = 4 needs all 255 registers per thread, so ONE
// CTA of 8 warps fills the register file (8 x 32 x 255) and still gives every scheduler two warps to alternate between.
constexpr int kWarpsU4 = 8;
constexpr int kMinCtasU2 = 2;
template <int U> constexpr int inner_warps() { return U <= 2 ? kWarpsPerCta : kWarpsU4; }


// Per-warp shared memory: [stage rows | test-phase weight image (aliased)] [Adam m, v] [lane configuration] [reduction]
template <int SD, int AD, int U, bool ROW = false>
struct SmemWarp {
    using SL = StageLayout<SD>;
    static constexpr int PUP = SD + 1 + AD;           // per-unit record of the test-phase weight image (scalar reads, broadcast)
    static constexpr int STAGE_ONE_F = SL::ROWS * SL::STAGE_F;
    static constexpr int STAGE_F = 2 * STAGE_ONE_F;   // double buffer: the gather of round k+1 overlaps the compute of round k
    static constexpr int QW_F = (U * 32 * PUP + 3) / 4 * 4;
    static constexpr int BUF_F = STAGE_F > QW_F ? STAGE_F : QW_F;
    static constexpr int MV_F = 2 * (U * (SD + 1 + AD) + AD) * 32;
    static constexpr int CFG_F = (sizeof(le_lane_cfg) + 15) / 16 * 4;
    static constexpr int RED_F = LaneCore<SD, AD, U, QACT_TANH, ROW>::SMEM_RED_F;   // reduction buffers, or the row-owner region
    static constexpr int FLOATS = BUF_F + MV_F + CFG_F + RED_F;
    static constexpr int OFF_MV = BUF_F, OFF_CFG = BUF_F + MV_F, OFF_RED = BUF_F + MV_F + CFG_F;
    static_assert(FLOATS % 4 == 0 && OFF_RED % 4 == 0 && STAGE_ONE_F % 4 == 0, "float4 accesses of the stage / reduction buffer need 16-byte alignment");
};

__device__ __forceinline__ float4 ld_cg_f4(const float4* p) { return __ldcg(p); }

// le_trace.qgap: (q_best - q_second) / max(|q_best|, |q_second|, 1e-12) of a greedy action choice
template <int AD>
__device__ __forceinline__ float relative_q_gap(const float (&q)[AD], int best) {
    float second = -3.4e38f;
#pragma unroll
    for (int a = 0; a < AD; ++a)
        if (a != best && q[a] > second) second = q[a];
    return (q[best] - second) / fmaxf(fmaxf(fabsf(q[best]), fabsf(second)), 1e-12f);
}

// AverageMeter._mean (utils.py:103-105) over the per-lane reward list in global memory
__device__ __forceinline__ double mean_window(const double* vals, int len, int num, int ignore_last) {
    int lo = len - num - ignore_last; if (lo < 0) lo = 0;
    int hi = len - ignore_last; if (hi < 0) hi = 0;
    double s = 0.0;
    for (int i = lo; i < hi; ++i) s += __ldcg(vals + i);   // written by another thread of this warp/CTA: read through L2
    return s / ((double)(hi - lo) + 1e-9);
}

// env_solved (agents/base_agent.py:49-62), checked after each episode past init_episodes: the mean of the last
// early_out_num episode values reaches solved_reward; on a virtual (SE) env without a test env, the mean stops moving instead
__device__ __forceinline__ bool env_solved(const double* rewards, int n_ep, int episode, const le_lane_cfg& c) {
    if (episode < c.init_episodes) return false;
    const double avg = mean_window(rewards, n_ep, c.early_out_num, 0);
    if ((!c.use_test_env) && c.env_kind == LE_ENV_SE) {
        const double avg_last = mean_window(rewards, n_ep, c.early_out_num, c.early_out_num);
        return (fabs(avg - avg_last) / (fabs(avg_last) + 1e-9) < c.early_out_virtual_diff) &&
               (episode >= c.init_episodes + c.early_out_num);
    }
    return avg >= c.solved_reward;
}

// eps-greedy schedule of the DDQN agents (agents/DDQN.py:112-117): eps_init in episode 0, then decayed and floored at eps_min
__device__ __forceinline__ double eps_schedule(double eps, int episode, const le_lane_cfg& c) {
    if (episode == 0) return c.eps_init;
    eps *= c.eps_decay;
    return eps < c.eps_min ? c.eps_min : eps;
}

// One replay row (registers, HBM layout) -> shared-memory stage (same layout)
template <int SD>
__device__ __forceinline__ void stage_row(float* dst, const float (&rowv)[RowLayout<SD>::ROWF]) {
    using RL = RowLayout<SD>;
    float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int q = 0; q < RL::ROW_VEC; ++q) d4[q] = make_float4(rowv[4 * q], rowv[4 * q + 1], rowv[4 * q + 2], rowv[4 * q + 3]);
}

__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* gptr) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Multi-warp lanes (W > 1, inner_loop_mw_kernel): shared state of one CTA = one lane.  The leader warp (warp 0) runs the lane's
// control flow; for every DDQN.learn it publishes a command and the W warps split the minibatch into 32-row passes.
struct MwShared {
    int cmd;                 // 0: exit, 1: learn, 2: new lane (configuration is in the leader's shared memory)
    int lane_id, rb_size, pad;
    long long learn_iters;
    float b2[4], tb2[4];     // output biases of the online / target net (registers of the leader)
    unsigned long long pack_mbar;   // mbarrier of the TMA bulk copy that stages the lane's SE / RN pack
};
// TMA bulk copy global -> shared memory, completion on an mbarrier (cp.async.bulk; SASS UBLKCP + SYNCS)
__device__ __forceinline__ void mbar_init(uint32_t mbar, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\tLE_MBAR_WAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra LE_MBAR_DONE_%=;\n\tbra LE_MBAR_WAIT_%=;\n\tLE_MBAR_DONE_%=:\n\t}" ::"r"(mbar), "r"(parity) : "memory");
}

template <int W>
__device__ __forceinline__ void mw_bar(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(W * 32) : "memory"); }
template <int U> constexpr int mw_warps() { return U <= 2 ? 8 : (U <= 4 ? 6 : 4); }
// Cluster lanes (CL = 2, inner_loop_mwc_kernel): ONE lane per thread-block cluster of two CTAs = two SMs.  CTA 0 holds the leader warp and
// kMwcWarps - 1 workers, CTA 1 the same number of workers; the minibatch passes alternate between the two SMs (one working warp per
// scheduler), the weight records and the command block are replicated into CTA 1 through distributed shared memory, the workers of CTA 1
// write their gradient sums straight into CTA 0's exchange buffer, and the two barriers of a learn() are cluster barriers.
constexpr int kMwcWarps = 5;
__device__ __forceinline__ void cluster_bar() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

template <int SD, int AD, int U, int ACT, int W = 1, int CL = 1>
struct FusedLane {
    static constexpr int NPART = CL == 1 ? W : 2 * (W - 1);          // participants of a learn(): pass p goes to participant p % NPART
    static constexpr int NEXS = CL == 1 ? W - 1 : NPART;             // exchange slots (CL == 1: the leader keeps its share in registers)
    static __device__ __forceinline__ void lane_bar(int id) { if constexpr (CL == 1) mw_bar<W>(id); else cluster_bar(); }
    using Core = LaneCore<SD, AD, U, ACT, (W > 1)>;
    using RL = RowLayout<SD>;
    using SW = SmemWarp<SD, AD, U, (W > 1)>;
    using SL0 = StageLayout<SD>;
    // multi-warp lanes: per-worker shared memory = a 32-row stage + the row-owner scratch; exchange = gradients, bias gradients, loss
    static constexpr int MW_STAGE_F = 32 * SL0::STAGE_F;
    static constexpr int MW_WORKER_F = MW_STAGE_F + Core::ROW_SCRATCH_F;
    static constexpr int MW_NEX = U * (SD + 1 + AD) + AD + 1;
    static constexpr int MW_EX_F = NEXS * MW_NEX * 32;
    static constexpr int MW_SH_F = (sizeof(MwShared) + 15) / 16 * 4;
    static constexpr int MW_CTA_F = SW::FLOATS + (W - 1) * MW_WORKER_F + MW_EX_F + MW_SH_F;

    // This warp's share of one DDQN.learn: passes w, w + W, ... of 32 sampled rows each (same Philox blocks as the single-warp
    // gather: block = row / 4 of the minibatch).  Gradients accumulate in core.a*, returns the warp's share of sum(delta^2).
    static __device__ __forceinline__ float mw_td_share(Core& core, int part, const float* wrec, float* stage, float* scratch, const float* ring,
                                                        int rb_size, long long learn_iters, uint32_t k0, uint32_t k1, const LearnScalars& ls, int lane) {
        core.zero_grads();
        float loss_part = 0.f;
        const int B = ls.batch;
        const int npass = (B + 31) >> 5;
        const uint32_t stage_sa = (uint32_t)__cvta_generic_to_shared(stage);
        for (int p = part; p < npass; p += NPART) {
            const int nrows = min(32, B - 32 * p);
            if (lane < 8) {
                const u32x4 wv = philox4x32_10((uint32_t)learn_iters, (uint32_t)(8 * p + lane), LE_P_SAMPLE, 0u, k0, k1);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const int rr = 4 * lane + kk;
                    if (rr < nrows) {
                        const uint32_t idx = __umulhi(pick(wv, kk), (uint32_t)rb_size);
                        const float* src = ring + (int64_t)idx * RL::ROWF;
#pragma unroll
                        for (int q = 0; q < RL::ROW_VEC; ++q) cp_async16(stage_sa + (uint32_t)((rr * SL0::STAGE_F + 4 * q) * 4), src + 4 * q);
                    } else {
                        float4* z = reinterpret_cast<float4*>(stage + rr * SL0::STAGE_F);
#pragma unroll
                        for (int q = 0; q < RL::ROW_VEC; ++q) z[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
            }
            cp_async_commit();
            cp_async_wait<0>();
            __syncwarp();
            loss_part += core.td_rows_rowown(stage, wrec, scratch, nrows, ls, lane);
            __syncwarp();
        }
        return loss_part;
    }
    // worker warps of a multi-warp lane
    // lead_smem: THIS CTA's copy of the leader region (weight records); ex / cfgp: the exchange buffer and lane configuration of the
    // leader's CTA (distributed shared memory for the workers of CTA 1)
    static __device__ void mw_worker(const RunParams& P, int slot, int w, int part, float* lead_smem, float* my_smem, MwShared* sh, float* ex,
                                     const le_lane_cfg* cfgp, int lane) {
        Core core;
        core.bind(lead_smem + SW::OFF_RED, lane);
        float* stage = my_smem;
        float* scratch = my_smem + MW_STAGE_F;
        Core::init_row_scratch(scratch, lane);
        const float* ring = P.rings + (int64_t)slot * P.ring_stride;
        const le_lane_cfg& c = *cfgp;
        LearnScalars ls;
        uint32_t k0 = 0, k1 = 0;
        for (;;) {
            lane_bar(1);
            const int cmd = sh->cmd;
            if (cmd == 0) break;
            if (cmd == 2) {
                fill_learn_scalars(ls, c);
                k0 = P.keys[2 * sh->lane_id]; k1 = P.keys[2 * sh->lane_id + 1];
            } else {
#pragma unroll
                for (int a = 0; a < AD; ++a) { core.b2[a] = sh->b2[a]; core.tb2[a] = sh->tb2[a]; }
                core.publish_weights(nullptr, lane);
                const float lp = mw_td_share(core, part, lead_smem + SW::OFF_RED, stage, scratch, ring, sh->rb_size, sh->learn_iters, k0, k1, ls, lane);
                float* e = ex + (CL == 1 ? w - 1 : part) * MW_NEX * 32 + lane;
                int k = 0;
#pragma unroll
                for (int u = 0; u < U; ++u) {
#pragma unroll
                    for (int i = 0; i < SD; ++i) e[32 * (k++)] = core.g_w1(u, i);
                    e[32 * (k++)] = core.g_b1(u);
#pragma unroll
                    for (int a = 0; a < AD; ++a) e[32 * (k++)] = core.g_w2(u, a);
                }
#pragma unroll
                for (int a = 0; a < AD; ++a) e[32 * (k++)] = core.gb2[a];
                e[32 * k] = lp;
            }
            lane_bar(2);
        }
    }

    // BaseAgent.test: greedy rollouts on the real env, one episode per thread, weights broadcast from smem.
    static __device__ __forceinline__ double run_test(const Core& core, float* smem, const le_lane_cfg& c, float slope,
                                                      uint32_t k0, uint32_t k1, int test_call, int lane,
                                                      double* ep_out /* [test_episodes] or nullptr */, int32_t* len_out, int64_t& test_steps) {
        constexpr int PUP = SW::PUP;
        __syncwarp();
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float* rec = smem + (lane + 32 * u) * PUP;
#pragma unroll
            for (int i = 0; i < SD; ++i) rec[i] = core.w1_on(u, i);
            rec[SD] = core.b1_on(u);
#pragma unroll
            for (int a = 0; a < AD; ++a) rec[SD + 1 + a] = core.w2_on(u, a);
        }
        __syncwarp();
        const int H = c.q_hidden;
        double sum = 0.0;
        int steps = 0;
        for (int ep0 = 0; ep0 < c.test_episodes; ep0 += 32) {
            const int ep = ep0 + lane;
            const bool active = ep < c.test_episodes;
            double st[4];
            real_reset(c.real_env, philox4x32_10((uint32_t)test_call, (uint32_t)ep, LE_P_RESET_TEST, 0u, k0, k1), st);
            float obs[SD];
            real_obs<SD>(c.real_env, st, obs);
            int elapsed = 0;
            float ep_rew = 0.f;
            int ep_steps = 0;
            bool running = active;
            const int K = c.same_action_num > 1 ? c.same_action_num : 1;
            for (int t = 0; t < c.max_steps; t += K) {   // agents/base_agent.py:193
                if (!__any_sync(LE_FULL_MASK, running)) break;
                if (running) {
                    float q[AD];
#pragma unroll
                    for (int a = 0; a < AD; ++a) q[a] = 0.f;
                    for (int j = 0; j < H; ++j) {
                        const float* rec = smem + j * PUP;
                        float z = rec[SD];
#pragma unroll
                        for (int i = 0; i < SD; ++i) z = fmaf(rec[i], obs[i], z);
                        const float h = act_one<ACT>(z, slope);
#pragma unroll
                        for (int a = 0; a < AD; ++a) q[a] = fmaf(h, rec[SD + 1 + a], q[a]);
                    }
#pragma unroll
                    for (int a = 0; a < AD; ++a) q[a] += core.b2[a];
                    const int act = Core::argmax_first(q);  // select_test_action agents/DDQN.py:106-110
                    float r, d;
                    real_step<SD>(c.real_env, c.max_steps, st, elapsed, act, obs, r, d);
                    if (K > 1) {   // EnvWrapper.step real branch (envs/env_wrapper.py:56-61): python-float reward sum, break on done
                        double rsum = (double)r;
                        for (int k = 1; k < K && !(d > 0.5f); ++k) {
                            float rk;
                            real_step<SD>(c.real_env, c.max_steps, st, elapsed, act, obs, rk, d);
                            rsum += (double)rk;
                        }
                        r = (float)rsum;
                    }
                    ep_rew += r;
                    steps += 1;
                    ep_steps += 1;
                    if (d > 0.5f) running = false;
                }
            }
            if (active) {
                sum += (double)ep_rew;
                if (ep_out) ep_out[ep] = (double)ep_rew;
                if (len_out) len_out[ep] = ep_steps;
            }
        }
        sum = warp_allreduce_sum(sum);
        int tot = steps;
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) tot += __shfl_xor_sync(LE_FULL_MASK, tot, m);
        test_steps += tot;
        __syncwarp();
        return sum / (double)c.test_episodes;  // statistics.mean
    }

    static __device__ void run(const RunParams& P, int lane_id, int slot, float* smem, int lane, MwShared* sh = nullptr, float* ex = nullptr,
                               float4* pack_smem = nullptr, uint32_t pack_parity = 0, MwShared* sh_r = nullptr, float* wrec_r = nullptr) {
        using SL = StageLayout<SD>;
        float* mv = smem + SW::OFF_MV;
        {   // lane configuration -> shared memory (read on demand instead of pinning ~46 registers)
            const uint32_t* src = reinterpret_cast<const uint32_t*>(P.cfg + (P.n_cfg == 1 ? 0 : lane_id));
            uint32_t* dst = reinterpret_cast<uint32_t*>(smem + SW::OFF_CFG);
            for (int i = lane; i < (int)(sizeof(le_lane_cfg) / 4); i += 32) dst[i] = src[i];
            __syncwarp();
        }
        const le_lane_cfg& c = *reinterpret_cast<const le_lane_cfg*>(smem + SW::OFF_CFG);
        const uint32_t k0 = P.keys[2 * lane_id], k1 = P.keys[2 * lane_id + 1];
        const float4* pack = P.env_pack + (int64_t)(P.env_index ? P.env_index[lane_id] : 0) * P.env_pack_stride;
        constexpr bool kPackSh = W > 1;     // multi-warp lanes: the SE / RN pack is staged in shared memory when it fits (else W == 1 code path below)
        bool pack_staged = false;
        if constexpr (W > 1) {
            if (P.mw_pack_f4 > 0 && pack_smem != nullptr) {
                // one TMA bulk copy per lane: weights of the member's SE / RN stay on chip for the whole calc_score
                const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&sh->pack_mbar);
                const uint32_t bytes = (uint32_t)P.mw_pack_f4 * 16u;
                __syncwarp();
                if (lane == 0) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // earlier generic-proxy reads of the buffer are done
                    mbar_expect_tx(mbar, bytes);
                    bulk_g2s((uint32_t)__cvta_generic_to_shared(pack_smem), pack, bytes, mbar);
                }
                mbar_wait(mbar, pack_parity);
                pack = pack_smem;
                pack_staged = true;
            }
        }
        const bool env_tanh = c.env_act == LE_ACT_TANH;
        const int H = c.q_hidden;
        float* ring = P.rings + (int64_t)slot * P.ring_stride;
        const int ring_cap = P.ring_cap;
        double* rewards = P.rewards + (int64_t)lane_id * P.rew_stride;
        int32_t* lengths = P.lengths + (int64_t)lane_id * P.rew_stride;
        double* test_rewards = P.test_rewards + (int64_t)lane_id * P.test_stride;
        const bool tracing = P.trace.cap > 0 && lane_id == P.trace_lane;

        Core core;
        core.bind(smem + SW::OFF_RED, lane);
        if (P.q_init) core.load_net(P.q_init + (int64_t)lane_id * P.q_stride, H, lane, 0);
        else core.init_online(H, lane, k0, k1);
        core.copy_online_to_target();  // model_target.load_state_dict(model.state_dict())   agents/DDQN.py:36
        Core::init_row_region(smem + SW::OFF_RED, lane);
        core.publish_weights(smem + SW::OFF_RED, lane);
        auto replicate_weights = [&]() {   // cluster lanes: CTA 1 reads its own copy of the weight records
            if constexpr (CL > 1) {
                const float4* src = reinterpret_cast<const float4*>(smem + SW::OFF_RED);
                float4* dst = reinterpret_cast<float4*>(wrec_r);
                for (int k = lane; k < Core::ROW_WREC_F / 4; k += 32) dst[k] = src[k];
            }
        };
        replicate_weights();
        Core::zero_moments(mv, lane);
        LearnScalars ls;
        fill_learn_scalars(ls, c);
        if constexpr (W > 1) {   // workers pick up the lane's configuration and keys
            if (lane == 0) {
                sh->cmd = 2; sh->lane_id = lane_id;
                if constexpr (CL > 1) { sh_r->cmd = 2; sh_r->lane_id = lane_id; }
            }
            lane_bar(1);
            lane_bar(2);
        }

        int rb_ptr = 0, rb_size = 0;
        int64_t train_steps = 0, learn_iters = 0, test_steps = 0;
        int test_calls = 0, n_ep = 0, timed_out = 0;
        double eps = c.eps_init;
        const bool rule_virtual = (!c.use_test_env) && c.env_kind == LE_ENV_SE;

        for (int episode = 0; episode < c.train_episodes; ++episode) {
            if (c.step_budget > 0 && train_steps >= c.step_budget) { timed_out = 1; break; }  // time_is_up analog
            if (episode == 0) eps = c.eps_init;                                              // agents/DDQN.py:112-117
            else { eps *= c.eps_decay; if (eps < c.eps_min) eps = c.eps_min; }
            double st[4];
            real_reset(c.real_env, philox4x32_10((uint32_t)episode, 0u, LE_P_RESET_TRAIN, 0u, k0, k1), st);
            float state[SD];
            real_obs<SD>(c.real_env, st, state);
            int elapsed = 0, ep_len = 0;
            float ep_rew = 0.f;
            const int K = c.same_action_num > 1 ? c.same_action_num : 1;
            for (int t = 0; t < c.max_steps; t += K) {   // agents/base_agent.py:104
                // ---- select_train_action (agents/DDQN.py:97-104)
                const u32x4 wa = philox4x32_10((uint32_t)train_steps, 0u, LE_P_ACT, 0u, k0, k1);
                const bool explore = ((double)(wa.x >> 8) * (1.0 / 16777216.0)) < eps;
                int action;
                float qgap = __int_as_float(0x7fc00000);
                if (explore) action = (int)__umulhi(wa.y, (uint32_t)AD);
                else {
                    float q[AD];
                    core.q_forward_row(state, ls.slope, q);
                    action = Core::argmax_first(q);
                    if (tracing) qgap = relative_q_gap<AD>(q, action);
                }
                // ---- env.step
                float ns[SD], r, d;
                if (c.env_kind == LE_ENV_SE) {
                    if (kPackSh && pack_staged) se_step_row<SD, AD, kPackSh>(pack, c.env_hidden, env_tanh, state, action, lane, ns, r, d);
                    else se_step_row<SD, AD>(pack, c.env_hidden, env_tanh, state, action, lane, ns, r, d);
                    // same_action_num > 1 (envs/env_wrapper.py:24-30): chained SE steps, fp32 reward sum, no break on done
                    for (int k = 1; k < K; ++k) {
                        float cur[SD], rk;
#pragma unroll
                        for (int i = 0; i < SD; ++i) cur[i] = ns[i];
                        if (kPackSh && pack_staged) se_step_row<SD, AD, kPackSh>(pack, c.env_hidden, env_tanh, cur, action, lane, ns, rk, d);
                        else se_step_row<SD, AD>(pack, c.env_hidden, env_tanh, cur, action, lane, ns, rk, d);
                        r += rk;
                    }
                } else {
                    // real branch (envs/env_wrapper.py:56-61): python-float reward sum over same_action_num steps, break on done
                    float cur[SD];
#pragma unroll
                    for (int i = 0; i < SD; ++i) cur[i] = state[i];
                    double rsum = 0.0;
                    for (int k = 0; k < K; ++k) {
                        float rr, rk;
                        real_step<SD>(c.real_env, c.max_steps, st, elapsed, action, ns, rr, d);
                        if (c.env_kind == LE_ENV_RN && c.rn_type != 0) {
                            float ps, ps2;
                            if (kPackSh && pack_staged) rn_phi2<SD, kPackSh>(pack, c.env_hidden, env_tanh, cur, ns, lane, ps, ps2);
                            else rn_phi2<SD>(pack, c.env_hidden, env_tanh, cur, ns, lane, ps, ps2);
                            rk = rn_combine(c.rn_type, ls.gamma, rr, ps, ps2);
                        } else rk = rr;
                        if (K == 1) { r = rk; break; }
                        rsum += (double)rk;
                        r = (float)rsum;
#pragma unroll
                        for (int i = 0; i < SD; ++i) cur[i] = ns[i];
                        if (d > 0.5f) break;
                    }
                }
                // ---- replay_buffer.add (utils.py:24-32): row [s a s' r d] in the 16B-aligned layout RL
                {
                    float rowv[RL::ROWF];
#pragma unroll
                    for (int i = 0; i < RL::ROWF; ++i) rowv[i] = 0.f;
#pragma unroll
                    for (int i = 0; i < SD; ++i) { rowv[RL::OFF_S + i] = state[i]; rowv[RL::OFF_S2 + i] = ns[i]; }
                    rowv[RL::OFF_A] = __int_as_float(action); rowv[RL::OFF_R] = r; rowv[RL::OFF_D] = d;
                    float4* dst = reinterpret_cast<float4*>(ring + (int64_t)rb_ptr * RL::ROWF);
#pragma unroll
                    for (int q = 0; q < RL::ROW_VEC; ++q)
                        if (lane == q) __stcg(dst + q, make_float4(rowv[4 * q], rowv[4 * q + 1], rowv[4 * q + 2], rowv[4 * q + 3]));
                    rb_ptr = (rb_ptr + 1 == ring_cap) ? 0 : rb_ptr + 1;
                    rb_size = rb_size + 1 < ring_cap ? rb_size + 1 : ring_cap;
                }
#pragma unroll
                for (int i = 0; i < SD; ++i) state[i] = ns[i];
                ep_rew += r;
                ep_len += K;   // episode_length += same_action_num (agents/base_agent.py:123)
                // ---- learn (agents/DDQN.py:60-95)
                float loss = __int_as_float(0x7fc00000);
                if (episode >= c.init_episodes) {
                    float loss_part = 0.f;
                    const int B = ls.batch;
                    if constexpr (W > 1) {
                        if (lane == 0) {
                            auto msg = [&](MwShared* m) {
                                m->cmd = 1; m->rb_size = rb_size; m->learn_iters = learn_iters;
#pragma unroll
                                for (int a = 0; a < AD; ++a) { m->b2[a] = core.b2[a]; m->tb2[a] = core.tb2[a]; }
                            };
                            msg(sh);
                            if constexpr (CL > 1) msg(sh_r);
                        }
                        lane_bar(1);     // the appended row, the weights and the command are visible to every warp of the lane
                        if constexpr (CL == 1) loss_part = mw_td_share(core, 0, smem + SW::OFF_RED, smem, smem + SW::OFF_RED + Core::ROW_WREC_F, ring, rb_size, learn_iters, k0, k1, ls, lane);
                        else core.zero_grads();
                        lane_bar(2);     // every participant's gradients are in the exchange buffer: add them in participant order
                        for (int w = 0; w < NEXS; ++w) {
                            const float* e = ex + w * MW_NEX * 32 + lane;
                            int k = 0;
#pragma unroll
                            for (int u = 0; u < U; ++u) {
#pragma unroll
                                for (int i = 0; i < SD; ++i) core.a1[u][i].x += e[32 * (k++)];
                                core.ab1[u].x += e[32 * (k++)];
#pragma unroll
                                for (int a = 0; a < AD; ++a) core.a2[u][a].x += e[32 * (k++)];
                            }
#pragma unroll
                            for (int a = 0; a < AD; ++a) core.gb2[a] += e[32 * (k++)];
                            loss_part += e[32 * k];
                        }
                    } else {
                    __syncwarp();  // the appended row is visible to the whole warp
                    core.zero_grads();
                    // replay_buffer.sample: idx = randint(0, size, B) on the P_SAMPLE stream (utils.py:35).  Thread t < 16
                    // gathers the 4 rows of Philox block (round*16 + t) with 16-byte cp.async (global -> shared, no
                    // registers); round k+1 is in flight while round k is computed.
                    const uint32_t stage_sa = (uint32_t)__cvta_generic_to_shared(smem);
                    auto gather = [&](int sc, int buf) {
                        const int nrows = min(SL::ROWS, B - sc * SL::ROWS);
                        const int nfill = (nrows + Core::R - 1) / Core::R * Core::R;
                        if (4 * lane < nfill) {
                            const u32x4 w = philox4x32_10((uint32_t)learn_iters, (uint32_t)(sc * (SL::ROWS / 4) + lane), LE_P_SAMPLE, 0u, k0, k1);
#pragma unroll
                            for (int kk = 0; kk < 4; ++kk) {
                                const int rr = 4 * lane + kk;
                                const uint32_t dst = stage_sa + (uint32_t)((buf * SW::STAGE_ONE_F + rr * SL::STAGE_F) * 4);
                                if (rr < nrows) {
                                    const uint32_t idx = __umulhi(pick(w, kk), (uint32_t)rb_size);
                                    const float* src = ring + (int64_t)idx * RL::ROWF;
#pragma unroll
                                    for (int q = 0; q < RL::ROW_VEC; ++q) cp_async16(dst + 16 * q, src + 4 * q);
                                } else {
                                    float4* z = reinterpret_cast<float4*>(smem + buf * SW::STAGE_ONE_F + rr * SL::STAGE_F);
#pragma unroll
                                    for (int q = 0; q < RL::ROW_VEC; ++q) z[q] = make_float4(0.f, 0.f, 0.f, 0.f);
                                }
                            }
                        }
                        cp_async_commit();
                    };
                    const int n_rounds = (B + SL::ROWS - 1) / SL::ROWS;
                    gather(0, 0);
                    for (int sc = 0; sc < n_rounds; ++sc) {
                        const int nrows = min(SL::ROWS, B - sc * SL::ROWS);
                        if (sc + 1 < n_rounds) { gather(sc + 1, (sc + 1) & 1); cp_async_wait<1>(); }
                        else cp_async_wait<0>();
                        __syncwarp();
                        loss_part += core.td_rows(smem + (sc & 1) * SW::STAGE_ONE_F, smem + SW::OFF_RED, nrows, ls, lane);
                        __syncwarp();
                    }
                    }
                    loss = warp_allreduce_sum(loss_part) / (float)B;
                    core.adam_polyak(ls, mv, lane);
                    core.publish_weights(smem + SW::OFF_RED, lane);
                    if constexpr (W > 1) replicate_weights();
                    learn_iters += 1;
                }
                if (tracing && train_steps < P.trace.cap && lane == 0) {
                    const int64_t i = train_steps;
                    P.trace.action[i] = action; P.trace.explore[i] = explore ? 1 : 0;
                    P.trace.reward[i] = r; P.trace.done[i] = d; P.trace.loss[i] = loss;
                    if (P.trace.qgap) P.trace.qgap[i] = qgap;
#pragma unroll
                    for (int k = 0; k < SD; ++k) P.trace.next_state[i * SD + k] = ns[k];
                }
                train_steps += 1;
                if (d > 0.5f) break;
            }
            // ---- episode bookkeeping (agents/base_agent.py:131-148)
            double ep_value;
            if (c.use_test_env) ep_value = run_test(core, smem, c, ls.slope, k0, k1, test_calls++, lane, nullptr, nullptr, test_steps);
            else ep_value = (double)ep_rew;
            if (lane == 0) { lengths[n_ep] = ep_len; rewards[n_ep] = ep_value; }
            n_ep += 1;
            __syncwarp();
            if (episode >= c.init_episodes) {  // env_solved (agents/base_agent.py:49-62)
                const double avg = mean_window(rewards, n_ep, c.early_out_num, 0);
                bool solved;
                if (rule_virtual) {
                    const double avg_last = mean_window(rewards, n_ep, c.early_out_num, c.early_out_num);
                    solved = (fabs(avg - avg_last) / (fabs(avg_last) + 1e-9) < c.early_out_virtual_diff) &&
                             (episode >= c.init_episodes + c.early_out_num);
                } else solved = avg >= c.solved_reward;
                if (solved) break;
            }
        }
        double score = 0.0;
        if (c.final_test)
            score = run_test(core, smem, c, ls.slope, k0, k1, test_calls++, lane, test_rewards,
                             P.test_lengths ? P.test_lengths + (int64_t)lane_id * P.test_stride : nullptr, test_steps);
        if (P.q_final) core.store_net(P.q_final + (int64_t)lane_id * P.q_stride, H, lane, 0);
        if (lane == 0) {
            le_lane_out o;
            o.n_episodes = n_ep; o.timed_out = timed_out; o.train_steps = train_steps; o.learn_iters = learn_iters;
            o.test_steps = test_steps; o.score = score;
            P.out[lane_id] = o;
        }
    }
};

template <int SD, int AD, int U, int ACT>
__global__ void __launch_bounds__(inner_warps<U>() * 32, (U <= 2 ? kMinCtasU2 : 1)) inner_loop_kernel(const RunParams P) {
    using SW = SmemWarp<SD, AD, U>;
    extern __shared__ __align__(16) float smem_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x * inner_warps<U>() + warp;
    float* smem = smem_dyn + warp * SW::FLOATS;
    // Lane queue: the first lane of every warp slot is static (lane_id == slot, so with n_lanes <= slots a lane's replay ring
    // is the ring of slot lane_id: agents.py reads it back), every further lane comes from the global counter.
    bool first = true;
    for (;;) {
        int lane_id = slot;
        if (!first) {
            if (lane == 0) lane_id = (int)(gridDim.x * inner_warps<U>()) + atomicAdd(P.work_counter, 1);
            lane_id = __shfl_sync(LE_FULL_MASK, lane_id, 0);
        }
        first = false;
        if (lane_id >= P.n_lanes) break;
        FusedLane<SD, AD, U, ACT>::run(P, lane_id, slot, smem, lane);
        __syncwarp();
    }
}

// Multi-warp lanes: ONE lane per CTA of mw_warps<U>() warps (small populations: fewer lanes than SMs).  Warp 0 runs the lane
// (FusedLane<..., W>::run); the minibatch of every DDQN.learn is split into 32-row passes over all warps (row-owner TD update on
// the lane's shared weight records), the gradients meet in shared memory and warp 0 takes the Adam / Polyak step.
template <int SD, int AD, int U, int ACT>
__global__ void __launch_bounds__(mw_warps<U>() * 32, 1) inner_loop_mw_kernel(const RunParams P) {
    constexpr int W = mw_warps<U>();
    using FL = FusedLane<SD, AD, U, ACT, W>;
    extern __shared__ __align__(16) float smem_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x;
    float* ex = smem_dyn + FL::SW::FLOATS + (W - 1) * FL::MW_WORKER_F;
    MwShared* sh = reinterpret_cast<MwShared*>(ex + FL::MW_EX_F);
    float4* pack_smem = reinterpret_cast<float4*>(smem_dyn + FL::MW_CTA_F);   // P.mw_pack_f4 float4s (0: not staged)
    if (warp == 0) {
        if (lane == 0) {
            mbar_init((uint32_t)__cvta_generic_to_shared(&sh->pack_mbar), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        uint32_t pack_parity = 0;
        bool first = true;
        for (;;) {
            int lane_id = slot;
            if (!first) {
                if (lane == 0) lane_id = (int)gridDim.x + atomicAdd(P.work_counter, 1);
                lane_id = __shfl_sync(LE_FULL_MASK, lane_id, 0);
            }
            first = false;
            if (lane_id >= P.n_lanes) break;
            FL::run(P, lane_id, slot, smem_dyn, lane, sh, ex, pack_smem, pack_parity);
            if (P.mw_pack_f4 > 0) pack_parity ^= 1u;
            __syncwarp();
        }
        if (lane == 0) sh->cmd = 0;
        mw_bar<W>(1);
    } else {
        FL::mw_worker(P, slot, warp, warp, smem_dyn, smem_dyn + FL::SW::FLOATS + (warp - 1) * FL::MW_WORKER_F, sh, ex,
                      reinterpret_cast<const le_lane_cfg*>(smem_dyn + FL::SW::OFF_CFG), lane);
    }
}

// Cluster lanes: one lane per thread-block cluster of two CTAs (two SMs), see kMwcWarps above.  Launched with cluster dimension 2.
template <int SD, int AD, int U, int ACT>
__global__ void __launch_bounds__(kMwcWarps * 32, 1) inner_loop_mwc_kernel(const RunParams P) {
    namespace cg = cooperative_groups;
    constexpr int W = kMwcWarps;
    using FL = FusedLane<SD, AD, U, ACT, W, 2>;
    extern __shared__ __align__(16) float smem_dyn[];
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x >> 1, n_slots = gridDim.x >> 1;
    float* ex = smem_dyn + FL::SW::FLOATS + (W - 1) * FL::MW_WORKER_F;
    MwShared* sh = reinterpret_cast<MwShared*>(ex + FL::MW_EX_F);
    float4* pack_smem = reinterpret_cast<float4*>(smem_dyn + FL::MW_CTA_F);
    // the same offsets in the other CTA of the cluster (distributed shared memory)
    float* smem_0 = cluster.map_shared_rank(smem_dyn, 0);
    float* smem_1 = cluster.map_shared_rank(smem_dyn, 1);
    float* ex_0 = smem_0 + (ex - smem_dyn);
    MwShared* sh_1 = reinterpret_cast<MwShared*>(smem_1 + (reinterpret_cast<float*>(sh) - smem_dyn));
    cluster_bar();   // both CTAs of the cluster are running before either touches the other's shared memory
    if (rank == 0 && warp == 0) {
        if (lane == 0) {
            mbar_init((uint32_t)__cvta_generic_to_shared(&sh->pack_mbar), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        uint32_t pack_parity = 0;
        bool first = true;
        for (;;) {
            int lane_id = slot;
            if (!first) {
                if (lane == 0) lane_id = n_slots + atomicAdd(P.work_counter, 1);
                lane_id = __shfl_sync(LE_FULL_MASK, lane_id, 0);
            }
            first = false;
            if (lane_id >= P.n_lanes) break;
            FL::run(P, lane_id, slot, smem_dyn, lane, sh, ex, pack_smem, pack_parity, sh_1, smem_1 + FL::SW::OFF_RED);
            if (P.mw_pack_f4 > 0) pack_parity ^= 1u;
            __syncwarp();
        }
        if (lane == 0) { sh->cmd = 0; sh_1->cmd = 0; }
        cluster_bar();
    } else if (warp >= 1) {
        FL::mw_worker(P, slot, warp, 2 * (warp - 1) + rank, smem_dyn, smem_dyn + FL::SW::FLOATS + (warp - 1) * FL::MW_WORKER_F, sh, ex_0,
                      reinterpret_cast<const le_lane_cfg*>(smem_0 + FL::SW::OFF_CFG), lane);
    } else {   // warp 0 of CTA 1: follows the barriers
        for (;;) {
            cluster_bar();
            if (sh->cmd == 0) break;
            cluster_bar();
        }
    }
    cluster_bar();   // no CTA leaves while the other may still touch its shared memory
}

}  // namespace le
