// le_cta_lane.cuh — the agent loop of the CTA-per-lane kernels (BaseAgent.train / test, agents/base_agent.py:64-227): one
// 256-thread CTA runs one lane.  The loop owns what every agent shares — lane claim, episodes, the SE / RN / real env step,
// the replay ring pointers, the trace record, the batched test rollouts, episode bookkeeping and the early-out rule — and
// calls the hooks of an agent type for the rest:
//   const le_lane_cfg& begin_lane(lane_id, k0, k1)   configuration, networks, parameter init or copy-in, Adam state
//   void begin_episode(episode)                      per-episode schedules (DDQN's eps)
//   int  train_action(state, episode, train_steps, tracing, explore, qgap, box)   select_train_action; `box` is free scratch
//   void store_row(row_index, state, action, next_state, r, d)                    replay_buffer.add (the agent's row format)
//   float learn(learn_iters, rb_size)                 sample + update, returns the loss
//   float* test_obs()                                 [64][SD] observation rows of the batched test forward
//   int  test_action(M, test_call, step, ep0, running)   select_test_action of row threadIdx.x (meaningful when running)
//   void end_lane(lane_id)                            final parameters out
// Every thread of the CTA calls every hook; scalars are computed redundantly by all threads (uniform), warp 0 runs the
// SE / RN mat-vec.
#pragma once
#include "le_inner_loop.cuh"

namespace le {

constexpr int kGThreads = 256;

template <int SD, int AD, typename Agent>
__device__ __forceinline__ void cta_lane_loop(const RunParams& P, Agent& ag) {
    __shared__ __align__(16) float box[16];   // state row / env step results broadcast
    __shared__ int ibox[4];
    __shared__ double dred[kGThreads / 32];
    __shared__ int sred[kGThreads / 32];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    bool first_lane = true;   // the first lane of a CTA slot is static (lane_id == slot), the rest come from the queue counter
    for (;;) {
        __syncthreads();
        if (tid == 0) ibox[0] = first_lane ? (int)blockIdx.x : (int)gridDim.x + atomicAdd(P.work_counter, 1);
        __syncthreads();
        const int lane_id = ibox[0];
        first_lane = false;
        if (lane_id >= P.n_lanes) break;
        const uint32_t k0 = P.keys[2 * lane_id], k1 = P.keys[2 * lane_id + 1];
        const le_lane_cfg& c = ag.begin_lane(lane_id, k0, k1);
        const float4* pack = P.env_pack + (int64_t)(P.env_index ? P.env_index[lane_id] : 0) * P.env_pack_stride;
        const bool env_tanh = c.env_act == LE_ACT_TANH;
        double* rewards = P.rewards + (int64_t)lane_id * P.rew_stride;
        int32_t* lengths = P.lengths + (int64_t)lane_id * P.rew_stride;
        double* test_rewards = P.test_rewards + (int64_t)lane_id * P.test_stride;
        const bool tracing = P.trace.cap > 0 && lane_id == P.trace_lane;
        const int K = c.same_action_num > 1 ? c.same_action_num : 1;

        // test rollouts on the real env, episodes = rows of one batched forward per step
        auto run_test = [&](int test_call, double* ep_out, int32_t* len_out, int64_t& test_steps) -> double {
            float* obs_rows = ag.test_obs();
            double total = 0.0;
            for (int ep0 = 0; ep0 < c.test_episodes; ep0 += 64) {
                const int M = min(64, c.test_episodes - ep0);
                double st[4] = {0, 0, 0, 0};
                float obs[SD];
                int elapsed = 0, ep_steps = 0;
                float ep_rew = 0.f;
                bool running = tid < M;
                if (tid < M) {
                    real_reset(c.real_env, philox4x32_10((uint32_t)test_call, (uint32_t)(ep0 + tid), LE_P_RESET_TEST, 0u, k0, k1), st);
                    real_obs<SD>(c.real_env, st, obs);
#pragma unroll
                    for (int i = 0; i < SD; ++i) obs_rows[tid * SD + i] = obs[i];
                }
                for (int t = 0; t < c.max_steps; t += K) {
                    if (!__syncthreads_or(running ? 1 : 0)) break;
                    const int a = ag.test_action(M, test_call, t / K, ep0, running);
                    if (running) {
                        float r, d;
                        real_step<SD>(c.real_env, c.max_steps, st, elapsed, a, obs, r, d);
                        if (K > 1) {
                            double rsum = (double)r;
                            for (int k = 1; k < K && !(d > 0.5f); ++k) {
                                float rk;
                                real_step<SD>(c.real_env, c.max_steps, st, elapsed, a, obs, rk, d);
                                rsum += (double)rk;
                            }
                            r = (float)rsum;
                        }
#pragma unroll
                        for (int i = 0; i < SD; ++i) obs_rows[tid * SD + i] = obs[i];
                        ep_rew += r;
                        ep_steps += 1;
                        if (d > 0.5f) running = false;
                    }
                }
                __syncthreads();
                if (tid < M) {
                    if (ep_out) ep_out[ep0 + tid] = (double)ep_rew;
                    if (len_out) len_out[ep0 + tid] = ep_steps;
                }
                // episode rewards are small integers / short fp32 sums: an fp32 CTA sum would round; sum in double via shared memory
                const double dv = warp_allreduce_sum((tid < M) ? (double)ep_rew : 0.0);
                int sv = (tid < M) ? ep_steps : 0;
#pragma unroll
                for (int mm = 16; mm > 0; mm >>= 1) sv += __shfl_xor_sync(LE_FULL_MASK, sv, mm);
                __syncthreads();
                if (lane == 0) { dred[warp] = dv; sred[warp] = sv; }
                __syncthreads();
                for (int q = 0; q < kGThreads / 32; ++q) { total += dred[q]; test_steps += sred[q]; }
                __syncthreads();
            }
            return total / (double)c.test_episodes;
        };

        int rb_ptr = 0, rb_size = 0;
        int64_t train_steps = 0, learn_iters = 0, test_steps = 0;
        int test_calls = 0, n_ep = 0, timed_out = 0;
        for (int episode = 0; episode < c.train_episodes; ++episode) {
            if (c.step_budget > 0 && train_steps >= c.step_budget) { timed_out = 1; break; }
            ag.begin_episode(episode);
            double st[4];
            real_reset(c.real_env, philox4x32_10((uint32_t)episode, 0u, LE_P_RESET_TRAIN, 0u, k0, k1), st);
            float state[SD];
            real_obs<SD>(c.real_env, st, state);
            int elapsed = 0, ep_len = 0;
            float ep_rew = 0.f;
            for (int t = 0; t < c.max_steps; t += K) {
                bool explore;
                float qgap = __int_as_float(0x7fc00000);
                const int action = ag.train_action(state, episode, train_steps, tracing, explore, qgap, box);
                float ns[SD], r = 0.f, d = 0.f;
                if (c.env_kind == LE_ENV_SE) {
                    __syncthreads();
                    if (warp == 0) {   // same_action_num chained SE steps, fp32 reward sum (envs/env_wrapper.py:24-30)
                        float cur[SD], ns0[SD], r0 = 0.f, d0 = 0.f;
#pragma unroll
                        for (int i = 0; i < SD; ++i) cur[i] = state[i];
                        for (int k = 0; k < K; ++k) {
                            float rk;
                            se_step_row<SD, AD>(pack, c.env_hidden, env_tanh, cur, action, lane, ns0, rk, d0);
                            r0 = k == 0 ? rk : r0 + rk;
#pragma unroll
                            for (int i = 0; i < SD; ++i) cur[i] = ns0[i];
                        }
                        if (lane == 0) {
#pragma unroll
                            for (int i = 0; i < SD; ++i) box[i] = ns0[i];
                            box[SD] = r0; box[SD + 1] = d0;
                        }
                    }
                    __syncthreads();
#pragma unroll
                    for (int i = 0; i < SD; ++i) ns[i] = box[i];
                    r = box[SD]; d = box[SD + 1];
                    __syncthreads();
                } else {   // real branch: python-float reward sum, break on done (envs/env_wrapper.py:56-61)
                    float cur[SD];
#pragma unroll
                    for (int i = 0; i < SD; ++i) cur[i] = state[i];
                    double rsum = 0.0;
                    for (int k = 0; k < K; ++k) {
                        float rr, rk;
                        real_step<SD>(c.real_env, c.max_steps, st, elapsed, action, ns, rr, d);
                        if (c.env_kind == LE_ENV_RN && c.rn_type != 0) {
                            __syncthreads();
                            if (warp == 0) {
                                float ps, ps2;
                                rn_phi2<SD>(pack, c.env_hidden, env_tanh, cur, ns, lane, ps, ps2);
                                if (lane == 0) box[0] = rn_combine(c.rn_type, (float)c.gamma, rr, ps, ps2);
                            }
                            __syncthreads();
                            rk = box[0];
                            __syncthreads();
                        } else rk = rr;
                        rsum += (double)rk;
                        r = K == 1 ? rk : (float)rsum;
#pragma unroll
                        for (int i = 0; i < SD; ++i) cur[i] = ns[i];
                        if (d > 0.5f) break;
                    }
                }
                ag.store_row(rb_ptr, state, action, ns, r, d);   // replay_buffer.add
                rb_ptr = (rb_ptr + 1 == P.ring_cap) ? 0 : rb_ptr + 1;
                rb_size = rb_size + 1 < P.ring_cap ? rb_size + 1 : P.ring_cap;
#pragma unroll
                for (int i = 0; i < SD; ++i) state[i] = ns[i];
                ep_rew += r;
                ep_len += K;
                float loss = __int_as_float(0x7fc00000);
                if (episode >= c.init_episodes) {
                    loss = ag.learn(learn_iters, rb_size);
                    learn_iters += 1;
                }
                if (tracing && train_steps < P.trace.cap && tid == 0) {
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
            double ep_value;
            if (c.use_test_env) ep_value = run_test(test_calls++, nullptr, nullptr, test_steps);
            else ep_value = (double)ep_rew;
            __syncthreads();
            if (tid == 0) { lengths[n_ep] = ep_len; rewards[n_ep] = ep_value; __threadfence_block(); }
            n_ep += 1;
            __syncthreads();
            if (env_solved(rewards, n_ep, episode, c)) break;
        }
        double score = 0.0;
        if (c.final_test)
            score = run_test(test_calls++, test_rewards, P.test_lengths ? P.test_lengths + (int64_t)lane_id * P.test_stride : nullptr, test_steps);
        __syncthreads();
        ag.end_lane(lane_id);
        if (tid == 0) {
            le_lane_out o;
            o.n_episodes = n_ep; o.timed_out = timed_out; o.train_steps = train_steps; o.learn_iters = learn_iters;
            o.test_steps = test_steps; o.score = score;
            P.out[lane_id] = o;
        }
    }
}

}  // namespace le
