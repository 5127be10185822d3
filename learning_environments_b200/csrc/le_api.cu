// le_api.cu — the C ABI of include/le_b200.h: argument checking, kernel-set dispatch, NES kernels.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "le_general_api.h"
#include "le_td3_api.h"
#include "le_instance.cuh"

// ---------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void le_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace le {
void le_register_cp_tanh();
void le_register_cp_leaky();
void le_register_ac_tanh();
void le_register_ac_leaky();

static const InstanceOps* g_instances[64];
static int g_n_instances = 0;
void le_register_instance(const InstanceOps* ops) {
    if (g_n_instances < 64) g_instances[g_n_instances++] = ops;
}
static void ensure_registered() {
    static bool done = false;
    if (!done) {
        done = true;
        le_register_cp_tanh();
        le_register_cp_leaky();
        le_register_ac_tanh();
        le_register_ac_leaky();
    }
}
const InstanceOps* le_find_instance(int sd, int ad, int units_needed, int act) {
    ensure_registered();
    const InstanceOps* best = nullptr;
    for (int i = 0; i < g_n_instances; ++i) {
        const InstanceOps* o = g_instances[i];
        if (o->sd == sd && o->ad == ad && o->act == act && o->units >= units_needed && (!best || o->units < best->units)) best = o;
    }
    return best;
}

static int qact_of(const le_lane_cfg* c) {
    if (c->q_act == LE_ACT_TANH) return QACT_TANH;
    if (c->q_act == LE_ACT_RELU || c->q_act == LE_ACT_LEAKYRELU) return QACT_LEAKY;
    return -1;
}

static const InstanceOps* instance_for(const le_lane_cfg* c, int max_hidden) {
    const int act = qact_of(c);
    if (act < 0) {
        le_set_error("Q-net activation id %d is outside the compiled kernel set (tanh, relu, leakyrelu)", c->q_act);
        return nullptr;
    }
    const int units = (max_hidden + 31) / 32;
    const InstanceOps* o = le_find_instance(c->sd, c->ad, units, act);
    if (!o) le_set_error("no compiled kernel set for state_dim=%d action_dim=%d q_hidden=%d act=%d", c->sd, c->ad, max_hidden, c->q_act);
    return o;
}

// Critic_DQN with one hidden layer whose width fits a compiled warp-per-lane kernel set: 32*U hidden units, U in {2,4} and,
// for the CartPole shapes, U = 6 (DDQN_vary samples hidden_size in [19,171], agents/DDQN_vary.py:26-59)
static int max_register_hidden(const le_lane_cfg* c) { return (c->sd == 4 && c->ad == 2) ? 192 : 128; }
static bool is_register_resident(const le_lane_cfg* c) { return c->q_kind == LE_Q_DQN && c->q_layers <= 1 && c->q_hidden <= max_register_hidden(c); }
static int q_params_of(const le_lane_cfg* c) {
    return is_register_resident(c) ? c->q_hidden * (c->sd + c->ad + 1) + c->ad : general_q_params(c);
}

static int check_env_cfg(const le_lane_cfg* c) {
    if (c->env_kind != LE_ENV_SE && c->env_kind != LE_ENV_RN && c->env_kind != LE_ENV_REAL) {
        le_set_error("unknown env_kind %d", c->env_kind);
        return LE_EINVAL;
    }
    if (c->env_kind == LE_ENV_RN && !(c->rn_type == 0 || c->rn_type == 1 || c->rn_type == 2 || c->rn_type == 5 || c->rn_type == 6)) {
        // the reference raises ValueError('No info dict provided by environment') for info-vector types on
        // CartPole/Acrobot (envs/reward_env.py:91-92) and NotImplementedError for unknown ids (:50,:59)
        le_set_error("reward_env_type %d needs an info vector (or is unknown): not available for this environment", c->rn_type);
        return LE_EUNSUPPORTED;
    }
    if ((c->real_env == LE_REAL_CARTPOLE && (c->sd != 4 || c->ad != 2)) || (c->real_env == LE_REAL_ACROBOT && (c->sd != 6 || c->ad != 3)) ||
        (c->real_env != LE_REAL_CARTPOLE && c->real_env != LE_REAL_ACROBOT)) {
        le_set_error("real_env %d does not match state_dim=%d action_dim=%d", c->real_env, c->sd, c->ad);
        return LE_EINVAL;
    }
    return LE_OK;
}

// (sd, ad) of the two compiled environment shapes, CartPole (4, 2) and Acrobot (6, 3); check_env_cfg admits only these
static bool env_shape_compiled(int sd, int ad) { return (sd == 4 && ad == 2) || (sd == 6 && ad == 3); }

// the checks of the fields a learn() step reads (nets, minibatch, TD3 hyper-parameters); no CUDA call
static int td3_learn_check(const le_td3_cfg* cfg, const char* who) {
    const le_lane_cfg* c = &cfg->base;
    if (qact_of(c) < 0 || c->q_hidden < 1 || c->q_layers > 3 || cfg->policy_delay < 1 || !(cfg->gumbel_temp > 0.0) || c->ad > 4 ||
        c->batch_size < 1) {
        le_set_error("%s: configuration outside the compiled kernel set", who);
        return LE_EUNSUPPORTED;
    }
    if (!env_shape_compiled(c->sd, c->ad)) { le_set_error("no compiled kernel set for state_dim=%d action_dim=%d", c->sd, c->ad); return LE_EUNSUPPORTED; }
    return LE_OK;
}

// the checks shared by the TD3 lane entry points, on the (maxima) configuration; no CUDA call
static int td3_check(const le_td3_cfg* cfg, const char* who) {
    const le_lane_cfg* c = &cfg->base;
    int rc = check_env_cfg(c);
    if (rc != LE_OK) return rc;
    if (c->env_kind == LE_ENV_RN) { le_set_error("%s: reward-network training envs are not built for TD3 lanes", who); return LE_EUNSUPPORTED; }
    if (c->train_episodes < 0 || c->test_episodes < 1 || c->max_steps < 1) {
        le_set_error("%s: configuration outside the compiled kernel set", who);
        return LE_EUNSUPPORTED;
    }
    return td3_learn_check(cfg, who);
}

// ---- NES kernels ------------------------------------------------------------------------------------
// Box-Muller in fp64 on Philox word pairs (oracle/philox.py normals): normal p of member `member`.
__device__ __forceinline__ void normals4(uint32_t blk, uint32_t member, uint32_t seed, uint32_t gen, float (&z)[4]) {
    const u32x4 w = philox4x32_10(blk, member, LE_P_NOISE, 0u, seed, gen);
    const double inv = 1.0 / 4294967296.0, twopi = 2.0 * 3.141592653589793;
    {
        const double u1 = ((double)w.x + 1.0) * inv, u2 = (double)w.y * inv;
        const double r = sqrt(-2.0 * log(u1));
        double s, c;
        sincos(__dmul_rn(twopi, u2), &s, &c);
        z[0] = (float)__dmul_rn(r, c);
        z[1] = (float)__dmul_rn(r, s);
    }
    {
        const double u1 = ((double)w.z + 1.0) * inv, u2 = (double)w.w * inv;
        const double r = sqrt(-2.0 * log(u1));
        double s, c;
        sincos(__dmul_rn(twopi, u2), &s, &c);
        z[2] = (float)__dmul_rn(r, c);
        z[3] = (float)__dmul_rn(r, s);
    }
}

// get_random_noise + add_noise (agents/GTN_worker.py:156-175): out[(m*3+v)][P], v: 0 theta, 1 +eps, 2 -eps
__global__ void nes_perturb_kernel(const float* __restrict__ theta, int P, int member_offset, int n_members, uint32_t seed,
                                   uint32_t gen, float noise_std, float* __restrict__ out) {
    const int nblk = (P + 3) / 4;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < (int64_t)nblk * n_members; t += (int64_t)gridDim.x * blockDim.x) {
        const int mloc = (int)(t / nblk), blk = (int)(t % nblk);
        float z[4];
        normals4((uint32_t)blk, (uint32_t)(member_offset + mloc), seed, gen, z);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = blk * 4 + k;
            if (p < P) {
                const float th = theta[p];
                const float e = __fmul_rn(z[k], noise_std);  // torch.normal(0,1) * noise_std (a rounded fp32 tensor)
                float* o = out + (int64_t)mloc * 3 * P + p;
                o[0] = th;
                o[P] = __fadd_rn(th, e);               // l_orig.weight + l_eps.weight   (no FMA contraction)
                o[2 * (int64_t)P] = __fsub_rn(th, e);  // l_orig.weight - l_eps.weight
            }
        }
    }
}

__global__ void nes_noise_kernel(int P, int member_offset, int n_members, uint32_t seed, uint32_t gen, float noise_std,
                                 float* __restrict__ eps) {
    const int nblk = (P + 3) / 4;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < (int64_t)nblk * n_members; t += (int64_t)gridDim.x * blockDim.x) {
        const int mloc = (int)(t / nblk), blk = (int)(t % nblk);
        float z[4];
        normals4((uint32_t)blk, (uint32_t)(member_offset + mloc), seed, gen, z);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = blk * 4 + k;
            if (p < P) eps[(int64_t)mloc * P + p] = __fmul_rn(z[k], noise_std);
        }
    }
}

// update_env (agents/GTN_master.py:267-298).  The reference accumulates theta += ss * w_i * eps_i SEQUENTIALLY in member order
// in fp32, so the adds of one parameter form a serial chain; what is expensive is regenerating eps_i (Philox + fp64
// Box-Muller: two log + two sincos per 4 normals).  A CTA owns kNesPT blocks of 4 parameters; its kNesMG "member groups"
// (threads) generate the terms coef_i * eps_i of a TILE of kNesMG members in parallel into shared memory, then the kNesPT
// threads of group 0 add the tile in member order: the fp32 accumulation order equals the reference's loop for any grid /
// tile / GPU count (bit-identical theta on 1/2/4/8 ranks), while the normal generation runs kNesMG-wide.
constexpr int kNesPT = 4, kNesMG = 256;
template <bool FULL>
__global__ void __launch_bounds__(kNesPT * kNesMG)
nes_update_kernel(float* __restrict__ theta, int P, int member_lo, int member_hi, uint32_t seed, uint32_t gen, float noise_std,
                  float one_minus_wd, const float* __restrict__ coef, const float* __restrict__ sign) {
    __shared__ float4 terms[2][kNesMG][kNesPT];
    const int nblk = (P + 3) / 4;
    const int pt = threadIdx.x % kNesPT, g = threadIdx.x / kNesPT;
    const int blk = blockIdx.x * kNesPT + pt;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (FULL && g == 0 && blk < nblk) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = blk * 4 + k;
            // l_orig.weight * (1 - weight_decay): python float (1 - wd) applied as an fp32 scalar
            acc[k] = p < P ? __fmul_rn(theta[p], one_minus_wd) : 0.f;
        }
    }
    int buf = 0;
    for (int i0 = member_lo; i0 < member_hi; i0 += kNesMG, buf ^= 1) {
        const int i = i0 + g;
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < member_hi && blk < nblk) {
            const float cf = coef[i];
            if (cf != 0.f) {   // a zero coefficient adds an exact zero in the reference's loop
                float z[4];
                normals4((uint32_t)blk, (uint32_t)i, seed, gen, z);
                const float sg = sign[i];
                // eps (already carrying its sign), then ss * score_transform * eps
                t.x = __fmul_rn(cf, __fmul_rn(__fmul_rn(z[0], noise_std), sg));
                t.y = __fmul_rn(cf, __fmul_rn(__fmul_rn(z[1], noise_std), sg));
                t.z = __fmul_rn(cf, __fmul_rn(__fmul_rn(z[2], noise_std), sg));
                t.w = __fmul_rn(cf, __fmul_rn(__fmul_rn(z[3], noise_std), sg));
            }
        }
        terms[buf][g][pt] = t;
        __syncthreads();   // one barrier per tile: the other buffer is only rewritten after the NEXT barrier
        if (g == 0) {
            const int n = min(kNesMG, member_hi - i0);
#pragma unroll 8
            for (int m = 0; m < n; ++m) {
                const float4 v = terms[buf][m][pt];
                acc[0] = __fadd_rn(acc[0], v.x);   // l_orig.weight + ss*score_transform*l_eps.weight, member order
                acc[1] = __fadd_rn(acc[1], v.y);
                acc[2] = __fadd_rn(acc[2], v.z);
                acc[3] = __fadd_rn(acc[3], v.w);
            }
        }
    }
    if (g == 0 && blk < nblk) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = blk * 4 + k;
            if (p < P) theta[p] = acc[k];
        }
    }
}

__global__ void real_env_step_kernel(int real_env, int max_steps, double* __restrict__ state, int32_t* __restrict__ elapsed,
                                     const int32_t* __restrict__ action, float* __restrict__ obs_out, float* __restrict__ reward,
                                     float* __restrict__ done, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double st[4] = {state[4 * i], state[4 * i + 1], state[4 * i + 2], state[4 * i + 3]};
    int el = elapsed[i];
    float r, d;
    if (real_env == LE_REAL_CARTPOLE) {
        float obs[4];
        real_step<4>(real_env, max_steps, st, el, action[i], obs, r, d);
        for (int k = 0; k < 4; ++k) obs_out[4 * i + k] = obs[k];
    } else {
        float obs[6];
        real_step<6>(real_env, max_steps, st, el, action[i], obs, r, d);
        for (int k = 0; k < 6; ++k) obs_out[6 * i + k] = obs[k];
    }
    for (int k = 0; k < 4; ++k) state[4 * i + k] = st[k];
    elapsed[i] = el;
    reward[i] = r;
    done[i] = d;
}

// parameters of one SE / RN env network (envs/virtual_env.py, envs/reward_env.py); 0 for the real envs
static int env_param_count(const le_lane_cfg* c) {
    const int H = c->env_hidden;
    if (c->env_kind == LE_ENV_SE) return 3 * H * (c->sd + c->ad + 1) + H * (c->sd + 2) + c->sd + 2;
    if (c->env_kind == LE_ENV_RN) return H * (c->sd + 2) + 1;
    return 0;
}

// ---- environment kernels: compiled once per environment shape, dispatched on sd ---------------------------------------

// floats per env of the packed SE / RN layout the lane kernels read (real envs: one float4, never read)
static int64_t env_pack_stride_f(const le_lane_cfg* c) {
    const int H = c->env_hidden;
    if (c->env_kind == LE_ENV_SE) return 4 * (c->sd == 4 ? SePack<4, 2>::pack_vec4(H) : SePack<6, 3>::pack_vec4(H));
    if (c->env_kind == LE_ENV_RN) return 4 * (c->sd == 4 ? RnPack<4>::pack_vec4(H) : RnPack<6>::pack_vec4(H));
    return 4;
}

static int64_t ring_row_floats(int sd) { return sd == 4 ? RowLayout<4>::ROWF : RowLayout<6>::ROWF; }

template <int SD, int AD>
static cudaError_t launch_pack_env(const le_lane_cfg* c, const float* theta, int n_env, float* pack, int64_t stride_f, cudaStream_t st) {
    const int64_t total = stride_f * n_env;
    const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    if (c->env_kind == LE_ENV_SE)
        pack_se_kernel<SD, AD><<<grid, 256, 0, st>>>(theta, env_param_count(c), n_env, c->env_hidden, act_slope(c->env_act, c->env_slope[0]),
                                                     act_slope(c->env_act, c->env_slope[1]), act_slope(c->env_act, c->env_slope[2]), pack,
                                                     stride_f);
    else
        pack_rn_kernel<SD><<<grid, 256, 0, st>>>(theta, env_param_count(c), n_env, c->env_hidden, act_slope(c->env_act, c->env_slope[0]),
                                                 pack, stride_f);
    return cudaGetLastError();
}

// n_env SE / RN parameter vectors -> the packed layout (stride_f = env_pack_stride_f floats per env); real envs: nothing
static cudaError_t pack_env(const le_lane_cfg* c, const float* theta, int n_env, float* pack, int64_t stride_f, cudaStream_t st) {
    if (c->env_kind == LE_ENV_REAL) return cudaSuccess;
    return c->sd == 4 ? launch_pack_env<4, 2>(c, theta, n_env, pack, stride_f, st) : launch_pack_env<6, 3>(c, theta, n_env, pack, stride_f, st);
}

// SE / RN unit operators (one warp per row), sharing the device code of the lane kernels
template <int SD, int AD>
__global__ void se_forward_kernel(const float4* __restrict__ pack, int64_t pack_stride, int H, int is_tanh, int lanes_per_member,
                                  const float* __restrict__ state, const int32_t* __restrict__ action, float* __restrict__ ns_out,
                                  float* __restrict__ reward, float* __restrict__ done, int n) {
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    float s[SD], ns[SD], r, d;
#pragma unroll
    for (int i = 0; i < SD; ++i) s[i] = state[(int64_t)row * SD + i];
    se_step_row<SD, AD>(pack + (int64_t)(row / lanes_per_member) * pack_stride, H, is_tanh != 0, s, action[row], lane, ns, r, d);
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < SD; ++i) ns_out[(int64_t)row * SD + i] = ns[i];
        reward[row] = r;
        done[row] = d;
    }
}

template <int SD>
__global__ void rn_reward_kernel(const float4* __restrict__ pack, int64_t pack_stride, int H, int is_tanh, int rn_type, float gamma,
                                 int lanes_per_member, const float* __restrict__ s_in, const float* __restrict__ s2_in,
                                 const float* __restrict__ rr, float* __restrict__ out, int n) {
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    float s[SD], s2[SD];
#pragma unroll
    for (int i = 0; i < SD; ++i) { s[i] = s_in[(int64_t)row * SD + i]; s2[i] = s2_in[(int64_t)row * SD + i]; }
    float ps = 0.f, ps2 = 0.f;
    if (rn_type != 0) rn_phi2<SD>(pack + (int64_t)(row / lanes_per_member) * pack_stride, H, is_tanh != 0, s, s2, lane, ps, ps2);
    if (lane == 0) out[row] = rn_combine(rn_type, gamma, rr[row], ps, ps2);
}

// FP32 FFMA peak microbenchmark: the denominator of the fused kernel's roofline (MEASURED_PEAKS.json has no
// FP32 figure).  8 independent FMA chains per thread, 256 threads x 8 CTAs per SM.
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* out, int iters, float a, float b) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    const float s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456f) out[0] = s;
}

// Multi-warp lanes (inner_loop_mw_kernel) for small populations: a lane gets a whole CTA instead of one warp (2.7x shorter
// generations at the yaml's population of 16, profiles/r02_mw_lanes.txt); up to two lanes per SM queue on the CTAs before the
// warp-per-lane kernel, which runs every lane at once, is the faster choice.
// LE_MW=0 never, LE_MW=1 whenever the kernel set has the kernel (any lane count), default: auto.
static bool use_mw_lanes(const InstanceOps* ops, int n_lanes, int sms) {
    if (ops->mw_warps <= 1) return false;
    const char* e = getenv("LE_MW");
    if (e && e[0] == '0') return false;
    if (e && e[0] == '1') return true;
    return n_lanes <= 2 * sms;
}

// Cluster lanes when every lane can have two SMs to itself (the yaml's population of 16 = 48 lanes on 148 SMs): LE_MWC=0 disables.
static bool use_mwc_lanes(const InstanceOps* ops, int n_lanes, int sms) {
    if (ops->mwc_smem_bytes <= 0 || 2 * n_lanes > sms) return false;
    const char* e = getenv("LE_MW");
    if (e && e[0] == '0') return false;
    const char* c = getenv("LE_MWC");
    return !(c && c[0] == '0');
}

// replay ring rows: rb_size, but never more than a lane can add (every episode at max_steps, or the step budget plus one episode)
static int ring_capacity(const le_lane_cfg* c) {
    int64_t max_total = (int64_t)c->train_episodes * c->max_steps;
    if (c->step_budget > 0 && c->step_budget + c->max_steps < max_total) max_total = c->step_budget + c->max_steps;
    if (max_total < 1) max_total = 1;
    return (int)((int64_t)c->rb_size < max_total ? c->rb_size : max_total);
}

static int64_t round256(int64_t bytes) { return (bytes + 255) / 256 * 256; }

// The lane families: the warp-per-lane, multi-warp (one lane per CTA) and cluster (one lane per cluster of two CTAs) kernels of
// a register Q-net kernel set, the CTA-per-lane general DDQN kernel and the TD3 kernel.
enum class LaneFamily { Warp, MultiWarp, Cluster, General, Td3 };

// One launch of lanes.  Every family lays out its workspace the same way, each region 256-byte aligned:
//   [env pack: max(n_env, 1) x pack_stride_f floats | lane queue counter: 256 B | slots: `slots` x slot_bytes]
// A slot is the replay ring of a register lane, or everything a CTA-per-lane lane keeps in HBM (ring, nets, Adam state,
// activations).  With the slots last, a shorter workspace only cuts slots off the end: le_td3_run keeps fewer lanes resident.
struct LanePlan {
    LaneFamily family;
    const InstanceOps* ops;   // register kernel set of warp / multi-warp / cluster lanes, else null
    GeneralPlan gp;           // general lanes
    Td3Plan tp;               // TD3 lanes
    int grid, slots, ring_cap;
    int64_t pack_stride_f, slot_bytes, off_counter, off_slots, total_bytes;
};

// The configuration checks of the lane entry points, before any CUDA call.  c: the lane configuration that fixes the shapes
// (cfg 0 / the maxima); td3: its TD3 configuration for TD3 lanes, else null.  Sets pl->family (Warp for every register kernel
// set; plan_lanes picks among its kernels) and pl->ops.
static int check_lanes(const le_lane_cfg* c, const le_td3_cfg* td3, int n_lanes, const char* who, LanePlan* pl) {
    pl->ops = nullptr;
    if (td3) { pl->family = LaneFamily::Td3; return td3_check(td3, who); }
    const int rc = check_env_cfg(c);
    if (rc != LE_OK) return rc;
    if (c->batch_size < 1 || c->rb_size < 1 || c->train_episodes < 0 || c->test_episodes < 1 || c->max_steps < 1 || n_lanes < 1) {
        le_set_error("bad lane configuration (batch_size=%d rb_size=%d train_episodes=%d test_episodes=%d max_steps=%d n_lanes=%d)",
                     c->batch_size, c->rb_size, c->train_episodes, c->test_episodes, c->max_steps, n_lanes);
        return LE_EINVAL;
    }
    if (c->q_layers > 3) { le_set_error("Q-network hidden_layer=%d: the compiled kernel set covers up to 3 hidden layers", c->q_layers); return LE_EUNSUPPORTED; }
    if (is_register_resident(c)) {
        pl->family = LaneFamily::Warp;
        pl->ops = instance_for(c, c->q_hidden);
        return pl->ops ? LE_OK : LE_EUNSUPPORTED;
    }
    pl->family = LaneFamily::General;
    if (qact_of(c) < 0) { le_set_error("Q-net activation id %d is outside the compiled kernel set", c->q_act); return LE_EUNSUPPORTED; }
    return LE_OK;
}

// Sizes lanes that passed check_lanes for the current device: family, grid, resident slots and the workspace layout.
static int plan_lanes(const le_lane_cfg* c, const le_td3_cfg* td3, int n_lanes, int n_env, LanePlan* pl) {
    int dev = 0, sms = 0;
    LE_CUDA_CHECK(cudaGetDevice(&dev));
    LE_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    pl->ring_cap = ring_capacity(c);
    const InstanceOps* ops = pl->ops;
    int64_t slot_floats = (int64_t)pl->ring_cap * ring_row_floats(c->sd);   // register lanes: one replay ring
    if (pl->family == LaneFamily::Td3) {
        const int rc = td3_plan(td3, n_lanes, pl->ring_cap, sms, &pl->tp);
        if (rc != LE_OK) return rc;
        pl->grid = pl->slots = pl->tp.grid;
        slot_floats = pl->tp.slot_floats;
    } else if (pl->family == LaneFamily::General) {
        const int rc = general_plan(c, n_lanes, pl->ring_cap, sms, &pl->gp);
        if (rc != LE_OK) return rc;
        pl->grid = pl->slots = pl->gp.grid;
        slot_floats = pl->gp.slot_floats;
    } else if (use_mwc_lanes(ops, n_lanes, sms)) {
        pl->family = LaneFamily::Cluster;
        pl->grid = 2 * n_lanes;      // one cluster of two CTAs per lane
        pl->slots = n_lanes;
    } else if (use_mw_lanes(ops, n_lanes, sms)) {
        pl->family = LaneFamily::MultiWarp;
        pl->grid = pl->slots = n_lanes < sms ? n_lanes : sms;
    } else {
        int per_sm = ops->inner_max_ctas_per_sm();
        if (per_sm < 1) per_sm = 1;
        const int want = (n_lanes + ops->inner_warps - 1) / ops->inner_warps;
        pl->grid = want < sms * per_sm ? want : sms * per_sm;
        pl->slots = pl->grid * ops->inner_warps;
    }
    pl->pack_stride_f = env_pack_stride_f(c);
    pl->slot_bytes = slot_floats * (int64_t)sizeof(float);
    pl->off_counter = round256((int64_t)(n_env > 0 ? n_env : 1) * pl->pack_stride_f * 4);
    pl->off_slots = pl->off_counter + 256;
    // the TD3 size is td3_workspace_bytes: a slot region without padding, and possibly fewer slots
    pl->total_bytes = pl->off_slots + round256((int64_t)pl->slots * pl->slot_bytes);
    return LE_OK;
}

// le_td3_workspace_bytes of a planned TD3 launch.  A slot of the widest vary_hp shapes (hidden 1530 x 3 layers) is ~0.3 GB:
// when every resident lane's slot does not fit 90 % of the free device memory, ask for fewer slots (the lane queue runs the
// rest on them).
static int64_t td3_workspace_bytes(const LanePlan& pl) {
    size_t free_b = 0, total_b = 0;
    LE_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const int64_t room = (int64_t)(0.9 * (double)free_b) - pl.off_slots;
    int64_t slots = pl.slots;
    if (slots * pl.slot_bytes > room) slots = room / pl.slot_bytes > 1 ? room / pl.slot_bytes : 1;
    return pl.off_slots + slots * pl.slot_bytes;
}

// Packs the env into the workspace, zeroes the lane queue counter and fills the RunParams fields every lane family reads;
// the entry points add their own.
static int start_lanes(const LanePlan& pl, const le_lane_cfg* c, const float* env_theta, int n_env, const int32_t* env_index,
                       const uint32_t* keys, int n_lanes, le_lane_out* out, double* rewards, int32_t* lengths, double* test_rewards,
                       char* ws, const le_trace* trace, int trace_lane, cudaStream_t st, RunParams* P) {
    LE_CUDA_CHECK(pack_env(c, env_theta, n_env, (float*)ws, pl.pack_stride_f, st));
    LE_CUDA_CHECK(cudaMemsetAsync(ws + pl.off_counter, 0, sizeof(int), st));
    memset(P, 0, sizeof(*P));
    P->env_pack = (const float4*)ws; P->env_pack_stride = pl.pack_stride_f / 4;
    P->env_index = env_index; P->keys = keys;
    P->n_lanes = n_lanes; P->out = out; P->rewards = rewards; P->lengths = lengths; P->test_rewards = test_rewards;
    P->rew_stride = c->train_episodes > 0 ? c->train_episodes : 1; P->test_stride = c->test_episodes;
    P->ring_cap = pl.ring_cap;
    P->work_counter = (int*)(ws + pl.off_counter);
    if (trace && trace->cap > 0) { P->trace = *trace; P->trace_lane = trace_lane; }
    return LE_OK;
}

}  // namespace le

using namespace le;

// Owns the private stream and the device arena of a *_host entry point: every early return (LE_CUDA_CHECK) releases both.
// The arena holds one 256-byte aligned segment per host array (add) and the call's device-only regions (reserve).
struct HostCall {
    struct Seg { const void* src; void* dst_host; size_t bytes; size_t off; };
    cudaStream_t st = nullptr;
    char* arena = nullptr;
    std::vector<Seg> segs;
    size_t total = 0;
    ~HostCall() {
        if (arena) cudaFreeAsync(arena, st);
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
    }
    // segment of `bytes`: filled from host `src` before the run, copied to host `dst` after it (either may be null)
    size_t add(const void* src, void* dst, size_t bytes) {
        segs.push_back(Seg{src, dst, bytes, total});
        total += (bytes + 255) / 256 * 256;
        return segs.size() - 1;
    }
    size_t reserve(size_t bytes) { const size_t off = total; total += bytes; return off; }
    char* dp(size_t i) const { return segs[i].bytes ? arena + segs[i].off : nullptr; }
    // creates the stream, allocates the arena and copies the inputs in
    int stage_in() {
        LE_CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        LE_CUDA_CHECK(cudaMallocAsync((void**)&arena, total, st));
        for (auto& s : segs)
            if (s.src && s.bytes) LE_CUDA_CHECK(cudaMemcpyAsync(arena + s.off, s.src, s.bytes, cudaMemcpyHostToDevice, st));
        return LE_OK;
    }
    // after a run that returned rc: copies the outputs out (rc == LE_OK) and waits for the stream
    int stage_out(int rc, const char* who) {
        if (rc == LE_OK) {
            for (auto& s : segs)
                if (s.dst_host && s.bytes) {
                    cudaError_t e = cudaMemcpyAsync(s.dst_host, arena + s.off, s.bytes, cudaMemcpyDeviceToHost, st);
                    if (e != cudaSuccess) { le_set_error("D2H copy failed: %s", cudaGetErrorString(e)); rc = LE_ECUDA; break; }
                }
        }
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess && rc == LE_OK) { le_set_error("%s: %s", who, cudaGetErrorString(e)); rc = LE_ECUDA; }
        return rc;
    }
};

// The segments both *_run_host entries stage: the lane configurations, env parameters, env index and keys in; per-lane results,
// reward / length histories and test rewards out; and the arrays of an optional trace.
struct LaneSegs { size_t cfg, th, ei, key, out, rw, ln, tr, trace[6]; int tcap; };

static LaneSegs add_lane_segs(HostCall& hc, const void* cfgs, size_t cfg_bytes, const le_lane_cfg* c, const float* env_theta, int n_env,
                              const int32_t* env_index, const uint32_t* keys, int n_lanes, le_lane_out* out, double* rewards,
                              int32_t* lengths, double* test_rewards, const le_trace* trace) {
    const int rs = c->train_episodes > 0 ? c->train_episodes : 1;
    LaneSegs s;
    s.cfg = hc.add(cfgs, nullptr, cfg_bytes);
    s.th = hc.add(env_theta, nullptr, env_theta ? sizeof(float) * (size_t)env_param_count(c) * n_env : 0);
    s.ei = hc.add(env_index, nullptr, env_index ? sizeof(int32_t) * n_lanes : 0);
    s.key = hc.add(keys, nullptr, sizeof(uint32_t) * 2 * n_lanes);
    s.out = hc.add(nullptr, out, sizeof(le_lane_out) * n_lanes);
    s.rw = hc.add(nullptr, rewards, sizeof(double) * (size_t)rs * n_lanes);
    s.ln = hc.add(nullptr, lengths, sizeof(int32_t) * (size_t)rs * n_lanes);
    s.tr = hc.add(nullptr, test_rewards, sizeof(double) * (size_t)c->test_episodes * n_lanes);
    s.tcap = trace && trace->cap > 0 ? trace->cap : 0;
    if (s.tcap) {   // 4-byte entries, one per step (next_state, k = 2: sd per step)
        void* const dst[6] = {trace->action, trace->explore, trace->next_state, trace->reward, trace->done, trace->loss};
        for (int k = 0; k < 6; ++k) s.trace[k] = hc.add(nullptr, dst[k], 4 * (size_t)s.tcap * (k == 2 ? c->sd : 1));
    }
    return s;
}

// HostCall::stage_in, then zeroes the reward / length histories and marks the trace (untouched entries read -1 / NaN);
// *tr: the trace with device pointers (cap 0 without one)
static int stage_lane_segs(HostCall& hc, const LaneSegs& s, le_trace* tr) {
    const int rc = hc.stage_in();
    if (rc != LE_OK) return rc;
    LE_CUDA_CHECK(cudaMemsetAsync(hc.dp(s.rw), 0, hc.segs[s.rw].bytes, hc.st));
    LE_CUDA_CHECK(cudaMemsetAsync(hc.dp(s.ln), 0, hc.segs[s.ln].bytes, hc.st));
    memset(tr, 0, sizeof(*tr));
    if (s.tcap) {
        for (int k = 0; k < 6; ++k) LE_CUDA_CHECK(cudaMemsetAsync(hc.dp(s.trace[k]), 0xff, hc.segs[s.trace[k]].bytes, hc.st));
        tr->cap = s.tcap;
        tr->action = (int32_t*)hc.dp(s.trace[0]); tr->explore = (int32_t*)hc.dp(s.trace[1]); tr->next_state = (float*)hc.dp(s.trace[2]);
        tr->reward = (float*)hc.dp(s.trace[3]); tr->done = (float*)hc.dp(s.trace[4]); tr->loss = (float*)hc.dp(s.trace[5]);
    }
    return LE_OK;
}

extern "C" {

int le_version(void) { return LE_VERSION; }
const char* le_last_error(void) { return g_err; }
int le_sizeof_lane_cfg(void) { return (int)sizeof(le_lane_cfg); }

int le_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, char* name, int name_cap) {
    cudaDeviceProp p;
    LE_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (name && name_cap > 0) { strncpy(name, p.name, name_cap - 1); name[name_cap - 1] = 0; }
    return LE_OK;
}

// Measured FP32 FFMA throughput in TFLOP/s (2 flop per FMA), best of `reps` timed launches on `stream`.
int le_bench_ffma(int iters, int reps, double* tflops_out, void* stream) {
    if (iters < 1 || reps < 1 || !tflops_out) { le_set_error("le_bench_ffma: bad arguments"); return LE_EINVAL; }
    int dev = 0, sms = 0;
    LE_CUDA_CHECK(cudaGetDevice(&dev));
    LE_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cudaStream_t st = (cudaStream_t)stream;
    float* out = nullptr;
    LE_CUDA_CHECK(cudaMalloc((void**)&out, 4));
    cudaEvent_t e0, e1;
    LE_CUDA_CHECK(cudaEventCreate(&e0));
    LE_CUDA_CHECK(cudaEventCreate(&e1));
    const int grid = sms * 8;
    double best = 0.0;
    for (int r = 0; r < reps + 1; ++r) {
        LE_CUDA_CHECK(cudaEventRecord(e0, st));
        ffma_peak_kernel<<<grid, 256, 0, st>>>(out, iters, 0.999f, 0.001f);
        LE_CUDA_CHECK(cudaEventRecord(e1, st));
        LE_CUDA_CHECK(cudaEventSynchronize(e1));
        float ms = 0.f;
        LE_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 128.0 * (double)iters * 256.0 * (double)grid;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (r > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    *tflops_out = best;
    return LE_OK;
}

// ---- unit operators ----------------------------------------------------------------------------------
int le_se_forward(const le_lane_cfg* cfg, const float* theta_dev, int pop, int lanes_per_member, const float* state_dev,
                  const int32_t* action_dev, float* next_state_dev, float* reward_dev, float* done_dev, void* stream) {
    if (!cfg || pop < 1 || lanes_per_member < 1) { le_set_error("le_se_forward: bad arguments"); return LE_EINVAL; }
    if (check_env_cfg(cfg) != LE_OK) return LE_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    le_lane_cfg c = *cfg;
    c.env_kind = LE_ENV_SE;
    const int H = c.env_hidden, n = pop * lanes_per_member, is_tanh = c.env_act == LE_ACT_TANH;
    const int64_t stride_f = env_pack_stride_f(&c);
    float* pack = nullptr;
    LE_CUDA_CHECK(cudaMallocAsync((void**)&pack, (size_t)pop * stride_f * 4, st));
    LE_CUDA_CHECK(pack_env(&c, theta_dev, pop, pack, stride_f, st));
    if (c.sd == 4)
        se_forward_kernel<4, 2><<<(n + 3) / 4, 128, 0, st>>>((const float4*)pack, stride_f / 4, H, is_tanh, lanes_per_member, state_dev,
                                                             action_dev, next_state_dev, reward_dev, done_dev, n);
    else
        se_forward_kernel<6, 3><<<(n + 3) / 4, 128, 0, st>>>((const float4*)pack, stride_f / 4, H, is_tanh, lanes_per_member, state_dev,
                                                             action_dev, next_state_dev, reward_dev, done_dev, n);
    LE_CUDA_CHECK(cudaGetLastError());
    LE_CUDA_CHECK(cudaFreeAsync(pack, st));
    return LE_OK;
}

int le_rn_reward(const le_lane_cfg* cfg, const float* theta_dev, int pop, int lanes_per_member, const float* state_dev,
                 const float* next_state_dev, const float* real_reward_dev, float* reward_dev, void* stream) {
    if (!cfg || pop < 1 || lanes_per_member < 1) { le_set_error("le_rn_reward: bad arguments"); return LE_EINVAL; }
    le_lane_cfg c = *cfg;
    c.env_kind = LE_ENV_RN;
    int rc = check_env_cfg(&c);
    if (rc != LE_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int H = c.env_hidden, n = pop * lanes_per_member, is_tanh = c.env_act == LE_ACT_TANH;
    const int64_t stride_f = env_pack_stride_f(&c);
    float* pack = nullptr;
    LE_CUDA_CHECK(cudaMallocAsync((void**)&pack, (size_t)pop * stride_f * 4, st));
    LE_CUDA_CHECK(pack_env(&c, theta_dev, pop, pack, stride_f, st));
    if (c.sd == 4)
        rn_reward_kernel<4><<<(n + 3) / 4, 128, 0, st>>>((const float4*)pack, stride_f / 4, H, is_tanh, c.rn_type, (float)c.gamma,
                                                         lanes_per_member, state_dev, next_state_dev, real_reward_dev, reward_dev, n);
    else
        rn_reward_kernel<6><<<(n + 3) / 4, 128, 0, st>>>((const float4*)pack, stride_f / 4, H, is_tanh, c.rn_type, (float)c.gamma,
                                                         lanes_per_member, state_dev, next_state_dev, real_reward_dev, reward_dev, n);
    LE_CUDA_CHECK(cudaGetLastError());
    LE_CUDA_CHECK(cudaFreeAsync(pack, st));
    return LE_OK;
}

int le_qnet_forward(const le_lane_cfg* cfg, const float* q_theta_dev, int n, const float* state_dev, float* q_out_dev,
                    int32_t* argmax_dev, void* stream) {
    if (!cfg || n < 1) { le_set_error("le_qnet_forward: bad arguments"); return LE_EINVAL; }
    if (cfg->q_layers > 3) { le_set_error("le_qnet_forward: hidden_layer > 3"); return LE_EUNSUPPORTED; }
    if (!is_register_resident(cfg)) {
        if (qact_of(cfg) < 0 || !env_shape_compiled(cfg->sd, cfg->ad)) { le_set_error("le_qnet_forward: unsupported Q-network"); return LE_EUNSUPPORTED; }
        return general_qnet_forward(cfg, q_theta_dev, n, state_dev, q_out_dev, argmax_dev, (cudaStream_t)stream);
    }
    const InstanceOps* ops = instance_for(cfg, cfg->q_hidden);
    if (!ops) return LE_EUNSUPPORTED;
    const int Pq = cfg->q_hidden * (cfg->sd + cfg->ad + 1) + cfg->ad;
    LE_CUDA_CHECK(ops->launch_qnet_forward(q_theta_dev, Pq, cfg->q_hidden, cfg->q_act == LE_ACT_LEAKYRELU ? 0.01f : 0.f, state_dev,
                                           q_out_dev, argmax_dev, n, (cudaStream_t)stream));
    return LE_OK;
}

int le_real_env_step(int real_env, int max_steps, double* state_dev, int32_t* elapsed_dev, const int32_t* action_dev, float* obs_dev,
                     float* reward_dev, float* done_dev, int n, void* stream) {
    if ((real_env != LE_REAL_CARTPOLE && real_env != LE_REAL_ACROBOT) || n < 1) { le_set_error("le_real_env_step: bad arguments"); return LE_EINVAL; }
    real_env_step_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(real_env, max_steps, state_dev, elapsed_dev, action_dev,
                                                                             obs_dev, reward_dev, done_dev, n);
    LE_CUDA_CHECK(cudaGetLastError());
    return LE_OK;
}

int le_td_update(const le_lane_cfg* cfg, float* q_theta_dev, float* q_target_dev, float* adam_m_dev, float* adam_v_dev,
                 int32_t* adam_t_dev, int n, const float* batch_rows_dev, float* loss_dev, void* stream) {
    if (!cfg || n < 1 || cfg->batch_size < 1) { le_set_error("le_td_update: bad arguments"); return LE_EINVAL; }
    if (cfg->q_layers > 3) { le_set_error("le_td_update: hidden_layer > 3"); return LE_EUNSUPPORTED; }
    const bool general = !is_register_resident(cfg);
    const InstanceOps* ops = general ? nullptr : instance_for(cfg, cfg->q_hidden);
    if (general && (qact_of(cfg) < 0 || !env_shape_compiled(cfg->sd, cfg->ad))) { le_set_error("le_td_update: unsupported Q-network"); return LE_EUNSUPPORTED; }
    if (!general && !ops) return LE_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    le_lane_cfg* cfg_dev = nullptr;
    LE_CUDA_CHECK(cudaMallocAsync((void**)&cfg_dev, sizeof(le_lane_cfg), st));
    LE_CUDA_CHECK(cudaMemcpyAsync(cfg_dev, cfg, sizeof(le_lane_cfg), cudaMemcpyHostToDevice, st));
    if (general) {
        const int rc = general_td_update(cfg, cfg_dev, q_theta_dev, q_target_dev, adam_m_dev, adam_v_dev, adam_t_dev, n, batch_rows_dev, loss_dev, st);
        cudaFreeAsync(cfg_dev, st);
        return rc;
    }
    const int Pq = cfg->q_hidden * (cfg->sd + cfg->ad + 1) + cfg->ad;
    LE_CUDA_CHECK(ops->launch_td_update(cfg_dev, q_theta_dev, q_target_dev, adam_m_dev, adam_v_dev, adam_t_dev, Pq, batch_rows_dev,
                                        cfg->batch_size, loss_dev, n, st));
    LE_CUDA_CHECK(cudaFreeAsync(cfg_dev, st));
    return LE_OK;
}

// ---- fused hot path -----------------------------------------------------------------------------------
int64_t le_inner_loop_workspace_bytes(const le_lane_cfg* cfg, int n_lanes, int n_env) {
    if (!cfg) { le_set_error("le_inner_loop_workspace_bytes: cfg is NULL"); return LE_EINVAL; }
    LanePlan pl;
    int rc = check_lanes(cfg, nullptr, n_lanes, "le_inner_loop_workspace_bytes", &pl);
    if (rc == LE_OK) rc = plan_lanes(cfg, nullptr, n_lanes, n_env, &pl);
    return rc == LE_OK ? pl.total_bytes : rc;
}

int le_inner_loop_run(const le_lane_cfg* cfg_dev, int n_cfg, const le_lane_cfg* cfg_host0, const float* env_theta_dev, int n_env,
                      const int32_t* env_index_dev, const uint32_t* keys_dev, const float* q_init_dev, float* q_final_dev, int n_lanes,
                      le_lane_out* out_dev, double* rewards_dev, int32_t* lengths_dev, double* test_rewards_dev, int32_t* test_lengths_dev,
                      void* workspace_dev, int64_t workspace_bytes, const le_trace* trace_host, int trace_lane, void* stream) {
    if (!cfg_dev || !cfg_host0 || !keys_dev || !out_dev || !rewards_dev || !lengths_dev || !test_rewards_dev || !workspace_dev ||
        (n_cfg != 1 && n_cfg != n_lanes)) {
        le_set_error("le_inner_loop_run: bad arguments (n_cfg must be 1 or n_lanes; no NULL outputs)");
        return LE_EINVAL;
    }
    const le_lane_cfg* c = cfg_host0;
    LanePlan pl;
    int rc = check_lanes(c, nullptr, n_lanes, "le_inner_loop_run", &pl);
    if (rc != LE_OK) return rc;
    if (c->env_kind != LE_ENV_REAL && (!env_theta_dev || n_env < 1)) { le_set_error("le_inner_loop_run: env_theta is required for SE/RN lanes"); return LE_EINVAL; }
    rc = plan_lanes(c, nullptr, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    if (workspace_bytes < pl.total_bytes) {
        le_set_error("le_inner_loop_run: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes, (long long)pl.total_bytes);
        return LE_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace_dev;
    RunParams P;
    rc = start_lanes(pl, c, env_theta_dev, n_env, env_index_dev, keys_dev, n_lanes, out_dev, rewards_dev, lengths_dev, test_rewards_dev, ws,
                     trace_host, trace_lane, st, &P);
    if (rc != LE_OK) return rc;
    P.cfg = cfg_dev; P.n_cfg = n_cfg;
    P.q_init = q_init_dev; P.q_final = q_final_dev; P.q_stride = q_params_of(c);
    P.test_lengths = test_lengths_dev;
    P.rings = (float*)(ws + pl.off_slots); P.ring_stride = pl.slot_bytes / 4;
    if (pl.family == LaneFamily::General) LE_CUDA_CHECK(general_launch(c, P, P.rings, pl.gp, st));
    else if (pl.family == LaneFamily::Warp) LE_CUDA_CHECK(pl.ops->launch_inner(P, pl.grid, st));
    else {
        // the member's SE / RN pack is staged in the CTA's shared memory by one TMA bulk copy per lane when it fits beside the lane state
        const bool cluster = pl.family == LaneFamily::Cluster;
        const int64_t pack_bytes = c->env_kind == LE_ENV_REAL ? 0 : pl.pack_stride_f * 4;
        const int64_t lane_smem = cluster ? pl.ops->mwc_smem_bytes : pl.ops->mw_smem_bytes;
        if (pack_bytes > 0 && lane_smem + pack_bytes <= 227 * 1024) P.mw_pack_f4 = (int)(pack_bytes / 16);
        if (cluster) LE_CUDA_CHECK(pl.ops->launch_inner_mwc(P, pl.slots, st));
        else LE_CUDA_CHECK(pl.ops->launch_inner_mw(P, pl.grid, st));
    }
    return LE_OK;
}

int le_inner_loop_plan(const le_lane_cfg* cfg, int n_lanes, int n_env, int* grid, int* slots, int* ring_cap, int* units,
                       int64_t* ring_offset_bytes) {
    LanePlan pl;
    int rc = check_lanes(cfg, nullptr, n_lanes, "le_inner_loop_plan", &pl);
    if (rc == LE_OK) rc = plan_lanes(cfg, nullptr, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    if (grid) *grid = pl.grid;
    if (slots) *slots = pl.slots;
    if (ring_cap) *ring_cap = pl.ring_cap;
    if (units) *units = pl.ops ? pl.ops->units : 0;
    if (ring_offset_bytes) *ring_offset_bytes = pl.off_slots;
    return LE_OK;
}

int le_inner_loop_run_host(const le_lane_cfg* cfgs, int n_cfg, const float* env_theta, int n_env, const int32_t* env_index,
                           const uint32_t* keys, const float* q_init, float* q_final, int n_lanes, le_lane_out* out, double* rewards,
                           int32_t* lengths, double* test_rewards, int device) {
    if (!cfgs || !keys || !out || !rewards || !lengths || !test_rewards || n_lanes < 1 || (n_cfg != 1 && n_cfg != n_lanes)) {
        le_set_error("le_inner_loop_run_host: bad arguments");
        return LE_EINVAL;
    }
    const le_lane_cfg* c = &cfgs[0];
    LanePlan pl;
    int rc = check_lanes(c, nullptr, n_lanes, "le_inner_loop_run_host", &pl);
    if (rc != LE_OK) return rc;
    LE_CUDA_CHECK(cudaSetDevice(device));
    rc = plan_lanes(c, nullptr, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    const int Pq = q_params_of(c);
    HostCall hc;
    const LaneSegs s = add_lane_segs(hc, cfgs, sizeof(le_lane_cfg) * n_cfg, c, env_theta, n_env, env_index, keys, n_lanes, out, rewards,
                                     lengths, test_rewards, nullptr);
    const size_t i_qi = hc.add(q_init, nullptr, q_init ? sizeof(float) * (size_t)Pq * n_lanes : 0);
    const size_t i_qf = hc.add(nullptr, q_final, q_final ? sizeof(float) * (size_t)Pq * n_lanes : 0);
    const size_t off_ws = hc.reserve((size_t)pl.total_bytes);
    le_trace tr;
    rc = stage_lane_segs(hc, s, &tr);
    if (rc != LE_OK) return rc;
    rc = le_inner_loop_run((const le_lane_cfg*)hc.dp(s.cfg), n_cfg, c, (const float*)hc.dp(s.th), n_env, (const int32_t*)hc.dp(s.ei),
                           (const uint32_t*)hc.dp(s.key), (const float*)hc.dp(i_qi), (float*)hc.dp(i_qf), n_lanes, (le_lane_out*)hc.dp(s.out),
                           (double*)hc.dp(s.rw), (int32_t*)hc.dp(s.ln), (double*)hc.dp(s.tr), nullptr, hc.arena + off_ws, pl.total_bytes, nullptr, 0,
                           hc.st);
    return hc.stage_out(rc, "le_inner_loop_run_host");   // ~HostCall frees the arena and destroys the stream
}

// ---- TD3_discrete_vary lanes ----------------------------------------------------------------------------
int le_td3_param_counts(const le_td3_cfg* cfg, int* p_actor, int* p_critic) {
    if (!cfg || cfg->base.q_hidden < 1) { le_set_error("le_td3_param_counts: bad arguments"); return LE_EINVAL; }
    const int sd = cfg->base.sd, ad = cfg->base.ad, H = cfg->base.q_hidden, L = cfg->base.q_layers > 1 ? cfg->base.q_layers : 1;
    if (p_actor) *p_actor = sd * H + H + (L - 1) * (H * H + H) + H * ad + ad;
    if (p_critic) *p_critic = (sd + ad) * H + H + (L - 1) * (H * H + H) + H + 1;
    return LE_OK;
}

int le_td3_learn(const le_td3_cfg* cfg, float* actor_dev, float* actor_target_dev, float* critic1_dev, float* critic1_target_dev,
                 float* critic2_dev, float* critic2_target_dev, float* adam_m_actor_dev, float* adam_v_actor_dev, float* adam_m_critic1_dev,
                 float* adam_v_critic1_dev, float* adam_m_critic2_dev, float* adam_v_critic2_dev, int32_t* counters_dev, int n,
                 const float* rows_dev, const float* policy_noise_dev, const float* expo_target_dev, const float* expo_actor_dev,
                 float* critic_loss_dev, void* stream) {
    float* const nets[6] = {actor_dev, actor_target_dev, critic1_dev, critic1_target_dev, critic2_dev, critic2_target_dev};
    float* const adam[6] = {adam_m_actor_dev, adam_v_actor_dev, adam_m_critic1_dev, adam_v_critic1_dev, adam_m_critic2_dev, adam_v_critic2_dev};
    bool any_null = !cfg || !counters_dev || !rows_dev || !policy_noise_dev || !expo_target_dev || !expo_actor_dev || !critic_loss_dev;
    for (int i = 0; i < 6; ++i) any_null = any_null || !nets[i] || !adam[i];
    if (any_null || n < 1 || cfg->base.batch_size < 1) { le_set_error("le_td3_learn: bad arguments"); return LE_EINVAL; }
    const int rc = td3_learn_check(cfg, "le_td3_learn");
    if (rc != LE_OK) return rc;
    return td3_learn(cfg, nets, adam, counters_dev, n, rows_dev, policy_noise_dev, expo_target_dev, expo_actor_dev, critic_loss_dev,
                     (cudaStream_t)stream);
}

int64_t le_td3_workspace_bytes(const le_td3_cfg* cfg_host0, int n_lanes, int n_env) {
    if (!cfg_host0 || n_lanes < 1) { le_set_error("le_td3_workspace_bytes: bad arguments"); return LE_EINVAL; }
    LanePlan pl;
    int rc = check_lanes(&cfg_host0->base, cfg_host0, n_lanes, "le_td3_workspace_bytes", &pl);
    if (rc == LE_OK) rc = plan_lanes(&cfg_host0->base, cfg_host0, n_lanes, n_env, &pl);
    return rc == LE_OK ? td3_workspace_bytes(pl) : rc;
}

int le_td3_run(const le_td3_cfg* cfg_dev, int n_cfg, const le_td3_cfg* cfg_host0, const float* env_theta_dev, int n_env,
               const int32_t* env_index_dev, const uint32_t* keys_dev, const float* actor_init_dev, const float* critic1_init_dev,
               const float* critic2_init_dev, int n_init, float* actor_final_dev, int n_lanes, le_lane_out* out_dev, double* rewards_dev,
               int32_t* lengths_dev, double* test_rewards_dev, void* workspace_dev, int64_t workspace_bytes, const le_trace* trace_host,
               int trace_lane, void* stream) {
    const bool any_init = actor_init_dev || critic1_init_dev || critic2_init_dev;
    const bool all_init = actor_init_dev && critic1_init_dev && critic2_init_dev;
    if (!cfg_dev || !cfg_host0 || !keys_dev || !out_dev || !rewards_dev || !lengths_dev || !test_rewards_dev || !workspace_dev || n_lanes < 1 ||
        (n_cfg != 1 && n_cfg != n_lanes) || any_init != all_init || (all_init && n_init != 1 && n_init != n_lanes)) {
        le_set_error("le_td3_run: bad arguments (n_cfg and n_init must be 1 or n_lanes; all three init arrays or none; no NULL outputs)");
        return LE_EINVAL;
    }
    const le_lane_cfg* c = &cfg_host0->base;
    LanePlan pl;
    int rc = check_lanes(c, cfg_host0, n_lanes, "le_td3_run", &pl);
    if (rc != LE_OK) return rc;
    if (c->env_kind == LE_ENV_SE && (!env_theta_dev || n_env < 1)) { le_set_error("le_td3_run: env_theta is required for SE lanes"); return LE_EINVAL; }
    rc = plan_lanes(c, cfg_host0, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    // resident lanes: as many slots as the workspace holds, up to the occupancy-bound grid
    const int64_t fit = workspace_bytes > pl.off_slots ? (workspace_bytes - pl.off_slots) / pl.slot_bytes : 0;
    if (fit < 1) {
        le_set_error("le_td3_run: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes, (long long)(pl.off_slots + pl.slot_bytes));
        return LE_EINVAL;
    }
    if (fit < pl.tp.grid) pl.tp.grid = (int)fit;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace_dev;
    RunParams P;
    rc = start_lanes(pl, c, env_theta_dev, n_env, env_index_dev, keys_dev, n_lanes, out_dev, rewards_dev, lengths_dev, test_rewards_dev, ws,
                     trace_host, trace_lane, st, &P);
    if (rc != LE_OK) return rc;
    cudaError_t le = td3_launch(cfg_dev, n_cfg, cfg_host0, P, (float*)(ws + pl.off_slots), pl.tp, actor_init_dev, critic1_init_dev,
                                critic2_init_dev, all_init && n_init == n_lanes && n_lanes > 1, actor_final_dev, st);
    if (le != cudaSuccess) { le_set_error("td3 launch failed: %s", cudaGetErrorString(le)); return LE_ECUDA; }
    return LE_OK;
}

int le_td3_run_host(const le_td3_cfg* cfg, const float* env_theta, int n_env, const int32_t* env_index, const uint32_t* keys,
                    const float* actor_init, const float* critic1_init, const float* critic2_init, int n_init, float* actor_final,
                    int n_lanes, le_lane_out* out, double* rewards, int32_t* lengths, double* test_rewards, const le_trace* trace_host,
                    int trace_lane, int device) {
    if (!cfg || !keys || !actor_init || !critic1_init || !critic2_init || !out || !rewards || !lengths || !test_rewards || n_lanes < 1 ||
        (n_init != 1 && n_init != n_lanes)) {
        le_set_error("le_td3_run_host: bad arguments");
        return LE_EINVAL;
    }
    const le_lane_cfg* c = &cfg->base;
    LanePlan pl;
    int rc = check_lanes(c, cfg, n_lanes, "le_td3_run_host", &pl);
    if (rc != LE_OK) return rc;
    if (c->env_kind == LE_ENV_SE && (!env_theta || n_env < 1)) { le_set_error("le_td3_run_host: env_theta is required for SE lanes"); return LE_EINVAL; }
    LE_CUDA_CHECK(cudaSetDevice(device));
    rc = plan_lanes(c, cfg, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    const int64_t ws_bytes = td3_workspace_bytes(pl);
    if (ws_bytes < 0) return (int)ws_bytes;
    HostCall hc;
    const LaneSegs s = add_lane_segs(hc, cfg, sizeof(le_td3_cfg), c, env_theta, n_env, env_index, keys, n_lanes, out, rewards, lengths,
                                     test_rewards, trace_host);
    const size_t i_a = hc.add(actor_init, nullptr, sizeof(float) * (size_t)pl.tp.p_actor * n_init);
    const size_t i_c1 = hc.add(critic1_init, nullptr, sizeof(float) * (size_t)pl.tp.p_critic * n_init);
    const size_t i_c2 = hc.add(critic2_init, nullptr, sizeof(float) * (size_t)pl.tp.p_critic * n_init);
    const size_t i_af = hc.add(nullptr, actor_final, actor_final ? sizeof(float) * (size_t)pl.tp.p_actor * n_lanes : 0);
    const size_t off_ws = hc.reserve((size_t)ws_bytes);
    le_trace tr;
    rc = stage_lane_segs(hc, s, &tr);
    if (rc != LE_OK) return rc;
    rc = le_td3_run((const le_td3_cfg*)hc.dp(s.cfg), 1, cfg, (const float*)hc.dp(s.th), n_env, (const int32_t*)hc.dp(s.ei),
                    (const uint32_t*)hc.dp(s.key), (const float*)hc.dp(i_a), (const float*)hc.dp(i_c1), (const float*)hc.dp(i_c2), n_init,
                    (float*)hc.dp(i_af), n_lanes, (le_lane_out*)hc.dp(s.out), (double*)hc.dp(s.rw), (int32_t*)hc.dp(s.ln), (double*)hc.dp(s.tr),
                    hc.arena + off_ws, ws_bytes, tr.cap ? &tr : nullptr, trace_lane, hc.st);
    return hc.stage_out(rc, "le_td3_run_host");   // ~HostCall frees the arena and destroys the stream
}

// ---- NES ----------------------------------------------------------------------------------------------
int le_nes_perturb(const float* theta_dev, int P, int pop, int member_offset, int n_members, uint32_t seed, uint32_t generation,
                   float noise_std, float* out_dev, void* stream) {
    if (!theta_dev || !out_dev || P < 1 || n_members < 1 || member_offset < 0 || member_offset + n_members > pop) {
        le_set_error("le_nes_perturb: bad arguments");
        return LE_EINVAL;
    }
    const int64_t work = (int64_t)((P + 3) / 4) * n_members;
    const int grid = (int)((work + 127) / 128 < 148 * 16 ? (work + 127) / 128 : 148 * 16);
    nes_perturb_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(theta_dev, P, member_offset, n_members, seed, generation, noise_std, out_dev);
    LE_CUDA_CHECK(cudaGetLastError());
    return LE_OK;
}

int le_nes_noise(int P, int member_offset, int n_members, uint32_t seed, uint32_t generation, float noise_std, float* eps_dev,
                 void* stream) {
    if (!eps_dev || P < 1 || n_members < 1 || member_offset < 0) { le_set_error("le_nes_noise: bad arguments"); return LE_EINVAL; }
    const int64_t work = (int64_t)((P + 3) / 4) * n_members;
    const int grid = (int)((work + 127) / 128 < 148 * 16 ? (work + 127) / 128 : 148 * 16);
    nes_noise_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(P, member_offset, n_members, seed, generation, noise_std, eps_dev);
    LE_CUDA_CHECK(cudaGetLastError());
    return LE_OK;
}

int le_nes_update(float* theta_dev, int P, int pop, uint32_t seed, uint32_t generation, float noise_std, double weight_decay,
                  const float* coef_dev, const float* sign_dev, void* stream) {
    if (!theta_dev || !coef_dev || !sign_dev || P < 1 || pop < 1) { le_set_error("le_nes_update: bad arguments"); return LE_EINVAL; }
    const int nblk = (P + 3) / 4;
    nes_update_kernel<true><<<(nblk + kNesPT - 1) / kNesPT, kNesPT * kNesMG, 0, (cudaStream_t)stream>>>(
        theta_dev, P, 0, pop, seed, generation, noise_std, (float)(1.0 - weight_decay), coef_dev, sign_dev);
    LE_CUDA_CHECK(cudaGetLastError());
    return LE_OK;
}

int le_nes_partial_update(float* delta_dev, int P, int member_lo, int member_hi, uint32_t seed, uint32_t generation, float noise_std,
                          const float* coef_dev, const float* sign_dev, void* stream) {
    if (!delta_dev || !coef_dev || !sign_dev || P < 1 || member_lo < 0 || member_hi < member_lo) { le_set_error("le_nes_partial_update: bad arguments"); return LE_EINVAL; }
    const int nblk = (P + 3) / 4;
    nes_update_kernel<false><<<(nblk + kNesPT - 1) / kNesPT, kNesPT * kNesMG, 0, (cudaStream_t)stream>>>(
        delta_dev, P, member_lo, member_hi, seed, generation, noise_std, 1.f, coef_dev, sign_dev);
    LE_CUDA_CHECK(cudaGetLastError());
    return LE_OK;
}

}  // extern "C"
