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

struct Plan {
    bool general;
    GeneralPlan gp;
    const InstanceOps* ops;
    int grid, slots, ring_cap;
    bool mw;   // multi-warp lanes: one lane per CTA
    bool mwc;  // cluster lanes: one lane per cluster of two CTAs (two SMs)
    int64_t ring_stride_f, pack_stride_f, pack_bytes, rings_bytes, total_bytes, off_rings, off_counter;
};

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

// parameters of one SE / RN env network (envs/virtual_env.py, envs/reward_env.py); 0 for the real envs
static int env_param_count(const le_lane_cfg* c) {
    const int H = c->env_hidden;
    if (c->env_kind == LE_ENV_SE) return 3 * H * (c->sd + c->ad + 1) + H * (c->sd + 2) + c->sd + 2;
    if (c->env_kind == LE_ENV_RN) return H * (c->sd + 2) + 1;
    return 0;
}

// n_env SE / RN parameter vectors -> the packed layout the lane kernels read (stride_f floats per env); real envs: nothing
static cudaError_t pack_env(const InstanceOps* ops, const le_lane_cfg* c, const float* theta, int n_env, float* pack, int64_t stride_f,
                            cudaStream_t st) {
    if (c->env_kind == LE_ENV_SE) {
        float slopes[3];
        for (int i = 0; i < 3; ++i) slopes[i] = act_slope(c->env_act, c->env_slope[i]);
        return ops->launch_pack_se(theta, env_param_count(c), n_env, c->env_hidden, slopes, pack, stride_f, st);
    }
    if (c->env_kind == LE_ENV_RN)
        return ops->launch_pack_rn(theta, env_param_count(c), n_env, c->env_hidden, act_slope(c->env_act, c->env_slope[0]), pack, stride_f, st);
    return cudaSuccess;
}

static int make_plan(const le_lane_cfg* c, int n_lanes, int n_env, Plan* pl) {
    { const int rc0 = check_env_cfg(c); if (rc0 != LE_OK) return rc0; }
    if (c->batch_size < 1 || c->rb_size < 1 || c->train_episodes < 0 || c->test_episodes < 1 || c->max_steps < 1 || n_lanes < 1) {
        le_set_error("bad lane configuration (batch_size=%d rb_size=%d train_episodes=%d test_episodes=%d max_steps=%d n_lanes=%d)",
                     c->batch_size, c->rb_size, c->train_episodes, c->test_episodes, c->max_steps, n_lanes);
        return LE_EINVAL;
    }
    pl->general = !is_register_resident(c);
    pl->mw = false;
    pl->mwc = false;
    if (c->q_layers > 3) { le_set_error("Q-network hidden_layer=%d: the compiled kernel set covers up to 3 hidden layers", c->q_layers); return LE_EUNSUPPORTED; }
    // the env-packing / unit kernels of any kernel set with the right (sd, ad) serve the general path too
    const InstanceOps* ops = pl->general ? le_find_instance(c->sd, c->ad, 1, QACT_TANH) : instance_for(c, c->q_hidden);
    if (!ops) { if (pl->general) le_set_error("no compiled kernel set for state_dim=%d action_dim=%d", c->sd, c->ad); return LE_EUNSUPPORTED; }
    if (pl->general && qact_of(c) < 0) { le_set_error("Q-net activation id %d is outside the compiled kernel set", c->q_act); return LE_EUNSUPPORTED; }
    int dev = 0, sms = 0;
    LE_CUDA_CHECK(cudaGetDevice(&dev));
    LE_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    pl->ring_cap = ring_capacity(c);
    pl->ops = ops;
    if (pl->general) {
        const int rc = general_plan(c, n_lanes, pl->ring_cap, sms, &pl->gp);
        if (rc != LE_OK) return rc;
        pl->grid = pl->gp.grid;
        pl->slots = pl->grid;
        pl->ring_stride_f = pl->gp.slot_floats;   // one slot = ring + parameters + activations
    } else if (use_mwc_lanes(ops, n_lanes, sms)) {
        pl->mw = true; pl->mwc = true;
        pl->grid = 2 * n_lanes;      // one cluster of two CTAs per lane
        pl->slots = n_lanes;
        pl->ring_stride_f = (int64_t)pl->ring_cap * ops->ring_row_floats();
    } else if (use_mw_lanes(ops, n_lanes, sms)) {
        pl->mw = true;
        pl->grid = n_lanes < sms ? n_lanes : sms;
        pl->slots = pl->grid;
        pl->ring_stride_f = (int64_t)pl->ring_cap * ops->ring_row_floats();
    } else {
        int per_sm = ops->inner_max_ctas_per_sm();
        if (per_sm < 1) per_sm = 1;
        const int want = (n_lanes + ops->inner_warps - 1) / ops->inner_warps;
        pl->grid = want < sms * per_sm ? want : sms * per_sm;
        pl->slots = pl->grid * ops->inner_warps;
        pl->ring_stride_f = (int64_t)pl->ring_cap * ops->ring_row_floats();
    }
    const int64_t pv4 = c->env_kind == LE_ENV_SE ? ops->se_pack_vec4(c->env_hidden) : (c->env_kind == LE_ENV_RN ? ops->rn_pack_vec4(c->env_hidden) : 1);
    pl->pack_stride_f = pv4 * 4;
    pl->pack_bytes = ((int64_t)(n_env > 0 ? n_env : 1) * pl->pack_stride_f * 4 + 255) / 256 * 256;
    pl->rings_bytes = ((int64_t)pl->slots * pl->ring_stride_f * 4 + 255) / 256 * 256;
    pl->off_rings = pl->pack_bytes;
    pl->off_counter = pl->off_rings + pl->rings_bytes;
    pl->total_bytes = pl->off_counter + 256;
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
    const InstanceOps* ops = le_find_instance(cfg->sd, cfg->ad, 1, QACT_TANH);
    if (!ops) { le_set_error("no compiled kernel set for state_dim=%d action_dim=%d", cfg->sd, cfg->ad); return LE_EUNSUPPORTED; }
    cudaStream_t st = (cudaStream_t)stream;
    le_lane_cfg c = *cfg;
    c.env_kind = LE_ENV_SE;
    const int H = c.env_hidden;
    const int64_t stride_f = ops->se_pack_vec4(H) * 4;
    float* pack = nullptr;
    LE_CUDA_CHECK(cudaMallocAsync((void**)&pack, (size_t)pop * stride_f * 4, st));
    LE_CUDA_CHECK(pack_env(ops, &c, theta_dev, pop, pack, stride_f, st));
    LE_CUDA_CHECK(ops->launch_se_forward((const float4*)pack, stride_f / 4, H, cfg->env_act == LE_ACT_TANH, lanes_per_member, state_dev,
                                         action_dev, next_state_dev, reward_dev, done_dev, pop * lanes_per_member, st));
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
    const InstanceOps* ops = le_find_instance(c.sd, c.ad, 1, QACT_TANH);
    if (!ops) { le_set_error("no compiled kernel set for state_dim=%d action_dim=%d", c.sd, c.ad); return LE_EUNSUPPORTED; }
    cudaStream_t st = (cudaStream_t)stream;
    const int H = c.env_hidden;
    const int64_t stride_f = ops->rn_pack_vec4(H) * 4;
    float* pack = nullptr;
    LE_CUDA_CHECK(cudaMallocAsync((void**)&pack, (size_t)pop * stride_f * 4, st));
    LE_CUDA_CHECK(pack_env(ops, &c, theta_dev, pop, pack, stride_f, st));
    LE_CUDA_CHECK(ops->launch_rn_reward((const float4*)pack, stride_f / 4, H, c.env_act == LE_ACT_TANH, c.rn_type, (float)c.gamma,
                                        lanes_per_member, state_dev, next_state_dev, real_reward_dev, reward_dev, pop * lanes_per_member, st));
    LE_CUDA_CHECK(cudaFreeAsync(pack, st));
    return LE_OK;
}

int le_qnet_forward(const le_lane_cfg* cfg, const float* q_theta_dev, int n, const float* state_dev, float* q_out_dev,
                    int32_t* argmax_dev, void* stream) {
    if (!cfg || n < 1) { le_set_error("le_qnet_forward: bad arguments"); return LE_EINVAL; }
    if (cfg->q_layers > 3) { le_set_error("le_qnet_forward: hidden_layer > 3"); return LE_EUNSUPPORTED; }
    if (!is_register_resident(cfg)) {
        if (qact_of(cfg) < 0 || !le_find_instance(cfg->sd, cfg->ad, 1, QACT_TANH)) { le_set_error("le_qnet_forward: unsupported Q-network"); return LE_EUNSUPPORTED; }
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
    const InstanceOps* ops = general ? le_find_instance(cfg->sd, cfg->ad, 1, QACT_TANH) : instance_for(cfg, cfg->q_hidden);
    if (!ops || qact_of(cfg) < 0) { if (general) le_set_error("le_td_update: unsupported Q-network"); return LE_EUNSUPPORTED; }
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
    Plan pl;
    if (!cfg) { le_set_error("le_inner_loop_workspace_bytes: cfg is NULL"); return LE_EINVAL; }
    int rc = make_plan(cfg, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    return pl.total_bytes;
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
    Plan pl;
    int rc = make_plan(cfg_host0, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    if (cfg_host0->env_kind != LE_ENV_REAL && (!env_theta_dev || n_env < 1)) { le_set_error("le_inner_loop_run: env_theta is required for SE/RN lanes"); return LE_EINVAL; }
    if (workspace_bytes < pl.total_bytes) {
        le_set_error("le_inner_loop_run: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes, (long long)pl.total_bytes);
        return LE_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace_dev;
    float* pack = (float*)ws;
    const le_lane_cfg* c = cfg_host0;
    LE_CUDA_CHECK(pack_env(pl.ops, c, env_theta_dev, n_env, pack, pl.pack_stride_f, st));
    int* counter = (int*)(ws + pl.off_counter);
    LE_CUDA_CHECK(cudaMemsetAsync(counter, 0, sizeof(int), st));
    RunParams P;
    memset(&P, 0, sizeof(P));
    P.cfg = cfg_dev; P.n_cfg = n_cfg;
    P.env_pack = (const float4*)pack; P.env_pack_stride = pl.pack_stride_f / 4;
    P.env_index = env_index_dev; P.keys = keys_dev;
    P.q_init = q_init_dev; P.q_final = q_final_dev;
    P.q_stride = q_params_of(c);
    P.n_lanes = n_lanes; P.out = out_dev; P.rewards = rewards_dev; P.lengths = lengths_dev; P.test_rewards = test_rewards_dev; P.test_lengths = test_lengths_dev;
    P.rew_stride = c->train_episodes > 0 ? c->train_episodes : 1;
    P.test_stride = c->test_episodes;
    P.rings = (float*)(ws + pl.off_rings); P.ring_stride = pl.ring_stride_f; P.ring_cap = pl.ring_cap;
    P.work_counter = counter;
    if (trace_host && trace_host->cap > 0) { P.trace = *trace_host; P.trace_lane = trace_lane; }
    if (pl.general) LE_CUDA_CHECK(general_launch(c, P, P.rings, pl.gp, st));
    else if (pl.mw) {
        // the member's SE / RN pack is staged in the CTA's shared memory by one TMA bulk copy per lane when it fits beside the lane state
        const int64_t pack_bytes = c->env_kind == LE_ENV_REAL ? 0 : pl.pack_stride_f * 4;
        const int64_t lane_smem = pl.mwc ? pl.ops->mwc_smem_bytes : pl.ops->mw_smem_bytes;
        if (pack_bytes > 0 && lane_smem + pack_bytes <= 227 * 1024) P.mw_pack_f4 = (int)(pack_bytes / 16);
        if (pl.mwc) LE_CUDA_CHECK(pl.ops->launch_inner_mwc(P, pl.slots, st));
        else LE_CUDA_CHECK(pl.ops->launch_inner_mw(P, pl.grid, st));
    }
    else LE_CUDA_CHECK(pl.ops->launch_inner(P, pl.grid, st));
    return LE_OK;
}

int le_inner_loop_plan(const le_lane_cfg* cfg, int n_lanes, int n_env, int* grid, int* slots, int* ring_cap, int* units,
                       int64_t* ring_offset_bytes) {
    Plan pl;
    int rc = make_plan(cfg, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    if (grid) *grid = pl.grid;
    if (slots) *slots = pl.slots;
    if (ring_cap) *ring_cap = pl.ring_cap;
    if (units) *units = pl.ops->units;
    if (ring_offset_bytes) *ring_offset_bytes = pl.off_rings;
    return LE_OK;
}

int le_inner_loop_run_host(const le_lane_cfg* cfgs, int n_cfg, const float* env_theta, int n_env, const int32_t* env_index,
                           const uint32_t* keys, const float* q_init, float* q_final, int n_lanes, le_lane_out* out, double* rewards,
                           int32_t* lengths, double* test_rewards, int device) {
    if (!cfgs || !keys || !out || !rewards || !lengths || !test_rewards || n_lanes < 1 || (n_cfg != 1 && n_cfg != n_lanes)) {
        le_set_error("le_inner_loop_run_host: bad arguments");
        return LE_EINVAL;
    }
    LE_CUDA_CHECK(cudaSetDevice(device));
    const le_lane_cfg* c = &cfgs[0];
    Plan pl;
    int rc = make_plan(c, n_lanes, n_env, &pl);
    if (rc != LE_OK) return rc;
    const int Pq = q_params_of(c);
    const int rs = c->train_episodes > 0 ? c->train_episodes : 1;
    HostCall hc;
    const size_t i_cfg = hc.add(cfgs, nullptr, sizeof(le_lane_cfg) * n_cfg);
    const size_t i_th = hc.add(env_theta, nullptr, env_theta ? sizeof(float) * (size_t)env_param_count(c) * n_env : 0);
    const size_t i_ei = hc.add(env_index, nullptr, env_index ? sizeof(int32_t) * n_lanes : 0);
    const size_t i_key = hc.add(keys, nullptr, sizeof(uint32_t) * 2 * n_lanes);
    const size_t i_qi = hc.add(q_init, nullptr, q_init ? sizeof(float) * (size_t)Pq * n_lanes : 0);
    const size_t i_qf = hc.add(nullptr, q_final, q_final ? sizeof(float) * (size_t)Pq * n_lanes : 0);
    const size_t i_out = hc.add(nullptr, out, sizeof(le_lane_out) * n_lanes);
    const size_t i_rw = hc.add(nullptr, rewards, sizeof(double) * (size_t)rs * n_lanes);
    const size_t i_ln = hc.add(nullptr, lengths, sizeof(int32_t) * (size_t)rs * n_lanes);
    const size_t i_tr = hc.add(nullptr, test_rewards, sizeof(double) * (size_t)c->test_episodes * n_lanes);
    const size_t off_ws = hc.reserve((size_t)pl.total_bytes);
    rc = hc.stage_in();
    if (rc != LE_OK) return rc;
    LE_CUDA_CHECK(cudaMemsetAsync(hc.arena + hc.segs[i_rw].off, 0, hc.segs[i_rw].bytes + hc.segs[i_ln].bytes, hc.st));
    rc = le_inner_loop_run((const le_lane_cfg*)hc.dp(i_cfg), n_cfg, c, (const float*)hc.dp(i_th), n_env, (const int32_t*)hc.dp(i_ei),
                           (const uint32_t*)hc.dp(i_key), (const float*)hc.dp(i_qi), (float*)hc.dp(i_qf), n_lanes, (le_lane_out*)hc.dp(i_out),
                           (double*)hc.dp(i_rw), (int32_t*)hc.dp(i_ln), (double*)hc.dp(i_tr), nullptr, hc.arena + off_ws, pl.total_bytes, nullptr, 0,
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

// the checks of the fields a learn() step reads (nets, minibatch, TD3 hyper-parameters); no CUDA call
static int td3_learn_check(const le_td3_cfg* cfg, const char* who) {
    const le_lane_cfg* c = &cfg->base;
    if (qact_of(c) < 0 || c->q_hidden < 1 || c->q_layers > 3 || cfg->policy_delay < 1 || !(cfg->gumbel_temp > 0.0) || c->ad > 4 ||
        c->batch_size < 1) {
        le_set_error("%s: configuration outside the compiled kernel set", who);
        return LE_EUNSUPPORTED;
    }
    if (!le_find_instance(c->sd, c->ad, 1, QACT_TANH)) { le_set_error("no compiled kernel set for state_dim=%d action_dim=%d", c->sd, c->ad); return LE_EUNSUPPORTED; }
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

// workspace layout of the TD3 entry points: [SE pack | lane queue counter | resident lane slots]
struct Td3Layout {
    Td3Plan tp;
    const InstanceOps* ops;
    int ring_cap;
    int64_t pack_stride_f, off_counter, off_slots, slot_bytes;
};

static int td3_layout(const le_td3_cfg* cfg, int n_lanes, int n_env, const char* who, Td3Layout* L) {
    const le_lane_cfg* c = &cfg->base;
    int rc = td3_check(cfg, who);
    if (rc != LE_OK) return rc;
    L->ops = le_find_instance(c->sd, c->ad, 1, QACT_TANH);
    int dev = 0, sms = 0;
    LE_CUDA_CHECK(cudaGetDevice(&dev));
    LE_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    L->ring_cap = ring_capacity(c);
    rc = td3_plan(cfg, n_lanes, L->ring_cap, sms, &L->tp);
    if (rc != LE_OK) return rc;
    L->pack_stride_f = (c->env_kind == LE_ENV_SE ? L->ops->se_pack_vec4(c->env_hidden) : 1) * 4;
    L->off_counter = ((int64_t)(n_env > 0 ? n_env : 1) * L->pack_stride_f * 4 + 255) / 256 * 256;
    L->off_slots = L->off_counter + 256;
    L->slot_bytes = L->tp.slot_floats * (int64_t)sizeof(float);
    return LE_OK;
}

int64_t le_td3_workspace_bytes(const le_td3_cfg* cfg_host0, int n_lanes, int n_env) {
    if (!cfg_host0 || n_lanes < 1) { le_set_error("le_td3_workspace_bytes: bad arguments"); return LE_EINVAL; }
    Td3Layout L;
    const int rc = td3_layout(cfg_host0, n_lanes, n_env, "le_td3_workspace_bytes", &L);
    if (rc != LE_OK) return rc;
    // a slot of the widest vary_hp shapes (hidden 1530 x 3 layers) is ~0.3 GB: when every resident lane's slot does not fit
    // 90 % of the free device memory, ask for fewer slots (the lane queue runs the rest on them)
    size_t free_b = 0, total_b = 0;
    LE_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const int64_t room = (int64_t)(0.9 * (double)free_b) - L.off_slots;
    int64_t slots = L.tp.grid;
    if (slots * L.slot_bytes > room) slots = room / L.slot_bytes > 1 ? room / L.slot_bytes : 1;
    return L.off_slots + slots * L.slot_bytes;
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
    Td3Layout L;
    int rc = td3_layout(cfg_host0, n_lanes, n_env, "le_td3_run", &L);
    if (rc != LE_OK) return rc;
    const le_lane_cfg* c = &cfg_host0->base;
    if (c->env_kind == LE_ENV_SE && (!env_theta_dev || n_env < 1)) { le_set_error("le_td3_run: env_theta is required for SE lanes"); return LE_EINVAL; }
    // resident lanes: as many slots as the workspace holds, up to the occupancy-bound grid
    const int64_t fit = workspace_bytes > L.off_slots ? (workspace_bytes - L.off_slots) / L.slot_bytes : 0;
    if (fit < 1) {
        le_set_error("le_td3_run: workspace too small (%lld < %lld bytes)", (long long)workspace_bytes, (long long)(L.off_slots + L.slot_bytes));
        return LE_EINVAL;
    }
    if (fit < L.tp.grid) L.tp.grid = (int)fit;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace_dev;
    LE_CUDA_CHECK(cudaMemsetAsync(ws + L.off_counter, 0, 256, st));
    LE_CUDA_CHECK(pack_env(L.ops, c, env_theta_dev, n_env, (float*)ws, L.pack_stride_f, st));
    RunParams P;
    memset(&P, 0, sizeof(P));
    P.env_pack = (const float4*)ws; P.env_pack_stride = L.pack_stride_f / 4;
    P.env_index = env_index_dev; P.keys = keys_dev;
    P.n_lanes = n_lanes; P.out = out_dev; P.rewards = rewards_dev; P.lengths = lengths_dev; P.test_rewards = test_rewards_dev;
    P.rew_stride = c->train_episodes > 0 ? c->train_episodes : 1; P.test_stride = c->test_episodes;
    P.ring_cap = L.ring_cap;
    P.work_counter = (int*)(ws + L.off_counter);
    if (trace_host && trace_host->cap > 0) { P.trace = *trace_host; P.trace_lane = trace_lane; }
    cudaError_t le = td3_launch(cfg_dev, n_cfg, cfg_host0, P, (float*)(ws + L.off_slots), L.tp, actor_init_dev, critic1_init_dev, critic2_init_dev,
                                all_init && n_init == n_lanes && n_lanes > 1, actor_final_dev, st);
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
    int rc = td3_check(cfg, "le_td3_run_host");
    if (rc != LE_OK) return rc;
    LE_CUDA_CHECK(cudaSetDevice(device));
    Td3Layout L;
    rc = td3_layout(cfg, n_lanes, n_env, "le_td3_run_host", &L);
    if (rc != LE_OK) return rc;
    if (c->env_kind == LE_ENV_SE && (!env_theta || n_env < 1)) { le_set_error("le_td3_run_host: env_theta is required for SE lanes"); return LE_EINVAL; }
    const int64_t ws_bytes = le_td3_workspace_bytes(cfg, n_lanes, n_env);
    if (ws_bytes < 0) return (int)ws_bytes;
    const int rs = c->train_episodes > 0 ? c->train_episodes : 1;
    const int tcap = trace_host ? trace_host->cap : 0;
    HostCall hc;
    const size_t i_cfg = hc.add(cfg, nullptr, sizeof(le_td3_cfg));
    const size_t i_th = hc.add(env_theta, nullptr, sizeof(float) * (size_t)env_param_count(c) * n_env);
    const size_t i_ei = hc.add(env_index, nullptr, env_index ? sizeof(int32_t) * n_lanes : 0);
    const size_t i_key = hc.add(keys, nullptr, sizeof(uint32_t) * 2 * n_lanes);
    const size_t i_a = hc.add(actor_init, nullptr, sizeof(float) * (size_t)L.tp.p_actor * n_init);
    const size_t i_c1 = hc.add(critic1_init, nullptr, sizeof(float) * (size_t)L.tp.p_critic * n_init);
    const size_t i_c2 = hc.add(critic2_init, nullptr, sizeof(float) * (size_t)L.tp.p_critic * n_init);
    const size_t i_af = hc.add(nullptr, actor_final, actor_final ? sizeof(float) * (size_t)L.tp.p_actor * n_lanes : 0);
    const size_t i_out = hc.add(nullptr, out, sizeof(le_lane_out) * n_lanes);
    const size_t i_rw = hc.add(nullptr, rewards, sizeof(double) * (size_t)rs * n_lanes);
    const size_t i_ln = hc.add(nullptr, lengths, sizeof(int32_t) * (size_t)rs * n_lanes);
    const size_t i_tr = hc.add(nullptr, test_rewards, sizeof(double) * (size_t)c->test_episodes * n_lanes);
    const size_t i_ta = hc.add(nullptr, tcap ? trace_host->action : nullptr, sizeof(int32_t) * (size_t)tcap);
    const size_t i_te = hc.add(nullptr, tcap ? trace_host->explore : nullptr, sizeof(int32_t) * (size_t)tcap);
    const size_t i_tn = hc.add(nullptr, tcap ? trace_host->next_state : nullptr, sizeof(float) * (size_t)tcap * c->sd);
    const size_t i_trw = hc.add(nullptr, tcap ? trace_host->reward : nullptr, sizeof(float) * (size_t)tcap);
    const size_t i_td = hc.add(nullptr, tcap ? trace_host->done : nullptr, sizeof(float) * (size_t)tcap);
    const size_t i_tl = hc.add(nullptr, tcap ? trace_host->loss : nullptr, sizeof(float) * (size_t)tcap);
    const size_t off_ws = hc.reserve((size_t)ws_bytes);
    rc = hc.stage_in();
    if (rc != LE_OK) return rc;
    char* arena = hc.arena;
    LE_CUDA_CHECK(cudaMemsetAsync(arena + hc.segs[i_rw].off, 0, hc.segs[i_rw].bytes + hc.segs[i_ln].bytes, hc.st));
    le_trace tr;
    memset(&tr, 0, sizeof(tr));
    if (tcap) {
        LE_CUDA_CHECK(cudaMemsetAsync(arena + hc.segs[i_ta].off, 0xff, off_ws - hc.segs[i_ta].off, hc.st));   /* untouched trace slots: -1 / NaN */
        tr.cap = tcap; tr.action = (int32_t*)hc.dp(i_ta); tr.explore = (int32_t*)hc.dp(i_te); tr.next_state = (float*)hc.dp(i_tn);
        tr.reward = (float*)hc.dp(i_trw); tr.done = (float*)hc.dp(i_td); tr.loss = (float*)hc.dp(i_tl);
    }
    rc = le_td3_run((const le_td3_cfg*)hc.dp(i_cfg), 1, cfg, (const float*)hc.dp(i_th), n_env, (const int32_t*)hc.dp(i_ei),
                    (const uint32_t*)hc.dp(i_key), (const float*)hc.dp(i_a), (const float*)hc.dp(i_c1), (const float*)hc.dp(i_c2), n_init,
                    (float*)hc.dp(i_af), n_lanes, (le_lane_out*)hc.dp(i_out), (double*)hc.dp(i_rw), (int32_t*)hc.dp(i_ln), (double*)hc.dp(i_tr),
                    arena + off_ws, ws_bytes, tcap ? &tr : nullptr, trace_lane, hc.st);
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
