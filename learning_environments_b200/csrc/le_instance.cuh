// le_instance.cuh — launchers for one compiled (SD, AD, U, ACT) register Q-net kernel set: the warp, multi-warp and
// cluster lane kernels and the Q-net unit operators.  The instantiations live in le_inst_*.cu (one translation unit per
// environment shape x activation so they compile in parallel); le_api.cu looks up the kernel set of a lane with
// le_find_instance().  The environment kernels (packing, SE / RN unit operators) depend on the shape only and are compiled
// once, in le_api.cu.
#pragma once
#include "le_inner_loop.cuh"

namespace le {

struct InstanceOps {
    int sd, ad, units, act;  // act: QACT_TANH / QACT_LEAKY
    int inner_warps;         // warps (= lane slots) per CTA of the fused kernel
    int mw_warps;            // warps per lane of the multi-warp (one lane per CTA) kernel; 0 if its shared memory does not fit
    int64_t mw_smem_bytes;   // its shared memory without the staged env pack (P.mw_pack_f4 * 16 bytes are added at launch)
    int64_t mwc_smem_bytes;  // cluster lanes (one lane per cluster of two CTAs): shared memory per CTA, 0 if not compiled for this kernel set
    cudaError_t (*launch_inner_mwc)(const RunParams& P, int n_slots, cudaStream_t st);
    cudaError_t (*launch_inner_mw)(const RunParams& P, int grid, cudaStream_t st);
    // fused persistent kernel
    int (*inner_max_ctas_per_sm)();
    cudaError_t (*launch_inner)(const RunParams& P, int grid, cudaStream_t st);
    // unit operators
    cudaError_t (*launch_qnet_forward)(const float* q_theta, int q_stride, int H, float slope, const float* state, float* q_out,
                                       int32_t* argmax, int n, cudaStream_t st);
    cudaError_t (*launch_td_update)(const le_lane_cfg* cfg_dev, float* th, float* thT, float* m, float* v, int32_t* t, int q_stride,
                                    const float* rows, int B, float* loss, int n, cudaStream_t st);
};

const InstanceOps* le_find_instance(int sd, int ad, int units_needed, int act);
void le_register_instance(const InstanceOps* ops);

// ------------------------------------------------------------------------------------------------------
// Q-net unit kernels (one warp per row / lane), sharing the device code of the fused kernel

template <int SD, int AD, int U, int ACT>
__global__ void qnet_forward_kernel(const float* __restrict__ q_theta, int q_stride, int H, float slope,
                                    const float* __restrict__ state, float* __restrict__ q_out, int32_t* __restrict__ argmax, int n) {
    using Core = LaneCore<SD, AD, U, ACT>;
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    // row-owner cores keep their weights in shared-memory records (4 warps per block, launch_qnet_forward)
    __shared__ float wrec[4][Core::kRow ? Core::ROW_WREC_F : 1];
    Core core;
    core.bind(wrec[(threadIdx.x >> 5) & 3], lane);
    core.load_net(q_theta + (int64_t)row * q_stride, H, lane, 0);
    core.publish_weights(nullptr, lane);
    float s[SD], q[AD];
#pragma unroll
    for (int i = 0; i < SD; ++i) s[i] = state[(int64_t)row * SD + i];
    core.q_forward_row(s, slope, q);
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < AD; ++a) q_out[(int64_t)row * AD + a] = q[a];
        argmax[row] = Core::argmax_first(q);
    }
}

// DDQN.learn on explicit minibatches: rows in the public packed order [s a s' r d] (2*SD+3 floats)
template <int SD, int AD, int U, int ACT>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
td_update_kernel(const le_lane_cfg* __restrict__ cfg_dev, float* th, float* thT, float* m, float* v, int32_t* tcount, int q_stride,
                 const float* __restrict__ rows, int B, float* __restrict__ loss_out, int n) {
    using Core = LaneCore<SD, AD, U, ACT>;
    using RL = RowLayout<SD>;
    using SL = StageLayout<SD>;
    using SW = SmemWarp<SD, AD, U>;
    extern __shared__ __align__(16) float smem_dyn[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int id = blockIdx.x * kWarpsPerCta + warp;
    if (id >= n) return;
    float* smem = smem_dyn + warp * SW::FLOATS;
    float* mv = smem + SW::OFF_MV;
    const le_lane_cfg c = *cfg_dev;
    const int H = c.q_hidden;
    Core core;
    core.bind(smem + SW::OFF_RED, lane);
    const int64_t o = (int64_t)id * q_stride;
    core.load_net(th + o, H, lane, 0);
    core.load_net(thT + o, H, lane, 1);
    Core::init_row_region(smem + SW::OFF_RED, lane);
    core.publish_weights(smem + SW::OFF_RED, lane);
    Core::load_moments(mv, m + o, v + o, H, lane);
    LearnScalars ls;
    fill_learn_scalars(ls, c);
    ls.batch = B;
    ls.norm = (float)(2.0 / (double)B);
    const int t0 = tcount[id];
    ls.b1pow = pow(c.beta1, (double)t0);
    ls.b2pow = pow(c.beta2, (double)t0);
    core.zero_grads();
    float loss_part = 0.f;
    constexpr int ROWP = 2 * SD + 3;
    const float* my_rows = rows + (int64_t)id * B * ROWP;
    for (int sc = 0; sc * SL::ROWS < B; ++sc) {
        const int nrows = min(SL::ROWS, B - sc * SL::ROWS);
        const int nfill = (nrows + Core::R - 1) / Core::R * Core::R;
        for (int rr = lane; rr < nfill; rr += 32) {
            const float* src = my_rows + (int64_t)(sc * SL::ROWS + rr) * ROWP;
            float rowv[RL::ROWF];
#pragma unroll
            for (int i = 0; i < RL::ROWF; ++i) rowv[i] = 0.f;
            if (rr < nrows) {
#pragma unroll
                for (int i = 0; i < SD; ++i) { rowv[RL::OFF_S + i] = src[i]; rowv[RL::OFF_S2 + i] = src[SD + 1 + i]; }
                rowv[RL::OFF_A] = __int_as_float((int)src[SD]); rowv[RL::OFF_R] = src[2 * SD + 1]; rowv[RL::OFF_D] = src[2 * SD + 2];
            }
            stage_row<SD>(smem + rr * SL::STAGE_F, rowv);
        }
        __syncwarp();
        loss_part += core.td_rows(smem, smem + SW::OFF_RED, nrows, ls, lane);
        __syncwarp();
    }
    const float loss = warp_allreduce_sum(loss_part) / (float)B;
    core.adam_polyak(ls, mv, lane);
    core.store_net(th + o, H, lane, 0);
    core.store_net(thT + o, H, lane, 1);
    __syncwarp();
    Core::store_moments(mv, m + o, v + o, H, lane);
    if (lane == 0) { loss_out[id] = loss; tcount[id] = t0 + 1; }
}

// ------------------------------------------------------------------------------------------------------
template <int SD, int AD, int U, int ACT>
struct InstanceImpl {
    static constexpr size_t kSmemBytes = (size_t)kWarpsPerCta * SmemWarp<SD, AD, U>::FLOATS * sizeof(float);          // unit kernels
    static constexpr int kInnerWarps = inner_warps<U>();
    static constexpr size_t kInnerSmemBytes = (size_t)kInnerWarps * SmemWarp<SD, AD, U>::FLOATS * sizeof(float);      // fused kernel
    static_assert(kInnerSmemBytes <= 227 * 1024, "per-CTA shared memory of the fused kernel exceeds 227 KB");
    static int inner_max_ctas_per_sm() {
        int nb = 0;
        cudaFuncSetAttribute(inner_loop_kernel<SD, AD, U, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInnerSmemBytes);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, inner_loop_kernel<SD, AD, U, ACT>, kInnerWarps * 32, kInnerSmemBytes);
        return nb;
    }
    static cudaError_t launch_inner(const RunParams& P, int grid, cudaStream_t st) {
        cudaError_t e = cudaFuncSetAttribute(inner_loop_kernel<SD, AD, U, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInnerSmemBytes);
        if (e != cudaSuccess) return e;
        inner_loop_kernel<SD, AD, U, ACT><<<grid, kInnerWarps * 32, kInnerSmemBytes, st>>>(P);
        return cudaGetLastError();
    }
    using MwLane = FusedLane<SD, AD, U, ACT, mw_warps<U>()>;
    static constexpr size_t kMwSmemBytes = (size_t)MwLane::MW_CTA_F * sizeof(float);
    static constexpr bool kMwOk = kMwSmemBytes <= 227 * 1024;
    static cudaError_t launch_inner_mw(const RunParams& P, int grid, cudaStream_t st) {
        if constexpr (kMwOk) {
            const size_t smem = kMwSmemBytes + (size_t)P.mw_pack_f4 * 16;
            cudaError_t e = cudaFuncSetAttribute(inner_loop_mw_kernel<SD, AD, U, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            inner_loop_mw_kernel<SD, AD, U, ACT><<<grid, mw_warps<U>() * 32, smem, st>>>(P);
            return cudaGetLastError();
        } else return cudaErrorInvalidConfiguration;
    }
    using MwcLane = FusedLane<SD, AD, U, ACT, kMwcWarps, 2>;
    static constexpr size_t kMwcSmemBytes = (size_t)MwcLane::MW_CTA_F * sizeof(float);
    static constexpr bool kMwcOk = U <= 4 && kMwcSmemBytes <= 200 * 1024;
    static cudaError_t launch_inner_mwc(const RunParams& P, int n_slots, cudaStream_t st) {
        if constexpr (kMwcOk) {
            const size_t smem = kMwcSmemBytes + (size_t)P.mw_pack_f4 * 16;
            cudaError_t e = cudaFuncSetAttribute(inner_loop_mwc_kernel<SD, AD, U, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(2 * n_slots); cfg.blockDim = dim3(kMwcWarps * 32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            return cudaLaunchKernelEx(&cfg, inner_loop_mwc_kernel<SD, AD, U, ACT>, P);
        } else return cudaErrorInvalidConfiguration;
    }
    static cudaError_t launch_qnet_forward(const float* q_theta, int q_stride, int H, float slope, const float* state, float* q_out,
                                           int32_t* argmax, int n, cudaStream_t st) {
        const int grid = (n + 3) / 4;
        qnet_forward_kernel<SD, AD, U, ACT><<<grid, 128, 0, st>>>(q_theta, q_stride, H, slope, state, q_out, argmax, n);
        return cudaGetLastError();
    }
    static cudaError_t launch_td_update(const le_lane_cfg* cfg_dev, float* th, float* thT, float* m, float* v, int32_t* t, int q_stride,
                                        const float* rows, int B, float* loss, int n, cudaStream_t st) {
        const int grid = (n + kWarpsPerCta - 1) / kWarpsPerCta;
        cudaError_t e = cudaFuncSetAttribute(td_update_kernel<SD, AD, U, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
        if (e != cudaSuccess) return e;
        td_update_kernel<SD, AD, U, ACT><<<grid, kWarpsPerCta * 32, kSmemBytes, st>>>(cfg_dev, th, thT, m, v, t, q_stride, rows, B, loss, n);
        return cudaGetLastError();
    }
    static const InstanceOps* ops() {
        static const InstanceOps o = {SD, AD, U, ACT, kInnerWarps, kMwOk ? mw_warps<U>() : 0, (int64_t)kMwSmemBytes, kMwcOk ? (int64_t)kMwcSmemBytes : 0, launch_inner_mwc, launch_inner_mw, inner_max_ctas_per_sm, launch_inner,
                                      launch_qnet_forward, launch_td_update};
        return &o;
    }
};

}  // namespace le
