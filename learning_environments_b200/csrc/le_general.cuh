// le_general.cuh — CTA-per-lane kernels for Q-networks that do not fit one warp's registers:
//   Critic_DuelingDQN (models/actor_critic.py:94-122, 11.5k .. 67k parameters), Critic_DQN with two hidden layers or
//   more than 128 hidden units (DDQN_vary tails, agents/DDQN_vary.py:26-59).
// One CTA (256 threads) owns one lane; parameters, Adam state, gradients and the minibatch activations live in the
// lane slot's HBM workspace (<= 2.5 MB per slot) and every dense layer with more than 16 rows is a 128x64x16
// shared-memory-tiled GEMM with an 8x4 register tile of packed fp32x2 accumulators per thread, operands streamed by cp.async
// (forward NT, input-gradient NN, weight-gradient TN through one strided routine; LE_TC=1: the tcgen05 routine of le_tc.cuh);
// <= 16 rows (acting, batched test rollouts) take a thin thread-per-column path.  The agent loop (episodes, env step, replay ring, tests, early-out) is
// cta_lane_loop of le_cta_lane.cuh, shared with the TD3 lanes; GeneralAgent supplies the DDQN pieces.
//
// Dueling coupling (models/actor_critic.py:121): q = V + (A - A.mean()) with the mean over the WHOLE batch tensor, so
// the forward needs a CTA-wide reduction before the TD error and the backward seeds dA = dq*[a=a_r] - sum(dq)/(B*AD).
#pragma once
#include <cstddef>
#include <type_traits>
#include "le_cta_lane.cuh"
#include "le_tc.cuh"

namespace le {

constexpr int kGTileM = 128, kGTileN = 64, kGChunk = 16, kGPad = 4;
constexpr int kGSmemFloats = 2 * kGChunk * (kGTileM + kGPad + kGTileN + kGPad);

struct GLayer { int in, out, act, w_off, b_off, y_off; };
struct GNet {
    int kind, nfeat, P, sum_out, sd, ad;
    float slope;
    GLayer feat[4], val[2], adv[2];
};

__host__ __device__ inline void gnet_add(GLayer* l, int in, int out, int act, int* p, int* y) {
    // activation columns of a layer start at a multiple of 4 floats: 16-byte aligned rows for the vector staging of the
    // tensor-core GEMM (the parameter offsets follow torch's state_dict order and stay unpadded)
    l->in = in; l->out = out; l->act = act; l->w_off = *p; *p += in * out; l->b_off = *p; *p += out; l->y_off = *y; *y += (out + 3) & ~3;
}
// same construction as oracle/le_oracle.c build_net (torch state_dict order)
__host__ __device__ inline void gnet_build(const le_lane_cfg* c, GNet* n) {
    int p = 0, y = 0;
    const int L = c->q_layers > 1 ? c->q_layers : 1, H = c->q_hidden;
    const int act = c->q_act == LE_ACT_TANH ? 1 : 2;
    n->kind = c->q_kind; n->sd = c->sd; n->ad = c->ad; n->nfeat = 0;
    n->slope = c->q_act == LE_ACT_LEAKYRELU ? 0.01f : 0.f;
    gnet_add(&n->feat[n->nfeat++], c->sd, H, act, &p, &y);
    for (int i = 1; i < L; ++i) gnet_add(&n->feat[n->nfeat++], H, H, act, &p, &y);
    if (c->q_kind == LE_Q_DQN) {
        gnet_add(&n->feat[n->nfeat++], H, c->ad, 0, &p, &y);
    } else {
        const int fd = c->q_feature_dim;
        gnet_add(&n->feat[n->nfeat++], H, fd, 0, &p, &y);
        gnet_add(&n->val[0], fd, fd, act, &p, &y);
        gnet_add(&n->val[1], fd, 1, 0, &p, &y);
        gnet_add(&n->adv[0], fd, fd, act, &p, &y);
        gnet_add(&n->adv[1], fd, c->ad, 0, &p, &y);
    }
    n->P = p; n->sum_out = y;
}

// 4-byte asynchronous global -> shared copy; !valid copies nothing and writes zero (src-size 0)
__device__ __forceinline__ void cp_async4_zfill(uint32_t saddr, const void* gptr, bool valid) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(saddr), "l"(gptr), "r"(valid ? 4 : 0) : "memory");
}

__device__ __forceinline__ void cp_async4(uint32_t saddr, const void* gptr) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(gptr) : "memory");
}

__device__ __forceinline__ float g_act(int act, float slope, float z) {
    if (act == 1) return tanh_one(z);
    if (act == 2) return fmaxf(z, slope * z);
    return z;
}
__device__ __forceinline__ float g_act_grad(int act, float slope, float h) {
    if (act == 1) return fmaf(-h, h, 1.f);
    if (act == 2) return h > 0.f ? 1.f : slope;
    return 1.f;
}

struct GActFn {
    __device__ __forceinline__ float operator()(int act, float slope, float z) const { return g_act(act, slope, z); }
};
// Dense contractions (>= 64 rows, both other extents >= 32: the hidden x hidden layers of the dueling / two-hidden-layer
// nets with the minibatch as rows, and their input / weight gradients) go to the tcgen05 tensor cores (le_tc.cuh, 3xTF32,
// fp32 accumulate in TMEM); everything with a short side (first layers K = sd, heads N <= 4, row counts <= 16) stays on
// the FFMA paths below.  `tcx` is null in kernels that do not own a TMEM allocation (TD3 lanes, single-row forward).
// TCX is tc::Ctx* in the tensor-core instantiations of the lane kernels and std::nullptr_t everywhere else: kernels that do
// not own a TMEM allocation contain no tcgen05 code at all (a kernel that allocates TMEM is limited to ONE resident CTA per SM
// by the runtime, measured with tools/ubench/occ_tmem.cu, so the FFMA instantiations keep their two CTAs per SM).
template <typename TCX>
__device__ __forceinline__ bool g_use_tc(TCX tcx, int I, int J, int L) {
    if constexpr (std::is_same<TCX, tc::Ctx*>::value) return tcx != nullptr && I >= 64 && J >= 32 && L >= 32;
    else return false;
}
template <typename TCX, typename... Args>
__device__ __forceinline__ void g_tc_gemm(TCX tcx, Args... args) {
    if constexpr (std::is_same<TCX, tc::Ctx*>::value) tc::gemm_3xtf32(*tcx, args..., GActFn());
}

// C[i*c_si + j*c_sj] (+)= sum_l A[i*a_si + l*a_sl] * B[l*b_sl + j*b_sj]  (+ bias[j], activation)   — whole CTA.
// 128x64 output tiles, K chunks of 16, 8x4 accumulators per thread.  The (tile, chunk) sequence is flattened and
// software-pipelined over two shared-memory stages: the operands of chunk s+1 travel global -> shared with cp.async
// while the FFMAs of chunk s run (one wait + one __syncthreads per chunk; the L2 latency of the operand stream is
// covered by 512 FFMA per thread).  Per-thread element coordinates inside a tile-chunk are loop invariants (element q
// of a thread is its first element plus q constant steps), so a chunk costs one base address per operand.  Warps whose
// 16 rows lie outside I skip the arithmetic.  The k-summation order per output element is ascending for every shape.
static __device__ __noinline__ void g_gemm(const float* __restrict__ A, int a_si, int a_sl, const float* __restrict__ B, int b_sl, int b_sj,
                                    float* __restrict__ C, int c_si, int c_sj, int I, int J, int L, const float* __restrict__ bias,
                                    int act, float slope, bool accumulate, float* sm) {
    constexpr int TM = kGTileM, TN = kGTileN, TK = kGChunk, LDA = TM + kGPad, LDB = TN + kGPad;
    constexpr int NA = TM * TK / kGThreads, NB = TN * TK / kGThreads;   // 8 + 4 elements per thread per chunk
    float* As = sm;                       // [2][TK][LDA]
    float* Bs = sm + 2 * TK * LDA;        // [2][TK][LDB]
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, warp = tid >> 5;
    const int n_jt = (J + TN - 1) / TN, n_lc = (L + TK - 1) / TK;
    const int total = ((I + TM - 1) / TM) * n_jt * n_lc;
    const bool akm = a_sl == 1, bkm = b_sl == 1;   // operand stored k-major (k contiguous) or not
    // element q of this thread inside a tile-chunk: A (ia + q*dia, la + q*dla), B (lb + q*dlb, jb + q*djb)
    const int ia = akm ? (tid >> 4) : (tid & (TM - 1)), la = akm ? (tid & (TK - 1)) : (tid / TM);
    const int dia = akm ? kGThreads / TK : 0, dla = akm ? 0 : kGThreads / TM;
    const int jb = bkm ? (tid >> 4) : (tid & (TN - 1)), lb = bkm ? (tid & (TK - 1)) : (tid / TN);
    const int djb = bkm ? kGThreads / TK : 0, dlb = bkm ? 0 : kGThreads / TN;
    const int64_t gdA = (int64_t)dia * a_si + (int64_t)dla * a_sl, gdB = (int64_t)dlb * b_sl + (int64_t)djb * b_sj;
    const int sA0 = la * LDA + ia, sdA = dla * LDA + dia, sB0 = lb * LDB + jb, sdB = dlb * LDB + djb;
    // operand stream: 4-byte cp.async straight into the shared-memory stage (any stride, transposing on the fly,
    // out-of-range elements zero-filled through src-size 0) — no staging registers, nothing for the compiler to spill
    const uint32_t sm_u32 = (uint32_t)__cvta_generic_to_shared(sm);
    auto issue = [&](int buf, int i0, int j0, int l0) {
        const float* a = A + (int64_t)(i0 + ia) * a_si + (int64_t)(l0 + la) * a_sl;
        const float* b = B + (int64_t)(l0 + lb) * b_sl + (int64_t)(j0 + jb) * b_sj;
        const uint32_t sa = sm_u32 + 4u * (uint32_t)(buf * TK * LDA + sA0);
        const uint32_t sb = sm_u32 + 4u * (uint32_t)(2 * TK * LDA + buf * TK * LDB + sB0);
        if (i0 + TM <= I && j0 + TN <= J && l0 + TK <= L) {   // interior chunk: no bounds tests, pointer increments only
#pragma unroll
            for (int q = 0; q < NA; ++q) { cp_async4(sa + 4u * (uint32_t)(q * sdA), a); a += gdA; }
#pragma unroll
            for (int q = 0; q < NB; ++q) { cp_async4(sb + 4u * (uint32_t)(q * sdB), b); b += gdB; }
        } else {
#pragma unroll
            for (int q = 0; q < NA; ++q) {
                const bool ok = i0 + ia + q * dia < I && l0 + la + q * dla < L;
                cp_async4_zfill(sa + 4u * (uint32_t)(q * sdA), ok ? a + q * gdA : A, ok);
            }
#pragma unroll
            for (int q = 0; q < NB; ++q) {
                const bool ok = j0 + jb + q * djb < J && l0 + lb + q * dlb < L;
                cp_async4_zfill(sb + 4u * (uint32_t)(q * sdB), ok ? b + q * gdB : B, ok);
            }
        }
        cp_async_commit();
    };
    float2 acc[8][2];   // packed fp32x2 accumulators: (a, 2c) and (a, 2c+1) share one FFMA2
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int c = 0; c < 2; ++c) acc[a][c] = make_float2(0.f, 0.f);
    issue(0, 0, 0, 0);
    cp_async_wait<0>();
    __syncthreads();
    int it = 0, jt = 0, lc = 0;   // current (tile row, tile column, chunk)
    for (int s = 0; s < total; ++s) {
        const int buf = s & 1;
        const int i0 = it * TM, j0 = jt * TN;
        const bool tile_done = lc == n_lc - 1;
        int nit = it, njt = jt, nlc = lc + 1;
        if (tile_done) { nlc = 0; njt = jt + 1; if (njt == n_jt) { njt = 0; nit = it + 1; } }
        if (s + 1 < total) issue(buf ^ 1, nit * TM, njt * TN, nlc * TK);   // stage buf^1 was last read before the previous barrier
        if (i0 + 16 * warp < I) {
            const float* as = As + buf * TK * LDA + 8 * ty;
            const float* bs = Bs + buf * TK * LDB + 4 * tx;
            // fragments of step l+1 are loaded before the 32 FFMAs of step l (register double buffer)
            float4 a0 = *reinterpret_cast<const float4*>(as), a1 = *reinterpret_cast<const float4*>(as + 4);
            float4 b4 = *reinterpret_cast<const float4*>(bs);
#pragma unroll
            for (int l = 0; l < TK; ++l) {
                float4 na0 = a0, na1 = a1, nb4 = b4;
                if (l + 1 < TK) {
                    na0 = *reinterpret_cast<const float4*>(as + (l + 1) * LDA);
                    na1 = *reinterpret_cast<const float4*>(as + (l + 1) * LDA + 4);
                    nb4 = *reinterpret_cast<const float4*>(bs + (l + 1) * LDB);
                }
                const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                const float2 bv[2] = {make_float2(b4.x, b4.y), make_float2(b4.z, b4.w)};
#pragma unroll
                for (int a = 0; a < 8; ++a)
#pragma unroll
                    for (int c = 0; c < 2; ++c) acc[a][c] = __ffma2_rn(make_float2(av[a], av[a]), bv[c], acc[a][c]);
                a0 = na0; a1 = na1; b4 = nb4;
            }
        }
        if (tile_done) {   // epilogue of tile (it, jt)
            float bj[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) bj[b] = (bias && j0 + 4 * tx + b < J) ? __ldcg(bias + j0 + 4 * tx + b) : 0.f;
            if (i0 + 16 * warp < I) {
                float* row0 = C + (int64_t)(i0 + 8 * ty) * c_si + (int64_t)(j0 + 4 * tx) * c_sj;
                if (accumulate) {   // all loads first: between stores the compiler must assume aliasing and would serialise them
#pragma unroll
                    for (int a = 0; a < 8; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            if (i0 + 8 * ty + a < I && j0 + 4 * tx + b < J) {
                                const float old = __ldcg(row0 + (int64_t)a * c_si + b * c_sj);
                                if (b & 1) acc[a][b >> 1].y += old; else acc[a][b >> 1].x += old;
                            }
                }
#pragma unroll
                for (int a = 0; a < 8; ++a) {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        if (i0 + 8 * ty + a < I && j0 + 4 * tx + b < J) {
                            float v = (b & 1) ? acc[a][b >> 1].y : acc[a][b >> 1].x;
                            if (bias) v += bj[b];
                            __stcg(row0 + (int64_t)a * c_si + b * c_sj, g_act(act, slope, v));
                        }
                    }
                }
            }
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int c = 0; c < 2; ++c) acc[a][c] = make_float2(0.f, 0.f);
        }
        it = nit; jt = njt; lc = nlc;
        cp_async_wait<0>();
        __syncthreads();
    }
}

// Dense layer forward for M <= MT rows (greedy action M = 1, batched test rollouts M <= 16): thread j owns output
// column j and streams its weight row W[j][:] (16-byte loads when the rows are aligned); the input rows sit in shared
// memory as Xs[k][m] and are read as broadcasts.  Same ascending-k fmaf chain per output as g_gemm.
// RS = 2 (layers with at most kGThreads / 2 outputs, MT >= 8): the two halves of the CTA take the two halves of the ROWS of the
// same output column — every output keeps its ascending-k chain (bit-identical results), each thread does half the FMAs and
// half the shared-memory reads, and all 256 threads work instead of 128.  The per-episode test() rollouts on the real env
// (agents/base_agent.py:134-136: test_episodes greedy episodes after EVERY training episode) run through this path: it is
// ~70 % of the warp-state samples of the Acrobot DuelingDDQN workload (profiles/r02_general_ffma.txt).
template <int MT, int RS>
__device__ __noinline__ void g_thin_fwd_impl(const GLayer& l, const float* __restrict__ th, const float* __restrict__ X, int xs, int M,
                                             float* __restrict__ acts, int S, float slope, float* sm) {
    constexpr int KB = (kGSmemFloats / MT) / 4 * 4 > 512 ? 512 : (kGSmemFloats / MT) / 4 * 4;
    constexpr int MR = MT / RS;                 // rows per thread
    constexpr int COLS = kGThreads / RS;        // output columns per pass
    const int tid = threadIdx.x;
    const int half = tid / COLS, jt = tid % COLS, m0 = half * MR;
    for (int o0 = 0; o0 < l.out; o0 += COLS) {
        const int j = o0 + jt;
        float acc[MR];
#pragma unroll
        for (int m = 0; m < MR; ++m) acc[m] = 0.f;
        for (int k0 = 0; k0 < l.in; k0 += KB) {
            const int kn = min(KB, l.in - k0);
            __syncthreads();
            for (int e = tid; e < kn * MT; e += kGThreads) {
                const int k = e / MT, m = e % MT;
                sm[e] = m < M ? __ldcg(X + (int64_t)m * xs + k0 + k) : 0.f;
            }
            __syncthreads();
            if (j < l.out && m0 < M) {
                const float* wr = th + l.w_off + (int64_t)j * l.in + k0;
                const bool vec = ((l.in | kn) & 3) == 0 && (reinterpret_cast<uintptr_t>(wr) & 15) == 0;
                auto mac = [&](int k, float w) {
                    if constexpr (MR == 1) acc[0] = fmaf(sm[k * MT + m0], w, acc[0]);
                    else {
#pragma unroll
                        for (int m4 = 0; m4 < MR / 4; ++m4) {
                            const float4 x = *reinterpret_cast<const float4*>(sm + k * MT + m0 + 4 * m4);
                            acc[4 * m4] = fmaf(x.x, w, acc[4 * m4]); acc[4 * m4 + 1] = fmaf(x.y, w, acc[4 * m4 + 1]);
                            acc[4 * m4 + 2] = fmaf(x.z, w, acc[4 * m4 + 2]); acc[4 * m4 + 3] = fmaf(x.w, w, acc[4 * m4 + 3]);
                        }
                    }
                };
                if (vec) {
                    // 16 independent 16-byte weight loads in flight per thread: the stream is L2-latency bound
#pragma unroll 16
                    for (int k = 0; k < kn; k += 4) {
                        const float4 w4 = __ldcg(reinterpret_cast<const float4*>(wr + k));
                        mac(k, w4.x); mac(k + 1, w4.y); mac(k + 2, w4.z); mac(k + 3, w4.w);
                    }
                } else {
#pragma unroll 8
                    for (int k = 0; k < kn; ++k) mac(k, __ldcg(wr + k));
                }
            }
        }
        if (j < l.out) {
            const float bj = __ldcg(th + l.b_off + j);
#pragma unroll
            for (int m = 0; m < MR; ++m)
                if (m0 + m < M) __stcg(acts + (int64_t)(m0 + m) * S + l.y_off + j, g_act(l.act, slope, acc[m] + bj));
        }
    }
    __syncthreads();
}

template <int MT>
__device__ __forceinline__ void g_thin_fwd(const GLayer& l, const float* __restrict__ th, const float* __restrict__ X, int xs, int M,
                                           float* __restrict__ acts, int S, float slope, float* sm) {
    if constexpr (MT >= 8) {
        if (l.out <= kGThreads / 2) { g_thin_fwd_impl<MT, 2>(l, th, X, xs, M, acts, S, slope, sm); return; }
    }
    g_thin_fwd_impl<MT, 1>(l, th, X, xs, M, acts, S, slope, sm);
}

// Dense layer forward with at most 4 output columns and many rows (dueling heads fd -> 1 / fd -> ad): thread b owns
// batch row b and streams X[b][:] (16-byte loads when aligned); the weights sit in shared memory as Ws[k][4] and are
// read as broadcasts.  Same ascending-k fmaf chain per output as g_gemm.
static __device__ __noinline__ void g_thinj_fwd(const GLayer& l, const float* __restrict__ th, const float* __restrict__ X, int xs, int B,
                                         float* __restrict__ acts, int S, float slope, float* sm) {
    constexpr int KB = 1024;
    static_assert(KB * 4 <= kGSmemFloats, "weight stage must fit the GEMM buffer");
    const int tid = threadIdx.x;
    for (int b0 = 0; b0 < B; b0 += kGThreads) {
        const int b = b0 + tid;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int k0 = 0; k0 < l.in; k0 += KB) {
            const int kn = min(KB, l.in - k0);
            __syncthreads();
            for (int e = tid; e < kn * 4; e += kGThreads) {
                const int k = e >> 2, j = e & 3;
                sm[e] = j < l.out ? __ldcg(th + l.w_off + (int64_t)j * l.in + k0 + k) : 0.f;
            }
            __syncthreads();
            if (b < B) {
                const float* xr = X + (int64_t)b * xs + k0;
                const bool vec = ((xs | kn | k0) & 3) == 0 && (reinterpret_cast<uintptr_t>(xr) & 15) == 0;
                auto mac = [&](int k, float x) {
                    const float4 w = *reinterpret_cast<const float4*>(sm + 4 * k);
                    acc[0] = fmaf(x, w.x, acc[0]); acc[1] = fmaf(x, w.y, acc[1]);
                    acc[2] = fmaf(x, w.z, acc[2]); acc[3] = fmaf(x, w.w, acc[3]);
                };
                if (vec) {
#pragma unroll 8
                    for (int k = 0; k < kn; k += 4) {
                        const float4 x4 = __ldcg(reinterpret_cast<const float4*>(xr + k));
                        mac(k, x4.x); mac(k + 1, x4.y); mac(k + 2, x4.z); mac(k + 3, x4.w);
                    }
                } else {
#pragma unroll 4
                    for (int k = 0; k < kn; ++k) mac(k, __ldcg(xr + k));
                }
            }
        }
        if (b < B) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (j < l.out) __stcg(acts + (int64_t)b * S + l.y_off + j, g_act(l.act, slope, acc[j] + __ldcg(th + l.b_off + j)));
        }
    }
    __syncthreads();
}

template <typename TCX = std::nullptr_t>
__device__ __forceinline__ void g_layer_fwd(const GLayer& l, const float* th, const float* X, int xs, int B, float* acts, int S,
                                            float slope, float* sm, TCX tcx = nullptr) {
    if (B == 1) { g_thin_fwd<1>(l, th, X, xs, B, acts, S, slope, sm); return; }
    if (B <= 16) { g_thin_fwd<16>(l, th, X, xs, B, acts, S, slope, sm); return; }
    if (l.out <= 4) { g_thinj_fwd(l, th, X, xs, B, acts, S, slope, sm); return; }
    if (g_use_tc(tcx, B, l.out, l.in)) {
        g_tc_gemm(tcx, X, xs, 1, th + l.w_off, 1, l.in, acts + l.y_off, S, 1, B, l.out, l.in, th + l.b_off, l.act, slope, false);
        return;
    }
    g_gemm(X, xs, 1, th + l.w_off, 1, l.in, acts + l.y_off, S, 1, B, l.out, l.in, th + l.b_off, l.act, slope, false, sm);
}

// all layers for B rows; returns nothing: activations are in `acts` (row stride S = net.sum_out)
template <typename TCX = std::nullptr_t>
static __device__ void g_net_forward(const GNet& n, const float* th, const float* X, int xs, int B, float* acts, float* sm, TCX tcx = nullptr) {
    const int S = n.sum_out;
    const float* in = X;
    int in_s = xs;
    for (int i = 0; i < n.nfeat; ++i) {
        g_layer_fwd(n.feat[i], th, in, in_s, B, acts, S, n.slope, sm, tcx);
        in = acts + n.feat[i].y_off;
        in_s = S;
    }
    if (n.kind == LE_Q_DUELING) {
        g_layer_fwd(n.val[0], th, in, S, B, acts, S, n.slope, sm, tcx);
        g_layer_fwd(n.val[1], th, acts + n.val[0].y_off, S, B, acts, S, n.slope, sm, tcx);
        g_layer_fwd(n.adv[0], th, in, S, B, acts, S, n.slope, sm, tcx);
        g_layer_fwd(n.adv[1], th, acts + n.adv[0].y_off, S, B, acts, S, n.slope, sm, tcx);
    }
}

// CTA-wide sum of one float per thread; result broadcast to all threads. red: >= 32 floats of shared memory.
__device__ __forceinline__ float g_block_sum(float v, float* red) {
    v = warp_allreduce_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kGThreads / 32; ++w) t += red[w];
    return t;
}

// q[b][a] for B rows from the activation record: DQN -> output layer; dueling -> V + (A - mean(A over batch x actions))
static __device__ void g_q_values(const GNet& n, const float* acts, int B, float* q, float* red) {
    const int S = n.sum_out, AD = n.ad;
    if (n.kind == LE_Q_DQN) {
        const int yo = n.feat[n.nfeat - 1].y_off;
        for (int e = threadIdx.x; e < B * AD; e += kGThreads) q[e] = acts[(int64_t)(e / AD) * S + yo + (e % AD)];
        __syncthreads();
        return;
    }
    const int ao = n.adv[1].y_off, vo = n.val[1].y_off;
    float part = 0.f;
    for (int e = threadIdx.x; e < B * AD; e += kGThreads) part += acts[(int64_t)(e / AD) * S + ao + (e % AD)];
    const float mean = g_block_sum(part, red) / (float)(B * AD);
    for (int e = threadIdx.x; e < B * AD; e += kGThreads) {
        const int b = e / AD, a = e % AD;
        q[e] = acts[(int64_t)b * S + vo] + (acts[(int64_t)b * S + ao + a] - mean);
    }
    __syncthreads();
}

// backward of one dense layer for B rows. dact holds dL/dY at l.y_off (overwritten by dZ); X/xs: the layer's input.
// dX (may be null) receives / accumulates dL/dX with row stride dxs.
template <typename TCX = std::nullptr_t>
static __device__ void g_layer_bwd(const GLayer& l, const float* th, float* grad, const float* X, int xs, const float* acts, float* dact,
                            int S, int B, float* dX, int dxs, bool dx_accumulate, float slope, float* sm, TCX tcx = nullptr) {
    // dZ = dY * act'(Y) in place, and db[o] = sum_b dZ[b][o]: thread (rg, o) walks rows rg, rg+RG, ... of column o
    // (coalesced across o, independent loads down the column), partial sums meet in shared memory in fixed order.
    for (int o0 = 0; o0 < l.out; o0 += kGThreads) {
        const int cw = min(l.out - o0, kGThreads), RG = kGThreads / cw;
        const int rg = threadIdx.x / cw, o = o0 + threadIdx.x % cw;
        float part = 0.f;
        if (rg < RG) {
            constexpr int UN = 8;   // rows in flight per thread: the loop is L2-latency bound, not bandwidth bound
            for (int b = rg; b < B; b += UN * RG) {
                float dy[UN], y[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const int bb = b + u * RG;
                    const int64_t at = (int64_t)(bb < B ? bb : b) * S + l.y_off + o;
                    dy[u] = __ldcg(dact + at);
                    y[u] = __ldcg(acts + at);
                }
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const int bb = b + u * RG;
                    if (bb < B) {
                        const float dz = dy[u] * g_act_grad(l.act, slope, y[u]);
                        __stcg(dact + (int64_t)bb * S + l.y_off + o, dz);
                        part += dz;
                    }
                }
            }
            sm[rg * cw + (o - o0)] = part;
        }
        __syncthreads();
        if (threadIdx.x < cw) {
            float t = 0.f;
            for (int r = 0; r < RG; ++r) t += sm[r * cw + threadIdx.x];
            grad[l.b_off + o0 + threadIdx.x] = t;
        }
        __syncthreads();
    }
    // dW[o][i] = sum_b dZ[b][o] * X[b][i]; the longer of (out, in) takes the 128-row side of the tile
    const bool tc_dw = g_use_tc(tcx, B, l.out, l.in);     // (rows of the contraction = B, extents out x in)
    if (tc_dw) {
        if (l.out >= l.in) g_tc_gemm(tcx, dact + l.y_off, 1, S, X, xs, 1, grad + l.w_off, l.in, 1, l.out, l.in, B, (const float*)nullptr, 0, 0.f, false);
        else g_tc_gemm(tcx, X, 1, xs, dact + l.y_off, S, 1, grad + l.w_off, 1, l.in, l.in, l.out, B, (const float*)nullptr, 0, 0.f, false);
    } else if (l.out >= l.in) g_gemm(dact + l.y_off, 1, S, X, xs, 1, grad + l.w_off, l.in, 1, l.out, l.in, B, nullptr, 0, 0.f, false, sm);
    else g_gemm(X, 1, xs, dact + l.y_off, S, 1, grad + l.w_off, 1, l.in, l.in, l.out, B, nullptr, 0, 0.f, false, sm);
    // dX[b][i] (+)= sum_o dZ[b][o] * W[o][i]
    if (dX) {
        if (g_use_tc(tcx, B, l.in, l.out))
            g_tc_gemm(tcx, dact + l.y_off, S, 1, th + l.w_off, l.in, 1, dX, dxs, 1, B, l.in, l.out, (const float*)nullptr, 0, 0.f, dx_accumulate);
        else g_gemm(dact + l.y_off, S, 1, th + l.w_off, l.in, 1, dX, dxs, 1, B, l.in, l.out, nullptr, 0, 0.f, dx_accumulate, sm);
    }
}

// Device-side view of one lane slot's workspace
struct GSlot {
    float *ring, *theta, *thetaT, *m, *v, *grad, *xs, *xs2, *misc, *actA, *actB, *dact, *q, *q2, *qT, *dq, *obs;
    int* astar;
};

// torch.optim.Adam step of one parameter vector (b1pow / b2pow: beta^t after the step count increment); with a target thT,
// also the Polyak update thT <- tau * th + (1 - tau) * thT.  Same operation order as LaneCore::adam_polyak.
static __device__ void g_adam(float* th, float* thT, float* m, float* v, const float* grad, int P, const LearnScalars& ls, double b1pow,
                              double b2pow) {
    const double bc1 = 1.0 - b1pow, bc2 = 1.0 - b2pow;
    const float neg_step = (float)(-(ls.lr / bc1));
    const float bc2s = (float)sqrt(bc2);
    constexpr int UN = 8;   // parameters in flight per thread (5 loads each)
    for (int p0 = threadIdx.x; p0 < P; p0 += UN * kGThreads) {
        float g[UN], mo[UN], vo[UN], t[UN], tt[UN];
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            const int p = p0 + u * kGThreads < P ? p0 + u * kGThreads : p0;
            g[u] = __ldcg(grad + p); mo[u] = __ldcg(m + p); vo[u] = __ldcg(v + p);
            t[u] = __ldcg(th + p);
            if (thT) tt[u] = __ldcg(thT + p);
        }
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            const int p = p0 + u * kGThreads;
            if (p < P) {
                float mm = mo[u] + ls.w1 * (g[u] - mo[u]);
                float vv = vo[u] * ls.beta2;
                vv = vv + (ls.w2 * g[u]) * g[u];
                __stcg(m + p, mm);
                __stcg(v + p, vv);
                bool exact = true;
                float up = adam_update_core(mm, vv, neg_step, bc2s, ls.eps, &exact);
                if (!exact) up = __fdiv_rn(neg_step * mm, __fdiv_rn(__fsqrt_rn(vv), bc2s) + ls.eps);
                const float pn = t[u] + up;
                __stcg(th + p, pn);
                if (thT) __stcg(thT + p, ls.tau * pn + ls.one_minus_tau * tt[u]);
            }
        }
    }
    __syncthreads();
}

// DDQN.learn / DuelingDDQN.learn on the B rows staged in slot.xs / xs2 / misc (misc = [a, r, d, pad] per row)
template <typename TCX = std::nullptr_t>
static __device__ float g_td_update(const GNet& n, const GSlot& w, int B, LearnScalars& ls, float* sm, float* red, TCX tcx = nullptr) {
    const int S = n.sum_out, AD = n.ad, SDs = n.sd;
    g_net_forward(n, w.theta, w.xs, SDs, B, w.actA, sm, tcx);    // q_values = model(states)            (activations kept)
    g_q_values(n, w.actA, B, w.q, red);
    g_net_forward(n, w.theta, w.xs2, SDs, B, w.actB, sm, tcx);   // next_q_values = model(next_states)
    g_q_values(n, w.actB, B, w.q2, red);
    g_net_forward(n, w.thetaT, w.xs2, SDs, B, w.actB, sm, tcx);  // model_target(next_states)
    g_q_values(n, w.actB, B, w.qT, red);
    float lpart = 0.f, gpart = 0.f;
    for (int b = threadIdx.x; b < B; b += kGThreads) {
        const int a = (int)w.misc[4 * b];
        int astar = 0;
        float best = w.q2[b * AD];
        for (int k = 1; k < AD; ++k)
            if (w.q2[b * AD + k] > best) { best = w.q2[b * AD + k]; astar = k; }
        const float y = w.misc[4 * b + 1] + (ls.gamma * w.qT[b * AD + astar]) * (1.f - w.misc[4 * b + 2]);
        const float delta = w.q[b * AD + a] - y;
        lpart = fmaf(delta, delta, lpart);
        const float dq = ls.norm * delta;
        w.dq[b] = dq;
        gpart += dq;
    }
    const float loss = g_block_sum(lpart, red) / (float)B;
    const float mean_g = g_block_sum(gpart, red) / (float)(B * AD);
    // seed dL/d(outputs)
    if (n.kind == LE_Q_DQN) {
        const int yo = n.feat[n.nfeat - 1].y_off;
        for (int e = threadIdx.x; e < B * AD; e += kGThreads) {
            const int b = e / AD, k = e % AD;
            w.dact[(int64_t)b * S + yo + k] = ((int)w.misc[4 * b] == k) ? w.dq[b] : 0.f;
        }
    } else {
        const int ao = n.adv[1].y_off, vo = n.val[1].y_off;
        for (int e = threadIdx.x; e < B * AD; e += kGThreads) {
            const int b = e / AD, k = e % AD;
            w.dact[(int64_t)b * S + ao + k] = (((int)w.misc[4 * b] == k) ? w.dq[b] : 0.f) - mean_g;
            if (k == 0) w.dact[(int64_t)b * S + vo] = w.dq[b];
        }
    }
    __syncthreads();
    const GLayer& lf = n.feat[n.nfeat - 1];
    if (n.kind == LE_Q_DUELING) {
        g_layer_bwd(n.val[1], w.theta, w.grad, w.actA + n.val[0].y_off, S, w.actA, w.dact, S, B, w.dact + n.val[0].y_off, S, false, n.slope, sm, tcx);
        g_layer_bwd(n.val[0], w.theta, w.grad, w.actA + lf.y_off, S, w.actA, w.dact, S, B, w.dact + lf.y_off, S, false, n.slope, sm, tcx);
        g_layer_bwd(n.adv[1], w.theta, w.grad, w.actA + n.adv[0].y_off, S, w.actA, w.dact, S, B, w.dact + n.adv[0].y_off, S, false, n.slope, sm, tcx);
        g_layer_bwd(n.adv[0], w.theta, w.grad, w.actA + lf.y_off, S, w.actA, w.dact, S, B, w.dact + lf.y_off, S, true, n.slope, sm, tcx);
    }
    for (int i = n.nfeat - 1; i >= 0; --i) {
        const GLayer& l = n.feat[i];
        const float* X = i > 0 ? w.actA + n.feat[i - 1].y_off : w.xs;
        const int xs = i > 0 ? S : SDs;
        g_layer_bwd(l, w.theta, w.grad, X, xs, w.actA, w.dact, S, B, i > 0 ? w.dact + n.feat[i - 1].y_off : nullptr, S, false, n.slope, sm, tcx);
    }
    ls.b1pow *= ls.beta1;
    ls.b2pow *= ls.beta2d;
    g_adam(w.theta, w.thetaT, w.m, w.v, w.grad, n.P, ls, ls.b1pow, ls.b2pow);
    return loss;
}

// greedy action of ONE state row (select_train/test_action); every thread takes the argmax, so the result is uniform
static __device__ int g_greedy_row(const GNet& n, const GSlot& w, const float* state_row /* [sd] in global memory */, float* sm, float* red) {
    g_net_forward(n, w.theta, state_row, n.sd, 1, w.actB, sm);
    g_q_values(n, w.actB, 1, w.q2, red);
    int best = 0;
    for (int k = 1; k < n.ad; ++k)
        if (w.q2[k] > w.q2[best]) best = k;
    return best;
}

struct GRunParams {
    RunParams rp;            // same lane-level inputs/outputs as the warp kernel
    GNet net;
    float* slots; int64_t slot_stride;   // floats per CTA slot
    int bmax;
};

__host__ __device__ inline int64_t gslot_floats(const GNet& n, int ring_cap, int rowf, int bmax, int64_t* offs /* [18] */) {
    const int Pp = (n.P + 3) / 4 * 4;
    const int64_t BS = (int64_t)bmax * n.sum_out;
    int64_t o = 0;
    int k = 0;
    auto take = [&](int64_t nfl) { offs[k++] = o; o += (nfl + 3) / 4 * 4; };
    take((int64_t)ring_cap * rowf);          // 0 ring
    take(Pp); take(Pp); take(Pp); take(Pp); take(Pp);   // 1..5 theta thetaT m v grad
    take((int64_t)bmax * n.sd); take((int64_t)bmax * n.sd); take((int64_t)bmax * 4);   // 6 xs, 7 xs2, 8 misc
    take(BS); take(BS); take(BS);            // 9 actA, 10 actB, 11 dact
    take((int64_t)bmax * n.ad); take((int64_t)bmax * n.ad); take((int64_t)bmax * n.ad);   // 12 q, 13 q2, 14 qT
    take(bmax); take((int64_t)64 * n.sd); take(bmax);   // 15 dq, 16 obs, 17 astar
    return o;
}

__device__ inline GSlot gslot_view(float* base, const GNet& n, int ring_cap, int rowf, int bmax) {
    int64_t offs[18];
    gslot_floats(n, ring_cap, rowf, bmax, offs);
    GSlot s;
    s.ring = base + offs[0]; s.theta = base + offs[1]; s.thetaT = base + offs[2]; s.m = base + offs[3]; s.v = base + offs[4];
    s.grad = base + offs[5]; s.xs = base + offs[6]; s.xs2 = base + offs[7]; s.misc = base + offs[8]; s.actA = base + offs[9];
    s.actB = base + offs[10]; s.dact = base + offs[11]; s.q = base + offs[12]; s.q2 = base + offs[13]; s.qT = base + offs[14];
    s.dq = base + offs[15]; s.obs = base + offs[16]; s.astar = reinterpret_cast<int*>(base + offs[17]);
    return s;
}

// torch default nn.Linear init of a general net from the P_QINIT stream (same stream as the CPU restatement)
static __device__ void g_init_layer(const GLayer& l, float* th, uint32_t k0, uint32_t k1) {
    const double bnd = 1.0 / sqrt((double)l.in);
    const int end = l.b_off + l.out;
    for (int p = l.w_off + threadIdx.x; p < end; p += kGThreads) {
        const u32x4 w = philox4x32_10((uint32_t)(p >> 2), 0u, LE_P_QINIT, 0u, k0, k1);
        th[p] = (float)((2.0 * (((double)pick(w, p & 3) + 0.5) * (1.0 / 4294967296.0)) - 1.0) * bnd);
    }
}

// DDQN / DuelingDDQN agent (agents/DDQN.py, agents/DuelingDDQN.py) as the hooks of cta_lane_loop: eps-greedy acting on
// the greedy row, replay rows in RowLayout<SD>, learn = g_td_update.  cfg / n: this lane's configuration and network in shared
// memory (per-lane q_hidden / q_layers under vary_hp).
template <int SD, int AD, typename TCX>
struct GeneralAgent {
    using RL = RowLayout<SD>;
    const RunParams& P;
    const GSlot w;   // sized for the maxima (cfg 0)
    le_lane_cfg& cfg;
    GNet& n;
    float* sm;
    float* red;
    TCX tcx;
    uint32_t k0, k1;
    LearnScalars ls;
    double eps;

    __device__ __forceinline__ const le_lane_cfg& begin_lane(int lane_id, uint32_t key0, uint32_t key1) {
        const int tid = threadIdx.x;
        k0 = key0; k1 = key1;
        {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(P.cfg + (P.n_cfg == 1 ? 0 : lane_id));
            uint32_t* dst = reinterpret_cast<uint32_t*>(&cfg);
            for (int i = tid; i < (int)(sizeof(le_lane_cfg) / 4); i += kGThreads) dst[i] = src[i];
        }
        __syncthreads();
        if (tid == 0) gnet_build(&cfg, &n);
        __syncthreads();
        if (P.q_init) { for (int p = tid; p < n.P; p += kGThreads) w.theta[p] = P.q_init[(int64_t)lane_id * P.q_stride + p]; }
        else {
            for (int i = 0; i < n.nfeat; ++i) g_init_layer(n.feat[i], w.theta, k0, k1);
            if (n.kind == LE_Q_DUELING) { g_init_layer(n.val[0], w.theta, k0, k1); g_init_layer(n.val[1], w.theta, k0, k1);
                                          g_init_layer(n.adv[0], w.theta, k0, k1); g_init_layer(n.adv[1], w.theta, k0, k1); }
        }
        __syncthreads();
        for (int p = tid; p < n.P; p += kGThreads) { w.thetaT[p] = w.theta[p]; w.m[p] = 0.f; w.v[p] = 0.f; }
        __syncthreads();
        fill_learn_scalars(ls, cfg);
        eps = cfg.eps_init;
        return cfg;
    }

    __device__ __forceinline__ void begin_episode(int episode) { eps = eps_schedule(eps, episode, cfg); }

    __device__ __forceinline__ int train_action(const float (&state)[SD], int, int64_t train_steps, bool tracing, bool& explore, float& qgap,
                                                float*) {
        const u32x4 wa = philox4x32_10((uint32_t)train_steps, 0u, LE_P_ACT, 0u, k0, k1);
        explore = ((double)(wa.x >> 8) * (1.0 / 16777216.0)) < eps;
        if (explore) return (int)__umulhi(wa.y, (uint32_t)AD);
        __syncthreads();
        if (threadIdx.x < SD) __stcg(w.xs + threadIdx.x, state[threadIdx.x]);   // operand rows are read with ld.global.cg: stage in the slot
        __syncthreads();
        const int action = g_greedy_row(n, w, w.xs, sm, red);
        if (tracing) {
            float q[AD];
#pragma unroll
            for (int k = 0; k < AD; ++k) q[k] = w.q2[k];
            qgap = relative_q_gap<AD>(q, action);
            __syncthreads();
        }
        return action;
    }

    __device__ __forceinline__ void store_row(int row, const float (&state)[SD], int action, const float (&ns)[SD], float r, float d) {
        float rowv[RL::ROWF];
#pragma unroll
        for (int i = 0; i < RL::ROWF; ++i) rowv[i] = 0.f;
#pragma unroll
        for (int i = 0; i < SD; ++i) { rowv[RL::OFF_S + i] = state[i]; rowv[RL::OFF_S2 + i] = ns[i]; }
        rowv[RL::OFF_A] = __int_as_float(action); rowv[RL::OFF_R] = r; rowv[RL::OFF_D] = d;
        float4* dst = reinterpret_cast<float4*>(w.ring + (int64_t)row * RL::ROWF);
#pragma unroll
        for (int q = 0; q < RL::ROW_VEC; ++q)
            if (threadIdx.x == q) __stcg(dst + q, make_float4(rowv[4 * q], rowv[4 * q + 1], rowv[4 * q + 2], rowv[4 * q + 3]));
    }

    __device__ __forceinline__ float learn(int64_t learn_iters, int rb_size) {
        __syncthreads();
        const int B = ls.batch;
        for (int b = threadIdx.x; b < B; b += kGThreads) {   // replay_buffer.sample on the P_SAMPLE stream
            const u32x4 wv = philox4x32_10((uint32_t)learn_iters, (uint32_t)(b >> 2), LE_P_SAMPLE, 0u, k0, k1);
            const uint32_t idx = __umulhi(pick(wv, b & 3), (uint32_t)rb_size);
            const float4* src = reinterpret_cast<const float4*>(w.ring + (int64_t)idx * RL::ROWF);
            float rowv[RL::ROWF];
#pragma unroll
            for (int q = 0; q < RL::ROW_VEC; ++q) { const float4 v4 = __ldcg(src + q); rowv[4 * q] = v4.x; rowv[4 * q + 1] = v4.y; rowv[4 * q + 2] = v4.z; rowv[4 * q + 3] = v4.w; }
#pragma unroll
            for (int i = 0; i < SD; ++i) { w.xs[b * SD + i] = rowv[RL::OFF_S + i]; w.xs2[b * SD + i] = rowv[RL::OFF_S2 + i]; }
            w.misc[4 * b] = (float)__float_as_int(rowv[RL::OFF_A]); w.misc[4 * b + 1] = rowv[RL::OFF_R]; w.misc[4 * b + 2] = rowv[RL::OFF_D];
        }
        __syncthreads();
        return g_td_update(n, w, B, ls, sm, red, tcx);
    }

    __device__ __forceinline__ float* test_obs() { return w.obs; }

    // greedy action of test row threadIdx.x
    __device__ __forceinline__ int test_action(int M, int, int, int, bool running) {
        g_net_forward(n, w.theta, w.obs, SD, M, w.actB, sm);
        g_q_values(n, w.actB, M, w.q2, red);
        int best = 0;
        if (running)
            for (int k = 1; k < AD; ++k)
                if (w.q2[threadIdx.x * AD + k] > w.q2[threadIdx.x * AD + best]) best = k;
        return best;
    }

    __device__ __forceinline__ void end_lane(int lane_id) {
        if (P.q_final) for (int p = threadIdx.x; p < n.P; p += kGThreads) P.q_final[(int64_t)lane_id * P.q_stride + p] = w.theta[p];
    }
};

// TC = false: two CTAs per SM, every dense layer on the FFMA GEMM.  TC = true: the CTA owns 128 TMEM columns and the dense
// hidden x hidden layers run on tcgen05 (one CTA per SM: the runtime's TMEM occupancy rule).
template <int SD, int AD, bool TC>
__global__ void __launch_bounds__(kGThreads, TC ? 1 : 2) general_loop_kernel(const GRunParams G) {
    __shared__ __align__(16) float sm[kGSmemFloats];
    __shared__ float red[32];
    __shared__ le_lane_cfg cfg_sm;
    __shared__ GNet net_sm;
    extern __shared__ __align__(128) unsigned char tc_smem[];   // TC: tc::kSmemBytes, operand parts of the tensor-core GEMM
    tc::Ctx tcs;
    if constexpr (TC) tcs = tc::ctx_create(tc_smem);
    typename std::conditional<TC, tc::Ctx*, std::nullptr_t>::type tcx = nullptr;
    if constexpr (TC) tcx = &tcs;
    GeneralAgent<SD, AD, decltype(tcx)> ag{G.rp, gslot_view(G.slots + (int64_t)blockIdx.x * G.slot_stride, G.net, G.rp.ring_cap, RowLayout<SD>::ROWF, G.bmax),
                                           cfg_sm, net_sm, sm, red, tcx};
    cta_lane_loop<SD, AD>(G.rp, ag);
    if constexpr (TC) tc::ctx_destroy(tcs);
}

// unit kernels on caller-owned canonical arrays (same layout as the slot's theta/thetaT/m/v)
template <int SD, int AD, bool TC>
__global__ void __launch_bounds__(kGThreads, TC ? 1 : 2)
general_td_update_kernel(const le_lane_cfg* __restrict__ cfg_dev, GNet n, float* th, float* thT, float* m, float* v, int32_t* tcount,
                         int q_stride, const float* __restrict__ rows, int B, float* __restrict__ loss_out, float* scratch,
                         int64_t scratch_stride) {
    __shared__ __align__(16) float sm[kGSmemFloats];
    __shared__ float red[32];
    extern __shared__ __align__(128) unsigned char tc_smem[];
    tc::Ctx tcs;
    if constexpr (TC) tcs = tc::ctx_create(tc_smem);
    typename std::conditional<TC, tc::Ctx*, std::nullptr_t>::type tcx = nullptr;
    if constexpr (TC) tcx = &tcs;
    const int id = blockIdx.x, tid = threadIdx.x;
    const le_lane_cfg c = *cfg_dev;
    GSlot w = gslot_view(scratch + (int64_t)id * scratch_stride, n, 0, 0, B);   // scratch arrays; parameters and Adam state are the caller's
    w.theta = th + (int64_t)id * q_stride; w.thetaT = thT + (int64_t)id * q_stride;
    w.m = m + (int64_t)id * q_stride; w.v = v + (int64_t)id * q_stride;
    constexpr int ROWP = 2 * SD + 3;
    const float* my_rows = rows + (int64_t)id * B * ROWP;
    for (int b = tid; b < B; b += kGThreads) {
        const float* src = my_rows + (int64_t)b * ROWP;
#pragma unroll
        for (int i = 0; i < SD; ++i) { w.xs[b * SD + i] = src[i]; w.xs2[b * SD + i] = src[SD + 1 + i]; }
        w.misc[4 * b] = src[SD]; w.misc[4 * b + 1] = src[2 * SD + 1]; w.misc[4 * b + 2] = src[2 * SD + 2];
    }
    __syncthreads();
    LearnScalars ls;
    fill_learn_scalars(ls, c);
    ls.batch = B;
    ls.norm = (float)(2.0 / (double)B);
    const int t0 = tcount[id];
    ls.b1pow = pow(c.beta1, (double)t0);
    ls.b2pow = pow(c.beta2, (double)t0);
    const float loss = g_td_update(n, w, B, ls, sm, red, tcx);
    if (tid == 0) { loss_out[id] = loss; tcount[id] = t0 + 1; }
    if constexpr (TC) tc::ctx_destroy(tcs);
}

template <int SD, int AD>
__global__ void __launch_bounds__(kGThreads)
general_qnet_forward_kernel(GNet n, const float* __restrict__ q_theta, int q_stride, const float* __restrict__ state,
                            float* __restrict__ q_out, int32_t* __restrict__ argmax, float* scratch, int64_t scratch_stride) {
    __shared__ __align__(16) float sm[kGSmemFloats];
    __shared__ float red[32];
    const int id = blockIdx.x;
    float* acts = scratch + (int64_t)id * scratch_stride;
    float* q = acts + n.sum_out;
    g_net_forward(n, q_theta + (int64_t)id * q_stride, state + (int64_t)id * SD, SD, 1, acts, sm);
    g_q_values(n, acts, 1, q, red);
    if (threadIdx.x == 0) {
        int best = 0;
        for (int k = 0; k < AD; ++k) { q_out[(int64_t)id * AD + k] = q[k]; if (q[k] > q[best]) best = k; }
        argmax[id] = best;
    }
}

}  // namespace le
