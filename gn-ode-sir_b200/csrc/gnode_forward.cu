// Forward rollout: encoder, fused Euler-step kernel, decoder (SURVEY 8a: a1-a9).
//
// One CTA owns a tile of 128 consecutive rows of the batch ((trial, node) pairs) and
// runs, per Euler step k (reference lines in brackets, ode_nn_ngraph_sim.py):
//   1. S_k tile  -> shared memory (UMMA K-major SWIZZLE_128B layout)
//   2. S' = sigmoid(S_k W^T + b)                        [:62-63]   -> shared memory
//   3. row-per-half-warp: AI = sum_nbrs I'_k            [:73]      (I'_k from HBM/L2)
//        dS,dI,dR ; y_{k+1} = y_k + dt f                [:75-77,96; torchdiffeq Euler]
//        -> HBM (coalesced); I_{k+1} stays in shared memory; decoder + softmax of
//        y_{k+1} -> probs[k+1]                          [:170-188]
//   4. I'_{k+1} = sigmoid(I_{k+1} W^T + b) -> HBM       (next step's aggregation operand)
// so one launch per step reads S,I,R,I' and writes S,I,R,I',probs exactly once; the
// grid-wide dependency (all of I'_k before any aggregation) is the launch boundary.
// The reference's R' = sigmoid(linear(R)) is never used (:66 vs :75-77) and is skipped.
#include <cooperative_groups.h>
#include <cuda.h>          // CUtensorMap (type and enums only: the encoder is resolved through the runtime, no libcuda link)
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "gnode_common.cuh"
#include "gnode_tile.cuh"
#include "gnode_umma.cuh"

#ifndef GNODE_DEFAULT_VARIANT
#define GNODE_DEFAULT_VARIANT 3
#endif

namespace gnode {

enum { MODE_STEP = 0, MODE_ENCODE = 1, MODE_IP = 2, MODE_RHS = 3 };

struct StepArgs {
    GnBatchView bv;
    const float* y_in;    // [3][M][H]
    float* y_out;         // [3][M][H]  STEP: y_{k+1}; ENCODE: y_0; RHS: f(y)
    const float* ip_in;   // [M][H]     I'_k
    float* ip_out;        // [M][H]     I'_{k+1}
    float* beta;          // [M]
    float* gamma;         // [M]
    const float* x;       // ENCODE: [M][ldx]
    int64_t ldx;
    float* probs;         // [M][3] slice of the produced state (dual kernel: of the INPUT state), or null
    float* hid_i;         // [M][4] linear3 pre-activations (no bias) of the I block: ENCODE writes I_0's, the dual step kernel updates in place; or null
    float* hid_r;         // [M][4] inference without an R plane (RF): W3 (S_0 + I_0 + R_0), constant over the rollout; hid(R_k) follows by
                          // the conserved sum (hid(R_k) = hid_r - hid(S_k) - hid(I_k)); ENCODE writes it; null = R is a full state plane
    float dt;
    long long* tbuf;      // phase timing accumulators (debug, env GNODE_DBG bit 7) or null
    int dbg;              // timing experiments only (env GNODE_DBG): bit0 no decode, 1 no gather, 2 no own loads, 3 no GEMM2, 4 no GEMM1
    int* counter;         // dynamic tile scheduler (one zeroed int per launch) or null = static striding
    gnode_params_t p;
    int relay_off;        // 1: hub rows are walked serially by one half-warp (gnode_set_hub_relay(0): the relay's bitwise check)
    int use_tma;          // dual kernel: I'_{k+1} tiles leave shared memory through TMA stores described by tm_ip_out
    // persistent rollout (dual kernel, cooperative launch): the kernel runs the Euler steps k0 .. k1-1 itself, with a
    // grid barrier between steps; per-step pointers are derived from the bases below (n_steps == 0: one step from the
    // fields above, ordinary launch)
    int k0, n_steps;
    float* traj;          // [T][3][M][H] or null (then the two ping-pong buffers st[])
    float* st[2];
    float* ipb[2];        // I' ping-pong
    float* probs_base;    // [T][M][3]
    const float* dt_dev;  // [T-1] device copy of the step sizes, or null: every step uses `dt`
    const int* out_slot;  // [T] output slot of every grid point (-1: not emitted), or null: slot(k) = (k - out_start) / out_stride
    int out_start, out_stride, n_out;   // arithmetic selection (identity: 0, 1, T)
    int* counters;        // one zeroed int per step (dynamic tile tickets)
    // training with auxiliary storage (step_stream_kernel): I'_k and AI_k = A I'_k of every step are kept for the reverse
    // sweep in aux[T][2][Mr + 1][H] (Mr = M rounded up to the tile; row Mr of every I' plane is the all-zero row)
    float* ai_out;        // one launch per step: AI_k plane, or null
    float* aux;           // persistent rollout: base of the buffer, or null
    int64_t aux_slot;     // floats per grid point = 2 (Mr + 1) H
    int ip_zrow;          // row index of the all-zero row of an I' plane (M for the ping-pong buffers)
    // Euler step 0 of a descriptor-fed inference rollout fused with the encoder (step_stream_kernel, OPT bit 7)
    const float* z_tbl;          // two-row table of trials_table_kernel
    const uint32_t* z_bitmap;    // bit g = row g is a seed row
    const float* z_beta;         // [n_inst]
    const float* z_gamma;        // [n_inst]
    alignas(64) CUtensorMap tm_ip_out;   // [M rows][64] fp32 over ip_out, box 32 x 128, SWIZZLE_128B
    alignas(64) CUtensorMap tm_ipb[2];   // the same over ipb[0] / ipb[1] (persistent rollout)
    // step_stream_kernel: the S_k tile arrives by TMA tensor loads (same box / swizzle = the UMMA operand layout)
    alignas(64) CUtensorMap tm_s_in;     // [M rows][64] fp32 over the S plane of y_in (one launch per step)
    alignas(64) CUtensorMap tm_sp[2];    // persistent rollout: over the S planes of st[0] / st[1], or [0] over the whole trajectory
    // weighted neighbour sum (step_stream_kernel, OPT bit 8): weight of entry e of instance i = edge_w[inst_e0[i] + e]
    const float* edge_w;
    const int64_t* inst_e0;
};

// output slot of grid point k (-1: its probabilities are not emitted)
__host__ __device__ __forceinline__ int out_slot_of(const StepArgs& a, int k) {
    if (a.out_slot) return a.out_slot[k];
    const int d = k - a.out_start;
    if (d < 0 || d % a.out_stride != 0) return -1;
    return d / a.out_stride < a.n_out ? d / a.out_stride : -1;
}

// shared-memory carve-up (bytes from a 1024-B aligned base; operand tiles need 1024-B alignment)
constexpr int SM_X = 0;                        // 32 KB  operand tile (S_k, then I_{k+1})
constexpr int SM_SP = 32768;                   // 32 KB  Xlo scratch / S' tile / I'_{k+1} staging
constexpr int SM_W = 65536;                    // 16 KB  FFMA: W [h][k] row-major; tensor path: Whi operand
constexpr int SM_WLO = SM_W + H * H * 4;       // 16 KB  tensor path: Wlo operand
constexpr int SM_B = SM_WLO + H * H * 4;       // bias [64]
constexpr int SM_W3 = SM_B + H * 4;            // linear3.weight [4][64]
constexpr int SM_W1 = SM_W3 + 4 * H * 4;       // linearS1.weight [64]
constexpr int SM_B1 = SM_W1 + H * 4;           // linearS1.bias [64]
constexpr int SM_SMALL = SM_B1 + H * 4;        // b3[4], w2[4], b2[1]
constexpr int SM_MBAR = SM_SMALL + 64;         // mbarrier (8 B) + TMEM base slot (4 B)
constexpr int SM_TOTAL = SM_MBAR + 16 + 1024;  // + slack for the manual 1024-B alignment

// kernel variants: bit 0 = tcgen05 3xTF32 transform (else FFMA), bit 1 = MUFU sigmoid (else expf + IEEE div)
constexpr int VAR_TC = 1, VAR_FASTSIG = 2;

// decoder + softmax of one row held 4 channels per lane by a half-warp
// (linear3 -> ReLU -> linearS2 -> softmax over {S,I,R}; ode_nn_ngraph_sim.py:172-187)
__device__ __forceinline__ void decode_row(float4 s, float4 i, float4 r, const float* W3s, const float* small,
                                           int l, bool valid, float* probs_row, float* hid_i_row = nullptr,
                                           float* hid_r_row = nullptr, const float* hid_r_in = nullptr) {
    float v[12];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        const float4 w = *reinterpret_cast<const float4*>(W3s + m * H + 4 * l);
        v[m] = dot4(s, w); v[4 + m] = dot4(i, w); v[8 + m] = dot4(r, w);
    }
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1)
#pragma unroll
        for (int m = 0; m < 12; ++m) v[m] += __shfl_xor_sync(0xffffffffu, v[m], off);
    if (l == 0 && valid && hid_i_row != nullptr) *reinterpret_cast<float4*>(hid_i_row) = make_float4(v[4], v[5], v[6], v[7]);
    // inference without an R plane: the row keeps hid(S_0 + I_0 + R_0) (written here by the encoder launch), and
    // hid(R_k) = that - hid(S_k) - hid(I_k) wherever probabilities are emitted (S + I + R is conserved, see the step kernels)
    if (l == 0 && valid && hid_r_row != nullptr)
        *reinterpret_cast<float4*>(hid_r_row) = make_float4((v[0] + v[4]) + v[8], (v[1] + v[5]) + v[9], (v[2] + v[6]) + v[10], (v[3] + v[7]) + v[11]);
    if (l == 0 && valid && hid_r_in != nullptr) {
        const float4 h = *reinterpret_cast<const float4*>(hid_r_in);
        v[8] = (h.x - v[0]) - v[4]; v[9] = (h.y - v[1]) - v[5]; v[10] = (h.z - v[2]) - v[6]; v[11] = (h.w - v[3]) - v[7];
    }
    if (l == 0 && valid && probs_row != nullptr) {
        const float* b3 = small; const float* w2 = small + 4; const float b2 = small[8];
        float o[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            float acc = b2;
#pragma unroll
            for (int m = 0; m < 4; ++m) acc = fmaf(w2[m], fmaxf(v[4 * c + m] + b3[m], 0.f), acc);
            o[c] = acc;
        }
        const float mx = fmaxf(o[0], fmaxf(o[1], o[2]));
        const float e0 = expf(o[0] - mx), e1 = expf(o[1] - mx), e2 = expf(o[2] - mx);
        const float inv = 1.0f / (e0 + e1 + e2);
        probs_row[0] = e0 * inv; probs_row[1] = e1 * inv; probs_row[2] = e2 * inv;
    }
}

template <int MODE, int VAR>
__global__ void __launch_bounds__(NTHREADS, 2) step_kernel(const StepArgs a) {
    constexpr bool TC = (VAR & VAR_TC) != 0;
    constexpr bool FAST = (VAR & VAR_FASTSIG) != 0;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Xs = smem + SM_X;
    unsigned char* SPs = smem + SM_SP;
    float* Ws = reinterpret_cast<float*>(smem + SM_W);
    float* bs = reinterpret_cast<float*>(smem + SM_B);
    float* W3s = reinterpret_cast<float*>(smem + SM_W3);
    float* w1s = reinterpret_cast<float*>(smem + SM_W1);
    float* b1s = reinterpret_cast<float*>(smem + SM_B1);
    float* small = reinterpret_cast<float*>(smem + SM_SMALL);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + SM_MBAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + SM_MBAR + 8);

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int l = tid & 15;           // 16-byte chunk of the row owned in the row-per-half-warp phases
    const int hw = tid >> 4;          // half-warp id 0..31
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;

    // parameters -> shared memory (once per CTA; the CTA is persistent over its tiles)
    umma::Ctx cx;
    if (TC) {
        umma::prepare_weights(a.p.lin_w, smem + SM_W, smem + SM_WLO, tid, NTHREADS);
        if (tid < 32) umma::tmem_alloc(tslot, umma::TMEM_COLS);          // warp 0 owns alloc / dealloc
        if (tid == 0) umma::mbar_init(mbar, 1);
        umma::fence_before_sync();
    } else {
        for (int i = tid; i < H * H / 4; i += NTHREADS)
            reinterpret_cast<float4*>(Ws)[i] = reinterpret_cast<const float4*>(a.p.lin_w)[i];
    }
    if (tid < H) bs[tid] = a.p.lin_b[tid];
    if (MODE == MODE_ENCODE && tid < H) { w1s[tid] = a.p.s1_w[tid]; b1s[tid] = a.p.s1_b[tid]; }
    if (MODE == MODE_ENCODE || MODE == MODE_STEP) {     // decoder weights (RHS / IP callers pass none)
        if (tid < 4 * H) W3s[tid] = a.p.l3_w[tid];
        if (tid < 4) { small[tid] = a.p.l3_b[tid]; small[4 + tid] = a.p.s2_w[tid]; }
        if (tid == 0) small[8] = a.p.s2_b[0];
    }
    __syncthreads();
    if (TC) {
        umma::fence_after_sync();
        cx.tmem = *tslot;
        cx.bar = mbar;
        cx.phase = 0;
        cx.whi = umma::smem_u32(smem + SM_W);
        cx.wlo = umma::smem_u32(smem + SM_WLO);
    }

    int* tile_slot = reinterpret_cast<int*>(smem + SM_MBAR + 12);
    for (int seq = blockIdx.x;; seq += gridDim.x) {
        if (a.counter != nullptr) {               // dynamic: next entry of the hub-first processing order
            if (tid == 0) *tile_slot = atomicAdd(a.counter, 1);
            __syncthreads();
            seq = *tile_slot;
        }
        if (seq >= a.bv.n_tiles) break;
        const int tile = a.bv.tile_order[seq];
        const int64_t tile0 = (int64_t)tile * TILE;

        if (MODE == MODE_STEP || MODE == MODE_RHS) {
            load_tile(Xs, a.y_in, tile0, M, tid);                 // S_k
            __syncthreads();
            if (TC) umma::gemm_sigmoid_tc<FAST>(cx, Xs, SPs, bs, tid);   // S'
            else gemm_sigmoid<FAST>(Xs, Ws, bs, SPs, tid);
            __syncthreads();
        } else if (MODE == MODE_IP) {
            load_tile(Xs, a.y_in + plane, tile0, M, tid);         // I
            __syncthreads();
        }

        if (MODE == MODE_STEP || MODE == MODE_RHS) {
            int inst = a.bv.tile_inst[tile];
#pragma unroll 1
            for (int it = 0; it < TILE / 32; ++it) {
                const int rr = hw + 32 * it;
                const int64_t g = tile0 + rr;
                const bool valid = g < M;
                int row0 = 0, e0 = 0, deg = 0;
                const int32_t* ci = nullptr;
                if (valid) {
                    while (inst + 1 < a.bv.n_inst && a.bv.inst[inst + 1].row0 <= g) ++inst;
                    const GnInstance I = a.bv.inst[inst];
                    row0 = I.row0; ci = I.colidx;
                    const int n = (int)(g - row0);
                    e0 = I.rowptr[n];
                    deg = I.rowptr[n + 1] - e0;
                }
                // ---- aggregation: sequential ascending-column sum (ode_nn_ngraph_sim.py:73)
                const float4 acc = gather_row(a.ip_in, ci, e0, deg, row0, l, lane);
                // ---- SIR derivative + Euler update (explicit _rn ops: no FMA contraction, the
                //      reference rounds after every ATen op; SURVEY Appendix A)
                float4 sn = make_float4(0.f, 0.f, 0.f, 0.f), in_ = sn, rn = sn;
                if (valid) {
                    const size_t off = (size_t)g * H + 4 * l;
                    const float4 ipo = ldg4(a.ip_in + off);
                    // the tensor path replaces the operand tile by its tf32 hi part: re-read S_k (L2 hit)
                    const float4 s = TC ? ldg4(a.y_in + off) : lds4(Xs, sw_off(rr, l));
                    const float4 sp = lds4(SPs, sw_off(rr, l));
                    const float4 iv = ldg4_stream(a.y_in + plane + off);
                    const float4 rv = ldg4_stream(a.y_in + 2 * plane + off);
                    const float nbe = -a.beta[g], ga = a.gamma[g], dt = a.dt;
#define GN_COMP(c)                                                                  \
    {                                                                               \
        const float dS = __fmul_rn(nbe, __fmul_rn(acc.c, sp.c));                    \
        const float dR = __fmul_rn(ga, ipo.c);                                      \
        const float dI = __fsub_rn(-dS, dR);                                        \
        if (MODE == MODE_RHS) { sn.c = dS; in_.c = dI; rn.c = dR; }                 \
        else {                                                                      \
            sn.c = __fadd_rn(s.c, __fmul_rn(dt, dS));                               \
            in_.c = __fadd_rn(iv.c, __fmul_rn(dt, dI));                             \
            rn.c = __fadd_rn(rv.c, __fmul_rn(dt, dR));                              \
        }                                                                           \
    }
                    GN_COMP(x) GN_COMP(y) GN_COMP(z) GN_COMP(w)
#undef GN_COMP
                    stg4_stream(a.y_out + off, sn);
                    stg4_stream(a.y_out + plane + off, in_);
                    stg4_stream(a.y_out + 2 * plane + off, rn);
                    if (MODE == MODE_STEP) sts4(Xs, sw_off(rr, l), in_);      // operand of the next GEMM
                }
                if (MODE == MODE_STEP && a.probs != nullptr)
                    decode_row(sn, in_, rn, W3s, small, l, valid, a.probs + (size_t)(valid ? g : 0) * 3);
            }
            __syncthreads();
        } else if (MODE == MODE_ENCODE) {
            // encoder: C0 = relu(c * w1 + b1) for c in {S0, I0, R0}  (ode_nn_ngraph_sim.py:151-156)
#pragma unroll 1
            for (int it = 0; it < TILE / 32; ++it) {
                const int rr = hw + 32 * it;
                const int64_t g = tile0 + rr;
                const bool valid = g < M;
                float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), i0 = s0, r0 = s0;
                if (valid) {
                    const float* xr = a.x + (size_t)g * a.ldx;
                    const float cs = xr[0], ci_ = xr[1], cr = xr[2];
                    if (l == 0) { a.beta[g] = xr[3]; a.gamma[g] = xr[4]; }
                    const float4 w = *reinterpret_cast<const float4*>(w1s + 4 * l);
                    const float4 b = *reinterpret_cast<const float4*>(b1s + 4 * l);
#define GN_ENC(c)                                                             \
    s0.c = fmaxf(__fadd_rn(__fmul_rn(cs, w.c), b.c), 0.f);                    \
    i0.c = fmaxf(__fadd_rn(__fmul_rn(ci_, w.c), b.c), 0.f);                   \
    r0.c = fmaxf(__fadd_rn(__fmul_rn(cr, w.c), b.c), 0.f);
                    GN_ENC(x) GN_ENC(y) GN_ENC(z) GN_ENC(w)
#undef GN_ENC
                    const size_t off = (size_t)g * H + 4 * l;
                    stg4_stream(a.y_out + off, s0);
                    stg4_stream(a.y_out + plane + off, i0);
                    if (a.hid_r == nullptr) stg4_stream(a.y_out + 2 * plane + off, r0);   // inference carries hid(R) only: no R plane
                }
                sts4(Xs, sw_off(rr, l), i0);
                if (a.probs != nullptr || a.hid_i != nullptr || a.hid_r != nullptr)
                    decode_row(s0, i0, r0, W3s, small, l, valid, a.probs ? a.probs + (size_t)(valid ? g : 0) * 3 : nullptr,
                               a.hid_i ? a.hid_i + (size_t)(valid ? g : 0) * 4 : nullptr,
                               a.hid_r ? a.hid_r + (size_t)(valid ? g : 0) * 4 : nullptr);
            }
            __syncthreads();
        }

        if (MODE != MODE_RHS) {
            if (TC) umma::gemm_sigmoid_tc<FAST>(cx, Xs, SPs, bs, tid);   // I'_{k+1}
            else gemm_sigmoid<FAST>(Xs, Ws, bs, SPs, tid);
            __syncthreads();
            store_tile(a.ip_out, SPs, tile0, M, tid);
            __syncthreads();
        }
    }
    if (TC) {
        umma::fence_before_sync();
        __syncthreads();
        if (tid < 32) umma::tmem_dealloc(cx.tmem, umma::TMEM_COLS);
    }
}


// ---- N4 fast path: the encoder launch of an inference rollout fed by trial descriptors.
// With I0 in {0, 1} on the seeds, S0 = 1 - I0, R0 = 0 (ode_nn_ngraph_sim.py:371-390) every row of the batch is one of TWO
// kinds, so encoder, I'_0 = sigmoid(W enc + b) and the decoder of grid point 0 are evaluated for those two rows only --
// by the SAME device functions the generic encoder launch runs per row (GN_ENC arithmetic, gemm_sigmoid[_tc] on a tile
// whose rows 0 / 1 are enc(0) / enc(1), decode_row), so the result is bitwise the dense path's -- and kept in a small
// table (trials_table_kernel, one CTA). The encoder launch itself becomes a stream of stores (fill_trials_kernel: every row
// as a susceptible row; seed_rows_kernel: the seed rows patched afterwards, O(rows + seeds)): S0, I0, I'_0 rows,
// beta / gamma, hid(I_0), hid(R_0), probs[0]; no dense x block is expanded or read.
// table layout (floats): kind k in {0 = susceptible, 1 = seed}
constexpr int TB_E = 0;        // enc(0)[64], enc(1)[64]
constexpr int TB_IP = 128;     // I'_0 of kind k [64] at TB_IP + 64 k
constexpr int TB_PR = 256;     // probs[0] of kind k [4] at TB_PR + 4 k
constexpr int TB_HI = 264;     // hid(I_0) of kind k [4] at TB_HI + 4 k
constexpr int TB_HR = 272;     // hid(R_0) [4]
constexpr int TB_FLOATS = 276;

template <int VAR>
__global__ void __launch_bounds__(NTHREADS, 1) trials_table_kernel(const gnode_params_t p, float* __restrict__ tbl_g) {
    constexpr bool TC = (VAR & VAR_TC) != 0;
    constexpr bool FAST = (VAR & VAR_FASTSIG) != 0;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Xs = smem + SM_X;
    unsigned char* SPs = smem + SM_SP;
    float* Ws = reinterpret_cast<float*>(smem + SM_W);
    float* bs = reinterpret_cast<float*>(smem + SM_B);
    float* W3s = reinterpret_cast<float*>(smem + SM_W3);
    float* w1s = reinterpret_cast<float*>(smem + SM_W1);
    float* b1s = reinterpret_cast<float*>(smem + SM_B1);
    float* small = reinterpret_cast<float*>(smem + SM_SMALL);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + SM_MBAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + SM_MBAR + 8);
    const int tid = threadIdx.x, l = tid & 15, hw = tid >> 4;

    umma::Ctx cx;
    if (TC) {
        umma::prepare_weights(p.lin_w, smem + SM_W, smem + SM_WLO, tid, NTHREADS);
        if (tid < 32) umma::tmem_alloc(tslot, umma::TMEM_COLS);
        if (tid == 0) umma::mbar_init(mbar, 1);
        umma::fence_before_sync();
    } else {
        for (int i = tid; i < H * H / 4; i += NTHREADS)
            reinterpret_cast<float4*>(Ws)[i] = reinterpret_cast<const float4*>(p.lin_w)[i];
    }
    if (tid < H) { bs[tid] = p.lin_b[tid]; w1s[tid] = p.s1_w[tid]; b1s[tid] = p.s1_b[tid]; }
    if (tid < 4 * H) W3s[tid] = p.l3_w[tid];
    if (tid < 4) { small[tid] = p.l3_b[tid]; small[4 + tid] = p.s2_w[tid]; }
    if (tid == 0) small[8] = p.s2_b[0];
    __syncthreads();
    if (TC) {
        umma::fence_after_sync();
        cx.tmem = *tslot; cx.bar = mbar; cx.phase = 0;
        cx.whi = umma::smem_u32(smem + SM_W); cx.wlo = umma::smem_u32(smem + SM_WLO);
    }
    // the two encoded vectors (this lane's 4 channels): e0 = enc(0), e1 = enc(1), op for op the generic encoder's
    // relu(c * w1 + b1) with explicit _rn ops
    float4 e0, e1;
    {
        const float4 w = *reinterpret_cast<const float4*>(w1s + 4 * l);
        const float4 b = *reinterpret_cast<const float4*>(b1s + 4 * l);
#define GN_ENC2(c)                                                      \
    e0.c = fmaxf(__fadd_rn(__fmul_rn(0.f, w.c), b.c), 0.f);             \
    e1.c = fmaxf(__fadd_rn(__fmul_rn(1.f, w.c), b.c), 0.f);
        GN_ENC2(x) GN_ENC2(y) GN_ENC2(z) GN_ENC2(w)
#undef GN_ENC2
    }
    // operand tile: row 0 = enc(I0 = 0), row 1 = enc(I0 = 1), the other rows zero
    for (int idx = tid; idx < TILE * CHUNKS; idx += NTHREADS) {
        const int rr = idx >> 4;
        sts4(Xs, sw_off(rr, idx & 15), rr == 0 ? e0 : (rr == 1 ? e1 : make_float4(0.f, 0.f, 0.f, 0.f)));
    }
    // decoder of the two kinds of rows (half-warps 0 and 1: both halves of warp 0 take part in the shuffles)
    if (tid < 32) {
        const bool seed = hw == 1;                           // row (S0, I0, R0) = seed ? (0, 1, 0) : (1, 0, 0)
        decode_row(seed ? e0 : e1, seed ? e1 : e0, e0, W3s, small, l, true, tbl_g + TB_PR + 4 * hw, tbl_g + TB_HI + 4 * hw,
                   seed ? nullptr : tbl_g + TB_HR);
        if (tid < 16) {
            *reinterpret_cast<float4*>(tbl_g + TB_E + 4 * l) = e0;
            *reinterpret_cast<float4*>(tbl_g + TB_E + 64 + 4 * l) = e1;
        }
    }
    __syncthreads();
    if (TC) umma::gemm_sigmoid_tc<FAST>(cx, Xs, SPs, bs, tid);
    else gemm_sigmoid<FAST>(Xs, Ws, bs, SPs, tid);
    __syncthreads();
    if (tid < 32) *reinterpret_cast<float4*>(tbl_g + TB_IP + 64 * hw + 4 * l) = lds4(SPs, sw_off(hw, l));
    if (TC) {
        umma::fence_before_sync();
        __syncthreads();
        if (tid < 32) umma::tmem_dealloc(cx.tmem, umma::TMEM_COLS);
    }
}

// every row of the batch written as a susceptible row (a warp per 32 consecutive rows: the three 256-byte rows by
// half-warps, then one thread per row for the scalars)
__global__ void __launch_bounds__(256) fill_trials_kernel(const StepArgs a, const float* __restrict__ tbl,
                                                          const float* __restrict__ beta_i, const float* __restrict__ gamma_i) {
    const int lane = threadIdx.x & 31, l = lane & 15, h = lane >> 4;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    const float4 s0 = *reinterpret_cast<const float4*>(tbl + TB_E + 64 + 4 * l);     // S0 = 1
    const float4 i0 = *reinterpret_cast<const float4*>(tbl + TB_E + 4 * l);          // I0 = 0
    const float4 ip = *reinterpret_cast<const float4*>(tbl + TB_IP + 4 * l);
    const float4 hi = *reinterpret_cast<const float4*>(tbl + TB_HI), hr = *reinterpret_cast<const float4*>(tbl + TB_HR);
    const float4 pr = *reinterpret_cast<const float4*>(tbl + TB_PR);
    const int64_t n_groups = ((int64_t)M + 31) / 32;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t grp = warp0; grp < n_groups; grp += n_warps) {
        const int64_t g0 = grp * 32;
#pragma unroll 4
        for (int j = 0; j < 16; ++j) {
            const int64_t g = g0 + 2 * j + h;
            if (g < M) {
                const size_t off = (size_t)g * H + 4 * l;
                stg4_stream(a.y_out + off, s0);
                stg4_stream(a.y_out + plane + off, i0);
                stg4_stream(a.ip_out + off, ip);
            }
        }
        const int64_t g = g0 + lane;
        if (g < M) {
            const int inst = find_instance(a.bv, g);
            a.beta[g] = beta_i[inst]; a.gamma[g] = gamma_i[inst];
            *reinterpret_cast<float4*>(a.hid_i + (size_t)g * 4) = hi;
            *reinterpret_cast<float4*>(a.hid_r + (size_t)g * 4) = hr;
            if (a.probs != nullptr) {
                float* out = a.probs + (size_t)g * 3;
                out[0] = pr.x; out[1] = pr.y; out[2] = pr.z;
            }
        }
    }
}

// the seed rows (I0 = 1, S0 = 0): a half-warp per seed entry; entries out of range are ignored (as gnode_expand_trials)
__global__ void __launch_bounds__(256) seed_rows_kernel(const StepArgs a, const float* __restrict__ tbl,
                                                        const int32_t* __restrict__ seeds, const int32_t* __restrict__ seed_ptr) {
    const int l = threadIdx.x & 15;
    const int total = seed_ptr[a.bv.n_inst];
    const size_t plane = (size_t)a.bv.M * H;
    const float4 s0 = *reinterpret_cast<const float4*>(tbl + TB_E + 4 * l);          // S0 = 0
    const float4 i0 = *reinterpret_cast<const float4*>(tbl + TB_E + 64 + 4 * l);     // I0 = 1
    const float4 ip = *reinterpret_cast<const float4*>(tbl + TB_IP + 64 + 4 * l);
    const int hw0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 4, n_hw = (gridDim.x * blockDim.x) >> 4;
    for (int e = hw0; e < total; e += n_hw) {
        int lo = 0, hi = a.bv.n_inst - 1;                    // instance that owns seed entry e
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (seed_ptr[mid] <= e) lo = mid; else hi = mid - 1;
        }
        const GnInstance I = a.bv.inst[lo];
        const int s = seeds[e];
        if (s < 0 || s >= I.n) continue;
        const int64_t g = I.row0 + s;
        const size_t off = (size_t)g * H + 4 * l;
        stg4_stream(a.y_out + off, s0);
        stg4_stream(a.y_out + plane + off, i0);
        stg4_stream(a.ip_out + off, ip);
        if (l == 0) {
            *reinterpret_cast<float4*>(a.hid_i + (size_t)g * 4) = *reinterpret_cast<const float4*>(tbl + TB_HI + 4);
            if (a.probs != nullptr) {
                float* out = a.probs + (size_t)g * 3;
                out[0] = tbl[TB_PR + 4]; out[1] = tbl[TB_PR + 5]; out[2] = tbl[TB_PR + 6];
            }
        }
    }
}

// bit g of the bitmap = global row g is a seed row (the bitmap is zeroed before); entries out of range are ignored
__global__ void __launch_bounds__(256) seed_bitmap_kernel(const GnBatchView bv, const int32_t* __restrict__ seeds,
                                                          const int32_t* __restrict__ seed_ptr, uint32_t* __restrict__ bitmap) {
    const int total = seed_ptr[bv.n_inst];
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        int lo = 0, hi = bv.n_inst - 1;                      // instance that owns seed entry e
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (seed_ptr[mid] <= e) lo = mid; else hi = mid - 1;
        }
        const GnInstance I = bv.inst[lo];
        const int s = seeds[e];
        if (s < 0 || s >= I.n) continue;
        const int64_t g = (int64_t)I.row0 + s;
        atomicOr(&bitmap[g >> 5], 1u << (g & 31));
    }
}

// small device helpers of the pipelined step kernels
__device__ __forceinline__ float ex2_approx(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// TMA tensor store of one box (shared memory -> global), bulk-group completion
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, const void* smem_src, int c0, int c1, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%1, %2}], [%3], %4;"
                 ::"l"(tm), "r"(c0), "r"(c1), "r"(umma::smem_u32(smem_src)), "l"(pol) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Fused Euler step, "dual" kernel (the production kernel for MODE_STEP).
//
// ONE CTA of 1024 threads per SM = two independent 512-thread halves, each running a phase pipeline (P1 .. P5
// below) on its own tiles (own operand tiles, CSR slice, mbarrier, TMEM accumulator, named barrier),
// while the W operand tiles, bias and decoder constants are shared. The shared-memory saved by not duplicating
// W pays for the N = 80 operand [W; W3]: the decoder's hidden layer (linear3, ode_nn_ngraph_sim.py:172-176) of
// the S and I blocks comes out of the two GEMMs that the step needs anyway, in accumulator columns 64..67:
//   GEMM1: S_k     [W; W3]^T -> S'_k         and hid(S_k)
//   GEMM2: I_{k+1} [W; W3]^T -> I'_{k+1}     and hid(I_{k+1})  -> HBM side buffer hid_i (16 B / row), read by step k+1
//   hid(R_k): 16 FMAs + a 5-shuffle butterfly per lane in the update phase (R has no GEMM)
// so the launch of step k emits probs[k] (the softmax of its INPUT state, one thread per row) instead of probs[k+1];
// the host decodes the last state with decode_kernel. Further:
//   * the tcgen05.commit mbarrier is awaited with a suspend-time hint (the hardware parks the warps; no spin loop);
//   * no tile starts with a chain of dependent loads: an idle warp resolves the next tile's metadata during the
//     second GEMM, the next tile's S rows are prefetched into registers during the I' store, and the CSR slice,
//     beta/gamma and S rows of a tile are all in flight together;
//   * the gather is specialised by the exact degree (1..12 rows per round trip) and reads an all-zero row for the
//     padding slots instead of predicating; no L2 bulk prefetch (measured: evicted before use on B200).
constexpr int D_THREADS = 1024;
constexpr int D_WHI = 0;
constexpr int D_WLO = umma::WB80_BYTES;
constexpr int D_B = 2 * umma::WB80_BYTES;                 // bias [64]
constexpr int D_W3 = D_B + H * 4;                         // linear3.weight [4][64] fp32 (hidden of R by FFMA)
constexpr int D_SMALL = D_W3 + 4 * H * 4;                 // b3[4], w2[4], b2
constexpr int D_TSLOT = D_SMALL + 64;                     // TMEM base slot
constexpr int D_SHARED = 43008;                           // shared part, rounded up to 1 KB (operand tiles need 1024-B alignment)
static_assert(D_TSLOT + 16 + 64 <= D_SHARED, "shared part overflows (TMEM slot + DStep)");
// up to 4*NB neighbour rows of one row, all loads issued before the first add (one memory round trip)
template <int NB>
__device__ __forceinline__ void gather_block(float4& acc, const float* __restrict__ lane_base, const int* cp, int j0, int deg, uint64_t pol) {
    float4 v[4 * NB];
#pragma unroll
    for (int k = 0; k < 4 * NB; ++k) {
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (j0 + k < deg) v[k] = ldg4_hint(lane_base + (size_t)(unsigned)cp[j0 + k] * H, pol);
    }
#pragma unroll
    for (int k = 0; k < 4 * NB; ++k) add4(acc, v[k]);
}

// Warp-uniform neighbour sum (both half-warps run the trip counts of the larger degree, loads predicated per row);
// sequential ascending-column accumulation; rows with up to 12 neighbours complete in one round trip.
template <int MAXB>       // MAXB = 3: up to 12 rows per round trip, 2: up to 8 (leaves registers for the own-row loads)
__device__ __forceinline__ float4 gather_smem_nb(const float* __restrict__ lane_base, const int* cp, int deg, uint64_t pol) {
    const int degm = max(deg, __shfl_xor_sync(0xffffffffu, deg, 16));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = 0;
    for (; degm - j > 4 * MAXB; j += 8) gather_block<2>(acc, lane_base, cp, j, deg, pol);
    const int rem = degm - j;
    if (MAXB >= 3 && rem > 8) gather_block<3>(acc, lane_base, cp, j, deg, pol);
    else if (rem > 4) gather_block<2>(acc, lane_base, cp, j, deg, pol);
    else if (rem > 0) gather_block<1>(acc, lane_base, cp, j, deg, pol);
    return acc;
}

// K neighbour rows, no predication: slots past the row's degree read the all-zero row `zrow` of the I' buffer
// (adding +0 is exact), so the loads need neither a zero-initialised destination nor a predicate.
// W: weighted, acc += fl(wp[j] v_j); the weights are read after the loads are issued (pad slots: weight 0, row 0)
template <int K, bool W = false>
__device__ __forceinline__ void gather_exact(float4& acc, const float* __restrict__ lane_base, const int* cp, int j0, int deg, int zrow, uint64_t pol,
                                             const float* wp = nullptr) {
    float4 v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int c = (j0 + k < deg) ? cp[j0 + k] : zrow;
        v[k] = ldg4_hint(lane_base + (size_t)(unsigned)c * H, pol);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if (W) v[k] = mul4((j0 + k < deg) ? wp[j0 + k] : 0.f, v[k]);
        add4(acc, v[k]);
    }
}

// Warp-uniform neighbour sum specialised by the pair's larger degree (1..12 in one round trip, longer rows in
// rounds of 8); sequential ascending-column accumulation per row.
__device__ __forceinline__ float4 gather_smem_z(const float* __restrict__ lane_base, const int* cp, int deg, int zrow, uint64_t pol) {
    const int degm = max(deg, __shfl_xor_sync(0xffffffffu, deg, 16));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = 0;
    for (; degm - j > 12; j += 8) gather_exact<8>(acc, lane_base, cp, j, deg, zrow, pol);
    switch (degm - j) {
        case 12: gather_exact<12>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 11: gather_exact<11>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 10: gather_exact<10>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 9: gather_exact<9>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 8: gather_exact<8>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 7: gather_exact<7>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 6: gather_exact<6>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 5: gather_exact<5>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 4: gather_exact<4>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 3: gather_exact<3>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 2: gather_exact<2>(acc, lane_base, cp, j, deg, zrow, pol); break;
        case 1: gather_exact<1>(acc, lane_base, cp, j, deg, zrow, pol); break;
        default: break;
    }
    return acc;
}

// Tile metadata of one pipeline (shared memory): everything the next tile needs, fetched by an otherwise idle warp
// while the current tile's second GEMM runs, so no tile starts with a chain of dependent global loads.
struct DTileMeta {
    const int32_t* rowptr;   // of the owning instance, already offset to the tile's first row
    const int32_t* colidx;   // of the owning instance
    int seq;                 // sequence number (>= n_tiles: no more tiles)
    int tile0;               // first global row
    int nrows;
    int i_row0;              // first global row of the owning instance
    int single;              // whole tile inside one instance
    int ebase, ecnt;         // CSR entry range of the tile (single tiles)
    int inst0;
};

// Compile-time geometry of the pipelined step kernel: NP independent tile pipelines per CTA (2 or 4), each of PT
// threads working on TR-row tiles (TR = UMMA M). The row-per-half-warp loops run 4 passes in both cases.
template <int NP>
struct PipeCfg {
    static constexpr int PT = D_THREADS / NP;              // threads per pipeline (512 / 256)
    static constexpr int TR = 256 / NP;                    // tile rows (128 / 64)
    static constexpr int RSTEP = PT / 16;                  // rows per pass (32 / 16)
    static constexpr int PASS = RSTEP * 128;               // byte offset between the passes' rows in an operand tile
    static constexpr int CAP = 3 * PT;                     // colidx entries staged per tile (3 per thread)
    static constexpr int HUB_DEG = 512;                    // longer rows: loads by the whole pipeline, adds relayed in order
    static constexpr int KBLK = TR * 128;                  // bytes of one K-block (32 fp32) of the A operand
    static constexpr int P_X = 0;                          // A operand hi / parked neighbour sums
    static constexpr int P_L = 2 * KBLK;                   // A operand lo / S' / I' staging
    static constexpr int P_MBAR = 4 * KBLK;                // mbarrier (8) + row-pair counter (4)
    static constexpr int P_META = P_MBAR + 16;             // DTileMeta of the coming tile (48 B)
    static constexpr int P_BG = P_META + 48;               // beta[TR], gamma[TR]
    static constexpr int P_RP = P_BG + 2 * TR * 4;         // rowptr slice [TR + 1] (+pad)
    static constexpr int P_HS = P_RP + TR * 4 + 32;        // hid(S_k) [TR][4]
    static constexpr int P_HR = P_HS + TR * 16;            // hid(R_k) [TR][4]
    static constexpr int P_CI = P_HR + TR * 16;            // colidx slice (instance-local ids) + 64 B over-read pad
    static constexpr int P_BYTES = ((P_CI + CAP * 4 + 64 + 1023) / 1024) * 1024;
    static constexpr int TOTAL = D_SHARED + NP * P_BYTES + 1024;
    static constexpr int TMEM_COLS = 512;                  // one [TR x 160] accumulator per pipeline, 256 columns apart
    static_assert(NP == 2, "the N = 160 accumulators of more than two pipelines do not fit the 512 TMEM columns");
    static_assert(TOTAL + 1024 <= 200704, "stay inside the 196 KB shared-memory carve-out (60 KB of L1 left)");
    static_assert(PT / 4 >= TR, "beta / gamma staging needs a quarter of the pipeline's threads per array");
    static_assert((TR + 2 + TR / 32) * 4 <= TR * 4 + 32, "hub mask lives in the pad behind the rowptr slice");
    // byte offset of the 16-byte chunk c4 of tile row r (canonical UMMA K-major SWIZZLE_128B, two K-blocks)
    static __device__ __forceinline__ int sw(int r, int c4) { return (c4 >> 3) * KBLK + (r << 7) + (((c4 & 7) ^ (r & 7)) << 4); }
};

// Operands of the Euler step in progress (shared memory, written by one thread per step): keeping them out of
// registers matters at the 64-register budget of the 1024-thread CTA.
struct DStep {
    const float* y_in; float* y_out;
    const float* ip_in; float* ip_out;
    float* probs; int* counter;
    const CUtensorMap* tm;
    float dt;
};

template <bool FAST, int NP, bool PERSIST, bool RF>
__global__ void __launch_bounds__(D_THREADS, 1) step_dual_kernel(const __grid_constant__ StepArgs a) {
    using C = PipeCfg<NP>;
    constexpr int PT = C::PT, TR = C::TR, RSTEP = C::RSTEP, PASS = C::PASS;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    const int tid = threadIdx.x;
    const int half = __shfl_sync(0xffffffffu, tid / PT, 0);          // pipeline index, provably warp-uniform
    const int t = tid & (PT - 1), lane = t & 31;
    const int warp = __shfl_sync(0xffffffffu, t >> 5, 0);            // warp index inside the half
    const int l = t & 15, hw = t >> 4;
    unsigned char* hb = smem + D_SHARED + half * C::P_BYTES;
    unsigned char* Xs = hb + C::P_X;
    unsigned char* Ls = hb + C::P_L;
    float* bs = reinterpret_cast<float*>(smem + D_B);
    float* W3s = reinterpret_cast<float*>(smem + D_W3);
    float* small = reinterpret_cast<float*>(smem + D_SMALL);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + D_TSLOT);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(hb + C::P_MBAR);
    int* row_ctr = reinterpret_cast<int*>(hb + C::P_MBAR + 8);
    DTileMeta* meta = reinterpret_cast<DTileMeta*>(hb + C::P_META);
    float* bg_s = reinterpret_cast<float*>(hb + C::P_BG);
    int* rp_s = reinterpret_cast<int*>(hb + C::P_RP);
    float* hs_s = reinterpret_cast<float*>(hb + C::P_HS);
    float* hr_s = reinterpret_cast<float*>(hb + C::P_HR);
    int* ci_s = reinterpret_cast<int*>(hb + C::P_CI);
    unsigned* hub_mask = reinterpret_cast<unsigned*>(rp_s + TR + 2);   // TR / 32 words in the pad behind the rowptr slice
    const int bar_id = 1 + half;
#define HSYNC() umma::bar_sync(bar_id, PT)

    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    const int n_tiles = (NP == 2 ? 1 : 2) * a.bv.n_tiles;          // units of TR rows
    const int off0 = C::sw(hw, l);
    // timing experiments: GNODE_DBG bit 8 (256) = gathered rows without evict_last, bit 9 (512) = streams without evict_first
    const uint64_t pol_keep = (a.dbg & 256) ? l2_policy_evict_normal() : l2_policy_evict_last();
    const uint64_t pol_stream = (a.dbg & 512) ? l2_policy_evict_normal() : l2_policy_evict_first();

    // per-step operands (ordinary launch: the StepArgs fields; persistent rollout: derived from the bases per step)
    // PERSIST = false (one launch per step): read straight from the kernel parameters
    DStep* stp = reinterpret_cast<DStep*>(smem + D_TSLOT + 16);
#define STP(f) (PERSIST ? stp->f : a.f)

    // one thread: draw the next sequence number and resolve its metadata (3 dependent loads of small tables)
    auto fetch_meta = [&](int k) {
        // first tile: static, CTA-major (a batch with fewer tiles than pipelines is spread one tile per SM, and the
        // launch starts without a burst of atomics); later tiles: dynamic ticket
        const int first = (a.dbg & 524288) ? NP * (int)blockIdx.x + half          // A/B: adjacent first tiles per CTA
                                           : (int)blockIdx.x + half * (int)gridDim.x;
        int seq = k == 0 ? first : (STP(counter) ? NP * (int)gridDim.x + atomicAdd(STP(counter), 1) : first + NP * k * (int)gridDim.x);
        if ((a.dbg & 2048) && half != 0) seq = n_tiles;               // timing experiment: one pipeline per SM
        DTileMeta m;
        m.seq = seq; m.rowptr = nullptr; m.colidx = nullptr;
        m.tile0 = 0; m.nrows = 0; m.i_row0 = 0; m.single = 0; m.ebase = 0; m.ecnt = 0; m.inst0 = 0;
        if (seq < n_tiles) {
            // NP == 4: the 128-row tiles of the batch tables are processed as two 64-row halves
            const int tile = a.bv.tile_order[NP == 2 ? seq : (seq >> 1)];
            const int4 tm = NP == 2 ? a.bv.tile_meta[tile] : a.bv.sub_meta[2 * tile + (seq & 1)];   // {ebase, ecnt, inst0, single}
            const GnInstance I = a.bv.inst[tm.z];
            m.tile0 = tile * TILE + (NP == 2 ? 0 : (seq & 1) * TR);
            m.nrows = max(0, min(TR, M - m.tile0));
            m.i_row0 = I.row0; m.single = tm.w; m.ebase = tm.x; m.ecnt = tm.y; m.inst0 = tm.z;
            m.rowptr = I.rowptr + (m.tile0 - I.row0);
            m.colidx = I.colidx;
        }
        *meta = m;
    };

    umma::prepare_weights160(a.p.lin_w, a.p.l3_w, smem + D_WHI, tid, D_THREADS);
    if (tid < 32) umma::tmem_alloc(tslot, C::TMEM_COLS);
    if (t == 0) umma::mbar_init(mbar, 1);
    umma::fence_before_sync();
    if (tid < H) bs[tid] = a.p.lin_b[tid];
    if (tid < 4 * H) W3s[tid] = a.p.l3_w[tid];
    if (tid < 4) { small[tid] = a.p.l3_b[tid]; small[4 + tid] = a.p.s2_w[tid]; }
    if (tid == 0) small[8] = a.p.s2_b[0];
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tslot + (uint32_t)half * 256u;             // this pipeline's [TR x 160] fp32 accumulator
    const uint32_t wop = umma::smem_u32(smem + D_WHI);
    const uint32_t xs_addr = umma::smem_u32(Xs), ls_addr = umma::smem_u32(Ls);
    // epilogue geometry. TR = 128: 16 warps = 4 TMEM lane quarters x 4 blocks of 16 columns, lane == tile row.
    // TR = 64 (measured with tools/umma_m64_probe.cu): rows 16q .. 16q+15 live in lanes 0..15 of quarter q, so 8 warps =
    // 4 quarters x 2 halves of 32 columns, and only lanes 0..15 hold rows.
    const int q = warp & 3, cq = warp >> 2;
    constexpr int NCB = (NP == 2) ? 1 : 2;                            // 16-column blocks per warp
    const bool erow_ok = (NP == 2) || lane < 16;
    const int erow = q * (TR / 4) + lane;                             // tile row this thread owns in the epilogues
    uint32_t phase = 0;
    int kfetch = 1;
    const int n_steps = PERSIST ? max(a.n_steps, 1) : 1;

    // S_k rows of the tile (4 rows x 16 B per thread)
    float4 sreg[4];
    auto load_s = [&](int tile0, int nrows) {
        const float* src = STP(y_in) + (size_t)tile0 * H + (size_t)hw * H + 4 * l;
#pragma unroll
        for (int i = 0; i < 4; ++i)
            sreg[i] = (hw + RSTEP * i < nrows) ? ldg4_hint(src + (size_t)i * RSTEP * H, pol_stream) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tprev = clock64();
#define GN_TICK(i) if (a.tbuf && tid == 0) { const long long tn = clock64(); tacc[i] += tn - tprev; tprev = tn; }
#pragma unroll 1
    for (int step = 0; step < n_steps; ++step) {
    if (PERSIST) {
    if (tid == 0) {
        DStep d;
        d.y_in = a.y_in; d.y_out = a.y_out; d.ip_in = a.ip_in; d.ip_out = a.ip_out;
        d.probs = a.probs; d.counter = a.counter; d.tm = &a.tm_ip_out; d.dt = a.dt;
        if (a.n_steps > 0) {                              // persistent rollout: operands of Euler step ks
            const int ks = a.k0 + step;
            const size_t plane3 = 3 * (size_t)M * H;
            d.y_in = a.traj ? a.traj + (size_t)ks * plane3 : a.st[ks & 1];
            d.y_out = a.traj ? a.traj + (size_t)(ks + 1) * plane3 : a.st[(ks + 1) & 1];
            d.ip_in = a.ipb[ks & 1]; d.ip_out = a.ipb[(ks + 1) & 1];
            const int slot = out_slot_of(a, ks);
            d.probs = (ks > 0 && slot >= 0) ? a.probs_base + (size_t)slot * M * 3 : nullptr;
            d.dt = a.dt_dev ? a.dt_dev[ks] : a.dt;
            d.counter = a.counters ? a.counters + ks + 1 : nullptr;
            d.tm = &a.tm_ipb[(ks + 1) & 1];
        }
        *stp = d;
    }
    __syncthreads();
    }
    if (t == 0) fetch_meta(0);
    kfetch = 1;
    HSYNC();
    for (;;) {
        const DTileMeta m = *meta;                                    // written before the last barrier passed
        if (m.seq >= n_tiles) break;
        const int tile0 = m.tile0, nrows = m.nrows, i_row0 = m.i_row0, ebase = m.ebase;
        const bool single = (m.single & 1) != 0;
        const bool relay = (m.single & 2) != 0 && !(a.dbg & 4194304) && !a.relay_off;   // the tile has isolated hub rows (host cost model)

        // ---- P1: operand tiles for GEMM1 (S_k rows); the tile's CSR slice, beta/gamma -> smem
        //      (every address is known from the metadata: all these loads are in flight together)
        {
            load_s(tile0, nrows);
            int rpv = 0, civ[3] = {0, 0, 0};
            float bgv = 0.f;
            const int ecnt = min(m.ecnt, C::CAP);
            if (single && t <= nrows) rpv = __ldg(m.rowptr + t);
            if (single) {
#pragma unroll
                for (int u = 0; u < 3; ++u) if (t + u * PT < ecnt) civ[u] = __ldg(m.colidx + ebase + t + u * PT);
            }
            if (t >= PT / 2 && t < PT / 2 + nrows) bgv = a.beta[tile0 + t - PT / 2];
            if (t >= 3 * PT / 4 && t < 3 * PT / 4 + nrows) bgv = a.gamma[tile0 + t - 3 * PT / 4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                sts4(Xs, off0 + i * PASS, sreg[i]);                          // raw fp32 = hi operand (the tensor core truncates)
                sts4(Ls, off0 + i * PASS, umma::tf32_trunc_lo4(sreg[i]));
            }
            umma::fence_proxy_async();
            if (t == 0) *row_ctr = 0;
            if (t < TR / 32) hub_mask[t] = 0u;
            if (single && t <= nrows) rp_s[t] = rpv;
            if (single) {
#pragma unroll
                for (int u = 0; u < 3; ++u) if (t + u * PT < ecnt) ci_s[t + u * PT] = civ[u];   // instance-local ids
            }
            if (t >= PT / 2 && t < PT / 2 + nrows) bg_s[t - PT / 2] = bgv;
            if (t >= 3 * PT / 4 && t < 3 * PT / 4 + nrows) bg_s[TR + t - 3 * PT / 4] = bgv;
        }
        HSYNC();                                                                // S1
        GN_TICK(0)
        // ---- P2: GEMM1 ; S' epilogue (+ hid(S_k))
        const bool do_g1 = !(a.dbg & 16), do_g2 = !(a.dbg & 8);       // timing experiments only
        if (do_g1 && t == 0) umma::issue_split_gemm160<TR>(tmem, mbar, wop, xs_addr, ls_addr);
        // rows longer than HUB_DEG are summed by the whole pipeline in P3a (in-order relay): mark them while the GEMM runs
        if (relay && t < nrows && rp_s[t + 1] - rp_s[t] > C::HUB_DEG) atomicOr(&hub_mask[t >> 5], 1u << (t & 31));
        if (do_g1) { umma::mbar_wait_suspend(mbar, phase); phase ^= 1; }        // hardware-suspended wait (no spinning)
        umma::fence_after_sync();
        if (do_g1) {
#pragma unroll
            for (int cb = 0; cb < NCB; ++cb) {
                const int c16 = NCB * cq + cb;                        // 16-column block
                float v[16];
                umma::tmem_ld16_sum(tmem + ((uint32_t)(q * 32) << 16) + 16 * c16, v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * c16 + 4 * j);
                    float4 o;
                    o.x = sigmoid_t<FAST>(v[4 * j + 0] + bb.x); o.y = sigmoid_t<FAST>(v[4 * j + 1] + bb.y);
                    o.z = sigmoid_t<FAST>(v[4 * j + 2] + bb.z); o.w = sigmoid_t<FAST>(v[4 * j + 3] + bb.w);
                    if (erow_ok) sts4(Ls, C::sw(erow, 4 * c16 + j), o);
                }
            }
            if (cq == 0) {
                float hv[4];
                umma::tmem_ld4_sum(tmem + ((uint32_t)(q * 32) << 16) + 64, hv);
                if (erow_ok) *reinterpret_cast<float4*>(hs_s + 4 * erow) = make_float4(hv[0], hv[1], hv[2], hv[3]);
            }
        }
        umma::fence_before_sync();
        HSYNC();                                                                // S2
        GN_TICK(1)
        // ---- P3a: neighbour sums AI -> parked in the (now dead) hi operand tile
        {
            const float* lane_base = STP(ip_in) + (size_t)i_row0 * H + 4 * l;
            const int zrow = M - i_row0;                     // the all-zero row that follows the I' rows
            if (single) {
                // row pairs: strided over the warps when the tile's CSR slice fits the staged window (no hub in the tile:
                // +1.3 % over tickets, same box), shared-memory tickets for hub tiles so that a long row does not leave
                // the other warps idle (GNODE_DBG bit 20: tickets always)
                const bool static_rows = m.ecnt <= C::CAP && (a.dbg & 1048576) == 0;
                int p = 0, sj = 1;
                if (static_rows) p = warp;
                else {
                    if (lane == 0) p = atomicAdd(row_ctr, 1);
                    p = __shfl_sync(0xffffffffu, p, 0);
                }
                while (p < TR / 2) {
                    int pn = 0;
                    if (static_rows) { pn = warp + (PT / 32) * sj; ++sj; }
                    else if (lane == 0) pn = atomicAdd(row_ctr, 1);
                    const int rr = 2 * p + (lane >> 4);
                    int e_rel = 0, deg = 0;
                    if (rr < nrows) { e_rel = rp_s[rr] - ebase; deg = (a.dbg & 2) ? 0 : rp_s[rr + 1] - rp_s[rr]; }
                    if (relay && deg > C::HUB_DEG) deg = 0;                    // hub row: in-order relay below
                    const int over = (e_rel + deg > C::CAP) ? 1 : 0;
                    float4 acc;
                    if (__any_sync(0xffffffffu, over))           // indices beyond the staged slice: same gather on the global list
                        acc = gather_smem_z(lane_base, m.colidx + ebase + e_rel, deg, zrow, pol_keep);
                    else
                        acc = gather_smem_z(lane_base, ci_s + e_rel, deg, zrow, pol_keep);
                    sts4(Xs, C::sw(rr, l), acc);
                    p = static_rows ? pn : __shfl_sync(0xffffffffu, pn, 0);
                }
                // Hub rows (power-law graphs: degrees in the thousands). One half-warp walking the row in rounds of 8 pays a
                // full memory round trip per round (~2.4k cycles under load: 0.5 ms for a 3k-degree row) while the rest of
                // the pipeline waits at the barrier. The sum must stay strictly sequential in ascending column order (the
                // order of the reference's CPU scatter_add_; a hub's ~1e3 sum amplifies any re-association to ~1e-3 in its
                // hidden state), but only the ADDS are serial: every half-warp of the pipeline LOADS 8 consecutive
                // neighbour rows of a 256-neighbour super-round at once, and the running sum is relayed through shared
                // memory from warp to warp in column order (lower half-warp, shuffle, upper half-warp, next warp). Bitwise
                // the same result as the serial walk, one memory round trip per 256 neighbours instead of per 8.
                // Several hub rows in ONE tile are walked concurrently by different warps in the serial scheme, while the relay
                // takes them one after the other (~7k cycles per super-round, mostly hand-offs): gnode_batch_create sets the
                // relay flag of a tile only where its cost model favours it (isolated hubs: 6-10x shorter tile).
                if (relay) {
                    HSYNC();                                             // every ordinary row is parked; the colidx slice is dead
                    volatile float* run = reinterpret_cast<volatile float*>(ci_s);          // [64] running sum
                    uint64_t* hbar = reinterpret_cast<uint64_t*>(ci_s + H);                  // one mbarrier per warp: "your turn"
                    if (t < PT / 32) umma::mbar_init(&hbar[t], 1);
                    HSYNC();
                    constexpr int SR = (PT / 16) * 8;                    // neighbours per super-round
                    int nsr_done = 0;                                    // super-rounds so far (phase bookkeeping)
#pragma unroll 1
                    for (int w = 0; w < TR / 32; ++w) {
                        unsigned mm = hub_mask[w];
                        while (mm) {
                            const int r = 32 * w + __ffs(mm) - 1;
                            mm &= mm - 1;
                            const int dg = rp_s[r + 1] - rp_s[r];
                            const int* cp = m.colidx + rp_s[r];
                            const int n_sr = (dg + SR - 1) / SR;
#pragma unroll 1
                            for (int sr = 0; sr < n_sr; ++sr) {
                                const int j0 = sr * SR + hw * 8;
                                float4 v[8];
#pragma unroll
                                for (int k = 0; k < 8; ++k) {
                                    const int c = (j0 + k < dg) ? cp[j0 + k] : zrow;
                                    v[k] = ldg4_hint(lane_base + (size_t)(unsigned)c * H, pol_keep);
                                }
                                // warp w > 0 is released by warp w - 1 of this super-round, warp 0 by the last warp of the previous one
                                if (warp > 0) umma::mbar_wait(&hbar[warp], (uint32_t)(nsr_done & 1));
                                else if (nsr_done > 0) umma::mbar_wait(&hbar[0], (uint32_t)((nsr_done - 1) & 1));
                                float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (!(sr == 0 && warp == 0)) {
                                    sum.x = run[4 * l + 0]; sum.y = run[4 * l + 1]; sum.z = run[4 * l + 2]; sum.w = run[4 * l + 3];
                                }
                                if (lane < 16) {
#pragma unroll
                                    for (int k = 0; k < 8; ++k) add4(sum, v[k]);
                                }
                                sum.x = __shfl_sync(0xffffffffu, sum.x, l); sum.y = __shfl_sync(0xffffffffu, sum.y, l);
                                sum.z = __shfl_sync(0xffffffffu, sum.z, l); sum.w = __shfl_sync(0xffffffffu, sum.w, l);
                                if (lane >= 16) {
#pragma unroll
                                    for (int k = 0; k < 8; ++k) add4(sum, v[k]);
                                    run[4 * l + 0] = sum.x; run[4 * l + 1] = sum.y; run[4 * l + 2] = sum.z; run[4 * l + 3] = sum.w;
                                    if (sr == n_sr - 1 && warp == PT / 32 - 1) sts4(Xs, C::sw(r, l), sum);
                                }
                                __syncwarp();
                                if (lane == 0) umma::mbar_arrive(&hbar[(warp + 1) & (PT / 32 - 1)]);   // release: orders the stores above
                                ++nsr_done;
                            }
                        }
                    }
                    HSYNC();
                    if (t < PT / 32) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(umma::smem_u32(&hbar[t])) : "memory");
                }
            } else {                                         // tile spans several (small) instances
                int inst = m.inst0;
#pragma unroll 1
                for (int it = 0; it < 4; ++it) {
                    const int rr = hw + RSTEP * it;
                    int row0 = 0, e0 = 0, deg = 0;
                    const int32_t* ci = nullptr;
                    if (rr < nrows) {
                        const int g = tile0 + rr;
                        while (inst + 1 < a.bv.n_inst && a.bv.inst[inst + 1].row0 <= g) ++inst;
                        const GnInstance I = a.bv.inst[inst];
                        row0 = I.row0; ci = I.colidx;
                        e0 = I.rowptr[g - row0];
                        deg = I.rowptr[g - row0 + 1] - e0;
                    }
                    const float4 acc = gather_row(STP(ip_in), ci, e0, deg, row0, l, lane);
                    sts4(Xs, off0 + it * PASS, acc);
                }
            }
        }
        HSYNC();                                                                // S2b: every AI row is parked
        GN_TICK(2)
        // ---- P3b: SIR update, stores; hid(R_k) -> smem; I_{k+1} hi/lo -> operand tiles. The lane's 4 x 4 linear3
        //      weights stay in registers for the four passes (the kernel is bound by LSU wavefronts: re-reading them
        //      from shared memory per row cost 8 of the 55 shared-memory wavefronts per row).
        {
            float4 s, iv, rv, ipo;
            auto load_own = [&](int it) {
                const int rr = hw + RSTEP * it;
                s = make_float4(1.f, 1.f, 1.f, 1.f); iv = s; rv = s; ipo = s;
                if (rr < nrows && !(a.dbg & 4)) {
                    const size_t off = (size_t)(tile0 + rr) * H + 4 * l;
                    s = ldg4_hint(STP(y_in) + off, pol_stream);
                    iv = ldg4_hint(STP(y_in) + plane + off, pol_stream);
                    if (!RF) rv = ldg4_hint(STP(y_in) + 2 * plane + off, pol_stream);
                    ipo = ldg4_hint(STP(ip_in) + off, pol_keep);
                }
            };
            load_own(0);
            const bool dec = !RF && STP(probs) != nullptr && !(a.dbg & 8192);   // RF: hid(R_k) follows from the conserved sum (P4)
            const bool b3 = (l & 8) != 0, b2 = (l & 4) != 0;
            const float4 w30 = *reinterpret_cast<const float4*>(W3s + 0 * H + 4 * l), w31 = *reinterpret_cast<const float4*>(W3s + 1 * H + 4 * l),
                         w32 = *reinterpret_cast<const float4*>(W3s + 2 * H + 4 * l), w33 = *reinterpret_cast<const float4*>(W3s + 3 * H + 4 * l);
#pragma unroll 1
            for (int it = 0; it < 4; ++it) {
                const int rr = hw + RSTEP * it;
                const bool valid = rr < nrows;
                float hv0 = 0.f, hv1 = 0.f, hv2 = 0.f, hv3 = 0.f;
                if (valid) {
                    const size_t off = (size_t)(tile0 + rr) * H + 4 * l;
                    const float4 acc = lds4(Xs, off0 + it * PASS);
                    const float4 sp = lds4(Ls, off0 + it * PASS);
                    const float nbe = -bg_s[rr], ga = bg_s[TR + rr], dt = STP(dt);
                    float4 sn, in_, rn;
#define GN_COMP(c)                                                                  \
    {                                                                               \
        const float dS = __fmul_rn(nbe, __fmul_rn(acc.c, sp.c));                    \
        const float dR = __fmul_rn(ga, ipo.c);                                      \
        const float dI = __fsub_rn(-dS, dR);                                        \
        sn.c = __fadd_rn(s.c, __fmul_rn(dt, dS));                                   \
        in_.c = __fadd_rn(iv.c, __fmul_rn(dt, dI));                                 \
        rn.c = __fadd_rn(rv.c, __fmul_rn(dt, dR));                                  \
    }
                    GN_COMP(x) GN_COMP(y) GN_COMP(z) GN_COMP(w)
#undef GN_COMP
                    if (!(a.dbg & 4096)) {
                    stg4_hint(STP(y_out) + off, sn, pol_stream);
                    stg4_hint(STP(y_out) + plane + off, in_, pol_stream);
                    if (!RF) stg4_hint(STP(y_out) + 2 * plane + off, rn, pol_stream);
                    }
                    sts4(Xs, off0 + it * PASS, in_);             // operand of GEMM2 (raw = hi, truncation split)
                    sts4(Ls, off0 + it * PASS, umma::tf32_trunc_lo4(in_));
                    if (dec) {                                   // partial linear3 products of R_k over this lane's 4 channels
                        const float4 dv = rv;
                        hv0 = dot4(dv, w30); hv1 = dot4(dv, w31); hv2 = dot4(dv, w32); hv3 = dot4(dv, w33);
                    }
                }
                if (it + 1 < 4) load_own(it + 1);
                if (dec) {
                    // halving butterfly over the 16 lanes of the row: lanes 0 / 4 / 8 / 12 end with hid(R)[0 / 1 / 2 / 3]
                    const float a0 = (b3 ? hv2 : hv0) + __shfl_xor_sync(0xffffffffu, b3 ? hv0 : hv2, 8);
                    const float a1 = (b3 ? hv3 : hv1) + __shfl_xor_sync(0xffffffffu, b3 ? hv1 : hv3, 8);
                    float c = (b2 ? a1 : a0) + __shfl_xor_sync(0xffffffffu, b2 ? a0 : a1, 4);
                    c += __shfl_xor_sync(0xffffffffu, c, 2);
                    c += __shfl_xor_sync(0xffffffffu, c, 1);
                    if (valid && (l & 3) == 0) hr_s[4 * rr + (l >> 2)] = c;
                }
            }
        }
        GN_TICK(3)
        float4 hI = make_float4(0.f, 0.f, 0.f, 0.f);     // hid(I_k) of row t (softmax threads): in flight across the barrier
        float4 hRg = hI;                                 // RF: hid(S_0 + I_0 + R_0) of row t (constant over the rollout)
        if (STP(probs) != nullptr && t < nrows) hI = *reinterpret_cast<const float4*>(a.hid_i + (size_t)(tile0 + t) * 4);
        if (RF && STP(probs) != nullptr && t < nrows) hRg = *reinterpret_cast<const float4*>(a.hid_r + (size_t)(tile0 + t) * 4);
        umma::fence_proxy_async();
        HSYNC();                                                                // S3 (every thread has read its copy of *meta)
        GN_TICK(4)
        // ---- P4: GEMM2 || metadata of the next tile (one thread of the idle warp 15) || softmax of the input state ;
        //      I' epilogue (+ hid(I_{k+1}))
        if (do_g2 && t == 0) umma::issue_split_gemm160<TR>(tmem, mbar, wop, xs_addr, ls_addr);
        if (t == PT - 32) fetch_meta(kfetch);
        ++kfetch;
        if (STP(probs) != nullptr && t < nrows) {           // one thread per row: probs[k] = softmax(decoder(S_k, I_k, R_k))
            const float4 hS = *reinterpret_cast<const float4*>(hs_s + 4 * t);
            // RF: R feeds nothing but the decoder's linear3 and S + I + R is conserved channel by channel (dS + dI + dR = 0,
            // ode_nn_ngraph_sim.py:75-77): hid(R_k) = W3 (S_0 + I_0 + R_0) - hid(S_k) - hid(I_k), the first term written once
            // by the encoder launch (4 floats per row), the other two riding on the transform's GEMMs
            const float4 hR = RF ? make_float4((hRg.x - hS.x) - hI.x, (hRg.y - hS.y) - hI.y, (hRg.z - hS.z) - hI.z, (hRg.w - hS.w) - hI.w)
                                 : *reinterpret_cast<const float4*>(hr_s + 4 * t);
            const float4 b3v = *reinterpret_cast<const float4*>(small);
            const float4 w2v = *reinterpret_cast<const float4*>(small + 4);
            const float b2v = small[8];
#define GN_DEC(h) fmaf(w2v.w, fmaxf(h.w + b3v.w, 0.f), fmaf(w2v.z, fmaxf(h.z + b3v.z, 0.f), fmaf(w2v.y, fmaxf(h.y + b3v.y, 0.f), fmaf(w2v.x, fmaxf(h.x + b3v.x, 0.f), b2v))))
            const float oS = GN_DEC(hS), oI = GN_DEC(hI), oR = GN_DEC(hR);
#undef GN_DEC
            const float mx = fmaxf(oS, fmaxf(oI, oR));
            const float eS = ex2_approx((oS - mx) * 1.4426950408889634f), eI = ex2_approx((oI - mx) * 1.4426950408889634f),
                        eR = ex2_approx((oR - mx) * 1.4426950408889634f);
            const float inv = rcp_approx(eS + eI + eR);
            float* pr = STP(probs) + (size_t)(tile0 + t) * 3;
            pr[0] = eS * inv; pr[1] = eI * inv; pr[2] = eR * inv;
        }
        if (do_g2) { umma::mbar_wait_suspend(mbar, phase); phase ^= 1; }
        umma::fence_after_sync();
        if (do_g2) {
#pragma unroll
            for (int cb = 0; cb < NCB; ++cb) {
                const int c16 = NCB * cq + cb;                        // 16-column block
                float v[16];
                umma::tmem_ld16_sum(tmem + ((uint32_t)(q * 32) << 16) + 16 * c16, v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * c16 + 4 * j);
                    float4 o;
                    o.x = sigmoid_t<FAST>(v[4 * j + 0] + bb.x); o.y = sigmoid_t<FAST>(v[4 * j + 1] + bb.y);
                    o.z = sigmoid_t<FAST>(v[4 * j + 2] + bb.z); o.w = sigmoid_t<FAST>(v[4 * j + 3] + bb.w);
                    if (erow_ok) sts4(Ls, C::sw(erow, 4 * c16 + j), o);
                }
            }
            if (cq == 0) {
                float hv[4];
                umma::tmem_ld4_sum(tmem + ((uint32_t)(q * 32) << 16) + 64, hv);
                if (erow_ok && erow < nrows) *reinterpret_cast<float4*>(a.hid_i + (size_t)(tile0 + erow) * 4) = make_float4(hv[0], hv[1], hv[2], hv[3]);
            }
        }
        umma::fence_before_sync();
        umma::fence_proxy_async();                       // the staged tile is read by the TMA (async proxy)
        HSYNC();                                                                // S4 (the next tile's metadata is published)
        GN_TICK(5)
        // ---- P5: I'_{k+1} tile -> HBM. TR = 128: two TMA tensor stores (one per 128-byte K-block of the swizzled staging
        //      tile; rows past M are clipped by the tensor bounds) issued by one thread, no LSU traffic; the tile may be
        //      overwritten once the bulk group has finished READING shared memory. Otherwise: coalesced LSU stores.
        if (NP == 2 && a.use_tma) {
            if (t == 0 && !(a.dbg & 16384)) {
                tma_store_2d((PERSIST ? stp->tm : &a.tm_ip_out), Ls, 0, tile0, pol_stream);
                tma_store_2d((PERSIST ? stp->tm : &a.tm_ip_out), Ls + C::KBLK, 32, tile0, pol_stream);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
        } else {
            float* dst = STP(ip_out) + (size_t)tile0 * H + (size_t)hw * H + 4 * l;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (hw + RSTEP * i < nrows && !(a.dbg & 16384)) stg4_hint(dst + (size_t)i * RSTEP * H, lds4(Ls, off0 + i * PASS), pol_stream);
        }
        HSYNC();                                                                // S5
        GN_TICK(6)
    }
    if (step + 1 < n_steps) {
        // every I' / state row of this step must be complete and visible before any pipeline gathers it: the TMA
        // stores are awaited in full (not only their shared-memory reads), then the grid barrier (its gpu-scope fence
        // also invalidates L1, which still holds lines of the ping-pong buffers from two steps ago)
        if (t == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __threadfence();
        cooperative_groups::this_grid().sync();
    }
    }
    if (a.tbuf && tid == 0)
        for (int i = 0; i < 8; ++i) atomicAdd((unsigned long long*)a.tbuf + i, (unsigned long long)tacc[i]);
#undef GN_TICK
#undef HSYNC
#undef STP
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc(*tslot, C::TMEM_COLS);
}

}  // namespace gnode
#include "gnode_step_stream.cuh"
namespace gnode {

// Decoder + softmax of one stored state (the last grid point of the dual-kernel rollout): probs = softmax over
// {S, I, R} of linearS2(relu(linear3(.)))  (ode_nn_ngraph_sim.py:170-188). Half-warp per row.
__global__ void __launch_bounds__(256) decode_kernel(const float* __restrict__ y, float* __restrict__ probs, int M, const gnode_params_t p,
                                                     const float* __restrict__ hid_r) {
    __shared__ __align__(16) float W3s[4 * H];
    __shared__ float small[16];
    const int tid = threadIdx.x, l = tid & 15;
    for (int i = tid; i < 4 * H; i += 256) W3s[i] = p.l3_w[i];
    if (tid < 4) { small[tid] = p.l3_b[tid]; small[4 + tid] = p.s2_w[tid]; }
    if (tid == 0) small[8] = p.s2_b[0];
    __syncthreads();
    const size_t plane = (size_t)M * H;
    for (int64_t base = ((int64_t)blockIdx.x * 8 + (tid >> 5)) * 2; base < M; base += (int64_t)gridDim.x * 16) {
        const int64_t g = base + ((tid >> 4) & 1);
        const bool valid = g < M;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f), i = s, r = s;
        if (valid) {
            const size_t off = (size_t)g * H + 4 * l;
            s = ldg4_stream(y + off); i = ldg4_stream(y + plane + off);
            if (hid_r == nullptr) r = ldg4_stream(y + 2 * plane + off);
        }
        decode_row(s, i, r, W3s, small, l, valid, probs + (size_t)(valid ? g : 0) * 3, nullptr, nullptr,
                   hid_r ? hid_r + (size_t)(valid ? g : 0) * 4 : nullptr);
    }
}

// 0 = FFMA + accurate sigmoid ... 3 = tcgen05 + MUFU sigmoid; chosen by gnode_set_variant() / GNODE_VARIANT
static int g_variant = -1;
static long long* g_tbuf = nullptr;      // phase-timing accumulators of step_dual_kernel (GNODE_DBG bit 7)

static int current_variant() {
    if (g_variant < 0) {
        const char* e = getenv("GNODE_VARIANT");
        g_variant = e ? (atoi(e) & 3) : GNODE_DEFAULT_VARIANT;
    }
    return g_variant;
}

template <int MODE, int VAR>
static int launch_step_v(const gnode_batch* b, const StepArgs& a, cudaStream_t stream) {
    static bool configured[64] = {false};
    if (!configured[b->device & 63]) {
        GN_CUDA(cudaFuncSetAttribute(step_kernel<MODE, VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL));
        configured[b->device & 63] = true;
    }
    const int grid = std::min(b->n_tiles, 2 * b->sm_count);
    step_kernel<MODE, VAR><<<grid, NTHREADS, SM_TOTAL, stream>>>(a);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

template <bool FAST, int NP, bool RF>
static int launch_step_dual(const gnode_batch* b, const StepArgs& a, cudaStream_t stream) {
    static bool configured[64] = {false};
    if (!configured[b->device & 63]) {
        GN_CUDA(cudaFuncSetAttribute(step_dual_kernel<FAST, NP, false, RF>, cudaFuncAttributeMaxDynamicSharedMemorySize, PipeCfg<NP>::TOTAL));
        GN_CUDA(cudaFuncSetAttribute(step_dual_kernel<FAST, NP, true, RF>, cudaFuncAttributeMaxDynamicSharedMemorySize, PipeCfg<NP>::TOTAL));
        configured[b->device & 63] = true;
    }
    const int units = (NP == 2 ? 1 : 2) * b->n_tiles;
    const int grid = std::min(units, b->sm_count);          // small batches: one tile per SM before a second pipeline is used
    if (a.n_steps > 0) {                                    // persistent rollout: all CTAs co-resident (1 per SM), grid barriers inside
        void* params[] = {const_cast<StepArgs*>(&a)};
        GN_CUDA(cudaLaunchCooperativeKernel((const void*)step_dual_kernel<FAST, NP, true, RF>, dim3(grid), dim3(D_THREADS), params,
                                            (size_t)PipeCfg<NP>::TOTAL, stream));
        gnode::g_launches++;
        return GNODE_OK;
    }
    step_dual_kernel<FAST, NP, false, RF><<<grid, D_THREADS, PipeCfg<NP>::TOTAL, stream>>>(a);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

template <bool FAST, bool RF, int OPT>
static int launch_step_stream(const gnode_batch* b, const StepArgs& a, cudaStream_t stream) {
    static bool configured[64] = {false};
    if (!configured[b->device & 63]) {
        GN_CUDA(cudaFuncSetAttribute(step_stream_kernel<FAST, false, RF, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, StreamCfg::TOTAL));
        GN_CUDA(cudaFuncSetAttribute(step_stream_kernel<FAST, true, RF, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, StreamCfg::TOTAL));
        configured[b->device & 63] = true;
    }
    const int grid = std::min(b->n_tiles, b->sm_count);
    if (a.n_steps > 0) {
        void* params[] = {const_cast<StepArgs*>(&a)};
        GN_CUDA(cudaLaunchCooperativeKernel((const void*)step_stream_kernel<FAST, true, RF, OPT>, dim3(grid), dim3(D_THREADS), params,
                                            (size_t)StreamCfg::TOTAL, stream));
        gnode::g_launches++;
        return GNODE_OK;
    }
    step_stream_kernel<FAST, false, RF, OPT><<<grid, D_THREADS, StreamCfg::TOTAL, stream>>>(a);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

// Euler step 0 of a descriptor-fed inference rollout, fused with the encoder (OPT bit 7 of step_stream_kernel)
template <bool FAST, int OPT>
static int launch_step_stream_zero(const gnode_batch* b, const StepArgs& a, cudaStream_t stream) {
    static bool configured[64] = {false};
    if (!configured[b->device & 63]) {
        GN_CUDA(cudaFuncSetAttribute(step_stream_kernel<FAST, false, true, OPT | 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, StreamCfg::TOTAL));
        configured[b->device & 63] = true;
    }
    const int grid = std::min(b->n_tiles, b->sm_count);
    step_stream_kernel<FAST, false, true, OPT | 128><<<grid, D_THREADS, StreamCfg::TOTAL, stream>>>(a);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

// 5 = pipelined kernel with the TMA-fed S stream (default), 6 = 5 without the deferred store wait, 7 = 5 with 3xTF32 (the
// lo x lo term of the 4-term split product dropped: +2 % speed, per-product error 2^-21 + 2^-21 instead of 2^-21 + 2^-22;
// still inside the 1e-5 bar on every golden, tools/kernel_error_table.py), 3 = the same pipeline with LDG-fed operands
// (round 1; also the fallback when no tensor map can be encoded), 0 = generic
static int g_step_kernel = -1;
static int step_kernel_choice() {
    if (g_step_kernel < 0) { const char* e = getenv("GNODE_STEP_KERNEL"); g_step_kernel = e ? std::min(std::max(atoi(e), 0), 12) : 5; }
    return g_step_kernel;
}

// Inference (no stored trajectory) with the pipelined step kernels carries no R plane at all: R feeds nothing but the
// decoder's linear3 (ode_nn_ngraph_sim.py:172-176) and dS + dI + dR = 0 (:75-77), i.e. S + I + R is conserved channel by
// channel, so hid(R_k) = W3 (S_0 + I_0 + R_0) - hid(S_k) - hid(I_k). The first term is four floats per row written once by
// the encoder launch, the other two ride on the transform's GEMMs: nothing of R is computed, read or written per step.
// (Until round 3 hid(R) was advanced by linearity, hid(R_{k+1}) = hid(R_k) + dt gamma W3 I'_k: 16 FMAs, a butterfly and
// a 32-byte read-modify-write per row and step, 4 % of the step.) 512 of the 2060 algorithmic bytes per node-step are not
// moved; the roofline denominator stays 2060 (SURVEY 8d). GNODE_R_STATE=full / gnode_set_r_state(0) keeps the R plane
// (bitwise the training forward); training always stores R (the decoder's weight gradient needs it).
static int g_r_state = -1;
static int r_state_choice() {
    if (g_r_state < 0) { const char* e = getenv("GNODE_R_STATE"); g_r_state = (e && (!strcmp(e, "full") || !strcmp(e, "0"))) ? 0 : 1; }
    return g_r_state;
}

// persistent (cooperative, one launch per rollout) vs one launch per Euler step: -1 = by batch size (default), 0 / 1 forced
static int g_persistent = -2;
static int persistent_choice() {
    if (g_persistent < -1) { const char* e = getenv("GNODE_PERSISTENT"); g_persistent = e ? (atoi(e) != 0 ? 1 : 0) : -1; }
    return g_persistent;
}

static bool persistent_forced() { return persistent_choice() == 1; }
static int g_hub_relay = 1;

// GNODE_DBG (timing experiments of the older step kernels) is read once per process
static int debug_flags() {
    static const int flags = getenv("GNODE_DBG") ? atoi(getenv("GNODE_DBG")) : 0;
    return flags;
}

// the dual kernel emits probs[k] of its INPUT state and needs the hid_i side buffer (tensor-core variants only)
static bool use_dual() { return (current_variant() & VAR_TC) && step_kernel_choice() >= 3; }

template <int MODE>
static int launch_step(const gnode_batch* b, const StepArgs& a, cudaStream_t stream) {
    const int var = current_variant();
    if (MODE == MODE_STEP && a.edge_w) {                       // weighted neighbour sum: the default step kernel only
        if (!use_dual() || step_kernel_choice() != 5 || a.use_tma != 2) {
            set_error("gnode_rollout_forward_weighted: the weighted neighbour sum runs only on step kernel 5 with TMA-fed "
                      "operands (tensor-core variant, tensor maps available); current step kernel %d, variant %d",
                      step_kernel_choice(), var);
            return GNODE_ERR_UNSUPPORTED;
        }
        const bool fast = (var & VAR_FASTSIG) != 0, rf = a.hid_r != nullptr;
        return fast ? (rf ? launch_step_stream<true, true, 321>(b, a, stream) : launch_step_stream<true, false, 321>(b, a, stream))
                    : (rf ? launch_step_stream<false, true, 321>(b, a, stream) : launch_step_stream<false, false, 321>(b, a, stream));
    }
    if (MODE == MODE_STEP && use_dual()) {
        if (step_kernel_choice() >= 5 && a.use_tma == 2) {      // TMA-fed S stream (6: without the deferred store wait)
            const bool fast = (var & VAR_FASTSIG) != 0, rf = a.hid_r != nullptr;
#define GN_SS(O) (fast ? (rf ? launch_step_stream<true, true, O>(b, a, stream) : launch_step_stream<true, false, O>(b, a, stream)) \
                       : (rf ? launch_step_stream<false, true, O>(b, a, stream) : launch_step_stream<false, false, O>(b, a, stream)))
            if (step_kernel_choice() == 7) return GN_SS(97);              // 3xTF32: the lo x lo term of the split product dropped
#ifdef GNODE_ABLATIONS                                           // A/B and timing-only kernels: tools/ab_bench.py kernel=8..12
            if (fast && rf && a.n_steps == 0) {
                if (step_kernel_choice() == 8) return launch_step_stream<true, true, 69>(b, a, stream);   // no MMAs
                if (step_kernel_choice() == 9) return launch_step_stream<true, true, 73>(b, a, stream);   // no lo-operand pass
                if (step_kernel_choice() == 10) return launch_step_stream<true, true, 17>(b, a, stream);  // round 2h: N = 80 operands, 32 MMAs per GEMM, rna split
                if (step_kernel_choice() == 11) return launch_step_stream<true, true, 1>(b, a, stream);   // N = 160, 4 terms, rna split packed in place
                if (step_kernel_choice() == 12) return launch_step_stream<true, true, 33>(b, a, stream);  // N = 160, 3xTF32, rna split
            }
#endif
            return step_kernel_choice() == 6 ? GN_SS(64) : GN_SS(65);
#undef GN_SS
        }
        if (a.hid_r != nullptr) return (var & VAR_FASTSIG) ? launch_step_dual<true, 2, true>(b, a, stream) : launch_step_dual<false, 2, true>(b, a, stream);
        return (var & VAR_FASTSIG) ? launch_step_dual<true, 2, false>(b, a, stream) : launch_step_dual<false, 2, false>(b, a, stream);
    }
    switch (var) {
        case 0: return launch_step_v<MODE, 0>(b, a, stream);
        case 1: return launch_step_v<MODE, 1>(b, a, stream);
        case 2: return launch_step_v<MODE, 2>(b, a, stream);
        default: return launch_step_v<MODE, 3>(b, a, stream);
    }
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// [rows][64] fp32 row-major, box = 32 floats (one 128-byte swizzle span) x 128 rows
bool encode_rows_map(CUtensorMap* tm, float* base, size_t rows) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc || rows == 0) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)H, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)H * sizeof(float)};
    const cuuint32_t box[2] = {32, (cuuint32_t)TILE};
    const cuuint32_t estr[2] = {1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace gnode

using namespace gnode;

extern "C" int gnode_set_variant(int variant) {
    if (variant < 0 || variant > 3) { set_error("gnode_set_variant: variant must be 0..3"); return GNODE_ERR_ARG; }
    g_variant = variant;
    return GNODE_OK;
}
extern "C" int gnode_get_variant(void) { return current_variant(); }
extern "C" int gnode_set_step_kernel(int kernel) {
#ifdef GNODE_ABLATIONS
    if (kernel >= 8 && kernel <= 12) { g_step_kernel = kernel; return GNODE_OK; }
#endif
    if (kernel < 0 || kernel > 7 || kernel == 1 || kernel == 2 || kernel == 4) { set_error("gnode_set_step_kernel: kernel must be 0, 3, 5, 6 or 7"); return GNODE_ERR_ARG; }
    g_step_kernel = kernel;
    return GNODE_OK;
}
extern "C" int gnode_get_step_kernel(void) { return step_kernel_choice(); }
extern "C" int gnode_set_r_state(int hidden) {
    if (hidden < 0 || hidden > 1) { set_error("gnode_set_r_state: 0 = full R plane, 1 = hidden pre-activations only"); return GNODE_ERR_ARG; }
    g_r_state = hidden;
    return GNODE_OK;
}
extern "C" int gnode_get_r_state(void) { return r_state_choice(); }
extern "C" int gnode_set_persistent(int mode) {
    if (mode < -1 || mode > 1) { set_error("gnode_set_persistent: -1 = by batch size, 0 = one launch per step, 1 = one cooperative launch"); return GNODE_ERR_ARG; }
    g_persistent = mode;
    return GNODE_OK;
}
extern "C" int gnode_get_persistent(void) { return persistent_choice(); }
extern "C" int gnode_set_hub_relay(int on) {
    if (on < 0 || on > 1) { set_error("gnode_set_hub_relay: 0 or 1"); return GNODE_ERR_ARG; }
    g_hub_relay = on;
    return GNODE_OK;
}
extern "C" int gnode_get_hub_relay(void) { return g_hub_relay; }
extern "C" int gnode_debug_phase_cycles(long long* out8) {
    if (!out8) return GNODE_ERR_ARG;
    for (int i = 0; i < 8; ++i) out8[i] = 0;
    if (!g_tbuf) return GNODE_OK;
    GN_CUDA(cudaDeviceSynchronize());
    GN_CUDA(cudaMemcpy(out8, g_tbuf, 64, cudaMemcpyDeviceToHost));
    GN_CUDA(cudaMemset(g_tbuf, 0, 64));
    return GNODE_OK;
}


extern "C" size_t gnode_rollout_workspace_bytes(gnode_batch_t b, int with_traj) {
    if (!b) return 0;
    const size_t M = (size_t)b->M;
    size_t bytes = 2 * align_up(M * sizeof(float), 256);          // beta, gamma
    bytes += 4096;                                                // tile-scheduler counters (one int per launch)
    bytes += 4096;                                                // device copy of the step sizes (persistent rollout, non-uniform grids)
    bytes += 4096;                                                // device copy of the output slots (persistent rollout, irregular selections)
    bytes += 2 * align_up((M + 1) * H * sizeof(float), 256);      // I' ping-pong (+ one all-zero row each)
    bytes += 2 * align_up(M * 4 * sizeof(float), 256);            // hid_i, hid_r: linear3 pre-activations of the I / R block
    if (!with_traj) bytes += 2 * align_up(3 * M * H * sizeof(float), 256);  // state ping-pong
    return bytes;
}

namespace gnode {

// the handle's device must be the calling thread's current device (kernels are launched on it with the handle's pointers)
int check_current_device(const gnode_batch* b, const char* what) {
    int dev = -1;
    GN_CUDA(cudaGetDevice(&dev));
    if (dev != b->device) {
        set_error("%s: the batch lives on device %d but the current device is %d", what, b->device, dev);
        return GNODE_ERR_ARG;
    }
    return GNODE_OK;
}

int make_out_sel(int T, const int32_t* out_steps, int32_t n_out, OutSel* o, const char* what) {
    o->slot.assign((size_t)T, -1);
    if (!out_steps) {
        for (int k = 0; k < T; ++k) o->slot[k] = k;
        o->n_out = T; o->start = 0; o->stride = 1; o->arithmetic = true;
        return GNODE_OK;
    }
    if (n_out < 1 || n_out > T) { set_error("%s: n_out = %d outside [1, T = %d]", what, n_out, T); return GNODE_ERR_ARG; }
    for (int i = 0; i < n_out; ++i) {
        if (out_steps[i] < 0 || out_steps[i] >= T || (i > 0 && out_steps[i] <= out_steps[i - 1])) {
            set_error("%s: out_steps must be strictly ascending grid indices in [0, %d)", what, T);
            return GNODE_ERR_ARG;
        }
        o->slot[out_steps[i]] = i;
    }
    o->n_out = n_out; o->start = out_steps[0];
    o->stride = n_out > 1 ? out_steps[1] - out_steps[0] : 1;
    o->arithmetic = true;
    for (int i = 1; i < n_out; ++i) if (out_steps[i] - out_steps[i - 1] != o->stride) o->arithmetic = false;
    return GNODE_OK;
}

// trial descriptors of a descriptor-fed inference rollout (gnode_rollout_forward_trials) and 2 KB of device scratch
struct TrialDesc {
    const int32_t* seeds; const int32_t* seed_ptr;
    const float* beta; const float* gamma;
    float* table;          // TB_FLOATS floats
    uint32_t* bitmap;      // one bit per row of the batch (fused step 0)
};
constexpr size_t TRIALS_TABLE_BYTES = 4096;

// GNODE_TRIALS_ENCODE (A/B, read once): "dense" keeps the expansion into the dense block + the generic encoder launch,
// "fill" the descriptor-fed encoder launch without fusing Euler step 0 into it; default: both
static int trials_encode_mode() {
    static const int mode = [] {
        const char* e = getenv("GNODE_TRIALS_ENCODE");
        return !e ? 2 : !strcmp(e, "dense") ? 0 : !strcmp(e, "fill") ? 1 : 2;
    }();
    return mode;
}
static bool trials_fast_enabled() { return trials_encode_mode() != 0; }
// the descriptor-fed encoder writes no R plane and no trajectory: inference with R carried as hid(R) only
static bool trials_fast_applies(const float* traj, int32_t T) {
    return trials_fast_enabled() && use_dual() && !traj && T > 1 && r_state_choice() == 1;
}

// head of the trials workspace: the dense [M][GNODE_TRIAL_LDX] block of the expansion path, or the two-row table
static size_t trials_block_bytes(const gnode_batch* b) {
    static_assert(TB_FLOATS * sizeof(float) <= TRIALS_TABLE_BYTES, "table");
    return align_up(std::max((size_t)b->M * GNODE_TRIAL_LDX * sizeof(float), TRIALS_TABLE_BYTES + ((size_t)b->M + 31) / 32 * 4), 256);
}

template <int VAR>
static int launch_trials_table(const gnode_batch* b, const gnode_params_t& p, float* table, cudaStream_t stream) {
    static bool configured[64] = {false};
    if (!configured[b->device & 63]) {
        GN_CUDA(cudaFuncSetAttribute(trials_table_kernel<VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL));
        configured[b->device & 63] = true;
    }
    trials_table_kernel<VAR><<<1, NTHREADS, SM_TOTAL, stream>>>(p, table);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

static int launch_trials_table_v(const gnode_batch* b, const gnode_params_t& p, float* table, cudaStream_t stream) {
    switch (current_variant()) {
        case 0: return launch_trials_table<0>(b, p, table, stream);
        case 1: return launch_trials_table<1>(b, p, table, stream);
        case 2: return launch_trials_table<2>(b, p, table, stream);
        default: return launch_trials_table<3>(b, p, table, stream);
    }
}

static int launch_encode_trials(const gnode_batch* b, const StepArgs& a, const TrialDesc& td, cudaStream_t stream) {
    const int64_t groups = ((int64_t)b->M + 31) / 32;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((groups + 7) / 8, (int64_t)b->sm_count * 8));
    fill_trials_kernel<<<grid, 256, 0, stream>>>(a, td.table, td.beta, td.gamma);
    GN_LAUNCH_CHECK();
    seed_rows_kernel<<<std::max(1, std::min(b->n_inst, b->sm_count * 8)), 256, 0, stream>>>(a, td.table, td.seeds, td.seed_ptr);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

static int rollout_forward_impl(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p, int32_t T,
                                const float* dt_host, const OutSel& sel, float* traj, float* aux, int32_t* aux_filled,
                                float* probs, void* workspace, size_t workspace_bytes, cudaStream_t stream,
                                const TrialDesc* td = nullptr, const float* edge_w = nullptr) {
    if (aux_filled) *aux_filled = 0;
    if (edge_w && (td || !use_dual() || step_kernel_choice() != 5 || tensor_map_encoder() == nullptr)) {
        set_error("gnode_rollout_forward_weighted: the weighted neighbour sum runs only on step kernel 5 (current: %d) with "
                  "the tensor-core variant (current: %d) and tensor maps (%s)", step_kernel_choice(), current_variant(),
                  tensor_map_encoder() ? "available" : "not available on this driver");
        return GNODE_ERR_UNSUPPORTED;
    }
    if (workspace_bytes < gnode_rollout_workspace_bytes(b, traj != nullptr)) {
        set_error("gnode_rollout_forward: workspace too small (%zu < %zu)", workspace_bytes,
                  gnode_rollout_workspace_bytes(b, traj != nullptr));
        return GNODE_ERR_ARG;
    }
    int rc = check_current_device(b, "gnode_rollout_forward");
    if (rc) return rc;
    const size_t M = (size_t)b->M;
    unsigned char* ws = (unsigned char*)workspace;
    float* beta = (float*)ws;  ws += align_up(M * sizeof(float), 256);
    float* gamma = (float*)ws; ws += align_up(M * sizeof(float), 256);
    int* counters = (int*)ws;  ws += 4096;
    float* dt_dev = (float*)ws; ws += 4096;
    int* slot_dev = (int*)ws; ws += 4096;
    GN_CUDA(cudaMemsetAsync(counters, 0, 4096, stream));
    float* ip[2];
    ip[0] = (float*)ws; ws += align_up((M + 1) * H * sizeof(float), 256);
    ip[1] = (float*)ws; ws += align_up((M + 1) * H * sizeof(float), 256);
    GN_CUDA(cudaMemsetAsync(ip[0] + M * H, 0, H * sizeof(float), stream));      // row M: the zero row padded gather slots read
    GN_CUDA(cudaMemsetAsync(ip[1] + M * H, 0, H * sizeof(float), stream));
    float* hid_i = (float*)ws; ws += align_up(M * 4 * sizeof(float), 256);
    float* hid_r = (float*)ws; ws += align_up(M * 4 * sizeof(float), 256);
    float* st[2] = {nullptr, nullptr};
    if (!traj) {
        st[0] = (float*)ws; ws += align_up(3 * M * H * sizeof(float), 256);
        st[1] = (float*)ws;
    }
    auto state = [&](int k) -> float* { return traj ? traj + (size_t)k * 3 * M * H : st[k & 1]; };
    auto out = [&](int k) -> float* { return sel.slot[k] >= 0 ? probs + (size_t)sel.slot[k] * M * 3 : nullptr; };
    // Auxiliary storage for the reverse sweep (training, stream kernel): the I' plane of EVERY grid point stays in
    // aux[k][0] (the step writes I'_{k+1} anyway: no extra traffic) and AI_k = A I'_k goes to aux[k][1] (256 B per row
    // and step more), so that the reverse sweep neither recomputes I' nor repeats the neighbour gather of A I'.
    const size_t Mr = (M + TILE - 1) / TILE * TILE, Ms = Mr + 1;
    const size_t aux_slot = 2 * Ms * H;
    const bool aux_on = aux && traj && T > 1 && use_dual() && step_kernel_choice() >= 5 && !(debug_flags() & 32768) &&
                        tensor_map_encoder() != nullptr;
    if (aux_on) {
        for (int k = 0; k < 2; ++k) ip[k] = nullptr;
        // the all-zero rows (index Mr of every I' plane)
        GN_CUDA(cudaMemset2DAsync(aux + Mr * H, aux_slot * sizeof(float), 0, H * sizeof(float), (size_t)T, stream));
    }
    auto ipk = [&](int k) -> float* { return aux_on ? aux + (size_t)k * aux_slot : ip[k & 1]; };

    StepArgs a{};
    a.bv = gn_view(b);
    a.p = *p;
    a.beta = beta; a.gamma = gamma;
    a.x = x; a.ldx = ldx;
    a.y_in = nullptr; a.ip_in = nullptr;
    a.y_out = state(0); a.ip_out = ipk(0);
    a.ai_out = nullptr; a.aux = nullptr; a.aux_slot = (int64_t)aux_slot; a.ip_zrow = aux_on ? (int)Mr : (int)M;
    a.probs = out(0); a.dt = 0.f;
    a.out_slot = nullptr; a.out_start = sel.start; a.out_stride = sel.stride; a.n_out = sel.n_out;
    a.dbg = debug_flags();
    a.relay_off = g_hub_relay ? 0 : 1;
    a.edge_w = edge_w; a.inst_e0 = b->d_inst_e0;
    a.tbuf = nullptr;
    if (a.dbg & 128) {
        if (!g_tbuf) { GN_CUDA(cudaMalloc(&g_tbuf, 64)); GN_CUDA(cudaMemset(g_tbuf, 0, 64)); }
        a.tbuf = g_tbuf;
    }
    a.counter = (a.dbg & 64) ? nullptr : counters;
    const bool dual = use_dual();
    const bool stream_kernel = dual && step_kernel_choice() >= 5;
    a.use_tma = 0;
    CUtensorMap tm_ip[2];
    const bool have_tma = dual && !(a.dbg & 32768) &&
                          (aux_on ? encode_rows_map(&tm_ip[0], aux, (size_t)T * 2 * Ms)        // persistent rollout: one map over the buffer
                                  : (encode_rows_map(&tm_ip[0], ip[0], M) && encode_rows_map(&tm_ip[1], ip[1], M)));
    a.hid_i = dual ? hid_i : nullptr;
    const bool rfree = dual && !traj && T > 1 && r_state_choice() == 1;
    a.hid_r = rfree ? hid_r : nullptr;
    // Persistent rollout: ONE cooperative launch runs all T-1 Euler steps (see below); decided here because the
    // descriptor-fed encoder fuses Euler step 0 only into the launch-per-step form
    const int persistent_mode = persistent_choice();
    const bool persistent_ok = persistent_mode < 0 ? b->n_tiles <= 32 * b->sm_count : persistent_mode != 0;
    int coop = 0;
    if (dual && persistent_ok && T > 2 && T - 1 <= 1023 && !(a.dbg & 64) && (!aux_on || (size_t)T * 2 * Ms < ((size_t)1 << 31)))
        GN_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, b->device));
    bool step0_fused = false;
    if (td) {                                         // descriptor-fed: two kinds of rows
        if (!rfree) { set_error("gnode_rollout_forward_trials: internal: descriptor encoder without hid(R) state"); return GNODE_ERR_ARG; }
        rc = launch_trials_table_v(b, a.p, td->table, stream);
        if (rc) return rc;
        const int sk = step_kernel_choice();
        step0_fused = trials_encode_mode() == 2 && !coop && stream_kernel && have_tma && (sk == 5 || sk == 7);
        if (step0_fused) {
            // encoder + Euler step 0 in one launch: y_0 and I'_0 are never written (step_stream_kernel, OPT bit 7)
            GN_CUDA(cudaMemsetAsync(td->bitmap, 0, (M + 31) / 32 * 4, stream));
            seed_bitmap_kernel<<<std::max(1, std::min(b->n_inst, b->sm_count * 8)), 256, 0, stream>>>(a.bv, td->seeds, td->seed_ptr, td->bitmap);
            GN_LAUNCH_CHECK();
            a.z_tbl = td->table; a.z_bitmap = td->bitmap; a.z_beta = td->beta; a.z_gamma = td->gamma;
            a.y_in = nullptr; a.ip_in = nullptr; a.y_out = state(1); a.ip_out = ipk(1);
            a.use_tma = 2; a.tm_ip_out = tm_ip[1];
            a.probs = out(0); a.dt = dt_host[0];
            a.n_steps = 0; a.k0 = 0;
            a.counter = (a.dbg & 64) ? nullptr : counters + 1;
            const bool fast = (current_variant() & VAR_FASTSIG) != 0;
            rc = sk == 7 ? (fast ? launch_step_stream_zero<true, 97>(b, a, stream) : launch_step_stream_zero<false, 97>(b, a, stream))
                         : (fast ? launch_step_stream_zero<true, 65>(b, a, stream) : launch_step_stream_zero<false, 65>(b, a, stream));
        } else
            rc = launch_encode_trials(b, a, *td, stream);   // a stream of stores: y_0, I'_0, probs[0], hid(I_0), hid(R_0)
    } else
        rc = launch_step<MODE_ENCODE>(b, a, stream);  // y_0, I'_0, probs[0] (+ hid(I_0))
    if (rc) return rc;
    a.n_steps = 0; a.k0 = 0;
    // Persistent rollout: ONE cooperative launch runs all T-1 Euler steps with a grid barrier between them (no per-step
    // launch, weight operands and TMEM stay resident).
    // Default: batches of up to 16 tiles per pipeline (~600k rows), where a launch per step costs >= 2 % ; larger batches
    // keep one launch per step (the persistent variant reads its per-step operands from shared memory: -1 % there).
    // gnode_set_persistent / GNODE_PERSISTENT=1 / 0 forces it on / off.
    if (coop) {
        // step sizes / output slots: carried in the kernel parameters when the grid is uniform and the selection an
        // arithmetic progression (the reference's np.arange grid and int(i/deltaT) selection); otherwise copied to the
        // workspace (a pageable source makes that copy block the host until it is staged)
        bool uniform = true;
        for (int k = 1; k + 1 < T; ++k) if (dt_host[k] != dt_host[0]) uniform = false;
        a.dt_dev = nullptr;
        if (!uniform) {
            GN_CUDA(cudaMemcpyAsync(dt_dev, dt_host, sizeof(float) * (size_t)(T - 1), cudaMemcpyHostToDevice, stream));
            a.dt_dev = dt_dev;
        }
        if (!sel.arithmetic) {
            GN_CUDA(cudaMemcpyAsync(slot_dev, sel.slot.data(), sizeof(int) * (size_t)T, cudaMemcpyHostToDevice, stream));
            a.out_slot = slot_dev;
        }
        a.n_steps = T - 1; a.k0 = 0;
        a.traj = traj; a.st[0] = st[0]; a.st[1] = st[1];
        a.ipb[0] = ip[0]; a.ipb[1] = ip[1];
        a.aux = aux_on ? aux : nullptr;
        a.probs_base = probs; a.counters = counters;
        a.use_tma = have_tma ? 1 : 0;
        if (have_tma) { a.tm_ipb[0] = tm_ip[0]; a.tm_ipb[1] = tm_ip[1]; }
        if (have_tma && stream_kernel) {                  // S_k tiles by TMA: maps over the S planes (or the whole trajectory)
            const bool ok = traj ? encode_rows_map(&a.tm_sp[0], traj, (size_t)T * 3 * M)
                                 : (encode_rows_map(&a.tm_sp[0], st[0], M) && encode_rows_map(&a.tm_sp[1], st[1], M));
            if (ok && (!traj || (size_t)T * 3 * M < ((size_t)1 << 31))) a.use_tma = 2;
        }
        a.y_in = state(0); a.y_out = state(1); a.ip_in = ipk(0); a.ip_out = ipk(1); a.probs = nullptr; a.dt = dt_host[0];
        if (aux_on && a.use_tma != 2) { set_error("gnode_rollout_forward: tensor maps over the auxiliary buffer could not be encoded"); return GNODE_ERR_CUDA; }
        rc = launch_step<MODE_STEP>(b, a, stream);
        if (rc == GNODE_ERR_CUDA && !persistent_forced()) {
            // e.g. cudaErrorCooperativeLaunchTooLarge under MPS / green-context SM limits: clear it, one launch per step
            (void)cudaGetLastError();
            coop = 0;
            a.n_steps = 0;
        } else if (rc) return rc;
    }
    a.aux = nullptr;
    if (!coop)
    for (int k = step0_fused ? 1 : 0; k + 1 < T; ++k) {
        a.y_in = state(k); a.y_out = state(k + 1);
        a.ip_in = ipk(k); a.ip_out = ipk(k + 1);
        a.ai_out = aux_on ? ipk(k) + Ms * H : nullptr;
        a.use_tma = 0;
        if (have_tma && !aux_on) { a.use_tma = 1; a.tm_ip_out = tm_ip[(k + 1) & 1]; }
        if (have_tma && aux_on && encode_rows_map(&a.tm_ip_out, ipk(k + 1), M)) a.use_tma = 1;     // rows past M clipped
        if (a.use_tma == 1 && stream_kernel && encode_rows_map(&a.tm_s_in, state(k), M)) a.use_tma = 2;
        if (aux_on && a.use_tma != 2) { set_error("gnode_rollout_forward: tensor maps over the auxiliary buffer could not be encoded"); return GNODE_ERR_CUDA; }
        // dual kernel: step k decodes its input state k (k = 0 is the encoder's); the others decode their output
        a.probs = dual ? (k > 0 ? out(k) : nullptr) : out(k + 1);
        a.dt = dt_host[k];
        a.counter = (k + 1 < 1024 && !(a.dbg & 64)) ? counters + (k + 1) : nullptr;
        rc = launch_step<MODE_STEP>(b, a, stream);
        if (rc) return rc;
    }
    if (dual && T > 1 && out(T - 1)) {                     // the last grid state
        const int grid = (int)std::min<int64_t>(((int64_t)M + 15) / 16, (int64_t)b->sm_count * 16);
        decode_kernel<<<grid, 256, 0, stream>>>(state(T - 1), out(T - 1), (int)M, *p, a.hid_r);
        GN_LAUNCH_CHECK();
    }
    if (aux_filled) *aux_filled = aux_on ? 1 : 0;
    return GNODE_OK;
}

// ---- N4: compact trial descriptors -> the five live columns of the reference's dense input block -----------------
// x[r] = {S0, I0, R0, beta, gamma} with I0 = 1 on the seeds, S0 = 1 - I0, R0 = 0 (ode_nn_ngraph_sim.py:371-390)
__global__ void __launch_bounds__(256) expand_trials_kernel(const GnBatchView bv, const float* __restrict__ beta,
                                                            const float* __restrict__ gamma, float* __restrict__ x, int64_t ldx) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < bv.M; r += (int64_t)gridDim.x * blockDim.x) {
        const int i = find_instance(bv, r);
        float* xr = x + (size_t)r * ldx;
        xr[0] = 1.f; xr[1] = 0.f; xr[2] = 0.f; xr[3] = beta[i]; xr[4] = gamma[i];
    }
}
__global__ void __launch_bounds__(256) seed_trials_kernel(const GnBatchView bv, const int32_t* __restrict__ seeds,
                                                          const int32_t* __restrict__ seed_ptr, float* __restrict__ x, int64_t ldx) {
    const int total = seed_ptr[bv.n_inst];
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        int lo = 0, hi = bv.n_inst - 1;                      // instance that owns seed entry e
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (seed_ptr[mid] <= e) lo = mid; else hi = mid - 1;
        }
        const GnInstance I = bv.inst[lo];
        const int s = seeds[e];
        if (s < 0 || s >= I.n) continue;                     // out of range: ignored (the host wrapper validates)
        float* xr = x + (size_t)(I.row0 + s) * ldx;
        xr[0] = 0.f; xr[1] = 1.f;
    }
}

}  // namespace gnode

extern "C" int gnode_rollout_forward(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                     int32_t T, const float* dt_host, float* traj, float* probs,
                                     void* workspace, size_t workspace_bytes, void* stream_) {
    return gnode_rollout_forward_sel(b, x, ldx, p, T, dt_host, nullptr, 0, traj, probs, workspace, workspace_bytes, stream_);
}

extern "C" int gnode_rollout_forward_sel(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                         int32_t T, const float* dt_host, const int32_t* out_steps, int32_t n_out,
                                         float* traj, float* probs, void* workspace, size_t workspace_bytes, void* stream_) {
    if (!b || !x || !p || !probs || !workspace || T < 1 || ldx < 5 || (T > 1 && !dt_host)) {
        set_error("gnode_rollout_forward: bad arguments (T=%d ldx=%lld)", T, (long long)ldx);
        return GNODE_ERR_ARG;
    }
    OutSel sel;
    int rc = make_out_sel(T, out_steps, n_out, &sel, "gnode_rollout_forward_sel");
    if (rc) return rc;
    return rollout_forward_impl(b, x, ldx, p, T, dt_host, sel, traj, nullptr, nullptr, probs, workspace, workspace_bytes, (cudaStream_t)stream_);
}

extern "C" size_t gnode_rollout_aux_bytes(gnode_batch_t b, int32_t T) {
    if (!b || T < 1) return 0;
    const size_t Mr = ((size_t)b->M + TILE - 1) / TILE * TILE;
    return (size_t)T * 2 * (Mr + 1) * H * sizeof(float);
}

extern "C" int gnode_rollout_forward_aux(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                         int32_t T, const float* dt_host, const int32_t* out_steps, int32_t n_out,
                                         float* traj, float* aux, int32_t* aux_filled, float* probs, void* workspace,
                                         size_t workspace_bytes, void* stream_) {
    if (!b || !x || !p || !probs || !workspace || T < 1 || ldx < 5 || (T > 1 && !dt_host) || (aux && (!traj || !aux_filled))) {
        set_error("gnode_rollout_forward_aux: bad arguments (T=%d ldx=%lld)", T, (long long)ldx);
        return GNODE_ERR_ARG;
    }
    OutSel sel;
    int rc = make_out_sel(T, out_steps, n_out, &sel, "gnode_rollout_forward_aux");
    if (rc) return rc;
    return rollout_forward_impl(b, x, ldx, p, T, dt_host, sel, traj, aux, aux_filled, probs, workspace, workspace_bytes, (cudaStream_t)stream_);
}

extern "C" int gnode_rollout_forward_weighted(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                              int32_t T, const float* dt_host, const int32_t* out_steps, int32_t n_out,
                                              float* traj, float* aux, int32_t* aux_filled, float* probs,
                                              const float* edge_w, void* workspace, size_t workspace_bytes, void* stream_) {
    if (!b || !x || !p || !probs || !workspace || T < 1 || ldx < 5 || (T > 1 && !dt_host) || (aux && (!traj || !aux_filled))) {
        set_error("gnode_rollout_forward_weighted: bad arguments (T=%d ldx=%lld)", T, (long long)ldx);
        return GNODE_ERR_ARG;
    }
    OutSel sel;
    int rc = make_out_sel(T, out_steps, n_out, &sel, "gnode_rollout_forward_weighted");
    if (rc) return rc;
    return rollout_forward_impl(b, x, ldx, p, T, dt_host, sel, traj, aux, aux_filled, probs, workspace, workspace_bytes,
                                (cudaStream_t)stream_, nullptr, edge_w);
}

extern "C" int gnode_expand_trials(gnode_batch_t b, const int32_t* seeds, const int32_t* seed_ptr, const float* beta,
                                   const float* gamma, float* x, int64_t ldx, void* stream_) {
    if (!b || !seeds || !seed_ptr || !beta || !gamma || !x || ldx < 5) {
        set_error("gnode_expand_trials: bad arguments (ldx=%lld)", (long long)ldx);
        return GNODE_ERR_ARG;
    }
    int rc = check_current_device(b, "gnode_expand_trials");
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int grid = (int)std::min<int64_t>((b->M + 255) / 256, (int64_t)b->sm_count * 8);
    expand_trials_kernel<<<grid, 256, 0, stream>>>(gn_view(b), beta, gamma, x, ldx);
    GN_LAUNCH_CHECK();
    seed_trials_kernel<<<std::max(1, std::min(b->n_inst, b->sm_count * 8)), 256, 0, stream>>>(gn_view(b), seeds, seed_ptr, x, ldx);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

extern "C" size_t gnode_rollout_trials_workspace_bytes(gnode_batch_t b, int with_traj) {
    if (!b) return 0;
    return gnode_rollout_workspace_bytes(b, with_traj) + gnode::trials_block_bytes(b);
}

extern "C" int gnode_rollout_forward_trials(gnode_batch_t b, const int32_t* seeds, const int32_t* seed_ptr,
                                            const float* beta, const float* gamma, const gnode_params_t* p, int32_t T,
                                            const float* dt_host, const int32_t* out_steps, int32_t n_out, float* traj,
                                            float* probs, void* workspace, size_t workspace_bytes, void* stream_) {
    if (!b || !workspace || workspace_bytes < gnode_rollout_trials_workspace_bytes(b, traj != nullptr)) {
        set_error("gnode_rollout_forward_trials: workspace missing or too small");
        return GNODE_ERR_ARG;
    }
    const size_t xbytes = gnode::trials_block_bytes(b);
    float* x = (float*)workspace;
    if (gnode::trials_fast_applies(traj, T)) {
        // every row is one of two kinds: no dense block, the encoder launch is a stream of stores (trials_table_kernel)
        if (!seeds || !seed_ptr || !beta || !gamma || !p || !probs || T < 1 || !dt_host) {
            set_error("gnode_rollout_forward_trials: bad arguments (T=%d)", T);
            return GNODE_ERR_ARG;
        }
        gnode::OutSel sel;
        int rc = gnode::make_out_sel(T, out_steps, n_out, &sel, "gnode_rollout_forward_trials");
        if (rc) return rc;
        // the table and the seed bitmap live where the dense block would
        const gnode::TrialDesc td{seeds, seed_ptr, beta, gamma, x, (uint32_t*)((unsigned char*)workspace + gnode::TRIALS_TABLE_BYTES)};
        return gnode::rollout_forward_impl(b, nullptr, 0, p, T, dt_host, sel, traj, nullptr, nullptr, probs,
                                           (unsigned char*)workspace + xbytes, workspace_bytes - xbytes, (cudaStream_t)stream_, &td);
    }
    int rc = gnode_expand_trials(b, seeds, seed_ptr, beta, gamma, x, GNODE_TRIAL_LDX, stream_);
    if (rc) return rc;
    return gnode_rollout_forward_sel(b, x, GNODE_TRIAL_LDX, p, T, dt_host, out_steps, n_out, traj, probs,
                                     (unsigned char*)workspace + xbytes, workspace_bytes - xbytes, stream_);
}

extern "C" int gnode_odefunc_eval(gnode_batch_t b, const float* y, const float* beta, const float* gamma,
                                  const gnode_params_t* p, float* dy, float* scratch, void* stream_) {
    if (!b || !y || !beta || !gamma || !p || !dy || !scratch) {
        set_error("gnode_odefunc_eval: null argument");
        return GNODE_ERR_ARG;
    }
    if (int rc = check_current_device(b, "gnode_odefunc_eval")) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    StepArgs a{};
    a.bv = gn_view(b);
    a.p = *p;
    a.beta = const_cast<float*>(beta); a.gamma = const_cast<float*>(gamma);
    a.x = nullptr; a.ldx = 0; a.probs = nullptr; a.hid_i = nullptr; a.hid_r = nullptr; a.dt = 0.f; a.counter = nullptr; a.dbg = 0; a.tbuf = nullptr; a.use_tma = 0; a.n_steps = 0;
    a.y_in = y; a.y_out = nullptr; a.ip_in = nullptr; a.ip_out = scratch;
    int rc = launch_step<MODE_IP>(b, a, stream);       // I' of every row first (grid-wide dependency)
    if (rc) return rc;
    a.ip_in = scratch; a.ip_out = nullptr; a.y_out = dy;
    return launch_step<MODE_RHS>(b, a, stream);
}
