// Backward: reverse sweep over the stored trajectory (SURVEY 8a: a10; 3C).
//
// Replaces torchdiffeq's OdeintAdjointMethod.backward (entered from loss.backward(),
// ode_nn_ngraph_sim.py:245) plus autograd of the encoder (:151-156) and decoder (:172-187).
//
// With f the right-hand side (ode_nn_ngraph_sim.py:58-96) and cotangent a = (aS, aI, aR):
//   q    = aI - aS
//   gAI  = beta * q * S'                      gS' = beta * q * AI
//   gI'  = A^T gAI + gamma * (aR - aI)
//   gzS  = gS' * S'(1-S')                     gzI = gI' * I'(1-I')
//   vS   = gzS W ; vI = gzI W ; vR = 0        (VJP wrt the state)
//   vW   = gzS^T S + gzI^T I ; vb = sum_rows(gzS + gzI)
// grad_mode ADJOINT  (torchdiffeq semantics, what the reference trains with):
//   for j = T-1 .. 1:  a += D(y_j, gP_j);  a, g_theta += dt_{j-1} * VJP(y_j; a);   finally a += D(y_0, gP_0)
// grad_mode DISCRETE (exact gradient of the Euler loop):
//   a = D(y_{T-1}, gP_{T-1});  for j = T-2 .. 0:  (v, v_theta) = VJP(y_j; a);  a += D(y_j, gP_j) + dt_j v
// where D(y, gP) is the decoder+softmax backward. Then the encoder backward on a_0.
//
// Per reverse step four launches (two grid-wide dependencies: I' before A I', gAI before A^T gAI):
//   K1 bwd_transform_kernel : S' = sig(S_j W^T+b), I' = sig(I_j W^T+b)  (tcgen05)  -> Sp, Ip
//   K2 bwd_row_kernel       : AI = A I' ; a += D(y_j,gP_j) (adjoint mode) ; gAI   -> AI, G, a
//                             (discrete mode adds D in a separate row pass after K3)
//   K3a bwd_gz_kernel      : A^T gAI, gz* (in place over Sp / AI)
// Weighted sweeps (gnode_rollout_backward_weighted) gather sum_c w_rc I'[c] in K2 and sum_c w_cr gAI[c] in K3a (the
// weights in transpose order, permuted once per sweep by permute_weights_kernel); K3e's formula holds at any w.
//   K3e bwd_edge_kernel    : dL/dw_rc += dt * gAI[r] . I'[c] per stored entry of A (only when edge gradients are asked)
//   K3 bwd_vjp_kernel       : per-CTA vW / vb (FFMA), v = gz W into a (tcgen05)
// Parameter-gradient partial sums live in per-CTA slots (no atomics: bitwise reproducible) and are
// folded by reduce_partials_kernel at the end.
#include <algorithm>
#include <cstdlib>

#include "gnode_common.cuh"
#include "gnode_tile.cuh"
#include "gnode_umma.cuh"

namespace gnode {

constexpr int ROW_THREADS = 256;                 // K2 / K4 block size (16 half-warps)
constexpr int DEC_COUNT = 4 * H + 4 + 4 + 1;     // linear3.weight, linear3.bias, linearS2.weight, linearS2.bias
constexpr int LIN_COUNT = H * H + H;             // odefunc.linear.weight, bias
constexpr int ENC_COUNT = 2 * H;                 // linearS1.weight, bias

// Sum over the 16 lanes of a half-warp, in a fixed order (all 32 lanes of the warp must call it).
__device__ __forceinline__ float halfwarp_sum(float v) {
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

struct BwdArgs {
    GnBatchView bv;
    const float* x; int64_t ldx;   // beta = x[:,3], gamma = x[:,4]; encoder inputs x[:,0:3]
    const float* y;                // [3][M][H] state y_j
    const float* gP;               // [M][3] dL/dprobs at time j (may be null: no decoder term)
    float* a;                      // [3][M][H] adjoint (in place)
    float* Sp; float* Ip; float* AI; float* G;   // [M][H] scratch
    const float* Ipf; const float* AIf;          // [M][H] I'_j and AI_j = A I'_j kept by the forward (auxiliary storage), or null
    float* part;                   // per-block partial sums of this kernel family
    float* gx; int64_t ldgx;       // dL/dx [M][ldgx] (columns 0..4) or null: no input gradient
    float dt;
    int only_dec;                  // 1: only a += D(y, gP)
    gnode_params_t p;
    // weighted neighbour sum (the W instantiations): weight of forward entry e of instance i = ew[inst_e0[i] + e], of
    // transpose entry k = ewT[inst_e0[i] + k] (ew permuted by the graph's transpose map)
    const float* ew; const float* ewT; const int64_t* inst_e0;
};

// ---------------------------------------------------------------- K1
// S' and I' of the stored state, recomputed with the forward's tcgen05 4-term tf32 split product (gnode_umma.cuh).
constexpr int K1_SM_X = 0, K1_SM_O = 32768, K1_SM_WHI = 65536, K1_SM_WLO = K1_SM_WHI + H * H * 4,
              K1_SM_B = K1_SM_WLO + H * H * 4, K1_SM_BAR = K1_SM_B + H * 4, K1_SM_TOTAL = K1_SM_BAR + 16 + 1024;

__global__ void __launch_bounds__(NTHREADS, 2) bwd_transform_kernel(const BwdArgs a) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Xs = smem + K1_SM_X;
    unsigned char* Os = smem + K1_SM_O;
    float* bs = reinterpret_cast<float*>(smem + K1_SM_B);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + K1_SM_BAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + K1_SM_BAR + 8);
    const int tid = threadIdx.x;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    umma::prepare_weights(a.p.lin_w, smem + K1_SM_WHI, smem + K1_SM_WLO, tid, NTHREADS);
    if (tid < 32) umma::tmem_alloc(tslot, umma::TMEM_COLS);
    if (tid == 0) umma::mbar_init(mbar, 1);
    umma::fence_before_sync();
    if (tid < H) bs[tid] = a.p.lin_b[tid];
    __syncthreads();
    umma::fence_after_sync();
    umma::Ctx cx;
    cx.tmem = *tslot; cx.bar = mbar; cx.phase = 0;
    cx.whi = umma::smem_u32(smem + K1_SM_WHI); cx.wlo = umma::smem_u32(smem + K1_SM_WLO);
    for (int tile = blockIdx.x; tile < a.bv.n_tiles; tile += gridDim.x) {
        const int64_t tile0 = (int64_t)tile * TILE;
#pragma unroll 1
        for (int comp = 0; comp < 2; ++comp) {
            load_tile(Xs, a.y + comp * plane, tile0, M, tid);
            __syncthreads();
            umma::gemm_sigmoid_tc<false>(cx, Xs, Os, bs, tid);      // Xs -> tf32 hi, Os: lo, then the result
            __syncthreads();
            store_tile(comp == 0 ? a.Sp : a.Ip, Os, tile0, M, tid);
            __syncthreads();
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc(cx.tmem, umma::TMEM_COLS);
}

// ---------------------------------------------------------------- K1' (auxiliary storage)
// With I'_j and AI_j kept by the forward, everything that depends on S' alone leaves this tile kernel directly:
//   G = gAI = beta (aI - aS) S'  -> G      gzS = beta (aI - aS) AI S'(1 - S')  -> Sp
// (bwd_row_kernel's gather of A I' and the S' round trip through HBM are gone; I' is not recomputed.)
__global__ void __launch_bounds__(NTHREADS, 2) bwd_transform_g_kernel(const BwdArgs a) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* Xs = smem + K1_SM_X;
    unsigned char* Os = smem + K1_SM_O;
    float* bs = reinterpret_cast<float*>(smem + K1_SM_B);
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + K1_SM_BAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + K1_SM_BAR + 8);
    const int tid = threadIdx.x;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    umma::prepare_weights(a.p.lin_w, smem + K1_SM_WHI, smem + K1_SM_WLO, tid, NTHREADS);
    if (tid < 32) umma::tmem_alloc(tslot, umma::TMEM_COLS);
    if (tid == 0) umma::mbar_init(mbar, 1);
    umma::fence_before_sync();
    if (tid < H) bs[tid] = a.p.lin_b[tid];
    __syncthreads();
    umma::fence_after_sync();
    umma::Ctx cx;
    cx.tmem = *tslot; cx.bar = mbar; cx.phase = 0;
    cx.whi = umma::smem_u32(smem + K1_SM_WHI); cx.wlo = umma::smem_u32(smem + K1_SM_WLO);
    for (int tile = blockIdx.x; tile < a.bv.n_tiles; tile += gridDim.x) {
        const int64_t tile0 = (int64_t)tile * TILE;
        load_tile(Xs, a.y, tile0, M, tid);
        __syncthreads();
        umma::gemm_sigmoid_tc<false>(cx, Xs, Os, bs, tid);      // Xs -> tf32 hi, Os: lo, then S'
        __syncthreads();
#pragma unroll 2
        for (int i = 0; i < 4; ++i) {
            const int idx = tid + i * NTHREADS;
            const int rr = idx >> 4, c4 = idx & 15;
            const int64_t g = tile0 + rr;
            float gb = 0.f;
            if (g < M) {
                const size_t off = (size_t)g * H + 4 * c4;
                const float4 aS = ldg4(a.a + off), aI = ldg4(a.a + plane + off), ai = ldg4_stream(a.AIf + off);
                const float be = a.x[(size_t)g * a.ldx + 3];
                const float4 sp = lds4(Os, sw_off(rr, c4));
                float4 G, gz;
#define GN_G(c)                                                     \
    {                                                               \
        const float q = aI.c - aS.c;                                \
        G.c = be * q * sp.c;                                        \
        gz.c = be * q * ai.c * sp.c * (1.0f - sp.c);                \
    }
                GN_G(x) GN_G(y) GN_G(z) GN_G(w)
#undef GN_G
                stg4(a.G + off, G);
                stg4(a.Sp + off, gz);
                if (a.gx) gb = (aI.x - aS.x) * ai.x * sp.x + (aI.y - aS.y) * ai.y * sp.y +
                               (aI.z - aS.z) * ai.z * sp.z + (aI.w - aS.w) * ai.w * sp.w;
            }
            // dL/dbeta of the row += dt * sum_h (aI - aS) AI S' (half-warp reduction; one lane per row adds)
            if (a.gx) {
                gb = halfwarp_sum(gb);
                if (g < M && c4 == 0) a.gx[(size_t)g * a.ldgx + 3] += a.dt * gb;
            }
        }
        __syncthreads();
    }
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc(cx.tmem, umma::TMEM_COLS);
}

// ---------------------------------------------------------------- decoder backward for one row
// Row held 4 channels per lane by a half-warp. Returns d = D(y, gP) for the lane's channels and
// accumulates the decoder parameter gradients into per-thread registers.
struct DecAcc {
    float w3[16];     // [m][j]: d linear3.weight[m][4l+j]
    float b3[4], w2[4], b2;
};

__device__ __forceinline__ void decoder_backward_row(const float4 (&c)[3], const float* gP_row, const float* W3s,
                                                     const float* small, int l, bool valid, float4 (&d)[3],
                                                     DecAcc& acc) {
    float hid[12];
    float4 w3[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        w3[m] = *reinterpret_cast<const float4*>(W3s + m * H + 4 * l);
#pragma unroll
        for (int k = 0; k < 3; ++k) hid[4 * k + m] = dot4(c[k], w3[m]);
    }
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1)
#pragma unroll
        for (int m = 0; m < 12; ++m) hid[m] += __shfl_xor_sync(0xffffffffu, hid[m], off);
    const float* b3 = small; const float* w2 = small + 4; const float b2 = small[8];
    float o[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float s = b2;
#pragma unroll
        for (int m = 0; m < 4; ++m) { hid[4 * k + m] += b3[m]; s = fmaf(w2[m], fmaxf(hid[4 * k + m], 0.f), s); }
        o[k] = s;
    }
    const float mx = fmaxf(o[0], fmaxf(o[1], o[2]));
    float P[3] = {expf(o[0] - mx), expf(o[1] - mx), expf(o[2] - mx)};
    const float inv = 1.0f / (P[0] + P[1] + P[2]);
    float g[3] = {0.f, 0.f, 0.f};
    if (valid && gP_row != nullptr) { g[0] = gP_row[0]; g[1] = gP_row[1]; g[2] = gP_row[2]; }
    float dotgp = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) { P[k] *= inv; dotgp = fmaf(g[k], P[k], dotgp); }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float go = P[k] * (g[k] - dotgp);                // softmax backward
        float4 dk = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const float act = fmaxf(hid[4 * k + m], 0.f);
            const float gh = (hid[4 * k + m] > 0.f) ? go * w2[m] : 0.f;   // ReLU backward
            dk.x = fmaf(gh, w3[m].x, dk.x); dk.y = fmaf(gh, w3[m].y, dk.y);
            dk.z = fmaf(gh, w3[m].z, dk.z); dk.w = fmaf(gh, w3[m].w, dk.w);
            acc.w3[4 * m + 0] = fmaf(gh, c[k].x, acc.w3[4 * m + 0]); acc.w3[4 * m + 1] = fmaf(gh, c[k].y, acc.w3[4 * m + 1]);
            acc.w3[4 * m + 2] = fmaf(gh, c[k].z, acc.w3[4 * m + 2]); acc.w3[4 * m + 3] = fmaf(gh, c[k].w, acc.w3[4 * m + 3]);
            if (l == 0) { acc.b3[m] += gh; acc.w2[m] = fmaf(go, act, acc.w2[m]); }
        }
        if (l == 0) acc.b2 += go;
        d[k] = dk;
    }
}

// ---------------------------------------------------------------- K2
// (3 CTAs per SM at 80 registers; 2 CTAs at 128 registers without spills, and issuing the own-row loads before the
// gather, measured no better: profiles/r1e_ab_backward.log)
template <bool W>
__global__ void __launch_bounds__(ROW_THREADS, 3) bwd_row_kernel(const BwdArgs a) {
    __shared__ float W3s[4 * H];
    __shared__ float small[12];
    __shared__ float red[ROW_THREADS / 16][16][17];   // [half-warp][lane][16 w3 values (+pad)]
    __shared__ float red0[ROW_THREADS / 16][9];       // lane-0 values: b3[4], w2[4], b2
    const int tid = threadIdx.x, lane = tid & 31, l = tid & 15, hw = tid >> 4;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    for (int i = tid; i < 4 * H; i += ROW_THREADS) W3s[i] = a.p.l3_w[i];
    if (tid < 4) { small[tid] = a.p.l3_b[tid]; small[4 + tid] = a.p.s2_w[tid]; }
    if (tid == 0) small[8] = a.p.s2_b[0];
    __syncthreads();

    DecAcc acc;
#pragma unroll
    for (int i = 0; i < 16; ++i) acc.w3[i] = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc.b3[i] = 0.f; acc.w2[i] = 0.f; }
    acc.b2 = 0.f;

    const int hw_per_grid = gridDim.x * (ROW_THREADS / 16);
    // warp-uniform trip count: both half-warps of a warp walk rows r and r+1
    const int64_t n_iter = (M + hw_per_grid - 1) / hw_per_grid;
    for (int64_t it = 0; it < n_iter; ++it) {
        const int64_t g = it * hw_per_grid + (int64_t)blockIdx.x * (ROW_THREADS / 16) + hw;
        const bool valid = g < M;
        const size_t off = (size_t)(valid ? g : 0) * H + 4 * l;
        float4 AI = make_float4(0.f, 0.f, 0.f, 0.f);
        float be = 0.f;
        int row0 = 0, e0 = 0, deg = 0;
        const int32_t* ci = nullptr;
        const float* wp = nullptr;
        if (!a.only_dec) {
            if (valid) {
                int inst = a.bv.tile_inst[g / TILE];                 // owner of the tile's first row, then walk forward
                while (inst + 1 < a.bv.n_inst && a.bv.inst[inst + 1].row0 <= g) ++inst;
                const GnInstance I = a.bv.inst[inst];
                row0 = I.row0; ci = I.colidx;
                const int n = (int)(g - row0);
                e0 = I.rowptr[n];
                deg = I.rowptr[n + 1] - e0;
                be = a.x[(size_t)g * a.ldx + 3];
                if (W) wp = a.ew + a.inst_e0[inst];
            }
            AI = gather_row<W>(a.Ip, ci, e0, deg, row0, l, lane, wp);
        }
        // Grid points without a cotangent (sparse dL/dprobs: only the rows int(i/deltaT) enter the loss) have D = 0:
        // no decoder backward, the state planes are not read and the adjoint is not rewritten
        const bool dec = a.gP != nullptr;                     // kernel argument: uniform
        float4 c[3], d[3];
        if (dec) {
#pragma unroll
            for (int k = 0; k < 3; ++k) c[k] = valid ? ldg4_stream(a.y + k * plane + off) : make_float4(0.f, 0.f, 0.f, 0.f);
            decoder_backward_row(c, valid ? a.gP + (size_t)g * 3 : nullptr, W3s, small, l, valid, d, acc);
        }
        if (valid) {
            float4 av[3];
            av[0] = ldg4(a.a + off); av[1] = ldg4(a.a + plane + off);
            if (dec) {
                av[2] = ldg4(a.a + 2 * plane + off);
#pragma unroll
                for (int k = 0; k < 3; ++k) { av[k].x += d[k].x; av[k].y += d[k].y; av[k].z += d[k].z; av[k].w += d[k].w; }
            }
            if (!a.only_dec) {
                const float4 sp = ldg4(a.Sp + off);
                float4 G;
                G.x = be * (av[1].x - av[0].x) * sp.x; G.y = be * (av[1].y - av[0].y) * sp.y;
                G.z = be * (av[1].z - av[0].z) * sp.z; G.w = be * (av[1].w - av[0].w) * sp.w;
                stg4(a.G + off, G);
                stg4(a.AI + off, AI);
            }
            if (dec) {
#pragma unroll
                for (int k = 0; k < 3; ++k) stg4(a.a + k * plane + off, av[k]);
            }
        }
    }
    if (a.gP == nullptr) return;                               // no decoder gradients were accumulated
    // block reduction in a fixed order (deterministic), then this block's slot += result
#pragma unroll
    for (int i = 0; i < 16; ++i) red[hw][l][i] = acc.w3[i];
    if (l == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { red0[hw][i] = acc.b3[i]; red0[hw][4 + i] = acc.w2[i]; }
        red0[hw][8] = acc.b2;
    }
    __syncthreads();
    float* slot = a.part + (size_t)blockIdx.x * DEC_COUNT;
    if (tid < 4 * H) {                               // entry (m, h): h = 4*lane16 + j
        const int m = tid / H, h = tid % H;
        float s = 0.f;
        for (int w = 0; w < ROW_THREADS / 16; ++w) s += red[w][h >> 2][4 * m + (h & 3)];
        slot[tid] += s;
    }
    if (tid < 9) {
        float s = 0.f;
        for (int w = 0; w < ROW_THREADS / 16; ++w) s += red0[w][tid];
        slot[4 * H + tid] += s;
    }
}

// ---------------------------------------------------------------- decoder backward alone
// a += D(y_j, gP_j) for every row (grid points with a cotangent, auxiliary-storage sweep and discrete mode): the
// streaming part of bwd_row_kernel without its gather. The six row operands (y and a planes) are requested together, so
// an iteration pays one memory round trip instead of two (bwd_row_kernel reads the adjoint after the decoder's shuffles).
__global__ void __launch_bounds__(ROW_THREADS, 2) bwd_dec_kernel(const BwdArgs a) {
    __shared__ float W3s[4 * H];
    __shared__ float small[12];
    __shared__ float red[ROW_THREADS / 16][16][17];   // [half-warp][lane][16 w3 values (+pad)]
    __shared__ float red0[ROW_THREADS / 16][9];       // lane-0 values: b3[4], w2[4], b2
    const int tid = threadIdx.x, l = tid & 15, hw = tid >> 4;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    for (int i = tid; i < 4 * H; i += ROW_THREADS) W3s[i] = a.p.l3_w[i];
    if (tid < 4) { small[tid] = a.p.l3_b[tid]; small[4 + tid] = a.p.s2_w[tid]; }
    if (tid == 0) small[8] = a.p.s2_b[0];
    __syncthreads();
    DecAcc acc;
#pragma unroll
    for (int i = 0; i < 16; ++i) acc.w3[i] = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc.b3[i] = 0.f; acc.w2[i] = 0.f; }
    acc.b2 = 0.f;
    const int hw_per_grid = gridDim.x * (ROW_THREADS / 16);
    const int64_t n_iter = (M + hw_per_grid - 1) / hw_per_grid;      // warp-uniform trip count (full-mask shuffles inside)
    for (int64_t it = 0; it < n_iter; ++it) {
        const int64_t g = it * hw_per_grid + (int64_t)blockIdx.x * (ROW_THREADS / 16) + hw;
        const bool valid = g < M;
        const size_t off = (size_t)(valid ? g : 0) * H + 4 * l;
        float4 c[3], av[3], d[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            c[k] = valid ? ldg4_stream(a.y + k * plane + off) : make_float4(0.f, 0.f, 0.f, 0.f);
            av[k] = valid ? ldg4(a.a + k * plane + off) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        decoder_backward_row(c, valid ? a.gP + (size_t)g * 3 : nullptr, W3s, small, l, valid, d, acc);
        if (valid) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                av[k].x += d[k].x; av[k].y += d[k].y; av[k].z += d[k].z; av[k].w += d[k].w;
                stg4(a.a + k * plane + off, av[k]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) red[hw][l][i] = acc.w3[i];
    if (l == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) { red0[hw][i] = acc.b3[i]; red0[hw][4 + i] = acc.w2[i]; }
        red0[hw][8] = acc.b2;
    }
    __syncthreads();
    float* slot = a.part + (size_t)blockIdx.x * DEC_COUNT;
    if (tid < 4 * H) {
        const int m = tid / H, h = tid % H;
        float s = 0.f;
        for (int w = 0; w < ROW_THREADS / 16; ++w) s += red[w][h >> 2][4 * m + (h & 3)];
        slot[tid] += s;
    }
    if (tid < 9) {
        float s = 0.f;
        for (int w = 0; w < ROW_THREADS / 16; ++w) s += red0[w][tid];
        slot[4 * H + tid] += s;
    }
}

// ---------------------------------------------------------------- K3a
// Row kernel (half-warp per row, grid-stride): A^T gAI, then the cotangents wrt the pre-activations
//   gzI = (A^T gAI + gamma (aR - aI)) I'(1-I')      gzS = beta (aI - aS) AI S'(1-S')
// written IN PLACE over the row's own S' (Sp <- gzS) and AI (AI <- gzI): both are read only by this row's threads.
// Separate from the tile kernel so that this latency-bound gather runs at row-kernel occupancy.
// AUX: gzS was written by bwd_transform_g_kernel; I' comes from the forward's auxiliary storage. W: A^T of the weighted sum
template <bool AUX, bool W>
__global__ void __launch_bounds__(ROW_THREADS, 3) bwd_gz_kernel(const BwdArgs a) {
    const int tid = threadIdx.x, lane = tid & 31, l = tid & 15, hw = tid >> 4;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    const int hw_per_grid = gridDim.x * (ROW_THREADS / 16);
    const int64_t n_iter = (M + hw_per_grid - 1) / hw_per_grid;        // warp-uniform trip count
    for (int64_t it = 0; it < n_iter; ++it) {
        const int64_t g = it * hw_per_grid + (int64_t)blockIdx.x * (ROW_THREADS / 16) + hw;
        const bool valid = g < M;
        const size_t off = (size_t)(valid ? g : 0) * H + 4 * l;
        int row0 = 0, e0 = 0, deg = 0;
        const int32_t* ci = nullptr;
        const float* wp = nullptr;
        float be = 0.f, ga = 0.f;
        float4 aS, aI, aR, sp, ip, ai;
        if (valid) {
            aI = ldg4(a.a + plane + off); aR = ldg4(a.a + 2 * plane + off);
            if (AUX) {
                ip = ldg4_stream(a.Ipf + off);
                aS = aI; sp = ip; ai = ip;                     // unused
            } else {
                aS = ldg4(a.a + off);
                sp = ldg4(a.Sp + off); ip = ldg4_stream(a.Ip + off); ai = ldg4(a.AI + off);
            }
            int inst = a.bv.tile_inst[g / TILE];
            while (inst + 1 < a.bv.n_inst && a.bv.inst[inst + 1].row0 <= g) ++inst;
            const GnInstance I = a.bv.inst[inst];
            row0 = I.row0; ci = I.colidx_t;
            const int n = (int)(g - row0);
            e0 = I.rowptr_t[n];
            deg = I.rowptr_t[n + 1] - e0;
            be = a.x[(size_t)g * a.ldx + 3];
            ga = a.x[(size_t)g * a.ldx + 4];
            if (W) wp = a.ewT + a.inst_e0[inst];
        }
        const float4 gsum = gather_row<W>(a.G, ci, e0, deg, row0, l, lane, wp);
        if (valid) {
            float4 gzs, gzi;
#define GN_GZ(c)                                                               \
    {                                                                          \
        const float q = aI.c - aS.c;                                           \
        const float gip = gsum.c + ga * (aR.c - aI.c);                         \
        gzi.c = gip * ip.c * (1.0f - ip.c);                                    \
        gzs.c = be * q * ai.c * sp.c * (1.0f - sp.c);                          \
    }
            GN_GZ(x) GN_GZ(y) GN_GZ(z) GN_GZ(w)
#undef GN_GZ
            if (!AUX) stg4(a.Sp + off, gzs);
            stg4(a.AI + off, gzi);
        }
        // dL/dgamma of the row += dt * sum_h (aR - aI) I'; without auxiliary storage dL/dbeta += dt * sum_h (aI - aS) AI S'
        // as well (with it, bwd_transform_g_kernel adds that term). Half-warp reductions, one lane per row adds.
        if (a.gx) {
            float sg = 0.f, sb = 0.f;
            if (valid) {
                sg = (aR.x - aI.x) * ip.x + (aR.y - aI.y) * ip.y + (aR.z - aI.z) * ip.z + (aR.w - aI.w) * ip.w;
                if (!AUX)
                    sb = (aI.x - aS.x) * ai.x * sp.x + (aI.y - aS.y) * ai.y * sp.y + (aI.z - aS.z) * ai.z * sp.z +
                         (aI.w - aS.w) * ai.w * sp.w;
            }
            sg = halfwarp_sum(sg);
            if (!AUX) sb = halfwarp_sum(sb);
            if (valid && l == 0) {
                float* gr = a.gx + (size_t)g * a.ldgx;
                if (!AUX) gr[3] += a.dt * sb;
                gr[4] += a.dt * sg;
            }
        }
    }
}

// ---------------------------------------------------------------- K3e: edge gradient (only when asked for)
// The forward's neighbour sum is AI[r] = sum_c w_rc I'[c] at w = 1, so per reverse step, at the same state and dt as the
// parameter VJP:   dL/dw_rc += dt * sum_h gAI[r,h] I'[c,h]   for every stored entry (r, c) of A.
// Row kernel over the forward CSR (not the transpose): a half-warp holds G[r] = gAI (4 channels per lane) and loads 8
// neighbour rows of I' per memory round trip, as gather_row does. Each edge's dot product is summed in a fixed order
// (lane partials, then the 16-lane butterfly) and one lane per edge adds it into ge: no atomics, bitwise reproducible.
// Launched after bwd_gz_kernel (which overwrites only Sp and AI: G and I' are intact) and before the tile kernel.
// Ipr: I' of the step (the forward's auxiliary storage, or the Ip scratch); inst_e0[i]: first entry of instance i in ge.
__global__ void __launch_bounds__(ROW_THREADS, 3) bwd_edge_kernel(const BwdArgs a, const float* __restrict__ Ipr,
                                                                   const int64_t* __restrict__ inst_e0,
                                                                   float* __restrict__ ge) {
    const int tid = threadIdx.x, lane = tid & 31, l = tid & 15, hw = tid >> 4;
    const int M = a.bv.M;
    const int hw_per_grid = gridDim.x * (ROW_THREADS / 16);
    const int64_t n_iter = (M + hw_per_grid - 1) / hw_per_grid;        // warp-uniform trip count (shuffles inside)
    for (int64_t it = 0; it < n_iter; ++it) {
        const int64_t g = it * hw_per_grid + (int64_t)blockIdx.x * (ROW_THREADS / 16) + hw;
        const bool valid = g < M;
        int row0 = 0, e0 = 0, deg = 0;
        const int32_t* ci = nullptr;
        float* out = nullptr;
        float4 gr = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) {
            gr = ldg4(a.G + (size_t)g * H + 4 * l);
            int inst = a.bv.tile_inst[g / TILE];
            while (inst + 1 < a.bv.n_inst && a.bv.inst[inst + 1].row0 <= g) ++inst;
            const GnInstance I = a.bv.inst[inst];
            row0 = I.row0; ci = I.colidx;
            const int n = (int)(g - row0);
            e0 = I.rowptr[n];
            deg = I.rowptr[n + 1] - e0;
            out = ge + inst_e0[inst] + e0;
        }
        const int degmax = max(deg, __shfl_xor_sync(0xffffffffu, deg, 16));
        for (int eb = 0; eb < degmax; eb += 16) {
            const int mine = (eb + l < deg) ? ci[e0 + eb + l] + row0 : -1;
            float res = 0.f;                                   // dot product of edge eb + l
#pragma unroll
            for (int jb = 0; jb < 16; jb += 8) {
                if (eb + jb < degmax) {
                    float4 v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int c = __shfl_sync(0xffffffffu, mine, (lane & 16) + jb + j);
                        v[j] = (c >= 0) ? ldg4(Ipr + (size_t)c * H + 4 * l) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float s = halfwarp_sum(dot4(gr, v[j]));
                        if (l == jb + j) res = s;
                    }
                }
            }
            if (eb + l < deg) out[eb + l] += a.dt * res;
        }
    }
}

// ---------------------------------------------------------------- weights in transpose order (weighted sweeps)
// wT[inst_e0[i] + k] = w[inst_e0[i] + tmap_i[k]]: transpose entry k of instance i is forward entry tmap_i[k] of its graph
__global__ void __launch_bounds__(256) permute_weights_kernel(const float* __restrict__ w, const int32_t* const* __restrict__ tmaps,
                                                              const int64_t* __restrict__ inst_e0, int n_inst, int64_t nnz,
                                                              float* __restrict__ wT) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
        int lo = 0, hi = n_inst - 1;                      // last instance with inst_e0 <= k (edgeless ones share their e0)
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (inst_e0[mid] <= k) lo = mid; else hi = mid - 1;
        }
        const int64_t e0 = inst_e0[lo];
        wT[k] = w[e0 + tmaps[lo][k - e0]];
    }
}

// ---------------------------------------------------------------- K3
// Shared memory: gzS | gzI | S_j | I_j tiles (fp32, swizzled) | W^T operand tiles (tf32 hi / lo). The state-VJP
// v = gz W runs on tcgen05 as the same 4-term tf32 split product as the forward transform: after the weight-gradient
// phase has consumed the raw tiles, gz is split IN PLACE (gz tile <- hi, the dead state tile <- lo).
constexpr int K3_SM_GS = 0, K3_SM_GI = 32768, K3_SM_XS = 65536, K3_SM_XI = 98304, K3_SM_WTHI = 131072,
              K3_SM_WTLO = K3_SM_WTHI + H * H * 4, K3_SM_BAR = K3_SM_WTLO + H * H * 4, K3_SM_TOTAL = K3_SM_BAR + 16 + 1024;

__global__ void __launch_bounds__(NTHREADS, 1) bwd_vjp_kernel(const BwdArgs a) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* GS = smem + K3_SM_GS;
    unsigned char* GI = smem + K3_SM_GI;
    unsigned char* XS = smem + K3_SM_XS;
    unsigned char* XI = smem + K3_SM_XI;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + K3_SM_BAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + K3_SM_BAR + 8);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    // B operand of v[r][j] = sum_h gz[r][h] W[h][j]: row n = j, K index = h, i.e. W transposed
    for (int idx = tid; idx < H * CHUNKS; idx += NTHREADS) {
        const int n = idx >> 4, c4 = idx & 15;
        const float4 w = make_float4(a.p.lin_w[(4 * c4 + 0) * H + n], a.p.lin_w[(4 * c4 + 1) * H + n],
                                     a.p.lin_w[(4 * c4 + 2) * H + n], a.p.lin_w[(4 * c4 + 3) * H + n]);
        float4 hi, lo;
        umma::tf32_split4(w, hi, lo);
        sts4(smem + K3_SM_WTHI, umma::swb_off(n, c4), hi);
        sts4(smem + K3_SM_WTLO, umma::swb_off(n, c4), lo);
    }
    umma::fence_proxy_async();
    if (tid < 32) umma::tmem_alloc(tslot, 128);        // two [128 x 64] fp32 accumulators: vS, vI
    if (tid == 0) umma::mbar_init(mbar, 2);            // one phase = the commits of both GEMMs
    umma::fence_before_sync();

    // weight-gradient accumulators, register-blocked 8 (h) x 4 (j) so that one row costs 3 shared-memory loads per 32
    // FMAs (the previous 1 x 8 blocking was bound by the shared-memory queue: mio_throttle 36 %). Thread = (part:
    // gzS (x) S or gzI (x) I, row group of 64 rows, h block of 8, 16-byte column chunk); the four partial sums per
    // output element are folded through shared memory at the end of the kernel, in a fixed order.
    const int wpart = tid >> 8, wrg = (tid >> 7) & 1, whb = (tid >> 4) & 7, wjq = tid & 15;
    float gw[32], gb[8];
#pragma unroll
    for (int i = 0; i < 32; ++i) gw[i] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) gb[i] = 0.f;
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t wthi = umma::smem_u32(smem + K3_SM_WTHI), wtlo = umma::smem_u32(smem + K3_SM_WTLO);
    uint32_t phase = 0;

    for (int tile = blockIdx.x; tile < a.bv.n_tiles; tile += gridDim.x) {
        const int64_t tile0 = (int64_t)tile * TILE;
        // gz tiles (written by bwd_gz_kernel over Sp / AI) and state tiles -> shared memory
        for (int idx = tid; idx < TILE * CHUNKS; idx += NTHREADS) {
            const int rr = idx >> 4, c4 = idx & 15;
            const int64_t g = tile0 + rr;
            const int so = sw_off(rr, c4);
            if (g < M) {
                const size_t go = (size_t)g * H + 4 * c4;
                cp_async16(GS + so, a.Sp + go);
                cp_async16(GI + so, a.AI + go);
                cp_async16(XS + so, a.y + go);
                cp_async16(XI + so, a.y + plane + go);
            } else {
                const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                sts4(GS, so, z); sts4(GI, so, z); sts4(XS, so, z); sts4(XI, so, z);
            }
        }
        cp_async_wait_all();
        __syncthreads();
        // ---- vW[h][j] += sum_r gzS[r][h] S[r][j] + gzI[r][h] I[r][j] ; vb[h] += sum_r gzS + gzI   (fp32 FFMA)
        {
            const unsigned char* Gt = wpart == 0 ? GS : GI;
            const unsigned char* Xt = wpart == 0 ? XS : XI;
#pragma unroll 2
            for (int r = 64 * wrg; r < 64 * wrg + 64; ++r) {
                const float4 g0 = lds4(Gt, sw_off(r, 2 * whb)), g1 = lds4(Gt, sw_off(r, 2 * whb + 1));
                const float4 xv = lds4(Xt, sw_off(r, wjq));
                const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                for (int hh = 0; hh < 8; ++hh) {
                    gw[4 * hh + 0] = fmaf(g[hh], xv.x, gw[4 * hh + 0]); gw[4 * hh + 1] = fmaf(g[hh], xv.y, gw[4 * hh + 1]);
                    gw[4 * hh + 2] = fmaf(g[hh], xv.z, gw[4 * hh + 2]); gw[4 * hh + 3] = fmaf(g[hh], xv.w, gw[4 * hh + 3]);
                }
                if (wjq == 0) {
#pragma unroll
                    for (int hh = 0; hh < 8; ++hh) gb[hh] += g[hh];
                }
            }
        }
        __syncthreads();
        // ---- v = gz W on tcgen05: split gz in place (gz tile <- hi, state tile <- lo), two GEMMs, one mbarrier phase
        for (int idx = tid; idx < TILE * CHUNKS; idx += NTHREADS) {
            const int off = sw_off(idx >> 4, idx & 15);
            float4 hi, lo;
            umma::tf32_split4(lds4(GS, off), hi, lo);
            sts4(GS, off, hi); sts4(XS, off, lo);
            umma::tf32_split4(lds4(GI, off), hi, lo);
            sts4(GI, off, hi); sts4(XI, off, lo);
        }
        umma::fence_proxy_async();
        __syncthreads();
        if (tid == 0) {
            umma::issue_split_gemm_to(tmem, mbar, wthi, wtlo, umma::smem_u32(GS), umma::smem_u32(XS));
            umma::issue_split_gemm_to(tmem + 64, mbar, wthi, wtlo, umma::smem_u32(GI), umma::smem_u32(XI));
        }
        umma::mbar_wait(mbar, phase);
        phase ^= 1;
        umma::fence_after_sync();
        // ---- a += dt * v: warp (q = lane quarter, cq = 16-column block), thread = tile row; aS from vS, aI from vI (vR = 0)
        {
            const int q = warp & 3, cq = warp >> 2;
            const int64_t g = tile0 + q * 32 + lane;
#pragma unroll
            for (int comp = 0; comp < 2; ++comp) {
                float v[16];
                umma::tmem_ld16(tmem + 64 * comp + ((uint32_t)(q * 32) << 16) + 16 * cq, v);
                if (g < M) {
                    float* row = a.a + comp * plane + (size_t)g * H + 16 * cq;
#pragma unroll
                    for (int jj = 0; jj < 16; jj += 4) {
                        float4 cur = ldg4(row + jj);
                        cur.x = fmaf(a.dt, v[jj + 0], cur.x); cur.y = fmaf(a.dt, v[jj + 1], cur.y);
                        cur.z = fmaf(a.dt, v[jj + 2], cur.z); cur.w = fmaf(a.dt, v[jj + 3], cur.w);
                        stg4(row + jj, cur);
                    }
                }
            }
        }
        umma::fence_before_sync();
        __syncthreads();
    }
    // fold the four partial sums (part x row group) of every output element: red[4][64][64] over the gz tiles,
    // red_b[4][64] over the S tile (the tile loop has ended with a block barrier)
    {
        float* red = reinterpret_cast<float*>(GS);
        float* red_b = reinterpret_cast<float*>(XS);
        const int pidx = tid >> 7;
#pragma unroll
        for (int hh = 0; hh < 8; ++hh)
            *reinterpret_cast<float4*>(red + ((size_t)pidx * H + 8 * whb + hh) * H + 4 * wjq) =
                make_float4(gw[4 * hh + 0], gw[4 * hh + 1], gw[4 * hh + 2], gw[4 * hh + 3]);
        if (wjq == 0) {
#pragma unroll
            for (int hh = 0; hh < 8; ++hh) red_b[pidx * H + 8 * whb + hh] = gb[hh];
        }
        __syncthreads();
        float* slot = a.part + (size_t)blockIdx.x * LIN_COUNT;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int o = tid * 8 + i;                      // output element (h, j) = (o / 64, o % 64)
            const float sum = ((red[o] + red[H * H + o]) + red[2 * H * H + o]) + red[3 * H * H + o];
            slot[o] += a.dt * sum;
        }
        if (tid < H) slot[H * H + tid] += a.dt * (((red_b[tid] + red_b[H + tid]) + red_b[2 * H + tid]) + red_b[3 * H + tid]);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc(tmem, 128);
}

// ---------------------------------------------------------------- K3, two CTAs per SM
// The same work as bwd_vjp_kernel with half the shared memory per CTA: the (gzS, S_j) and (gzI, I_j) pairs of a tile are
// processed one after the other through ONE gz tile and ONE state tile (96 KB per CTA with the W^T operand), by 256
// threads, so that two CTAs are resident per SM and the load / FFMA / tensor / read-modify-write phases of one overlap
// those of the other (bwd_vjp_kernel runs them back to back on one 512-thread CTA: 1.8 TB/s of its 2 KB per row).
constexpr int K3B_THREADS = 256;
constexpr int K3B_SM_G = 0, K3B_SM_X = 32768, K3B_SM_WTHI = 65536, K3B_SM_WTLO = K3B_SM_WTHI + H * H * 4,
              K3B_SM_BAR = K3B_SM_WTLO + H * H * 4, K3B_SM_TOTAL = K3B_SM_BAR + 16 + 1024;

// WGRAD = false: no parameter gradient wanted (input gradients only): the vW FFMA loop, the vb column sums and the fold
// into the slots are compiled out; the state VJP and the adjoint's read-modify-write are the same instructions.
template <bool WGRAD>
__global__ void __launch_bounds__(K3B_THREADS, 2) bwd_vjp2_kernel(const BwdArgs a) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    unsigned char* G = smem + K3B_SM_G;
    unsigned char* X = smem + K3B_SM_X;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(smem + K3B_SM_BAR);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(smem + K3B_SM_BAR + 8);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    // B operand of v[r][j] = sum_h gz[r][h] W[h][j]: row n = j, K index = h, i.e. W transposed
    for (int idx = tid; idx < H * CHUNKS; idx += K3B_THREADS) {
        const int n = idx >> 4, c4 = idx & 15;
        const float4 w = make_float4(a.p.lin_w[(4 * c4 + 0) * H + n], a.p.lin_w[(4 * c4 + 1) * H + n],
                                     a.p.lin_w[(4 * c4 + 2) * H + n], a.p.lin_w[(4 * c4 + 3) * H + n]);
        float4 hi, lo;
        umma::tf32_split4(w, hi, lo);
        sts4(smem + K3B_SM_WTHI, umma::swb_off(n, c4), hi);
        sts4(smem + K3B_SM_WTLO, umma::swb_off(n, c4), lo);
    }
    umma::fence_proxy_async();
    if (tid < 32) umma::tmem_alloc(tslot, 64);         // one [128 x 64] fp32 accumulator
    if (tid == 0) umma::mbar_init(mbar, 1);
    umma::fence_before_sync();

    // weight-gradient accumulators, register-blocked 8 (h) x 4 (j); thread = (row group of 64 rows, h block of 8,
    // 16-byte column chunk); both parts of a tile add into the same accumulators (vW = gzS^T S + gzI^T I)
    const int wrg = tid >> 7, whb = (tid >> 4) & 7, wjq = tid & 15;
    float gw[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) gw[i] = 0.f;
    // bias gradient vb[h] = sum_r gz[r][h]: column sums taken where the gz tile is split (every thread already reads
    // its 16-byte column chunk c4 = tid & 15 of rows (tid >> 4) + 16 k there), not in the FFMA loop
    float4 gbv = make_float4(0.f, 0.f, 0.f, 0.f);
    // FFMA loop addressing: rows are walked in blocks of 8 so that the swizzle term (r & 7) is a compile-time constant
    const int cg = (2 * whb) & 7, cx = wjq & 7;
    const unsigned char* Gb = G + ((2 * whb) >> 3) * (TILE * 128) + 64 * wrg * 128;
    const unsigned char* Xb = X + (wjq >> 3) * (TILE * 128) + 64 * wrg * 128;
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t wthi = umma::smem_u32(smem + K3B_SM_WTHI), wtlo = umma::smem_u32(smem + K3B_SM_WTLO);
    uint32_t phase = 0;

    // gz tile (written by bwd_gz_kernel / bwd_transform_g_kernel over Sp / AI) and the state tile of one (tile, part)
    // unit -> shared memory, asynchronously: the request for the NEXT unit is issued as soon as the GEMM has consumed
    // the current tiles, so that its latency hides behind the read-modify-write of the adjoint
    auto request_unit = [&](int tile, int part) {
        if (tile >= a.bv.n_tiles) return;
        const int64_t tile0 = (int64_t)tile * TILE;
        const float* gsrc = part == 0 ? a.Sp : a.AI;
        const float* xsrc = a.y + (size_t)part * plane;
        for (int idx = tid; idx < TILE * CHUNKS; idx += K3B_THREADS) {
            const int rr = idx >> 4, c4 = idx & 15;
            const int64_t g = tile0 + rr;
            const int so = sw_off(rr, c4);
            if (g < M) {
                const size_t go = (size_t)g * H + 4 * c4;
                cp_async16(G + so, gsrc + go);
                cp_async16(X + so, xsrc + go);
            } else {
                const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                sts4(G, so, z); sts4(X, so, z);
            }
        }
    };
    request_unit(blockIdx.x, 0);
    for (int tile = blockIdx.x; tile < a.bv.n_tiles; tile += gridDim.x) {
        const int64_t tile0 = (int64_t)tile * TILE;
#pragma unroll 1
        for (int part = 0; part < 2; ++part) {
            cp_async_wait_all();
            __syncthreads();
            // ---- vW[h][j] += sum_r gz[r][h] x[r][j] ; vb[h] += sum_r gz[r][h]   (fp32 FFMA)
#pragma unroll 1
            for (int r8 = 0; r8 < (WGRAD ? 8 : 0); ++r8) {      // (no trip without a parameter gradient)
                const unsigned char* gp = Gb + r8 * 1024;
                const unsigned char* xp = Xb + r8 * 1024;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int og = i * 128 + ((cg ^ i) << 4);
                    const float4 g0 = *reinterpret_cast<const float4*>(gp + og);
                    const float4 g1 = *reinterpret_cast<const float4*>(gp + (og ^ 16));
                    const float4 xv = *reinterpret_cast<const float4*>(xp + i * 128 + ((cx ^ i) << 4));
                    const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                    for (int hh = 0; hh < 8; ++hh) {
                        gw[4 * hh + 0] = fmaf(g[hh], xv.x, gw[4 * hh + 0]); gw[4 * hh + 1] = fmaf(g[hh], xv.y, gw[4 * hh + 1]);
                        gw[4 * hh + 2] = fmaf(g[hh], xv.z, gw[4 * hh + 2]); gw[4 * hh + 3] = fmaf(g[hh], xv.w, gw[4 * hh + 3]);
                    }
                }
            }
            __syncthreads();
            // ---- v = gz W on tcgen05: split gz in place (gz tile <- hi, the dead state tile <- lo)
            for (int idx = tid; idx < TILE * CHUNKS; idx += K3B_THREADS) {
                const int off = sw_off(idx >> 4, idx & 15);
                float4 hi, lo;
                const float4 gz = lds4(G, off);
                if (WGRAD) { gbv.x += gz.x; gbv.y += gz.y; gbv.z += gz.z; gbv.w += gz.w; }
                umma::tf32_split4(gz, hi, lo);
                sts4(G, off, hi); sts4(X, off, lo);
            }
            umma::fence_proxy_async();
            __syncthreads();
            if (tid == 0) umma::issue_split_gemm_to(tmem, mbar, wthi, wtlo, umma::smem_u32(G), umma::smem_u32(X));
            umma::mbar_wait(mbar, phase);
            phase ^= 1;
            umma::fence_after_sync();
            // the tensor core has read both tiles: the next unit may land there (generic-proxy writes after the async
            // proxy's reads are ordered by the mbarrier wait above)
            request_unit(part == 0 ? tile : tile + (int)gridDim.x, part ^ 1);
            // ---- a[part] += dt * v: warp (q = lane quarter, ch = 32-column half), thread = tile row (vR = 0)
            {
                const int q = warp & 3, ch = warp >> 2;
                const int64_t g = tile0 + q * 32 + lane;
#pragma unroll
                for (int cb = 0; cb < 2; ++cb) {
                    float v[16];
                    umma::tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + 32 * ch + 16 * cb, v);
                    if (g < M) {
                        float* row = a.a + (size_t)part * plane + (size_t)g * H + 32 * ch + 16 * cb;
#pragma unroll
                        for (int jj = 0; jj < 16; jj += 4) {
                            float4 cur = ldg4(row + jj);
                            cur.x = fmaf(a.dt, v[jj + 0], cur.x); cur.y = fmaf(a.dt, v[jj + 1], cur.y);
                            cur.z = fmaf(a.dt, v[jj + 2], cur.z); cur.w = fmaf(a.dt, v[jj + 3], cur.w);
                            stg4(row + jj, cur);
                        }
                    }
                }
            }
            umma::fence_before_sync();
            __syncthreads();
        }
    }
    // fold the two partial sums (row groups) of every output element: red[2][64][64] over the gz tile, red_b[16][64]
    // over the state tile (the tile loop has ended with a block barrier)
    if (WGRAD) {
        float* red = reinterpret_cast<float*>(G);
        float* red_b = reinterpret_cast<float*>(X);
#pragma unroll
        for (int hh = 0; hh < 8; ++hh)
            *reinterpret_cast<float4*>(red + ((size_t)wrg * H + 8 * whb + hh) * H + 4 * wjq) =
                make_float4(gw[4 * hh + 0], gw[4 * hh + 1], gw[4 * hh + 2], gw[4 * hh + 3]);
        *reinterpret_cast<float4*>(red_b + (tid >> 4) * H + 4 * (tid & 15)) = gbv;      // red_b[16 row classes][64]
        __syncthreads();
        float* slot = a.part + (size_t)blockIdx.x * LIN_COUNT;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int o = tid * 16 + i;                     // output element (h, j) = (o / 64, o % 64)
            slot[o] += a.dt * (red[o] + red[H * H + o]);
        }
        if (tid < H) {
            float sb = 0.f;
#pragma unroll
            for (int w = 0; w < 16; ++w) sb += red_b[w * H + tid];
            slot[H * H + tid] += a.dt * sb;
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc(tmem, 64);
}

// ---------------------------------------------------------------- K4: encoder backward
// y0 = relu(c * w1 + b1): d w1[h] = sum a0[h] [y0>0] c ; d b1[h] = sum a0[h] [y0>0]   (c in {S0,I0,R0})
// Input gradient (a.gx): dL/dc = sum_h a0[h] [y0>0] w1[h], stored into columns 0..2. Parameter partials only when a.part.
__global__ void __launch_bounds__(ROW_THREADS) bwd_encoder_kernel(const BwdArgs a) {
    __shared__ float red[ROW_THREADS / 16][16][9];
    const int tid = threadIdx.x, l = tid & 15, hw = tid >> 4;
    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    float gw[4] = {0.f, 0.f, 0.f, 0.f}, gb[4] = {0.f, 0.f, 0.f, 0.f};
    const float4 w1 = a.gx ? ldg4(a.p.s1_w + 4 * l) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int hw_per_grid = gridDim.x * (ROW_THREADS / 16);
    const int64_t n_iter = (M + hw_per_grid - 1) / hw_per_grid;        // warp-uniform trip count (shuffles inside)
    for (int64_t it = 0; it < n_iter; ++it) {
        const int64_t g = it * hw_per_grid + (int64_t)blockIdx.x * (ROW_THREADS / 16) + hw;
        const bool valid = g < M;
        float gc[3] = {0.f, 0.f, 0.f};
        if (valid) {
            const size_t off = (size_t)g * H + 4 * l;
            const float* xr = a.x + (size_t)g * a.ldx;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float c = xr[k];
                const float4 y0 = ldg4_stream(a.y + k * plane + off);
                const float4 av = ldg4_stream(a.a + k * plane + off);
                const float m0 = y0.x > 0.f ? av.x : 0.f, m1 = y0.y > 0.f ? av.y : 0.f;
                const float m2 = y0.z > 0.f ? av.z : 0.f, m3 = y0.w > 0.f ? av.w : 0.f;
                gw[0] = fmaf(m0, c, gw[0]); gw[1] = fmaf(m1, c, gw[1]); gw[2] = fmaf(m2, c, gw[2]); gw[3] = fmaf(m3, c, gw[3]);
                gb[0] += m0; gb[1] += m1; gb[2] += m2; gb[3] += m3;
                gc[k] = m0 * w1.x + m1 * w1.y + m2 * w1.z + m3 * w1.w;
            }
        }
        if (a.gx) {
#pragma unroll
            for (int k = 0; k < 3; ++k) gc[k] = halfwarp_sum(gc[k]);
            if (valid && l == 0) {
                float* gr = a.gx + (size_t)g * a.ldgx;
                gr[0] = gc[0]; gr[1] = gc[1]; gr[2] = gc[2];
            }
        }
    }
    if (!a.part) return;                                       // no parameter gradient wanted
#pragma unroll
    for (int i = 0; i < 4; ++i) { red[hw][l][i] = gw[i]; red[hw][l][4 + i] = gb[i]; }
    __syncthreads();
    float* slot = a.part + (size_t)blockIdx.x * ENC_COUNT;
    if (tid < 2 * H) {
        const int which = tid / H, h = tid % H;
        float s = 0.f;
        for (int w = 0; w < ROW_THREADS / 16; ++w) s += red[w][h >> 2][4 * which + (h & 3)];
        slot[tid] = s;
    }
}

// out[i] = sum over slots (fixed order)
__global__ void reduce_partials_kernel(const float* __restrict__ part, int n_slots, int count, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float s = 0.f;
    for (int k = 0; k < n_slots; ++k) s += part[(size_t)k * count + i];
    out[i] = s;
}

// Per-instance sums of grad_x columns 3 and 4 (the gradient of compact descriptors' beta[i], gamma[i]): one CTA per
// instance, every thread sums a fixed strided subset of the rows in row order, then a fixed-shape tree (no atomics).
constexpr int TG_THREADS = 256;
__global__ void __launch_bounds__(TG_THREADS) trials_grad_kernel(const GnBatchView bv, const float* __restrict__ gx,
                                                                 int64_t ldgx, float* __restrict__ gbeta,
                                                                 float* __restrict__ ggamma) {
    __shared__ float sb[TG_THREADS], sg[TG_THREADS];
    const int tid = threadIdx.x;
    const GnInstance I = bv.inst[blockIdx.x];
    float b = 0.f, g = 0.f;
    for (int n = tid; n < I.n; n += TG_THREADS) {
        const float* r = gx + (size_t)(I.row0 + n) * ldgx;
        b += r[3]; g += r[4];
    }
    sb[tid] = b; sg[tid] = g;
    __syncthreads();
#pragma unroll
    for (int w = TG_THREADS / 2; w >= 1; w >>= 1) {
        if (tid < w) { sb[tid] += sb[tid + w]; sg[tid] += sg[tid + w]; }
        __syncthreads();
    }
    if (tid == 0) { gbeta[blockIdx.x] = sb[0]; ggamma[blockIdx.x] = sg[0]; }
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// 2 (default) = bwd_vjp2_kernel (two 256-thread CTAs per SM, parts in sequence), 1 = bwd_vjp_kernel; env GNODE_BWD_VJP.
// (The weight gradient vW = gz^T X on tcgen05 was probed and not built: kind::tf32 takes MN-major operands only in the
// SWIZZLE_128B_BASE32B layout -- 32-byte swizzle granules; with the plain SWIZZLE_128B descriptor the instruction
// completes and leaves zeros, tools/umma_mn_probe.cu, profiles/r2k_umma_mn_probe.log -- while v = gz W needs the same gz
// tile K-major in plain SWIZZLE_128B: two copies of gz (hi and lo each) beside the split state tile = six operand
// tiles, 192 KB + the W^T operand, with one CTA per SM left to hide the loads.)
static int g_vjp_kernel = 0;
static int vjp_kernel_choice() {
    if (g_vjp_kernel == 0) {
        const int c = getenv("GNODE_BWD_VJP") ? atoi(getenv("GNODE_BWD_VJP")) : 2;
        g_vjp_kernel = (c >= 1 && c <= 2) ? c : 2;
    }
    return g_vjp_kernel;
}
static int launch_vjp(const BwdArgs& a, int grid, bool wgrad, cudaStream_t stream) {
    switch (vjp_kernel_choice()) {
        case 1: bwd_vjp_kernel<<<grid, NTHREADS, K3_SM_TOTAL, stream>>>(a); break;   // (computes its partials anyway)
        default:
            if (wgrad) bwd_vjp2_kernel<true><<<grid, K3B_THREADS, K3B_SM_TOTAL, stream>>>(a);
            else bwd_vjp2_kernel<false><<<grid, K3B_THREADS, K3B_SM_TOTAL, stream>>>(a);
            break;
    }
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}

struct BwdPlan {
    int grid_row, grid_tile1, grid_tile3;
    size_t off_a, off_sp, off_ip, off_ai, off_g, off_pdec, off_plin, off_penc, total;
};

static BwdPlan plan_backward(const gnode_batch* b) {
    BwdPlan p;
    const size_t M = (size_t)b->M;
    const int hw_per_block = ROW_THREADS / 16;
    p.grid_row = (int)std::min<int64_t>((b->M + hw_per_block - 1) / hw_per_block, (int64_t)b->sm_count * 8);
    p.grid_tile1 = std::min(b->n_tiles, 2 * b->sm_count);
    p.grid_tile3 = std::min(b->n_tiles, (vjp_kernel_choice() == 2 ? 2 : 1) * b->sm_count);
    size_t o = 0;
    p.off_a = o;  o += align_up(3 * M * H * sizeof(float), 256);
    p.off_sp = o; o += align_up(M * H * sizeof(float), 256);
    p.off_ip = o; o += align_up(M * H * sizeof(float), 256);
    p.off_ai = o; o += align_up(M * H * sizeof(float), 256);
    p.off_g = o;  o += align_up(M * H * sizeof(float), 256);
    p.off_pdec = o; o += align_up((size_t)p.grid_row * DEC_COUNT * sizeof(float), 256);
    p.off_plin = o; o += align_up((size_t)p.grid_tile3 * LIN_COUNT * sizeof(float), 256);
    p.off_penc = o; o += align_up((size_t)p.grid_row * ENC_COUNT * sizeof(float), 256);
    p.total = o;
    return p;
}

}  // namespace gnode

using namespace gnode;

extern "C" int gnode_set_bwd_kernel(int kernel) {
    if (kernel < 1 || kernel > 2) { set_error("gnode_set_bwd_kernel: kernel must be 1 or 2"); return GNODE_ERR_ARG; }
    g_vjp_kernel = kernel;
    return GNODE_OK;
}
extern "C" int gnode_get_bwd_kernel(void) { return vjp_kernel_choice(); }

extern "C" size_t gnode_backward_workspace_bytes(gnode_batch_t b) {
    if (!b) return 0;
    return plan_backward(b).total;
}

extern "C" int gnode_rollout_backward(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                      int32_t T, const float* dt_host, const float* traj, const float* grad_probs,
                                      int32_t grad_mode, float* grads_out, void* workspace, size_t workspace_bytes,
                                      void* stream_) {
    return gnode_rollout_backward_aux(b, x, ldx, p, T, dt_host, traj, nullptr, grad_probs, nullptr, 0, grad_mode, grads_out,
                                      workspace, workspace_bytes, stream_);
}

extern "C" int gnode_rollout_backward_sel(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                          int32_t T, const float* dt_host, const float* traj, const float* grad_probs,
                                          const int32_t* out_steps, int32_t n_out, int32_t grad_mode, float* grads_out,
                                          void* workspace, size_t workspace_bytes, void* stream_) {
    return gnode_rollout_backward_aux(b, x, ldx, p, T, dt_host, traj, nullptr, grad_probs, out_steps, n_out, grad_mode,
                                      grads_out, workspace, workspace_bytes, stream_);
}

extern "C" int gnode_rollout_backward_aux(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                          int32_t T, const float* dt_host, const float* traj, const float* aux,
                                          const float* grad_probs, const int32_t* out_steps, int32_t n_out,
                                          int32_t grad_mode, float* grads_out, void* workspace, size_t workspace_bytes,
                                          void* stream_) {
    return gnode_rollout_backward_input(b, x, ldx, p, T, dt_host, traj, aux, grad_probs, out_steps, n_out, grad_mode,
                                        grads_out, nullptr, 0, workspace, workspace_bytes, stream_);
}

extern "C" int gnode_rollout_backward_input(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                            int32_t T, const float* dt_host, const float* traj, const float* aux,
                                            const float* grad_probs, const int32_t* out_steps, int32_t n_out,
                                            int32_t grad_mode, float* grads_out, float* grad_x, int64_t ldgx,
                                            void* workspace, size_t workspace_bytes, void* stream_) {
    return gnode_rollout_backward_edges(b, x, ldx, p, T, dt_host, traj, aux, grad_probs, out_steps, n_out, grad_mode,
                                        grads_out, grad_x, ldgx, nullptr, workspace, workspace_bytes, stream_);
}

extern "C" size_t gnode_backward_weighted_workspace_bytes(gnode_batch_t b) {
    if (!b) return 0;
    return plan_backward(b).total + align_up((size_t)std::max<int64_t>(b->nnz_total, 1) * sizeof(float), 256);
}

extern "C" int gnode_rollout_backward_edges(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                            int32_t T, const float* dt_host, const float* traj, const float* aux,
                                            const float* grad_probs, const int32_t* out_steps, int32_t n_out,
                                            int32_t grad_mode, float* grads_out, float* grad_x, int64_t ldgx,
                                            float* grad_edge, void* workspace, size_t workspace_bytes, void* stream_) {
    return gnode_rollout_backward_weighted(b, x, ldx, p, T, dt_host, traj, aux, grad_probs, out_steps, n_out, grad_mode,
                                           grads_out, grad_x, ldgx, grad_edge, nullptr, workspace, workspace_bytes, stream_);
}

extern "C" int gnode_rollout_backward_weighted(gnode_batch_t b, const float* x, int64_t ldx, const gnode_params_t* p,
                                               int32_t T, const float* dt_host, const float* traj, const float* aux,
                                               const float* grad_probs, const int32_t* out_steps, int32_t n_out,
                                               int32_t grad_mode, float* grads_out, float* grad_x, int64_t ldgx,
                                               float* grad_edge, const float* edge_w, void* workspace,
                                               size_t workspace_bytes, void* stream_) {
    if (!b || !x || !p || !traj || !grad_probs || (!grads_out && !grad_x && !grad_edge) || (grad_x && ldgx < 5) ||
        !workspace || T < 1 || ldx < 5 || (T > 1 && !dt_host) ||
        (grad_mode != GNODE_GRAD_ADJOINT && grad_mode != GNODE_GRAD_DISCRETE)) {
        set_error("gnode_rollout_backward: bad arguments (T=%d ldx=%lld ldgx=%lld grad_mode=%d grads_out=%p grad_x=%p "
                  "grad_edge=%p)", T, (long long)ldx, (long long)ldgx, grad_mode, (void*)grads_out, (void*)grad_x,
                  (void*)grad_edge);
        return GNODE_ERR_ARG;
    }
    const bool wgrad = grads_out != nullptr;
    OutSel sel;
    int rc = make_out_sel(T, out_steps, n_out, &sel, "gnode_rollout_backward_sel");
    if (rc) return rc;
    if ((rc = check_current_device(b, "gnode_rollout_backward"))) return rc;
    const BwdPlan pl = plan_backward(b);
    const size_t ws_need = edge_w ? gnode_backward_weighted_workspace_bytes(b) : pl.total;
    if (workspace_bytes < ws_need) {
        set_error("gnode_rollout_backward: workspace too small (%zu < %zu)", workspace_bytes, ws_need);
        return GNODE_ERR_ARG;
    }
    if (edge_w && (rc = ensure_transpose_maps(b))) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    static bool configured[64] = {false};
    if (!configured[b->device & 63]) {
        GN_CUDA(cudaFuncSetAttribute(bwd_transform_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_SM_TOTAL));
        GN_CUDA(cudaFuncSetAttribute(bwd_transform_g_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_SM_TOTAL));
        GN_CUDA(cudaFuncSetAttribute(bwd_vjp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K3_SM_TOTAL));
        GN_CUDA(cudaFuncSetAttribute(bwd_vjp2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K3B_SM_TOTAL));
        GN_CUDA(cudaFuncSetAttribute(bwd_vjp2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, K3B_SM_TOTAL));
        configured[b->device & 63] = true;
    }
    const size_t M = (size_t)b->M;
    unsigned char* ws = (unsigned char*)workspace;
    // Launch-bound batches (the reference's own monitorer runs use batch sizes 1 and 8: 4 launches per reverse step of
    // a few microseconds each): the whole sweep is captured once into a CUDA graph, keyed by every pointer and scalar
    // that enters it, and replayed while the caller keeps handing over the same buffers (a training loop under torch's
    // caching allocator does). GNODE_BWD_GRAPH=0 disables it.
    static const bool graphs_on = !(getenv("GNODE_BWD_GRAPH") && atoi(getenv("GNODE_BWD_GRAPH")) == 0);
    uint64_t key = 0;
    bool use_graph = false, capturing = false;
    cudaStream_t user_stream = stream;
    if (graphs_on && b->n_tiles <= 4 * b->sm_count) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(stream, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone) {
            auto mix = [&](const void* ptr, size_t n) {
                const unsigned char* c = (const unsigned char*)ptr;
                if (key == 0) key = 1469598103934665603ull;
                for (size_t i = 0; i < n; ++i) { key ^= c[i]; key *= 1099511628211ull; }
            };
            // (grads_out == NULL, i.e. no parameter gradient, grad_x == NULL, grad_edge == NULL and edge_w == NULL are part of
            // the pointers; the weights' values are read inside the graph, so new values written in place are honoured)
            const void* ptrs[] = {x, traj, aux, grad_probs, grads_out, workspace, stream_, grad_x, grad_edge, edge_w};
            mix(ptrs, sizeof(ptrs)); mix(p, sizeof(*p)); mix(&ldx, sizeof(ldx)); mix(&T, sizeof(T));
            mix(&ldgx, sizeof(ldgx));
            mix(&grad_mode, sizeof(grad_mode)); mix(dt_host, sizeof(float) * (size_t)(T > 1 ? T - 1 : 0));
            mix(sel.slot.data(), sizeof(int) * sel.slot.size());
            const int vk = vjp_kernel_choice();
            mix(&vk, sizeof(vk));
            use_graph = true;
            for (auto& e : b->bwd_graphs)
                if (e.key == key) {
                    GN_CUDA(cudaGraphLaunch((cudaGraphExec_t)e.exec, stream));
                    gnode::g_launches += e.kernels;
                    return GNODE_OK;
                }
            // captured on a stream of the handle's own (the caller's may be the legacy default stream, which cannot be
            // captured); the instantiated graph is then launched into the caller's stream
            if (!b->capture_stream) {
                cudaStream_t cs_ = nullptr;
                GN_CUDA(cudaStreamCreateWithFlags(&cs_, cudaStreamNonBlocking));
                b->capture_stream = (void*)cs_;
            }
            user_stream = stream;
            stream = (cudaStream_t)b->capture_stream;
            GN_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
            capturing = true;
        }
    }
    const int64_t launches_before = gnode::g_launches;
    auto enqueue = [&]() -> int {
    BwdArgs a;
    a.bv = gn_view(b);
    a.x = x; a.ldx = ldx; a.p = *p;
    a.gx = grad_x; a.ldgx = ldgx;
    a.a = (float*)(ws + pl.off_a);
    a.Sp = (float*)(ws + pl.off_sp); a.Ip = (float*)(ws + pl.off_ip);
    a.AI = (float*)(ws + pl.off_ai); a.G = (float*)(ws + pl.off_g);
    float* pdec = (float*)(ws + pl.off_pdec);
    float* plin = (float*)(ws + pl.off_plin);
    float* penc = (float*)(ws + pl.off_penc);
    a.ew = edge_w; a.ewT = edge_w ? (float*)(ws + pl.total) : nullptr; a.inst_e0 = b->d_inst_e0;
    if (edge_w && b->nnz_total > 0) {            // the weights in transpose order, for the A^T gather of every step
        const int grid = (int)std::min<int64_t>((b->nnz_total + 255) / 256, (int64_t)b->sm_count * 8);
        permute_weights_kernel<<<grid, 256, 0, stream>>>(edge_w, b->d_inst_tmap, b->d_inst_e0, b->n_inst, b->nnz_total,
                                                         (float*)(ws + pl.total));
        GN_LAUNCH_CHECK();
    }
    // adjoint and partial-sum slots start at zero
    GN_CUDA(cudaMemsetAsync(ws + pl.off_a, 0, 3 * M * H * sizeof(float), stream));
    GN_CUDA(cudaMemsetAsync(ws + pl.off_pdec, 0, pl.off_penc - pl.off_pdec, stream));
    // dL/dbeta, dL/dgamma are sums over the reverse steps (columns 3, 4 of grad_x); the encoder stores columns 0..2
    if (grad_x) GN_CUDA(cudaMemset2DAsync(grad_x + 3, (size_t)ldgx * sizeof(float), 0, 2 * sizeof(float), M, stream));
    // dL/dw is a sum over the reverse steps as well (steps without an adjoint add nothing)
    if (grad_edge && b->nnz_total > 0)
        GN_CUDA(cudaMemsetAsync(grad_edge, 0, (size_t)b->nnz_total * sizeof(float), stream));
    auto edge_step = [&](const float* ip) -> int {
        if (!grad_edge) return GNODE_OK;
        bwd_edge_kernel<<<pl.grid_row, ROW_THREADS, 0, stream>>>(a, ip, b->d_inst_e0, grad_edge);
        GN_LAUNCH_CHECK();
        return GNODE_OK;
    };

    auto state = [&](int j) { return traj + (size_t)j * 3 * M * H; };
    // cotangent of grid point j, or null when its probabilities were not emitted (sparse dL/dprobs: the loss of the
    // reference consumes only the grid points int(i/deltaT), ode_nn.py:249-261)
    auto gp = [&](int j) -> const float* { return sel.slot[j] >= 0 ? grad_probs + (size_t)sel.slot[j] * M * 3 : nullptr; };
    auto dec_only = [&](int j) -> int {
        if (!gp(j)) return GNODE_OK;
        a.y = state(j); a.gP = gp(j); a.part = pdec; a.only_dec = 1; a.dt = 0.f;
        bwd_dec_kernel<<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
        GN_LAUNCH_CHECK();
        return GNODE_OK;
    };
    // auxiliary storage of the forward (gnode_rollout_forward_aux): aux[k][0] = I'_k (all k), aux[k][1] = A I'_k (k <= T-2)
    const size_t Mr = (M + TILE - 1) / TILE * TILE, aux_plane = (Mr + 1) * H;
    a.Ipf = nullptr; a.AIf = nullptr;
    auto vjp_step = [&](int j, float dt, bool with_decoder) -> int {
        if (aux && j <= T - 2) {
            // three launches, one neighbour gather: a += D(y_j, gP_j) ; S' -> (G, gzS) ; A^T G -> gzI ; tile kernel
            if (with_decoder) { const int rc2 = dec_only(j); if (rc2) return rc2; }
            a.y = state(j); a.gP = nullptr; a.dt = dt; a.only_dec = 0; a.part = nullptr;
            a.Ipf = aux + (size_t)j * 2 * aux_plane; a.AIf = a.Ipf + aux_plane;
            bwd_transform_g_kernel<<<pl.grid_tile1, NTHREADS, K1_SM_TOTAL, stream>>>(a);
            GN_LAUNCH_CHECK();
            if (edge_w) bwd_gz_kernel<true, true><<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
            else bwd_gz_kernel<true, false><<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
            GN_LAUNCH_CHECK();
            if (const int rc2 = edge_step(a.Ipf)) return rc2;
            a.part = plin;
            return launch_vjp(a, pl.grid_tile3, wgrad, stream);
        }
        a.y = state(j); a.gP = with_decoder ? gp(j) : nullptr; a.dt = dt; a.only_dec = 0;
        a.part = nullptr;
        bwd_transform_kernel<<<pl.grid_tile1, NTHREADS, K1_SM_TOTAL, stream>>>(a);
        GN_LAUNCH_CHECK();
        a.part = pdec;
        if (edge_w) bwd_row_kernel<true><<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
        else bwd_row_kernel<false><<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
        GN_LAUNCH_CHECK();
        a.part = nullptr;
        if (edge_w) bwd_gz_kernel<false, true><<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
        else bwd_gz_kernel<false, false><<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
        GN_LAUNCH_CHECK();
        if (const int rc2 = edge_step(a.Ip)) return rc2;
        a.part = plin;
        return launch_vjp(a, pl.grid_tile3, wgrad, stream);
    };
    int jmax = T - 1;                             // last grid point with a cotangent: the adjoint is zero beyond it
    while (jmax > 0 && sel.slot[jmax] < 0) --jmax;
    if (grad_mode == GNODE_GRAD_ADJOINT) {
        for (int j = jmax; j >= 1; --j)
            if ((rc = vjp_step(j, dt_host[j - 1], true))) return rc;
        if ((rc = dec_only(0))) return rc;
    } else {
        if ((rc = dec_only(T - 1))) return rc;
        for (int j = T - 2; j >= 0; --j) {       // D(y_j) must not enter the cotangent of the VJP at y_j
            // (the adjoint of y_{j+1} is still zero beyond the last grid point with a cotangent: no VJP to take there)
            if (j + 1 <= jmax && (rc = vjp_step(j, dt_host[j], false))) return rc;
            if ((rc = dec_only(j))) return rc;
        }
    }
    a.y = state(0); a.part = wgrad ? penc : nullptr;
    bwd_encoder_kernel<<<pl.grid_row, ROW_THREADS, 0, stream>>>(a);
    GN_LAUNCH_CHECK();
    // (without a parameter gradient the decoder kernels' partial sums are left unread in their slots)
    if (!wgrad) return GNODE_OK;
    // fold the per-block slots into the flat gradient vector (layout of include/gnode_b200.h)
    reduce_partials_kernel<<<(LIN_COUNT + 255) / 256, 256, 0, stream>>>(plin, pl.grid_tile3, LIN_COUNT,
                                                                        grads_out + GNODE_GRAD_OFF_LIN_W);
    GN_LAUNCH_CHECK();
    reduce_partials_kernel<<<1, 256, 0, stream>>>(penc, pl.grid_row, ENC_COUNT, grads_out + GNODE_GRAD_OFF_S1_W);
    GN_LAUNCH_CHECK();
    reduce_partials_kernel<<<(DEC_COUNT + 255) / 256, 256, 0, stream>>>(pdec, pl.grid_row, DEC_COUNT,
                                                                        grads_out + GNODE_GRAD_OFF_L3_W);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
    };
    rc = enqueue();
    if (!capturing) return rc;
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(stream, &graph);
    if (rc != GNODE_OK || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        if (rc == GNODE_OK) { set_error("gnode_rollout_backward: graph capture failed: %s", cudaGetErrorString(ce)); rc = GNODE_ERR_CUDA; }
        return rc;
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) { set_error("gnode_rollout_backward: cudaGraphInstantiate: %s", cudaGetErrorString(ie)); return GNODE_ERR_CUDA; }
    const int64_t kernels = gnode::g_launches - launches_before;          // counted while capturing; nothing ran yet
    if (b->bwd_graphs.size() >= 8) {                                       // small LRU: drop the oldest
        cudaGraphExecDestroy((cudaGraphExec_t)b->bwd_graphs.front().exec);
        b->bwd_graphs.erase(b->bwd_graphs.begin());
    }
    b->bwd_graphs.push_back({key, (void*)exec, kernels});
    GN_CUDA(cudaGraphLaunch(exec, user_stream));
    (void)use_graph;
    return GNODE_OK;
}

extern "C" int gnode_trials_grad(gnode_batch_t b, const float* grad_x, int64_t ldgx, float* grad_beta, float* grad_gamma,
                                 void* stream_) {
    if (!b || !grad_x || ldgx < 5 || !grad_beta || !grad_gamma) {
        set_error("gnode_trials_grad: bad arguments (ldgx=%lld)", (long long)ldgx);
        return GNODE_ERR_ARG;
    }
    int rc = check_current_device(b, "gnode_trials_grad");
    if (rc) return rc;
    if (b->n_inst == 0) return GNODE_OK;
    trials_grad_kernel<<<b->n_inst, TG_THREADS, 0, (cudaStream_t)stream_>>>(gn_view(b), grad_x, ldgx, grad_beta, grad_gamma);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}
