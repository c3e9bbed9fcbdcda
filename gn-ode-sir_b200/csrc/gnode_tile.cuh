// Tile-level device helpers shared by the forward and backward kernels.
#pragma once
#include "gnode_common.cuh"

namespace gnode {

// Z = X W^T (X: swizzled 128x64 tile, W: [h][k]) ; dst = sigmoid(Z + b), swizzled.
// 256 threads: thread (r0 = tid&63, q = tid>>6) owns rows r0, r0+64 x columns [16q,16q+16).
template <bool FAST>
__device__ __forceinline__ void gemm_sigmoid(const unsigned char* Xs, const float* Ws, const float* bs,
                                             unsigned char* dst, int tid) {
    if (tid >= 256) return;
    const int r0 = tid & 63, q = tid >> 6;
    float a0[16], a1[16];
#pragma unroll
    for (int h = 0; h < 16; ++h) { a0[h] = 0.f; a1[h] = 0.f; }
    const float* wq = Ws + (16 * q) * H;
#pragma unroll 2
    for (int c4 = 0; c4 < CHUNKS; ++c4) {
        const float4 xa = lds4(Xs, sw_off(r0, c4));
        const float4 xb = lds4(Xs, sw_off(r0 + 64, c4));
#pragma unroll
        for (int h = 0; h < 16; ++h) {
            const float4 w = *reinterpret_cast<const float4*>(wq + h * H + 4 * c4);
            a0[h] = fmaf(xa.x, w.x, a0[h]); a0[h] = fmaf(xa.y, w.y, a0[h]);
            a0[h] = fmaf(xa.z, w.z, a0[h]); a0[h] = fmaf(xa.w, w.w, a0[h]);
            a1[h] = fmaf(xb.x, w.x, a1[h]); a1[h] = fmaf(xb.y, w.y, a1[h]);
            a1[h] = fmaf(xb.z, w.z, a1[h]); a1[h] = fmaf(xb.w, w.w, a1[h]);
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * q + 4 * j);
        float4 o0, o1;
        o0.x = sigmoid_t<FAST>(a0[4 * j + 0] + bb.x); o0.y = sigmoid_t<FAST>(a0[4 * j + 1] + bb.y);
        o0.z = sigmoid_t<FAST>(a0[4 * j + 2] + bb.z); o0.w = sigmoid_t<FAST>(a0[4 * j + 3] + bb.w);
        o1.x = sigmoid_t<FAST>(a1[4 * j + 0] + bb.x); o1.y = sigmoid_t<FAST>(a1[4 * j + 1] + bb.y);
        o1.z = sigmoid_t<FAST>(a1[4 * j + 2] + bb.z); o1.w = sigmoid_t<FAST>(a1[4 * j + 3] + bb.w);
        sts4(dst, sw_off(r0, 4 * q + j), o0);
        sts4(dst, sw_off(r0 + 64, 4 * q + j), o1);
    }
}

// coalesced HBM rows -> swizzled tile (rows past M are zero-filled)
__device__ __forceinline__ void load_tile(unsigned char* dst, const float* src, int64_t tile0, int M, int tid) {
    for (int idx = tid; idx < TILE * CHUNKS; idx += NTHREADS) {
        const int rr = idx >> 4, c4 = idx & 15;
        const int64_t g = tile0 + rr;
        if (g < M) cp_async16(dst + sw_off(rr, c4), src + (size_t)g * H + 4 * c4);
        else sts4(dst, sw_off(rr, c4), make_float4(0.f, 0.f, 0.f, 0.f));
    }
    cp_async_wait_all();
}

__device__ __forceinline__ void store_tile(float* dst, const unsigned char* src, int64_t tile0, int M, int tid) {
    for (int idx = tid; idx < TILE * CHUNKS; idx += NTHREADS) {
        const int rr = idx >> 4, c4 = idx & 15;
        const int64_t g = tile0 + rr;
        if (g < M) stg4(dst + (size_t)g * H + 4 * c4, lds4(src, sw_off(rr, c4)));
    }
}

__device__ __forceinline__ float dot4(float4 a, float4 b) {
    return fmaf(a.w, b.w, fmaf(a.z, b.z, fmaf(a.y, b.y, a.x * b.x)));
}


// V = G W (G: swizzled 128x64 tile of cotangents wrt z, W: [h][j] row-major): v[r][j] = sum_h g[r][h] W[h][j].
// 256 threads (t = 0..255): thread (r0 = t&63, q = t>>6) owns rows r0, r0+64 x columns [16q,16q+16).
__device__ __forceinline__ void gemm_gw(const unsigned char* Gs, const float* Ws, int t, float (&a0)[16], float (&a1)[16]) {
    const int r0 = t & 63, q = t >> 6;
#pragma unroll
    for (int j = 0; j < 16; ++j) { a0[j] = 0.f; a1[j] = 0.f; }
#pragma unroll 2
    for (int hc = 0; hc < CHUNKS; ++hc) {
        const float4 ga = lds4(Gs, sw_off(r0, hc));
        const float4 gb = lds4(Gs, sw_off(r0 + 64, hc));
        const float gav[4] = {ga.x, ga.y, ga.z, ga.w};
        const float gbv[4] = {gb.x, gb.y, gb.z, gb.w};
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) {
            const float* wr = Ws + (4 * hc + hh) * H + 16 * q;
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4) {
                const float4 w = *reinterpret_cast<const float4*>(wr + jj);
                a0[jj + 0] = fmaf(gav[hh], w.x, a0[jj + 0]); a0[jj + 1] = fmaf(gav[hh], w.y, a0[jj + 1]);
                a0[jj + 2] = fmaf(gav[hh], w.z, a0[jj + 2]); a0[jj + 3] = fmaf(gav[hh], w.w, a0[jj + 3]);
                a1[jj + 0] = fmaf(gbv[hh], w.x, a1[jj + 0]); a1[jj + 1] = fmaf(gbv[hh], w.y, a1[jj + 1]);
                a1[jj + 2] = fmaf(gbv[hh], w.z, a1[jj + 2]); a1[jj + 3] = fmaf(gbv[hh], w.w, a1[jj + 3]);
            }
        }
    }
}

// instance that owns global row r (binary search over the small, cached instance table)
__device__ __forceinline__ int find_instance(const GnBatchView& bv, int64_t r) {
    int lo = 0, hi = bv.n_inst - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (bv.inst[mid].row0 <= r) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Sequential ascending-column neighbour sum of one row by a half-warp (lane l owns 16 B of
// the row); both half-warps of the warp iterate together (trip count = max of the two
// degrees) so that full-mask shuffles stay convergent. 8 neighbour rows in flight per lane.
// W: weighted sum, acc += fl(w_e src[c_e]) with w_e = wp[e0 + j] (the entries' weights in CSR order).
template <bool W = false>
__device__ __forceinline__ float4 gather_row(const float* __restrict__ src, const int32_t* ci, int e0, int deg,
                                              int row0, int l, int lane, const float* wp = nullptr) {
    const int degmax = max(deg, __shfl_xor_sync(0xffffffffu, deg, 16));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int eb = 0; eb < degmax; eb += 16) {
        const int mine = (eb + l < deg) ? ci[e0 + eb + l] + row0 : -1;
        const float mw = (W && eb + l < deg) ? wp[e0 + eb + l] : 0.f;
#pragma unroll
        for (int jb = 0; jb < 16; jb += 8) {
            if (eb + jb < degmax) {
                float4 v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = __shfl_sync(0xffffffffu, mine, (lane & 16) + jb + j);
                    v[j] = (c >= 0) ? ldg4(src + (size_t)c * H + 4 * l) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                if (W) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = mul4(__shfl_sync(0xffffffffu, mw, (lane & 16) + jb + j), v[j]);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) add4(acc, v[j]);
            }
        }
    }
    return acc;
}

}  // namespace gnode
