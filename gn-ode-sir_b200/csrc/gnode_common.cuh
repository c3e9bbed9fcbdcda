// Internal declarations shared by the kernels of libgnode_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/gnode_b200.h"

namespace gnode {

constexpr int H = GNODE_H;            // hidden width (64)
constexpr int TILE = 128;             // rows per CTA tile (== UMMA M, == TMEM lanes)
constexpr int NTHREADS = 512;         // 16 warps per CTA
constexpr int CHUNKS = H / 4;         // 16-byte chunks per row (16)

// ---- host side ------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

#define GN_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e_ = (call);                                                   \
        if (e_ != cudaSuccess) {                                                   \
            gnode::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call,          \
                             cudaGetErrorString(e_));                              \
            return GNODE_ERR_CUDA;                                                 \
        }                                                                          \
    } while (0)

#define GN_LAUNCH_CHECK()                                                          \
    do {                                                                           \
        gnode::g_launches++;                                                       \
        cudaError_t e_ = cudaGetLastError();                                       \
        if (e_ != cudaSuccess) {                                                   \
            gnode::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__,      \
                             cudaGetErrorString(e_));                              \
            return GNODE_ERR_CUDA;                                                 \
        }                                                                          \
    } while (0)

}  // namespace gnode

struct gnode_batch;
namespace gnode {
// Host-side description of which grid points are emitted: slot[k] = row block of `probs` for grid point k, or -1.
struct OutSel {
    std::vector<int> slot;
    int n_out = 0, start = 0, stride = 1;
    bool arithmetic = true;
};
int make_out_sel(int T, const int32_t* out_steps, int32_t n_out, OutSel* o, const char* what);
// GNODE_ERR_ARG unless the handle's device is the calling thread's current device
int check_current_device(const gnode_batch* b, const char* what);
// weighted reverse sweep: uploads (once) the transpose -> forward entry maps of the batch's graphs and the per-instance
// table of them (b->d_inst_tmap); a blocking call, made before any capture starts
int ensure_transpose_maps(gnode_batch* b);
}  // namespace gnode

// One graph: CSR pattern (and its transpose) resident in HBM.
struct gnode_graph {
    int32_t n = 0;
    int64_t nnz = 0;
    int32_t max_degree = 0;
    int32_t symmetric = 0;
    int32_t* d_rowptr = nullptr;    // [n+1]
    int32_t* d_colidx = nullptr;    // [nnz]
    int32_t* d_rowptr_t = nullptr;  // transpose (aliases the above when symmetric)
    int32_t* d_colidx_t = nullptr;
    std::vector<int32_t> h_rowptr;  // host copy (tile cost model at batch creation)
    // transpose entry k (of the counting sort below) is forward entry h_tmap[k]: the order a weight vector takes for the
    // A^T gather of the weighted reverse sweep (symmetric graphs too: the pattern is shared, the weights need not be)
    std::vector<int32_t> h_tmap;
    int32_t* d_tmap = nullptr;      // uploaded on first weighted use
    int device = 0;
};

// Device-visible description of one instance (one diagonal block).
struct GnInstance {
    const int32_t* rowptr;
    const int32_t* colidx;
    const int32_t* rowptr_t;
    const int32_t* colidx_t;
    int32_t row0;   // first global row
    int32_t n;      // rows in this instance
};

struct gnode_batch {
    int64_t M = 0;
    int32_t n_inst = 0;
    int32_t n_tiles = 0;
    int64_t nnz_total = 0;
    GnInstance* d_inst = nullptr;    // [n_inst]
    int64_t* d_inst_e0 = nullptr;    // [n_inst] first entry of each instance in the batch's edge vector (edge gradients)
    int32_t* d_tile_inst = nullptr;  // [n_tiles] instance that owns the first row of each tile
    int32_t* d_tile_order = nullptr; // [n_tiles] processing order: hub-heavy tiles first, then row-major
    int2* d_sched = nullptr;         // [n_tiles] by sequence number: {tile, first row of the look-ahead I' prefetch or -1}
    int4* d_tile_meta = nullptr;     // [n_tiles] {first CSR entry, entry count, owning instance, bit 0: inside one instance, bit 1: hub relay}
    int4* d_sub_meta = nullptr;      // [2 n_tiles] the same for the two 64-row halves of every tile
    uint8_t* d_tile_perm = nullptr;  // [n_tiles][64][4] work items of the gather: tile rows {a, b | c, d} summed by one warp in one round trip
    int device = 0;
    int sm_count = 0;
    // captured reverse sweeps of launch-bound batches (gnode_rollout_backward): key of all arguments -> cudaGraphExec_t
    struct BwdGraph { uint64_t key; void* exec; int64_t kernels; };
    std::vector<BwdGraph> bwd_graphs;
    void* capture_stream = nullptr;      // cudaStream_t used only to capture those graphs
    std::vector<gnode_graph*> graphs;    // the instances' graphs (the caller keeps them alive while the batch lives)
    const int32_t** d_inst_tmap = nullptr;   // [n_inst] graph's transpose map per instance (weighted sweeps), or null
};

// Kernel-side view of a batch.
struct GnBatchView {
    const GnInstance* inst;
    const int32_t* tile_inst;
    const int32_t* tile_order;
    const int2* sched;
    const int4* tile_meta;
    const int4* sub_meta;
    const uint8_t* tile_perm;
    int32_t n_inst;
    int32_t n_tiles;
    int32_t M;
};

inline GnBatchView gn_view(const gnode_batch* b) {
    GnBatchView v;
    v.inst = b->d_inst;
    v.tile_inst = b->d_tile_inst;
    v.tile_order = b->d_tile_order;
    v.sched = b->d_sched;
    v.tile_meta = b->d_tile_meta;
    v.sub_meta = b->d_sub_meta;
    v.tile_perm = b->d_tile_perm;
    v.n_inst = b->n_inst;
    v.n_tiles = b->n_tiles;
    v.M = (int32_t)b->M;
    return v;
}

#ifdef __CUDACC__
namespace gnode {

// Byte offset of the 16-byte chunk c4 (0..15) of tile row r (0..127) inside a
// 32 KB tile buffer laid out as the canonical UMMA K-major SWIZZLE_128B operand:
// two K-blocks of 32 fp32 (128 B), each [128 rows][128 B] with 16-B chunks XORed by
// (row & 7).  Thread-per-row and row-per-half-warp accesses are both conflict-free.
__device__ __forceinline__ int sw_off(int r, int c4) {
    return ((c4 >> 3) << 14) + (r << 7) + ((((c4 & 7) ^ (r & 7))) << 4);
}

// ---- packed fp32 pairs (sm_100: add / mul / fma .f32x2, SASS FADD2 / FMUL2 / FFMA2): two IEEE round-to-nearest operations
// per instruction -- the same bits as the scalar form, half the issue slots. The step kernels are bound by their chain of
// dependent phases and by issue slots, not by the FP32 pipe, so the row sums, the SIR update and the sigmoid run on pairs.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
// acc += v, component by component (the sequential row sums: same additions, same order)
__device__ __forceinline__ void add4(float4& acc, const float4& v) {
    unpack2(add2(pack2(acc.x, acc.y), pack2(v.x, v.y)), acc.x, acc.y);
    unpack2(add2(pack2(acc.z, acc.w), pack2(v.z, v.w)), acc.z, acc.w);
}

// w * v component by component, each product rounded on its own: scalar mul.rn is never contracted with the add that
// follows (the weighted neighbour sums add fl(w v) in the same order as the binary ones add v; w = 1 gives their bits)
__device__ __forceinline__ float4 mul4(float w, const float4& v) {
    return make_float4(__fmul_rn(w, v.x), __fmul_rn(w, v.y), __fmul_rn(w, v.z), __fmul_rn(w, v.w));
}

__device__ __forceinline__ float4 lds4(const unsigned char* base, int off) {
    return *reinterpret_cast<const float4*>(base + off);
}
__device__ __forceinline__ void sts4(unsigned char* base, int off, float4 v) {
    *reinterpret_cast<float4*>(base + off) = v;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// streaming (read-once / write-once) accesses: keep them out of L1
__device__ __forceinline__ float4 ldg4_stream(const float* p) { return __ldcs(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void stg4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void stg4_stream(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }

// ---- L2 eviction-priority hints (createpolicy + .L2::cache_hint): the I' rows that neighbours gather
// are kept (evict_last); state rows and outputs that are touched once stream through (evict_first)
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p; asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p; asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t p; asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ float4 ldg4_hint(const float* p, uint64_t pol) {
    float4 v;
    asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void stg4_hint(float* p, float4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;"
                 ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}
__device__ __forceinline__ void prefetch_l2_bulk_hint(const void* p, uint32_t bytes, uint64_t pol) {
    asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(p), "r"(bytes), "l"(pol) : "memory");
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// sigmoid(z) = 1 / (1 + exp(-z))   (nn.Sigmoid, ode_nn_ngraph_sim.py:63)
//   FAST = false: expf + IEEE division              (3.2 ulp measured on B200, tools/sigmoid_err.cu)
//   FAST = true : 2^t by MUFU.EX2 with the rounding error of t = -z*log2(e) compensated to first
//                 order, then MUFU.RCP                (4.6 ulp measured for |z| <= 40; 8 instructions)
template <bool FAST>
__device__ __forceinline__ float sigmoid_t(float z) {
    if (FAST) {
        const float c = -1.4426950408889634f, clo = -1.9259629911266175e-08f;   // -log2(e) = c + clo
        const float th = z * c;
        const float tl = fmaf(z, clo, fmaf(z, c, -th));
        float e, r;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(th));
        e = e * fmaf(tl, 0.6931471805599453f, 1.0f);      // (inf or 0) * ~1 stays inf or 0: no NaN at the tails
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
        return r;
    } else {
        return 1.0f / (1.0f + expf(-z));
    }
}

// The same sigmoid on a pair. FAST: op for op the scalar code above as the compiler emits it (the final 1 + e f is an FMA
// there), with the negations folded into the constants: fma(z, -c, th) = -fma(z, c, -th) exactly (it is the exact residual
// of the product) and fma(-tl, -ln2, 1) = fma(tl, ln2, 1) -- the same bits (tests/test_variants_gpu.py compares the kernels
// that use the pair form with the one that uses the scalar form).
template <bool FAST>
__device__ __forceinline__ f32x2 sigmoid2_t(f32x2 z) {
    float z0, z1;
    if (FAST) {
        const float c = -1.4426950408889634f, clo = -1.9259629911266175e-08f, ln2 = 0.6931471805599453f;
        const f32x2 th = mul2(z, pack2(c, c));
        const f32x2 r = fma2(z, pack2(-c, -c), th);
        const f32x2 ntl = fma2(z, pack2(-clo, -clo), r);
        const f32x2 f = fma2(ntl, pack2(-ln2, -ln2), pack2(1.0f, 1.0f));
        unpack2(th, z0, z1);
        float e0, e1, r0, r1;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(z0));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(z1));
        unpack2(fma2(pack2(e0, e1), f, pack2(1.0f, 1.0f)), z0, z1);
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(z0));
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(z1));
        return pack2(r0, r1);
    }
    unpack2(z, z0, z1);
    return pack2(sigmoid_t<false>(z0), sigmoid_t<false>(z1));
}

}  // namespace gnode
#endif
