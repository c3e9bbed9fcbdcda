// step_stream_kernel: the fused Euler step with the contiguous S_k stream fed by TMA (included by gnode_forward.cu).
//
// Same tile pipeline as step_dual_kernel (one 1024-thread CTA per SM = two 512-thread pipelines of 128-row tiles that
// share the [W; W3] operand), with these changes that take bytes and LSU work out of the step:
//   * the S_k tile of the NEXT tile is fetched by two TMA tensor loads (cp.async.bulk.tensor.2d, SWIZZLE_128B boxes of
//     32 x 128 fp32, SASS UTMALDG) issued by the otherwise idle metadata thread as soon as GEMM2 of the current tile
//     has finished reading the operand buffer: no registers, no LSU wavefronts and no L1 lines for this stream, and the
//     load's latency hides behind the I' epilogue and the tile turn-over;
//   * the tile lands directly in the canonical UMMA K-major operand layout and IS the `hi` operand: tcgen05.mma kind::tf32
//     reads only the top 19 bits of each 32-bit element (tools/umma_lowbits_probe.cu), i.e. the raw fp32 word is
//     hi = trunc_tf32(x) to the tensor core and still x to the row update that reads S_k from the same tile later. Nothing
//     is converted or written back; the threads only add lo = rna_tf32(x - hi) in the second tile (truncation split,
//     |x - hi - lo| <= 2^-21 |x|). S_k is read from HBM/L2 ONCE per step (step_dual_kernel: twice). The rna split packed in
//     place (round 2h: hi = rna_tf32(x) in the top bits, the low 13 bits of x kept: tf32_pack / tf32_unpack) stays as an A/B
//     variant: one more shared-memory store per element, +3 % time for half the split residual;
//   * [W; W3] is ONE B operand with its hi and lo parts stacked along N (N = 160, umma::issue_split_gemm160): every A tile
//     is read from shared memory once per GEMM instead of twice, 16 MMAs instead of 32. The tensor core fetches operands
//     over the shared-memory port the LSU uses: without any MMA the step is 12 % faster, with the stacked operand 2.7 %
//     (profiles/r2n_ab_ablations.log, r2o_ab_gemm_variants.log);
//   * the rows of a tile are gathered in degree-sorted groups (gnode_batch_create: tile_perm): the two half-warps of a warp
//     run the same trip count and few padding slots read the all-zero row, and rows with at most 6 neighbours are summed
//     two per half-warp in one memory round trip;
//   * the neighbour sum is folded into S' in place (AI * S', the first product of dS, ode_nn_ngraph_sim.py:75), so the
//     parked value needs no buffer of its own. (Measured and rejected: the gathering half-warp performing the whole row
//     update with its own I_k / I'_k rows requested together with the neighbour rows -- 1.64e9 vs 1.66e9 node-steps/s,
//     profiles/r2b_ab_step_kernels.log; the first row pair gathered while GEMM1 runs -- 1.667e9 vs 1.683e9; the own rows
//     of the first update pass requested before the barrier -- 1.687e9 vs 1.683e9, noise; profiles/r2d_ab_stream_overlaps.log.)
// Arithmetic of the update is the reference's, op for op (SURVEY appendix A); S, I, R and the probabilities are bitwise
// those of step_dual_kernel.
#pragma once

namespace gnode {

struct StreamCfg {
    static constexpr int PT = D_THREADS / 2;               // threads per pipeline
    static constexpr int TR = 128;                         // tile rows = UMMA M
    static constexpr int RSTEP = PT / 16;                  // rows per pass of the row-per-half-warp loops (32)
    static constexpr int PASS = RSTEP * 128;               // byte offset between the passes' rows in an operand tile
    static constexpr int CAP = 3 * PT;                     // colidx entries staged per tile (weighted: CAP / 2, and their weights)
    static constexpr int HUB_DEG = 512;
    static constexpr int KBLK = TR * 128;                  // bytes of one K-block (32 fp32) of the A operand
    static constexpr int P_X = 0;                          // raw S_k (= hi operand) -> I_{k+1} raw (= hi operand of GEMM2)
    static constexpr int P_L = 2 * KBLK;                   // lo operand -> S' -> AI * S' -> lo of I_{k+1} -> I'_{k+1} staging
    static constexpr int P_MBAR = 4 * KBLK;                // GEMM mbarrier (8) + row-pair counter (4) + pad (4) + S-load mbarrier (8)
                                                           // + weighted: the coming tile's weights, edge_w + inst_e0[inst] + ebase (8)
    static constexpr int P_META = P_MBAR + 32;             // DTileMeta of the coming tile (48 B)
    static constexpr int P_BG = P_META + 48;               // beta[TR], gamma[TR]
    static constexpr int P_RP = P_BG + 2 * TR * 4;         // rowptr slice [TR + 1] (+pad, hub mask)
    static constexpr int P_HS = P_RP + TR * 4 + 32;        // hid(S_k) [TR][4]
    static constexpr int P_HR = P_HS + TR * 16;            // hid(R_k) / W3 I'_k [TR][4]
    static constexpr int P_CI = P_HR + TR * 16;            // colidx slice + 64 B over-read pad
    static constexpr int P_PM = P_CI + CAP * 4 + 64;       // work items of the gather: [64] x {a, b | c, d} tile rows (256 B)
    static constexpr int P_ZK = P_PM;                      // step 0 from descriptors (no work items): seed flag of every tile row [TR]
    static constexpr int P_ZI = P_CI;                      // and, in tiles that span instances (no staged colidx slice), its instance [TR]
    static constexpr int P_BYTES = ((P_PM + 256 + 1023) / 1024) * 1024;
    static constexpr int TOTAL = D_SHARED + 2 * P_BYTES + 1024;
    static constexpr int TMEM_COLS = 512;                 // two [128 x 160] fp32 accumulators, 256 columns apart
    static_assert(TOTAL + 1024 <= 200704, "stay inside the 196 KB shared-memory carve-out (60 KB of L1 left)");
    static __device__ __forceinline__ int sw(int r, int c4) { return (c4 >> 3) * KBLK + (r << 7) + (((c4 & 7) ^ (r & 7)) << 4); }
};

// TMA tensor load of one box (global -> shared memory), completion counted in bytes on an mbarrier
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* tm, void* smem_dst, uint64_t* bar, int c0, int c1, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(umma::smem_u32(smem_dst)), "l"(tm), "r"(c0), "r"(c1), "r"(umma::smem_u32(bar)), "l"(pol) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(umma::smem_u32(bar)), "r"(bytes) : "memory");
}

// The fp32 tile that the TMA delivered is turned into the hi operand IN PLACE without losing the fp32 value: the tensor
// core reads only the top 19 bits of an element (tools/umma_lowbits_probe.cu: the low 13 mantissa bits are ignored,
// i.e. truncation), so the word  p = bits(rna_tf32(x)) | (bits(x) & 0x1FFF)  is seen by tcgen05.mma as hi = rna_tf32(x)
// -- the same hi as a separate operand tile would hold -- while x is recovered exactly as
// bits(x) = p - ((p & 0x1000) << 1)  (rounding up happened iff bit 12 of x is set; it added 0x2000 to the pattern).
// lo = rna_tf32(x - hi) as in the LDG-fed kernel: the split product is bitwise the same.
__device__ __forceinline__ float tf32_pack(float x, float& lo) {
    const float hi = umma::tf32_rna(x);
    lo = umma::tf32_rna(x - hi);
    return __uint_as_float(__float_as_uint(hi) | (__float_as_uint(x) & 0x1FFFu));
}
__device__ __forceinline__ float tf32_unpack(float p) {
    const uint32_t b = __float_as_uint(p);
    return __uint_as_float(b - ((b & 0x1000u) << 1));
}
__device__ __forceinline__ float4 tf32_pack4(float4 x, float4& lo) {
    return make_float4(tf32_pack(x.x, lo.x), tf32_pack(x.y, lo.y), tf32_pack(x.z, lo.z), tf32_pack(x.w, lo.w));
}
__device__ __forceinline__ float4 tf32_unpack4(float4 p) {
    return make_float4(tf32_unpack(p.x), tf32_unpack(p.y), tf32_unpack(p.z), tf32_unpack(p.w));
}

// neighbour sum specialised by the pair's larger degree: 1..MAXR rows in one round trip, longer rows in rounds of 8
// (W: weighted, the weight of neighbour j at wp[j])
template <int MAXR, bool W = false>
__device__ __forceinline__ float4 gather_smem_zm(const float* __restrict__ lane_base, const int* cp, int deg, int zrow, uint64_t pol,
                                                 const float* wp = nullptr) {
    const int degm = max(deg, __shfl_xor_sync(0xffffffffu, deg, 16));
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int j = 0;
    for (; degm - j > MAXR; j += 8) gather_exact<8, W>(acc, lane_base, cp, j, deg, zrow, pol, wp);
    switch (degm - j) {
        case 12: if (MAXR >= 12) gather_exact<12, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 11: if (MAXR >= 11) gather_exact<11, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 10: if (MAXR >= 10) gather_exact<10, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 9: if (MAXR >= 9) gather_exact<9, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 8: gather_exact<8, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 7: gather_exact<7, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 6: gather_exact<6, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 5: gather_exact<5, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 4: gather_exact<4, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 3: gather_exact<3, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 2: gather_exact<2, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        case 1: gather_exact<1, W>(acc, lane_base, cp, j, deg, zrow, pol, wp); break;
        default: break;
    }
    return acc;
}

// four-row item: the lane's chunks of two rows of at most D neighbours each, all 2 D loads in one round trip; each row is
// summed alone in ascending column order (slots past its degree read the all-zero row: + 0 is exact; W: weighted, the
// weights at wpa / wpb are read after the loads are issued, pad slots weigh 0)
template <int D, bool W = false>
__device__ __forceinline__ void gather_two_rows(const float* __restrict__ lane_base, const int* cpa, int da, const int* cpb, int db,
                                                int zrow, uint64_t pol, float4& sa, float4& sb, const float* wpa, const float* wpb) {
    float4 v[2 * D + 1];
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const int c = (k < da) ? cpa[k] : zrow;
        v[k] = ldg4_hint(lane_base + (size_t)(unsigned)c * H, pol);
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        const int c = (k < db) ? cpb[k] : zrow;
        v[D + k] = ldg4_hint(lane_base + (size_t)(unsigned)c * H, pol);
    }
    sa = make_float4(0.f, 0.f, 0.f, 0.f); sb = sa;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        if (W) v[k] = mul4(k < da ? wpa[k] : 0.f, v[k]);
        add4(sa, v[k]);
    }
#pragma unroll
    for (int k = 0; k < D; ++k) {
        if (W) v[D + k] = mul4(k < db ? wpb[k] : 0.f, v[D + k]);
        add4(sb, v[D + k]);
    }
}
template <bool W = false>
__device__ __forceinline__ void gather_quad(const float* __restrict__ lane_base, const int* cpa, int da, const int* cpb, int db,
                                            int dmax, int zrow, uint64_t pol, float4& sa, float4& sb,
                                            const float* wpa = nullptr, const float* wpb = nullptr) {
    sa = make_float4(0.f, 0.f, 0.f, 0.f); sb = sa;
    switch (dmax) {                                      // warp-uniform
        case 6: gather_two_rows<6, W>(lane_base, cpa, da, cpb, db, zrow, pol, sa, sb, wpa, wpb); break;
        case 5: gather_two_rows<5, W>(lane_base, cpa, da, cpb, db, zrow, pol, sa, sb, wpa, wpb); break;
        case 4: gather_two_rows<4, W>(lane_base, cpa, da, cpb, db, zrow, pol, sa, sb, wpa, wpb); break;
        case 3: gather_two_rows<3, W>(lane_base, cpa, da, cpb, db, zrow, pol, sa, sb, wpa, wpb); break;
        case 2: gather_two_rows<2, W>(lane_base, cpa, da, cpb, db, zrow, pol, sa, sb, wpa, wpb); break;
        case 1: gather_two_rows<1, W>(lane_base, cpa, da, cpb, db, zrow, pol, sa, sb, wpa, wpb); break;
        default: break;
    }
}

// per-step operands (persistent rollout: derived per Euler step by one thread)
struct SStep {
    const float* y_in; float* y_out;
    const float* ip_in; float* ip_out;
    float* probs; int* counter;
    const CUtensorMap* tm;        // I'_{k+1} store
    const CUtensorMap* tms;       // S_k load
    int srow0;                    // row coordinate of the S plane's first row in tms
    int iprow0;                   // row coordinate of the I'_{k+1} plane's first row in tm
    float* ai_out;                // training with auxiliary storage: AI_k = A I'_k of every row (read by the reverse sweep), or null
    float dt;
};

// OPT bit 0: no block barrier after the I' store (see P5); bit 7 (ZS): Euler step 0 of a descriptor-fed inference rollout
// fused with the encoder. There y_0 has two kinds of rows (seed: I0 = 1, S0 = 0; susceptible: S0 = 1, I0 = 0;
// ode_nn_ngraph_sim.py:371-390), so nothing is read but the CSR, a seed bitmap and the two-row table of
// trials_table_kernel: the S_0 tile is synthesised in shared memory, the neighbour sum is the same sequence of additions
// over the two possible I'_0 rows (bitwise the gather of the encoder's I'_0 plane), I_0 / I'_0 / hid(R_0) / probs[0] come
// from the table. Neither y_0 nor I'_0 is ever written: the launch stores y_1, I'_1, hid(I_1), hid(R_1), beta / gamma.
// OPT bit 8 (WGT): weighted neighbour sum AI[r] = sum over stored (r, c), ascending c, of fl(w_rc I'[c]) -- every product
// rounded on its own (mul4), then added in the binary kernel's order, so w = 1 gives the binary bits and w = 0 those of a
// graph without the entry. The staged window holds CAP / 2 column indices and their CAP / 2 weights; rows past it take the
// global-list path (column indices and weights from global memory), as rows past the whole window do in the binary kernel.
template <bool FAST, bool PERSIST, bool RF, int OPT>
__global__ void __launch_bounds__(D_THREADS, 1) step_stream_kernel(const __grid_constant__ StepArgs a) {
    using C = StreamCfg;
    constexpr bool ZS = (OPT & 128) != 0;
    constexpr bool WGT = (OPT & 256) != 0;
    static_assert(!(ZS && WGT), "step 0 from descriptors is not weighted");
    constexpr int CAPS = WGT ? C::CAP / 2 : C::CAP;                   // column indices staged per tile
    static_assert(!ZS || (RF && !PERSIST && (OPT & 64)), "step 0 from descriptors: inference without an R plane, one launch, raw S tile");
    constexpr int PT = C::PT, TR = C::TR, RSTEP = C::RSTEP, PASS = C::PASS;
    // The dynamic shared memory of this kernel starts at a 1024-byte boundary of the shared window (declared so, and
    // checked once): with a base the compiler knows, every operand-tile address is the symbol plus a constant instead of
    // an alignment term that was rematerialised (S2UR SR_CgaCtaId, ULEA, ULOP3 ...) at 23 places of the 64-register kernel.
    extern __shared__ __align__(1024) unsigned char smem_al[];
    unsigned char* smem = smem_al;
    if ((umma::smem_u32(smem_al) & 1023u) != 0u) __trap();
    const int tid = threadIdx.x;
    const int half = __shfl_sync(0xffffffffu, tid / PT, 0);          // pipeline index, provably warp-uniform
    const int t = tid & (PT - 1), lane = t & 31;
    const int warp = __shfl_sync(0xffffffffu, t >> 5, 0);            // warp index inside the pipeline
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
    uint64_t* sbar = reinterpret_cast<uint64_t*>(hb + C::P_MBAR + 16);
    DTileMeta* meta = reinterpret_cast<DTileMeta*>(hb + C::P_META);
    float* bg_s = reinterpret_cast<float*>(hb + C::P_BG);
    int* rp_s = reinterpret_cast<int*>(hb + C::P_RP);
    float* hs_s = reinterpret_cast<float*>(hb + C::P_HS);
    float* hr_s = reinterpret_cast<float*>(hb + C::P_HR);
    int* ci_s = reinterpret_cast<int*>(hb + C::P_CI);
    const float* wt_s = reinterpret_cast<const float*>(ci_s + CAPS);  // WGT: the staged entries' weights
    const float** wslot = reinterpret_cast<const float**>(hb + C::P_MBAR + 24);   // WGT: weights of the tile's entries
    unsigned* hub_mask = reinterpret_cast<unsigned*>(rp_s + TR + 2);
    const uint32_t* items_s = reinterpret_cast<const uint32_t*>(hb + C::P_PM);
    unsigned char* kind_s = hb + C::P_ZK;                             // ZS: 1 = seed row
    int* zinst_s = reinterpret_cast<int*>(hb + C::P_ZI);              // ZS: instance of every tile row
    const int bar_id = 1 + half;
#define HSYNC() umma::bar_sync(bar_id, PT)

    const int M = a.bv.M;
    const size_t plane = (size_t)M * H;
    const int n_tiles = a.bv.n_tiles;
    const int off0 = C::sw(hw, l);
    const uint64_t pol_keep = l2_policy_evict_last();
    const uint64_t pol_stream = l2_policy_evict_first();

    SStep* stp = reinterpret_cast<SStep*>(smem + D_TSLOT + 16);
    static_assert(D_TSLOT + 16 + sizeof(SStep) <= D_SHARED, "SStep overflows the shared part");
#define STP(f) (PERSIST ? stp->f : a.f)
#define STP_TM() (PERSIST ? stp->tm : &a.tm_ip_out)
#define STP_TMS() (PERSIST ? stp->tms : &a.tm_s_in)
#define STP_SROW0() (PERSIST ? stp->srow0 : 0)
#define STP_IPROW0() (PERSIST ? stp->iprow0 : 0)

    // one thread: draw the next sequence number and resolve its metadata (3 dependent loads of small tables)
    auto fetch_meta = [&](int k) {
        const int first = (int)blockIdx.x + half * (int)gridDim.x;
        const int seq = k == 0 ? first : (STP(counter) ? 2 * (int)gridDim.x + atomicAdd(STP(counter), 1) : first + 2 * k * (int)gridDim.x);
        DTileMeta m;
        m.seq = seq; m.rowptr = nullptr; m.colidx = nullptr;
        m.tile0 = 0; m.nrows = 0; m.i_row0 = 0; m.single = 0; m.ebase = 0; m.ecnt = 0; m.inst0 = 0;
        if (seq < n_tiles) {
            const int tile = a.bv.tile_order[seq];
            const int4 tm = a.bv.tile_meta[tile];                     // {ebase, ecnt, inst0, single}
            const GnInstance I = a.bv.inst[tm.z];
            m.tile0 = tile * TILE;
            m.nrows = max(0, min(TR, M - m.tile0));
            m.i_row0 = I.row0; m.single = tm.w; m.ebase = tm.x; m.ecnt = tm.y; m.inst0 = tm.z;
            m.rowptr = I.rowptr + (m.tile0 - I.row0);
            m.colidx = I.colidx;
        }
        *meta = m;
        if (WGT && seq < n_tiles) *wslot = a.edge_w + a.inst_e0[m.inst0] + m.ebase;
    };
    // the same thread: request the S_k rows of that tile (raw fp32, operand layout) into Xs
    auto issue_s_load = [&]() {
        if (ZS) {                                                     // nothing to load: P1 synthesises the S_0 rows
            if (meta->seq < n_tiles) umma::mbar_arrive(sbar);
            return;
        }
        if (meta->seq < n_tiles) {
            mbar_expect_tx(sbar, 2 * C::KBLK);
            const int r0 = STP_SROW0() + meta->tile0;
            tma_load_2d(STP_TMS(), Xs, sbar, 0, r0, pol_stream);
            tma_load_2d(STP_TMS(), Xs + C::KBLK, sbar, 32, r0, pol_stream);
        }
    };

    constexpr bool N160 = (OPT & 16) == 0;                            // OPT bit 4: the N = 80 operands of round 2h (A/B baseline)
    if (N160) umma::prepare_weights160(a.p.lin_w, a.p.l3_w, smem + D_WHI, tid, D_THREADS);
    else umma::prepare_weights80(a.p.lin_w, a.p.l3_w, smem + D_WHI, smem + D_WLO, tid, D_THREADS);
    if (tid < 32) umma::tmem_alloc(tslot, C::TMEM_COLS);
    if (t == 0) { umma::mbar_init(mbar, 1); umma::mbar_init(sbar, (OPT & 1) ? 2 : 1); }
    umma::fence_before_sync();
    if (tid < H) bs[tid] = a.p.lin_b[tid];
    if (tid < 4 * H) W3s[tid] = a.p.l3_w[tid];
    if (tid < 4) { small[tid] = a.p.l3_b[tid]; small[4 + tid] = a.p.s2_w[tid]; }
    if (tid == 0) small[8] = a.p.s2_b[0];
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tslot + (uint32_t)half * 256u;             // this pipeline's [128 x 160] fp32 accumulator
    const uint32_t wop = umma::smem_u32(smem + D_WHI);
    const uint32_t xs_addr = umma::smem_u32(Xs), ls_addr = umma::smem_u32(Ls);
    // one thread: the split product of the operand tiles (hi in Xs, lo in Ls) with [W; W3]. OPT bits 1, 2, 4, 5 are A/B and
    // timing variants (GNODE_ABLATIONS builds): 16 of the MMAs skipped / none issued / N = 80 operands / lo x lo term dropped
    auto issue_gemm = [&]() {
        if (OPT & 4) umma::mma_commit(mbar);
        else if (OPT & 32) umma::issue_split_gemm160_3term<TR>(tmem, mbar, wop, xs_addr, ls_addr);
        else if (N160) umma::issue_split_gemm160<TR, (OPT & 2) ? 1 : 0>(tmem, mbar, wop, xs_addr, ls_addr);
        else umma::issue_split_gemm80<TR, (OPT & 2) ? 2 : 0>(tmem, mbar, wop, wop + umma::WB80_BYTES, xs_addr, ls_addr);
    };
    const int q = warp & 3, cq = warp >> 2;                           // TMEM lane quarter, 16-column block
    const int erow = q * 32 + lane;                                   // tile row this thread owns in the epilogues
    uint32_t phase = 0, sphase = 0;
    int kfetch = 1;
    const int n_steps = PERSIST ? max(a.n_steps, 1) : 1;

    const bool b3 = (l & 8) != 0, b2 = (l & 4) != 0;
    // ZS: this lane's 16-byte chunk of enc(0), enc(1) and of the two I'_0 rows (trials_table_kernel)
    float4 ze0 = make_float4(0.f, 0.f, 0.f, 0.f), ze1 = ze0, zip0 = ze0, zip1 = ze0;
    if (ZS) {
        ze0 = *reinterpret_cast<const float4*>(a.z_tbl + TB_E + 4 * l);
        ze1 = *reinterpret_cast<const float4*>(a.z_tbl + TB_E + 64 + 4 * l);
        zip0 = *reinterpret_cast<const float4*>(a.z_tbl + TB_IP + 4 * l);
        zip1 = *reinterpret_cast<const float4*>(a.z_tbl + TB_IP + 64 + 4 * l);
    }
    auto seed_bit = [&](int64_t g) -> int { return (int)((a.z_bitmap[g >> 5] >> (g & 31)) & 1u); };

#pragma unroll 1
    for (int step = 0; step < n_steps; ++step) {
    if (PERSIST) {
        if (tid == 0) {
            SStep d;
            d.y_in = a.y_in; d.y_out = a.y_out; d.ip_in = a.ip_in; d.ip_out = a.ip_out;
            d.probs = a.probs; d.counter = a.counter; d.tm = &a.tm_ip_out; d.tms = &a.tm_s_in; d.srow0 = 0; d.dt = a.dt;
            d.iprow0 = 0; d.ai_out = a.ai_out;
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
                d.tms = a.traj ? &a.tm_sp[0] : &a.tm_sp[ks & 1];
                d.srow0 = a.traj ? ks * 3 * M : 0;
                if (a.aux) {                                  // I'_k / AI_k of every step are kept for the reverse sweep
                    d.ip_in = a.aux + (size_t)ks * a.aux_slot; d.ip_out = a.aux + (size_t)(ks + 1) * a.aux_slot;
                    d.ai_out = a.aux + (size_t)ks * a.aux_slot + a.aux_slot / 2;
                    d.tm = &a.tm_ipb[0];                      // one map over the whole buffer, rows = T * 2 * (Mr + 1)
                    d.iprow0 = (int)((size_t)(ks + 1) * (a.aux_slot / H));
                }
            }
            *stp = d;
        }
        __syncthreads();
    }
    if (t == 0) {
        fetch_meta(0);
        if (PERSIST) asm volatile("fence.proxy.async;" ::: "memory");   // state rows written by other SMs (generic proxy) -> TMA reads
        issue_s_load();
        if ((OPT & 1) && meta->seq < n_tiles) umma::mbar_arrive(sbar);   // second arrival: Ls is free (no TMA store pending)
    }
    kfetch = 1;
    HSYNC();
    for (;;) {
        const DTileMeta m = *meta;                                    // written before the last barrier passed
        if (m.seq >= n_tiles) break;
        const int tile0 = m.tile0, nrows = m.nrows, i_row0 = m.i_row0, ebase = m.ebase;
        const bool single = (m.single & 1) != 0;
        const bool relay = (m.single & 2) != 0 && !a.relay_off;       // the tile has isolated hub rows (host cost model)
        const float dt = STP(dt);

        // ---- P1: CSR slice, beta/gamma -> smem; lo operand of the TMA-loaded S_k tile
        {
            int rpv = 0, civ[3] = {0, 0, 0};
            float bgv = 0.f;
            uint32_t pmv = 0;
            if (!ZS && single && t < 64) pmv = __ldg(reinterpret_cast<const uint32_t*>(a.bv.tile_perm) + (size_t)(tile0 / TR) * 64 + t);
            const int ecnt = min(m.ecnt, CAPS);
            // slot i of the window: column index i (i < CAPS) or, weighted, the weight of entry i - CAPS
            auto staged = [&](int i) { return i < CAPS ? i < ecnt : (WGT && i - CAPS < ecnt); };
            if (single && t <= nrows) rpv = __ldg(m.rowptr + t);
            if (single) {
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const int i = t + u * PT;
                    if (i < CAPS) { if (i < ecnt) civ[u] = __ldg(m.colidx + ebase + i); }
                    else if (staged(i)) civ[u] = __float_as_int(__ldg(*wslot + (i - CAPS)));
                }
            }
            if (!ZS && t >= PT / 2 && t < PT / 2 + nrows) bgv = a.beta[tile0 + t - PT / 2];
            if (!ZS && t >= 3 * PT / 4 && t < 3 * PT / 4 + nrows) bgv = a.gamma[tile0 + t - 3 * PT / 4];
            int zi = m.inst0, zk = 0;
            float zg = 0.f;
            if (ZS && t < nrows) {                                    // row t: instance, seed flag, beta / gamma of its trial
                if (!single) zi = find_instance(a.bv, (int64_t)tile0 + t);
                zk = seed_bit((int64_t)tile0 + t);
                bgv = a.z_beta[zi]; zg = a.z_gamma[zi];
                a.beta[tile0 + t] = bgv; a.gamma[tile0 + t] = zg;
            }
            umma::mbar_wait(sbar, sphase); sphase ^= 1;               // the S_k tile has landed in Xs (ZS: Xs and Ls are free)
            if (ZS) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {                         // S_0 rows: enc(1 - I0), raw = hi operand; lo as below
                    const int rr = hw + i * RSTEP;
                    float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f);      // rows past M: zeros, as the TMA load delivers them
                    if (rr < nrows) s0 = seed_bit((int64_t)tile0 + rr) ? ze0 : ze1;
                    sts4(Xs, off0 + i * PASS, s0);
                    sts4(Ls, off0 + i * PASS, umma::tf32_trunc_lo4(s0));
                }
                if (t < nrows) { kind_s[t] = (unsigned char)zk; bg_s[t] = bgv; bg_s[TR + t] = zg; }
                if (t < nrows && !single) zinst_s[t] = zi;            // (aliases the colidx slice, which only single tiles stage)
            }
#pragma unroll
            for (int i = 0; i < ((OPT & 8) || ZS ? 0 : 4); ++i) {
                if (OPT & 64) { sts4(Ls, off0 + i * PASS, umma::tf32_trunc_lo4(lds4(Xs, off0 + i * PASS))); continue; }
                float4 lo;
                const float4 pk = tf32_pack4(lds4(Xs, off0 + i * PASS), lo);
                sts4(Xs, off0 + i * PASS, pk);
                sts4(Ls, off0 + i * PASS, lo);
            }
            umma::fence_proxy_async();
            if (t == 0) *row_ctr = 0;
            if (t < TR / 32) hub_mask[t] = 0u;
            if (single && t <= nrows) rp_s[t] = rpv;
            if (!ZS && single && t < 64) reinterpret_cast<uint32_t*>(hb + C::P_PM)[t] = pmv;
            if (single) {
#pragma unroll
                for (int u = 0; u < 3; ++u) if (staged(t + u * PT)) ci_s[t + u * PT] = civ[u];   // instance-local ids
            }
            if (!ZS && t >= PT / 2 && t < PT / 2 + nrows) bg_s[t - PT / 2] = bgv;
            if (!ZS && t >= 3 * PT / 4 && t < 3 * PT / 4 + nrows) bg_s[TR + t - 3 * PT / 4] = bgv;
        }
        HSYNC();                                                                // S1
        // ---- P2: GEMM1 ; S' epilogue (+ hid(S_k))
        if (t == 0) issue_gemm();
        if (relay && t < nrows && rp_s[t + 1] - rp_s[t] > C::HUB_DEG) atomicOr(&hub_mask[t >> 5], 1u << (t & 31));
        if (ZS && single) {
            // step 0 from descriptors: the staged column indices are replaced by the seed bits of those neighbours, all
            // looked up together while GEMM1 runs; the neighbour sums below then read shared memory only
            const int ecnt = min(m.ecnt, C::CAP);
            int zb[3] = {0, 0, 0};
#pragma unroll
            for (int u = 0; u < 3; ++u) if (t + u * PT < ecnt) zb[u] = seed_bit((int64_t)i_row0 + ci_s[t + u * PT]);
#pragma unroll
            for (int u = 0; u < 3; ++u) if (t + u * PT < ecnt) ci_s[t + u * PT] = zb[u];
        }
        // work items of the neighbour gather (gnode_batch_create): strided over the warps when the tile's CSR slice fits the
        // staged window, shared-memory tickets for hub tiles so that a long row does not leave the other warps idle
        const float* lane_base = STP(ip_in) + (size_t)i_row0 * H + 4 * l;
        const int zrow = a.ip_zrow - i_row0;                 // the all-zero row that follows the I' rows
        const bool static_rows = m.ecnt <= C::CAP;
        int sj = 0;
        auto draw_item = [&]() -> int {
            if (static_rows) { const int it = sj < 4 ? warp + (PT / 32) * sj : 64; ++sj; return it; }
            int it = 0;
            if (lane == 0) it = atomicAdd(row_ctr, 1);
            return __shfl_sync(0xffffffffu, it, 0);
        };
        // two-row item: tile row rr of this half-warp (0xFF = none), one round trip per 12 neighbours
        auto gather_pair = [&](int rr, bool& ok) -> float4 {
            int e_rel = 0, deg = 0;
            if (rr < nrows) { e_rel = rp_s[rr] - ebase; deg = rp_s[rr + 1] - rp_s[rr]; }
            const bool hubrow = relay && deg > C::HUB_DEG;                 // summed by the in-order relay below
            if (hubrow) deg = 0;
            ok = rr < nrows && !hubrow;
            const int over = (e_rel + deg > CAPS) ? 1 : 0;
            if (__any_sync(0xffffffffu, over))               // indices beyond the staged slice: same gather on the global list
                return gather_smem_zm<12, WGT>(lane_base, m.colidx + ebase + e_rel, deg, zrow, pol_keep, WGT ? *wslot + e_rel : nullptr);
            return gather_smem_zm<12, WGT>(lane_base, ci_s + e_rel, deg, zrow, pol_keep, WGT ? wt_s + e_rel : nullptr);
        };
        umma::mbar_wait_suspend(mbar, phase); phase ^= 1;
        umma::fence_after_sync();
        {
            if (N160) {                                  // accumulator halves, bias and sigmoid on component pairs
                f32x2 v2[8];
                umma::tmem_ld16_sum2(tmem + ((uint32_t)(q * 32) << 16) + 16 * cq, v2);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * cq + 4 * j);
                    float4 o;
                    unpack2(sigmoid2_t<FAST>(add2(v2[2 * j], pack2(bb.x, bb.y))), o.x, o.y);
                    unpack2(sigmoid2_t<FAST>(add2(v2[2 * j + 1], pack2(bb.z, bb.w))), o.z, o.w);
                    sts4(Ls, C::sw(erow, 4 * cq + j), o);
                }
            } else {
            float v[16];
            umma::tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + 16 * cq, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * cq + 4 * j);
                float4 o;
                o.x = sigmoid_t<FAST>(v[4 * j + 0] + bb.x); o.y = sigmoid_t<FAST>(v[4 * j + 1] + bb.y);
                o.z = sigmoid_t<FAST>(v[4 * j + 2] + bb.z); o.w = sigmoid_t<FAST>(v[4 * j + 3] + bb.w);
                sts4(Ls, C::sw(erow, 4 * cq + j), o);
            }
            }
            if (cq == 0) {
                float hv[4];
                if (N160) umma::tmem_ld4_sum(tmem + ((uint32_t)(q * 32) << 16) + 64, hv); else umma::tmem_ld4(tmem + ((uint32_t)(q * 32) << 16) + 64, hv);
                *reinterpret_cast<float4*>(hs_s + 4 * erow) = make_float4(hv[0], hv[1], hv[2], hv[3]);
            }
        }
        umma::fence_before_sync();
        HSYNC();                                                                // S2

        // the full-plane mode decodes R_k from its row; RF needs nothing per step: hid(R_k) follows from the conserved sum
        const bool dec = !RF && STP(probs) != nullptr;
        // own-row operands that still come from HBM/L2: I_k, I'_k (and R_k when the R plane is carried)
        // (`off` = float offset of the lane's chunk of the row in a state / I' plane; rows that do not exist keep whatever
        // the registers hold: update_row never reads them)
        auto load_own = [&](size_t off, bool ok, float4& iv, float4& rv, float4& ipo) {
            if (ok) {
                iv = ldg4_hint(STP(y_in) + plane + off, pol_stream);
                if (!RF) rv = ldg4_hint(STP(y_in) + 2 * plane + off, pol_stream);
                ipo = ldg4_hint(STP(ip_in) + off, pol_keep);
            }
        };
        // SIR update of tile row rr from tp = AI * S' (`ok` is uniform per half-warp): stores S,I(,R)_{k+1}; I_{k+1}
        // raw / lo -> operand tiles; returns the lane's partial linear3 products of R_k (RF: of I'_k) in hv
        auto update_row = [&](int rr, size_t off, bool ok, float4 tp, float4 iv, float4 rv, float4 ipo,
                              float4 w30, float4 w31, float4 w32, float4 w33, float (&hv)[4]) {
            hv[0] = 0.f; hv[1] = 0.f; hv[2] = 0.f; hv[3] = 0.f;
            if (ok) {
                const int o = C::sw(rr, l);
                const float4 s = (OPT & 64) ? lds4(Xs, o) : tf32_unpack4(lds4(Xs, o));
                const float nbe = -bg_s[rr], ga = bg_s[TR + rr];
                float4 sn, in_, rn;
                // dS = -beta (AI S'), dR = gamma I', dI = -dS - dR; y + dt dy, every product and sum rounded on its own
                // (the reference rounds after every ATen op). The PRODUCTS run on component pairs; the sums stay scalar
                // __fadd_rn: ptxas 12.9 fuses mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (one rounding) although both carry an
                // explicit rounding mode -- seen in the SASS of the R-free instantiation, 2.7e-6 on the fb-food golden.
                // dI = fl(-dS - dR) = -fl(dS + dR) and fl(dt dI) = fl(-dt fl(dS + dR)) (round-to-nearest is sign-symmetric):
                // the same bits as the all-scalar form.
                const f32x2 nbe2 = pack2(nbe, nbe), ga2 = pack2(ga, ga), dt2 = pack2(dt, dt), ndt2 = pack2(-dt, -dt);
#define GN_COMP2(a, b)                                                              \
    {                                                                               \
        const f32x2 dS = mul2(nbe2, pack2(tp.a, tp.b));                             \
        const f32x2 dR = mul2(ga2, pack2(ipo.a, ipo.b));                            \
        float dSa, dSb, dRa, dRb, pa, pb;                                           \
        unpack2(dS, dSa, dSb); unpack2(dR, dRa, dRb);                               \
        const f32x2 u = pack2(__fadd_rn(dSa, dRa), __fadd_rn(dSb, dRb));            \
        unpack2(mul2(dt2, dS), pa, pb);                                             \
        sn.a = __fadd_rn(s.a, pa); sn.b = __fadd_rn(s.b, pb);                       \
        unpack2(mul2(ndt2, u), pa, pb);                                             \
        in_.a = __fadd_rn(iv.a, pa); in_.b = __fadd_rn(iv.b, pb);                   \
        if (!RF) {                                                                  \
            unpack2(mul2(dt2, dR), pa, pb);                                         \
            rn.a = __fadd_rn(rv.a, pa); rn.b = __fadd_rn(rv.b, pb);                 \
        }                                                                           \
    }
                GN_COMP2(x, y) GN_COMP2(z, w)
#undef GN_COMP2
                stg4_hint(STP(y_out) + off, sn, pol_stream);
                stg4_hint(STP(y_out) + plane + off, in_, pol_stream);
                if (!RF) stg4_hint(STP(y_out) + 2 * plane + off, rn, pol_stream);
                float4 ilo;
                if (OPT & 64) { sts4(Xs, o, in_); ilo = umma::tf32_trunc_lo4(in_); }
                else sts4(Xs, o, tf32_pack4(in_, ilo));              // hi operand of GEMM2 (packed like the S tile)
                sts4(Ls, o, ilo);
                if (dec) {
                    const float4 dv = rv;
                    hv[0] = dot4(dv, w30); hv[1] = dot4(dv, w31); hv[2] = dot4(dv, w32); hv[3] = dot4(dv, w33);
                }
            }
        };
        // halving butterfly over the 16 lanes of the row: lanes 0 / 4 / 8 / 12 end with hid[0 / 1 / 2 / 3]
        // (full-mask shuffles: all 32 lanes of the warp call it)
        auto hid_bfly = [&](int rr, bool ok, const float (&hv)[4]) {
            if (dec) {
                const float a0 = (b3 ? hv[2] : hv[0]) + __shfl_xor_sync(0xffffffffu, b3 ? hv[0] : hv[2], 8);
                const float a1 = (b3 ? hv[3] : hv[1]) + __shfl_xor_sync(0xffffffffu, b3 ? hv[1] : hv[3], 8);
                float c = (b2 ? a1 : a0) + __shfl_xor_sync(0xffffffffu, b2 ? a0 : a1, 4);
                c += __shfl_xor_sync(0xffffffffu, c, 2);
                c += __shfl_xor_sync(0xffffffffu, c, 1);
                if (ok && (l & 3) == 0) hr_s[4 * rr + (l >> 2)] = c;
            }
        };
        // what the gathering half-warp does with the finished neighbour sum of row rr: AI * S' replaces S' in place
        float* const ai_out = STP(ai_out);
        auto finish_row = [&](int rr, bool ok, float4 acc) {
            if (!ok) return;                                 // rr may be 0xFF (no row): never form an address from it
            const int o = C::sw(rr, l);
            const float4 sp = lds4(Ls, o);
            if (ai_out != nullptr) stg4_hint(ai_out + (size_t)(tile0 + rr) * H + 4 * l, acc, pol_stream);
            sts4(Ls, o, make_float4(__fmul_rn(acc.x, sp.x), __fmul_rn(acc.y, sp.y), __fmul_rn(acc.z, sp.z), __fmul_rn(acc.w, sp.w)));
        };

        // ---- P3a: neighbour sums AI (sequential, ascending columns), folded into S' in place
        if (ZS) {
            // step 0 from descriptors: neighbour c contributes I'_0(seed) or I'_0(susceptible) -- the same additions in the
            // same order as the gather of an I'_0 plane, with a bitmap bit per neighbour instead of a 256-byte row
#pragma unroll 1
            for (int it = 0; it < 4; ++it) {
                const int rr = hw + RSTEP * it;
                int deg = 0, row0 = i_row0;
                const int32_t* cp = nullptr;
                const int* fl = nullptr;                     // seed bits of the row's neighbours in shared memory, or null
                if (rr < nrows) {
                    if (single) {
                        deg = rp_s[rr + 1] - rp_s[rr];
                        cp = m.colidx + rp_s[rr];
                        const int e_rel = rp_s[rr] - ebase;
                        if (e_rel + deg <= C::CAP) fl = ci_s + e_rel;
                    } else {
                        const GnInstance I = a.bv.inst[zinst_s[rr]];
                        const int n = tile0 + rr - I.row0;
                        row0 = I.row0;
                        deg = I.rowptr[n + 1] - I.rowptr[n];
                        cp = I.colidx + I.rowptr[n];
                    }
                }
                const int degm = max(deg, __shfl_xor_sync(0xffffffffu, deg, 16));
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int j0 = 0; j0 < degm; j0 += 16) {
                    int bit = 0;
                    if (j0 + l < deg) bit = fl ? fl[j0 + l] : seed_bit((int64_t)row0 + cp[j0 + l]);
                    const unsigned mine = (__ballot_sync(0xffffffffu, bit) >> (lane & 16)) & 0xFFFFu;
                    const int nj = min(16, deg - j0);
                    for (int j = 0; j < nj; ++j) {
                        const float4 v = ((mine >> j) & 1u) ? zip1 : zip0;
                        add4(acc, v);
                    }
                }
                finish_row(rr, rr < nrows, acc);
            }
        } else {
            if (single) {
                int it = draw_item();
                while (it < 64) {
                    const uint32_t rw = items_s[it];                       // tile rows {a, b | c, d}, 0xFF = none
                    if (rw == 0xFFFFFFFFu) break;                          // no more items (for this warp / in this tile)
                    const uint32_t mine = rw >> ((lane & 16) ? 16 : 0);
                    const int ra = (int)(mine & 0xFFu), rb = (int)((mine >> 8) & 0xFFu);
                    if ((rw & 0xFF00FF00u) != 0xFF00FF00u) {               // four rows of at most 6 neighbours: one round trip
                        const bool oka = ra < nrows, okb = rb < nrows;
                        int ea = 0, da = 0, eb = 0, db = 0;
                        if (oka) { ea = rp_s[ra] - ebase; da = rp_s[ra + 1] - rp_s[ra]; }
                        if (okb) { eb = rp_s[rb] - ebase; db = rp_s[rb + 1] - rp_s[rb]; }
                        int dmax = max(da, db);
                        dmax = max(dmax, __shfl_xor_sync(0xffffffffu, dmax, 16));
                        float4 sa, sb;
                        if (!WGT) gather_quad(lane_base, ci_s + ea, da, ci_s + eb, db, dmax, zrow, pol_keep, sa, sb);
                        else if (__any_sync(0xffffffffu, ea + da > CAPS || eb + db > CAPS)) {   // past the halved window
                            const float* wt = *wslot;
                            gather_quad<true>(lane_base, m.colidx + ebase + ea, da, m.colidx + ebase + eb, db, dmax, zrow, pol_keep,
                                              sa, sb, wt + ea, wt + eb);
                        } else
                            gather_quad<true>(lane_base, ci_s + ea, da, ci_s + eb, db, dmax, zrow, pol_keep, sa, sb, wt_s + ea, wt_s + eb);
                        finish_row(ra, oka, sa);
                        finish_row(rb, okb, sb);
                    } else {
                        bool ok;
                        const float4 acc = gather_pair(ra, ok);
                        finish_row(ra, ok, acc);
                    }
                    it = draw_item();
                }
                // Hub rows: loads by the whole pipeline (256 neighbours per round trip), adds relayed from warp to warp in
                // column order through shared memory -- bitwise the serial walk (see step_dual_kernel / DESIGN.md 3.1)
                if (relay) {
                    HSYNC();                                             // every ordinary row is done; the colidx slice is dead
                    volatile float* run = reinterpret_cast<volatile float*>(ci_s);          // [64] running sum
                    uint64_t* hbar = reinterpret_cast<uint64_t*>(ci_s + H);                  // one mbarrier per warp: "your turn"
                    if (t < PT / 32) umma::mbar_init(&hbar[t], 1);
                    HSYNC();
                    constexpr int SR = (PT / 16) * 8;                    // neighbours per super-round
                    int nsr_done = 0;
#pragma unroll 1
                    for (int w = 0; w < TR / 32; ++w) {
                        unsigned mm = hub_mask[w];
                        while (mm) {
                            const int r = 32 * w + __ffs(mm) - 1;
                            mm &= mm - 1;
                            const int dg = rp_s[r + 1] - rp_s[r];
                            const int* cp = m.colidx + rp_s[r];
                            const float* wp = WGT ? *wslot + (rp_s[r] - ebase) : nullptr;
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
                                if (WGT) {                                   // products before the relayed adds
#pragma unroll
                                    for (int k = 0; k < 8; ++k) v[k] = mul4((j0 + k < dg) ? wp[j0 + k] : 0.f, v[k]);
                                }
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
                                }
                                __syncwarp();
                                if (sr == n_sr - 1 && warp == PT / 32 - 1) {     // the row's sum is complete in the upper half-warp
                                    const bool ok = lane >= 16;
                                    finish_row(r, ok, sum);
                                }
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
                    const float4 acc = gather_row<WGT>(STP(ip_in), ci, e0, deg, row0, l, lane,
                                                       WGT ? a.edge_w + a.inst_e0[inst] : nullptr);
                    finish_row(rr, rr < nrows, acc);
                }
            }
        }
        {
            // S2b: every AI * S' row is parked. (With strided rows every half-warp updates exactly the rows it gathered and
            // the barrier could be skipped: measured, 1.668e9 vs 1.677e9 node-steps/s with it, profiles/r2j_ab_no_s2b_barrier.log
            // -- warps that run ahead only add update-phase loads to a memory system the gather already saturates.)
            HSYNC();
            // ---- P3b: SIR update (own I_k / I'_k rows one pass ahead in registers; S_k from the raw operand tile; the
            //      lane's 4 x 4 linear3 weights stay in registers for the four passes)
            const float4 w30 = lds4((const unsigned char*)W3s, 16 * l), w31 = lds4((const unsigned char*)W3s, 256 + 16 * l),
                         w32 = lds4((const unsigned char*)W3s, 512 + 16 * l), w33 = lds4((const unsigned char*)W3s, 768 + 16 * l);
            float4 iv = make_float4(1.f, 1.f, 1.f, 1.f), rv = iv, ipo = iv;
            size_t off_own = (size_t)(tile0 + hw) * H + 4 * l;       // this half-warp's row of the pass, advanced by RSTEP rows
            if (!ZS) load_own(off_own, hw < nrows, iv, rv, ipo);
#pragma unroll 1
            for (int it = 0; it < 4; ++it) {
                const int rr = hw + RSTEP * it;
                const bool ok = rr < nrows;
                float hv[4];
                if (ZS) {                                    // I_0 = enc(I0), I'_0 of the row's kind; no R plane
                    const bool sd = ok && kind_s[rr] != 0;
                    iv = sd ? ze1 : ze0; ipo = sd ? zip1 : zip0; rv = iv;
                }
                update_row(rr, off_own, ok, lds4(Ls, off0 + it * PASS), iv, rv, ipo, w30, w31, w32, w33, hv);
                off_own += (size_t)RSTEP * H;
                if (!ZS && it + 1 < 4) load_own(off_own, rr + RSTEP < nrows, iv, rv, ipo);
                hid_bfly(rr, ok, hv);
            }
        }
        float4 hI = make_float4(0.f, 0.f, 0.f, 0.f);     // hid(I_k) of row t (softmax threads): in flight across the barrier
        float4 hRg = hI;                                 // RF: hid(S_0 + I_0 + R_0) of row t (constant over the rollout)
        if (!ZS && STP(probs) != nullptr && t < nrows) hI = *reinterpret_cast<const float4*>(a.hid_i + (size_t)(tile0 + t) * 4);
        if (!ZS && RF && STP(probs) != nullptr && t < nrows) hRg = *reinterpret_cast<const float4*>(a.hid_r + (size_t)(tile0 + t) * 4);
        if (ZS) hRg = *reinterpret_cast<const float4*>(a.z_tbl + TB_HR);       // the same for both kinds of rows
        umma::fence_proxy_async();
        HSYNC();                                                                // S3 (every thread has read its copy of *meta)
        // ---- P4: GEMM2 || metadata of the next tile || softmax of the input state ; I' epilogue (+ hid(I_{k+1}))
        if (t == 0) issue_gemm();
        if (t == PT - 32) fetch_meta(kfetch);
        ++kfetch;
        if (ZS && t < nrows) *reinterpret_cast<float4*>(a.hid_r + (size_t)(tile0 + t) * 4) = hRg;   // written once, read when probs are emitted
        if (ZS && STP(probs) != nullptr && t < nrows) {     // probs[0] of the row's kind (decoder of the two rows: table)
            const float* pk = a.z_tbl + TB_PR + 4 * kind_s[t];
            float* pr = STP(probs) + (size_t)(tile0 + t) * 3;
            pr[0] = pk[0]; pr[1] = pk[1]; pr[2] = pk[2];
        }
        if (!ZS && STP(probs) != nullptr && t < nrows) {    // one thread per row: probs[k] = softmax(decoder(S_k, I_k, R_k))
            const float4 hS = *reinterpret_cast<const float4*>(hs_s + 4 * t);
            // RF: S + I + R is conserved channel by channel (dS + dI + dR = 0, ode_nn_ngraph_sim.py:75-77), so
            // hid(R_k) = W3 (S_0 + I_0 + R_0) - hid(S_k) - hid(I_k): no R plane and no per-step recurrence
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
        umma::mbar_wait_suspend(mbar, phase); phase ^= 1;
        umma::fence_after_sync();
        if (t == PT - 32) issue_s_load();                // GEMM2 has read Xs: the next tile's S_k rows may land there
        {
            if (N160) {                                  // accumulator halves, bias and sigmoid on component pairs
                f32x2 v2[8];
                umma::tmem_ld16_sum2(tmem + ((uint32_t)(q * 32) << 16) + 16 * cq, v2);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * cq + 4 * j);
                    float4 o;
                    unpack2(sigmoid2_t<FAST>(add2(v2[2 * j], pack2(bb.x, bb.y))), o.x, o.y);
                    unpack2(sigmoid2_t<FAST>(add2(v2[2 * j + 1], pack2(bb.z, bb.w))), o.z, o.w);
                    sts4(Ls, C::sw(erow, 4 * cq + j), o);
                }
            } else {
            float v[16];
            umma::tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + 16 * cq, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 bb = *reinterpret_cast<const float4*>(bs + 16 * cq + 4 * j);
                float4 o;
                o.x = sigmoid_t<FAST>(v[4 * j + 0] + bb.x); o.y = sigmoid_t<FAST>(v[4 * j + 1] + bb.y);
                o.z = sigmoid_t<FAST>(v[4 * j + 2] + bb.z); o.w = sigmoid_t<FAST>(v[4 * j + 3] + bb.w);
                sts4(Ls, C::sw(erow, 4 * cq + j), o);
            }
            }
            if (cq == 0) {
                float hv[4];
                if (N160) umma::tmem_ld4_sum(tmem + ((uint32_t)(q * 32) << 16) + 64, hv); else umma::tmem_ld4(tmem + ((uint32_t)(q * 32) << 16) + 64, hv);
                if (erow < nrows) *reinterpret_cast<float4*>(a.hid_i + (size_t)(tile0 + erow) * 4) = make_float4(hv[0], hv[1], hv[2], hv[3]);
            }
        }
        umma::fence_before_sync();
        umma::fence_proxy_async();                       // the staged tile is read by the TMA (async proxy)
        HSYNC();                                                                // S4 (the next tile's metadata is published)
        // ---- P5: I'_{k+1} tile -> HBM by two TMA tensor stores (rows past M are clipped by the tensor bounds)
        if (t == 0) {
            tma_store_2d(STP_TM(), Ls, 0, STP_IPROW0() + tile0, pol_stream);
            tma_store_2d(STP_TM(), Ls + C::KBLK, 32, STP_IPROW0() + tile0, pol_stream);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            // OPT bit 0: no block barrier here. The staged tile may be overwritten once the bulk group has read it; the next
            // tile's threads learn that through the S-load mbarrier, whose second arrival is this thread's (they wait on
            // it before their first write to Ls), so the store's read time overlaps the S load and the CSR staging.
            if ((OPT & 1) && meta->seq < n_tiles) umma::mbar_arrive(sbar);
        }
        if (!(OPT & 1)) HSYNC();                                                // S5
    }
    if (step + 1 < n_steps) {
        if (t == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __threadfence();
        cooperative_groups::this_grid().sync();
    }
    }
#undef HSYNC
#undef STP
#undef STP_TM
#undef STP_TMS
#undef STP_SROW0
#undef STP_IPROW0
    umma::fence_before_sync();
    __syncthreads();
    if (tid < 32) umma::tmem_dealloc(*tslot, C::TMEM_COLS);
}

}  // namespace gnode
