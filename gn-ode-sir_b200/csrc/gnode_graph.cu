// Graph / batch handles and the standalone neighbour aggregation (SURVEY 8a: a6, a7).
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstdarg>
#include <cstring>

#include "gnode_common.cuh"

namespace gnode {

static thread_local char t_err[1024] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
}

// out[r, :] = sum_{c in adj(r)} in[c, :]  -- one half-warp per row, 16 B per lane, the
// neighbours of a row are accumulated sequentially in ascending-column order
// (the order of the reference's CPU scatter_add_, ode_nn_ngraph_sim.py:73).
__global__ void __launch_bounds__(256) aggregate_kernel(GnBatchView bv, const float* __restrict__ in,
                                                         float* __restrict__ out, int transpose) {
    const int l = threadIdx.x & 15;
    const int hw_in_block = threadIdx.x >> 4;
    const int hw_per_block = blockDim.x >> 4;
    const unsigned hmask = 0xFFFFu << (threadIdx.x & 16);
    for (int64_t r = (int64_t)blockIdx.x * hw_per_block + hw_in_block; r < bv.M;
         r += (int64_t)gridDim.x * hw_per_block) {
        // instance lookup: binary search over row0 (n_inst is small and cached)
        int lo = 0, hi = bv.n_inst - 1;
        while (lo < hi) {
            int mid = (lo + hi + 1) >> 1;
            if (bv.inst[mid].row0 <= r) lo = mid; else hi = mid - 1;
        }
        const GnInstance I = bv.inst[lo];
        const int32_t* rp = transpose ? I.rowptr_t : I.rowptr;
        const int32_t* ci = transpose ? I.colidx_t : I.colidx;
        const int n = (int)(r - I.row0);
        const int e0 = rp[n], e1 = rp[n + 1];
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int e = e0; e < e1; e += 16) {
            const int mine = (e + l < e1) ? ci[e + l] : 0;
            const int cnt = min(16, e1 - e);
            for (int j = 0; j < cnt; ++j) {
                const int c = __shfl_sync(hmask, mine, j, 16) + I.row0;
                const float4 v = ldg4(in + (size_t)c * H + 4 * l);
                acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
            }
        }
        stg4(out + (size_t)r * H + 4 * l, acc);
    }
}

}  // namespace gnode

using namespace gnode;

extern "C" const char* gnode_last_error(void) { return t_err; }
extern "C" int gnode_version(void) { return 100; }
extern "C" int64_t gnode_launch_count(void) { return g_launches; }

extern "C" int gnode_graph_create(int32_t n, int64_t nnz, const int32_t* rowptr, const int32_t* colidx,
                                  gnode_graph_t* out) {
    if (!out || !rowptr || (nnz > 0 && !colidx) || n <= 0 || nnz < 0 || nnz > 0x7fffffffLL) {
        set_error("gnode_graph_create: bad arguments (n=%d nnz=%lld)", n, (long long)nnz);
        return GNODE_ERR_ARG;
    }
    if (rowptr[0] != 0 || rowptr[n] != nnz) {
        set_error("gnode_graph_create: rowptr[0]=%d rowptr[n]=%d do not match nnz=%lld", rowptr[0], rowptr[n],
                  (long long)nnz);
        return GNODE_ERR_ARG;
    }
    // validate the whole CSR before touching it: a malformed rowptr must not drive the per-row sort out of bounds
    for (int32_t r = 0; r < n; ++r)
        if (rowptr[r + 1] < rowptr[r] || rowptr[r + 1] > nnz) {
            set_error("gnode_graph_create: rowptr not monotone within [0, nnz] at row %d", r);
            return GNODE_ERR_ARG;
        }
    for (int64_t e = 0; e < nnz; ++e)
        if (colidx[e] < 0 || colidx[e] >= n) {
            set_error("gnode_graph_create: column index %d out of range at entry %lld", colidx[e], (long long)e);
            return GNODE_ERR_ARG;
        }
    std::vector<int32_t> ci(colidx, colidx + nnz);
    int32_t maxdeg = 0;
    for (int32_t r = 0; r < n; ++r) {
        std::sort(ci.begin() + rowptr[r], ci.begin() + rowptr[r + 1]);
        maxdeg = std::max(maxdeg, rowptr[r + 1] - rowptr[r]);
    }
    // transpose pattern by counting sort (rows ascending -> columns of A^T ascending)
    std::vector<int32_t> rpt(n + 1, 0), cit(nnz), tmap(nnz);
    for (int64_t e = 0; e < nnz; ++e) rpt[ci[e] + 1]++;
    for (int32_t r = 0; r < n; ++r) rpt[r + 1] += rpt[r];
    {
        std::vector<int32_t> fill(rpt.begin(), rpt.end() - 1);
        for (int32_t r = 0; r < n; ++r)
            for (int32_t e = rowptr[r]; e < rowptr[r + 1]; ++e) { tmap[fill[ci[e]]] = e; cit[fill[ci[e]]++] = r; }
    }
    const bool sym = (memcmp(rpt.data(), rowptr, sizeof(int32_t) * (n + 1)) == 0) &&
                     (nnz == 0 || memcmp(cit.data(), ci.data(), sizeof(int32_t) * nnz) == 0);

    gnode_graph* g = new gnode_graph();
    g->n = n; g->nnz = nnz; g->max_degree = maxdeg; g->symmetric = sym ? 1 : 0;
    g->h_rowptr.assign(rowptr, rowptr + n + 1);
    g->h_tmap.swap(tmap);
    // device side: any CUDA failure frees what was allocated so far together with the handle
    auto upload = [&]() -> int {
    GN_CUDA(cudaGetDevice(&g->device));
    const size_t nnz_alloc = (size_t)std::max<int64_t>(nnz, 1);
    GN_CUDA(cudaMalloc(&g->d_rowptr, sizeof(int32_t) * (n + 1)));
    GN_CUDA(cudaMalloc(&g->d_colidx, sizeof(int32_t) * nnz_alloc));
    GN_CUDA(cudaMemcpy(g->d_rowptr, rowptr, sizeof(int32_t) * (n + 1), cudaMemcpyHostToDevice));
    if (nnz) GN_CUDA(cudaMemcpy(g->d_colidx, ci.data(), sizeof(int32_t) * nnz, cudaMemcpyHostToDevice));
    if (sym) {
        g->d_rowptr_t = g->d_rowptr;
        g->d_colidx_t = g->d_colidx;
    } else {
        GN_CUDA(cudaMalloc(&g->d_rowptr_t, sizeof(int32_t) * (n + 1)));
        GN_CUDA(cudaMalloc(&g->d_colidx_t, sizeof(int32_t) * nnz_alloc));
        GN_CUDA(cudaMemcpy(g->d_rowptr_t, rpt.data(), sizeof(int32_t) * (n + 1), cudaMemcpyHostToDevice));
        if (nnz) GN_CUDA(cudaMemcpy(g->d_colidx_t, cit.data(), sizeof(int32_t) * nnz, cudaMemcpyHostToDevice));
    }
    return GNODE_OK;
    };
    const int rc = upload();
    if (rc != GNODE_OK) {
        if (g->d_rowptr_t == g->d_rowptr) { g->d_rowptr_t = nullptr; g->d_colidx_t = nullptr; }
        g->symmetric = 0;                        // free whichever of the four arrays exist, once each
        gnode_graph_destroy(g);
        return rc;
    }
    *out = g;
    return GNODE_OK;
}

extern "C" int gnode_graph_destroy(gnode_graph_t g) {
    if (!g) return GNODE_OK;
    if (!g->symmetric) {
        cudaFree(g->d_rowptr_t);
        cudaFree(g->d_colidx_t);
    }
    cudaFree(g->d_rowptr);
    cudaFree(g->d_colidx);
    cudaFree(g->d_tmap);
    delete g;
    return GNODE_OK;
}

extern "C" int gnode_graph_info(gnode_graph_t g, int32_t* n, int64_t* nnz, int32_t* max_degree, int32_t* symmetric) {
    if (!g) { set_error("gnode_graph_info: null graph"); return GNODE_ERR_ARG; }
    if (n) *n = g->n;
    if (nnz) *nnz = g->nnz;
    if (max_degree) *max_degree = g->max_degree;
    if (symmetric) *symmetric = g->symmetric;
    return GNODE_OK;
}

extern "C" int gnode_batch_create(const gnode_graph_t* inst_graphs, int32_t n_inst, gnode_batch_t* out) {
    if (!out || !inst_graphs || n_inst <= 0) {
        set_error("gnode_batch_create: bad arguments (n_inst=%d)", n_inst);
        return GNODE_ERR_ARG;
    }
    std::vector<GnInstance> inst(n_inst);
    std::vector<int64_t> inst_e0(n_inst);
    int64_t M = 0, nnz = 0;
    for (int32_t i = 0; i < n_inst; ++i) {
        const gnode_graph* g = inst_graphs[i];
        if (!g) { set_error("gnode_batch_create: instance %d has a null graph", i); return GNODE_ERR_ARG; }
        inst[i].rowptr = g->d_rowptr; inst[i].colidx = g->d_colidx;
        inst[i].rowptr_t = g->d_rowptr_t; inst[i].colidx_t = g->d_colidx_t;
        inst[i].row0 = (int32_t)M; inst[i].n = g->n;
        inst_e0[i] = nnz;
        M += g->n; nnz += g->nnz;
        if (M > 0x7fffff00LL) { set_error("gnode_batch_create: %lld rows exceed the int32 row space", (long long)M); return GNODE_ERR_ARG; }
    }
    gnode_batch* b = new gnode_batch();
    b->M = M; b->n_inst = n_inst; b->nnz_total = nnz;
    b->graphs.assign(inst_graphs, inst_graphs + n_inst);
    b->n_tiles = (int32_t)((M + TILE - 1) / TILE);
    std::vector<int32_t> tile_inst(b->n_tiles);
    std::vector<int64_t> tile_cost(b->n_tiles, 0);
    std::vector<int32_t> tile_maxdeg(b->n_tiles, 0);
    int32_t cur = 0;
    for (int32_t t = 0; t < b->n_tiles; ++t) {
        const int64_t r = (int64_t)t * TILE;
        while (cur + 1 < n_inst && inst[cur + 1].row0 <= r) ++cur;
        tile_inst[t] = cur;
        // cost model: neighbour rows gathered by the tile (the only non-uniform work)
        int32_t ii = cur;
        for (int64_t g = r; g < std::min<int64_t>(r + TILE, M); ++g) {
            while (ii + 1 < n_inst && inst[ii + 1].row0 <= g) ++ii;
            const std::vector<int32_t>& rp = inst_graphs[ii]->h_rowptr;
            const int64_t nloc = g - inst[ii].row0;
            tile_cost[t] += rp[nloc + 1] - rp[nloc];
            tile_maxdeg[t] = std::max(tile_maxdeg[t], rp[nloc + 1] - rp[nloc]);
        }
    }
    // Processing order for the dynamic tile scheduler: instance by instance (= trial by trial, so that concurrently
    // processed tiles share their trial's I' rows in L2), and inside an instance the tiles whose gather work exceeds
    // 4x the mean (hub tiles of power-law graphs) first, heaviest first, then the others in row-major order.
    // Instances smaller than a few tiles are grouped 64 at a time so that tiny graphs keep a row-major order.
    std::vector<int32_t> order;
    order.reserve(b->n_tiles);
    {
        const double mean = (double)nnz / std::max(1, b->n_tiles);
        std::vector<int32_t> heavy, light;
        auto flush = [&]() {
            std::stable_sort(heavy.begin(), heavy.end(), [&](int32_t x, int32_t y) { return tile_cost[x] > tile_cost[y]; });
            order.insert(order.end(), heavy.begin(), heavy.end());
            order.insert(order.end(), light.begin(), light.end());
            heavy.clear(); light.clear();
        };
        int32_t group_first_inst = 0;
        for (int32_t t = 0; t < b->n_tiles; ++t) {
            if (tile_inst[t] != group_first_inst && heavy.size() + light.size() >= 64) { flush(); group_first_inst = tile_inst[t]; }
            if ((double)tile_cost[t] > 4.0 * mean + 1024.0) heavy.push_back(t); else light.push_back(t);
        }
        flush();
    }
    {
        cudaError_t e = cudaGetDevice(&b->device);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&b->sm_count, cudaDevAttrMultiProcessorCount, b->device);
        if (e != cudaSuccess) { set_error("gnode_batch_create: %s", cudaGetErrorString(e)); delete b; return GNODE_ERR_CUDA; }
        for (int32_t i = 0; i < n_inst; ++i)
            if (inst_graphs[i]->device != b->device) {
                set_error("gnode_batch_create: graph of instance %d lives on device %d, the current device is %d", i,
                          inst_graphs[i]->device, b->device);
                delete b;
                return GNODE_ERR_ARG;
            }
    }
    // Tail control. A row is summed by ONE half-warp in rounds of 8 neighbours, strictly in ascending column order (the
    // order of the reference's CPU scatter_add_: hub sums of ~1e3 amplify any re-association to ~1e-3 in the hidden
    // state, so the row is not split across warps). A round costs ~2.4k cycles under load, i.e. a tile with a hub row of
    // degree d occupies its pipeline for about d / 128 ordinary tile times (measured: 0.65 ms for two 4k-degree rows),
    // whatever the other rows do. Such a tile must not START late: the hub tile of the last trials would otherwise run
    // on alone after every other pipeline has drained (measured: +0.6 ms per launch, -14 % at 64 trials with 3k-degree
    // hubs). Tiles whose estimated end passes the end of the launch are hoisted to the very front of the order (longest
    // first); all others keep the trial-by-trial order above.
    if (getenv("GNODE_NO_TAIL_HOIST") == nullptr) {
        const int64_t n = (int64_t)order.size();
        const int64_t P = 2 * (int64_t)std::max(1, b->sm_count);          // tile pipelines in flight
        std::vector<char> hoist(b->n_tiles, 0);
        std::vector<int32_t> front;
        for (int64_t q = 0; q < n; ++q) {
            const int32_t t = order[q];
            if (tile_maxdeg[t] < 256) continue;
            const int64_t len = tile_maxdeg[t] / 128 + 1;                  // in ordinary tile times
            if (q > n - P * (len + 1)) { hoist[t] = 1; front.push_back(t); }
        }
        if (!front.empty() && (int64_t)front.size() < n) {
            std::stable_sort(front.begin(), front.end(), [&](int32_t x, int32_t y) { return tile_maxdeg[x] > tile_maxdeg[y]; });
            std::vector<int32_t> reordered(front);
            reordered.reserve(order.size());
            for (int32_t t : order) if (!hoist[t]) reordered.push_back(t);
            order.swap(reordered);
        }
    }
    // device side: any CUDA failure frees what was allocated so far together with the handle
    auto upload = [&]() -> int {
    GN_CUDA(cudaMalloc(&b->d_inst, sizeof(GnInstance) * n_inst));
    GN_CUDA(cudaMalloc(&b->d_tile_inst, sizeof(int32_t) * b->n_tiles));
    GN_CUDA(cudaMalloc(&b->d_tile_order, sizeof(int32_t) * b->n_tiles));
    GN_CUDA(cudaMemcpy(b->d_inst, inst.data(), sizeof(GnInstance) * n_inst, cudaMemcpyHostToDevice));
    GN_CUDA(cudaMalloc(&b->d_inst_e0, sizeof(int64_t) * n_inst));
    GN_CUDA(cudaMemcpy(b->d_inst_e0, inst_e0.data(), sizeof(int64_t) * n_inst, cudaMemcpyHostToDevice));
    GN_CUDA(cudaMemcpy(b->d_tile_inst, tile_inst.data(), sizeof(int32_t) * b->n_tiles, cudaMemcpyHostToDevice));
    GN_CUDA(cudaMemcpy(b->d_tile_order, order.data(), sizeof(int32_t) * b->n_tiles, cudaMemcpyHostToDevice));
    {   // schedule entries: tile + the row where the same tile of the NEXT instance starts (I' look-ahead prefetch)
        std::vector<int2> sched(b->n_tiles);
        for (int32_t q = 0; q < b->n_tiles; ++q) {
            const int32_t t = order[q];
            const int64_t ahead = (int64_t)t * TILE + inst[tile_inst[t]].n;
            sched[q].x = t;
            sched[q].y = ahead < M ? (int32_t)ahead : -1;
        }
        GN_CUDA(cudaMalloc(&b->d_sched, sizeof(int2) * b->n_tiles));
        GN_CUDA(cudaMemcpy(b->d_sched, sched.data(), sizeof(int2) * b->n_tiles, cudaMemcpyHostToDevice));
    }
    {   // per-tile metadata of the pipelined step kernel, for 128-row tiles and for their 64-row halves
        auto build = [&](int rows, std::vector<int4>& tm) {
            const int64_t n = (M + rows - 1) / rows;
            int32_t ii = 0;
            for (int64_t u = 0; u < (int64_t)tm.size(); ++u) {
                tm[u] = make_int4(0, 0, 0, 0);
                if (u >= n) continue;                                  // second half of a partial last tile: empty
                const int64_t r0 = u * rows, r1 = std::min<int64_t>(r0 + rows, M);
                while (ii + 1 < n_inst && inst[ii + 1].row0 <= r0) ++ii;
                const bool single = r1 <= (int64_t)inst[ii].row0 + inst[ii].n;
                tm[u].z = ii; tm[u].w = single ? 1 : 0;
                if (single) {
                    const std::vector<int32_t>& rp = inst_graphs[ii]->h_rowptr;
                    tm[u].x = rp[r0 - inst[ii].row0];
                    tm[u].y = rp[r1 - inst[ii].row0] - tm[u].x;
                    // bit 1: sum the tile's hub rows (degree > 512) by the in-order relay of the pipelined step kernel.
                    // Cost model (cycles, measured): relay = 7k per super-round of 2 * rows neighbours, hub after hub;
                    // serial = ~2k per round of 8, hub rows on different warps side by side -> longest row decides.
                    // The relay is chosen only where it wins by 2x (isolated hubs), e.g. not for the first tile of a
                    // Barabasi-Albert graph, whose rows are all hubs.
                    int64_t super_rounds = 0, maxdeg = 0;
                    for (int64_t g = r0; g < r1; ++g) {
                        const int64_t d = rp[g - inst[ii].row0 + 1] - rp[g - inst[ii].row0];
                        maxdeg = std::max(maxdeg, d);
                        if (d > 512) super_rounds += (d + 2 * rows - 1) / (2 * rows);
                    }
                    if (super_rounds > 0 && 2 * 7000 * super_rounds < 2000 * (maxdeg / 8)) tm[u].w |= 2;
                }
            }
        };
        std::vector<int4> tm(b->n_tiles), sm(2 * (size_t)b->n_tiles);
        build(TILE, tm);
        build(TILE / 2, sm);
        GN_CUDA(cudaMalloc(&b->d_tile_meta, sizeof(int4) * tm.size()));
        GN_CUDA(cudaMemcpy(b->d_tile_meta, tm.data(), sizeof(int4) * tm.size(), cudaMemcpyHostToDevice));
        GN_CUDA(cudaMalloc(&b->d_sub_meta, sizeof(int4) * sm.size()));
        GN_CUDA(cudaMemcpy(b->d_sub_meta, sm.data(), sizeof(int4) * sm.size(), cudaMemcpyHostToDevice));
        // Work items of the neighbour gather (step_stream_kernel): uint8 rows[64][4] per tile. A warp sums the rows
        // {a, b} of an item in its lower half-warp and {c, d} in its upper one, all loads of the item in ONE memory round
        // trip (at most 12 neighbour rows per lane), and both half-warps run the trip count of the longer side (padding
        // slots read the all-zero row). So: the tile's rows are sorted by degree; rows with at most 6 neighbours go four
        // to an item (two per half-warp, 6 + 6 slots: half as many round trips for them -- 47 % of the rows of a
        // Barabasi-Albert graph with m = 5), the others two to an item with a neighbour of (nearly) the same degree
        // (b = d = 0xFF). Tiles whose CSR slice fits the staged window stride the items over the 16 warps (warp w takes
        // items w, w + 16, w + 32, w + 48): the items are dealt to the warps longest first, each to the warp with the
        // fewest round trips so far (a row of degree d > 12 needs 1 + ceil((d - 12) / 8) of them). Hub tiles draw items from
        // a ticket counter, longest first, and form no four-row items (their slice overflows the window). Unused item
        // slots are 0xFF. The sums themselves do not depend on the grouping: every row is still added up alone, in
        // ascending column order.
        const bool no_sort = getenv("GNODE_NO_PAIR_SORT") != nullptr;                          // A/B: rows 2p, 2p+1 as they come
        const bool no_quads = no_sort || getenv("GNODE_NO_QUADS") != nullptr;                  // A/B: two-row items only
        std::vector<uint8_t> perm((size_t)b->n_tiles * 256, 0xFF);
        std::vector<int32_t> deg(TILE), start(258);
        std::vector<uint8_t> sorted(TILE);
        struct Item { uint8_t r[4]; int32_t cost; };
        std::vector<Item> items;
        items.reserve(64);
        auto rounds = [](int32_t d) { return d <= 12 ? 1 : 1 + (d - 12 + 7) / 8; };
        for (int32_t t = 0; t < b->n_tiles; ++t) {
            uint8_t* out_items = perm.data() + (size_t)t * 256;
            const int64_t nr = std::min<int64_t>(TILE, M - (int64_t)t * TILE);
            if (!(tm[t].w & 1) || no_sort) {                                                   // rows as they come, two per item
                for (int p = 0; p < TILE / 2; ++p) { out_items[4 * p] = (uint8_t)(2 * p); out_items[4 * p + 2] = (uint8_t)(2 * p + 1); }
                continue;
            }
            const int32_t ii = tm[t].z;
            const std::vector<int32_t>& rp = inst_graphs[ii]->h_rowptr;
            const int64_t r0 = (int64_t)t * TILE - inst[ii].row0;
            std::fill(start.begin(), start.end(), 0);
            for (int r = 0; r < nr; ++r) { deg[r] = rp[r0 + r + 1] - rp[r0 + r]; start[std::min(deg[r], 255) + 1]++; }
            for (int k = 1; k < 258; ++k) start[k] += start[k - 1];
            for (int r = 0; r < nr; ++r) sorted[start[std::min(deg[r], 255)]++] = (uint8_t)r;   // ascending degree, stable
            const bool strided = tm[t].y <= 1536;
            items.clear();
            int pos = 0;
            if (strided && !no_quads)
                for (; pos + 4 <= nr && deg[sorted[pos + 3]] <= 6; pos += 4)
                    items.push_back(Item{{sorted[pos], sorted[pos + 1], sorted[pos + 2], sorted[pos + 3]}, 1});
            for (; pos < nr; pos += 2) {
                const bool two = pos + 1 < nr;
                items.push_back(Item{{sorted[pos], 0xFF, two ? sorted[pos + 1] : (uint8_t)0xFF, 0xFF},
                                     rounds(deg[two ? sorted[pos + 1] : sorted[pos]])});
            }
            std::stable_sort(items.begin(), items.end(), [](const Item& x, const Item& y) { return x.cost > y.cost; });
            if (!strided) {                                                                    // tickets: longest first
                for (size_t i = 0; i < items.size(); ++i) memcpy(out_items + 4 * i, items[i].r, 4);
                continue;
            }
            int32_t load[16] = {0}, cnt[16] = {0};
            for (const Item& it : items) {
                int best = -1;
                for (int w = 0; w < 16; ++w)
                    if (cnt[w] < 4 && (best < 0 || load[w] < load[best])) best = w;
                memcpy(out_items + 4 * (best + 16 * cnt[best]), it.r, 4);
                load[best] += it.cost; cnt[best]++;
            }
        }
        GN_CUDA(cudaMalloc(&b->d_tile_perm, perm.size()));
        GN_CUDA(cudaMemcpy(b->d_tile_perm, perm.data(), perm.size(), cudaMemcpyHostToDevice));
    }
    return GNODE_OK;
    };
    const int rc = upload();
    if (rc != GNODE_OK) { gnode_batch_destroy(b); return rc; }
    *out = b;
    return GNODE_OK;
}

extern "C" int gnode_batch_destroy(gnode_batch_t b) {
    if (!b) return GNODE_OK;
    for (auto& e : b->bwd_graphs) cudaGraphExecDestroy((cudaGraphExec_t)e.exec);
    if (b->capture_stream) cudaStreamDestroy((cudaStream_t)b->capture_stream);
    cudaFree(b->d_inst);
    cudaFree(b->d_inst_e0);
    cudaFree(b->d_inst_tmap);
    cudaFree(b->d_tile_inst);
    cudaFree(b->d_tile_order);
    cudaFree(b->d_sched);
    cudaFree(b->d_tile_meta);
    cudaFree(b->d_sub_meta);
    cudaFree(b->d_tile_perm);
    delete b;
    return GNODE_OK;
}

extern "C" int64_t gnode_batch_rows(gnode_batch_t b) { return b ? b->M : -1; }

namespace gnode {
int ensure_transpose_maps(gnode_batch* b) {
    if (b->d_inst_tmap) return GNODE_OK;
    std::vector<const int32_t*> maps(b->n_inst);
    for (int32_t i = 0; i < b->n_inst; ++i) {
        gnode_graph* g = b->graphs[i];
        if (!g->d_tmap) {
            int32_t* d = nullptr;
            GN_CUDA(cudaMalloc(&d, sizeof(int32_t) * (size_t)std::max<int64_t>(g->nnz, 1)));
            if (g->nnz) {
                const cudaError_t e = cudaMemcpy(d, g->h_tmap.data(), sizeof(int32_t) * g->nnz, cudaMemcpyHostToDevice);
                if (e != cudaSuccess) { cudaFree(d); GN_CUDA(e); }
            }
            g->d_tmap = d;
        }
        maps[i] = g->d_tmap;
    }
    const int32_t** d = nullptr;
    GN_CUDA(cudaMalloc(&d, sizeof(const int32_t*) * b->n_inst));
    const cudaError_t e = cudaMemcpy(d, maps.data(), sizeof(const int32_t*) * b->n_inst, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(d); GN_CUDA(e); }
    b->d_inst_tmap = d;
    return GNODE_OK;
}
}  // namespace gnode

extern "C" int gnode_aggregate(gnode_batch_t b, const float* in, float* out, int transpose, void* stream) {
    if (!b || !in || !out) { set_error("gnode_aggregate: null argument"); return GNODE_ERR_ARG; }
    if (int rc = check_current_device(b, "gnode_aggregate")) return rc;
    const int hw_per_block = 256 / 16;
    int64_t blocks = (b->M + hw_per_block - 1) / hw_per_block;
    blocks = std::min<int64_t>(blocks, (int64_t)b->sm_count * 16);
    aggregate_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(gn_view(b), in, out, transpose);
    GN_LAUNCH_CHECK();
    return GNODE_OK;
}
