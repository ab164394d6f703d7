// K3: cut-off (radius) search, two-pass count -> scan -> fill.
//
// Replaces `radius_neighbors_graph(target, radius)` of CutOffEdges.get_adjacency_matrix
// (/root/reference/src/anemoi/graphs/edges/builder.py:364-366; sklearn _binary_tree.pxi.tp:1902-1979:
// a point is a neighbour iff rdist <= sin^2(radius/2), inclusive).
// One warp per query; the lanes stride over the contiguous record run of each window row (coalesced
// LDG.128), classify on the FP32 FMA pipe against chord^2 = 4 sin^2(r/2) -/+ the FP32 error margin, and
// only the pairs inside the margin evaluate the reference's float64 haversine.  The fill pass repeats
// the scan and writes (src, dst) with a ballot prefix, so the output order is the scan order:
// deterministic, grouped by query.
//
// Low-degree searches (few candidates per query: the warp would idle) use the tile form of the KNN kernel instead:
// one warp per 32 queries, the union window staged through shared memory by TMA, every lane scanning it for its own
// query.  Hits of a query come out in the same order either way (window rows in face / row order, records in
// cell / index order), so the two forms are interchangeable bit for bit.
#include "agx_tile.cuh"

template <bool FILL>
__global__ void __launch_bounds__(256) k_radius(const float4* __restrict__ pts, const int* __restrict__ cell_start,
                                                const float2* __restrict__ ref_latlon, int cells,
                                                const float2* __restrict__ q_latlon, int64_t nq, float chord2_thr,
                                                float chord2_margin, double rdist_thr, int32_t* __restrict__ counts,
                                                const int64_t* __restrict__ offsets, int32_t* __restrict__ out_src,
                                                int32_t* __restrict__ out_dst, int64_t dst_base,
                                                unsigned long long* __restrict__ stats, const int64_t* __restrict__ src_map,
                                                const int64_t* __restrict__ dst_map) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float t_in = chord2_thr - chord2_margin, t_out = chord2_thr + chord2_margin;
    const AgxCap cap = agx_make_cap(t_out);
    unsigned long long n_f64 = 0, n_boundary = 0;
    for (int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < nq; q += warps) {
        const float2 ql = q_latlon[q];
        const float3 qv = agx_search_xyz(ql);
        int64_t out_pos = FILL ? offsets[q] : 0;
        const int32_t dst = dst_map ? (int32_t)dst_map[q] : (int32_t)(dst_base + q);
        int found = 0;
        // single-face fast path (the cap ends at least a cell inside the query's major face), else all six faces
        const int mface = agx_major_face(qv.x, qv.y, qv.z);
        int fi0, fi1, fj0, fj1;
        bool fast;
        {
            float fa, fb, fc;
            agx_face_frame(mface, qv.x, qv.y, qv.z, fa, fb, fc);
            fast = !cap.everything && agx_axis_window_major(fa, fc, cap, cells, fi0, fi1);
            fast = fast && agx_axis_window_major(fb, fc, cap, cells, fj0, fj1);
        }
        const int face_end = fast ? mface + 1 : 6;
        for (int face = fast ? mface : 0; face < face_end; ++face) {
            int i0 = fi0, i1 = fi1, j0 = fj0, j1 = fj1;
            if (!fast && !agx_face_window(face, qv, cap, cells, i0, i1, j0, j1)) continue;
            for (int i = i0; i <= i1; ++i) {
                int row = (face * cells + i) * cells;
                int s = __ldg(cell_start + row + j0), e = __ldg(cell_start + row + j1 + 1);
                for (int base = s; base < e; base += 32) {
                    int p = base + lane;
                    bool hit = false;
                    int ci = 0;
                    if (p < e) {
                        float4 c = __ldg(pts + p);
                        ci = __float_as_int(c.w);
                        float dx = qv.x - c.x, dy = qv.y - c.y, dz = qv.z - c.z;
                        float d = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
                        if (d <= t_in) {
                            hit = true;
                        } else if (d <= t_out) {
                            double r = agx_rdist64(ql, ref_latlon[ci]);
                            hit = r <= rdist_thr;
                            if (FILL) {
                                ++n_f64;
                                if (fabs(r - rdist_thr) <= AGX_TIE_TAU * rdist_thr) ++n_boundary;
                            }
                        }
                    }
                    unsigned m = __ballot_sync(0xffffffffu, hit);
                    if (FILL) {
                        if (hit) {
                            int64_t w = out_pos + __popc(m & ((1u << lane) - 1u));
                            out_src[w] = src_map ? (int32_t)src_map[ci] : ci;
                            out_dst[w] = dst;
                        }
                        out_pos += __popc(m);
                    } else {
                        found += __popc(m);
                    }
                }
            }
        }
        if (!FILL && lane == 0) counts[q] = found;
    }
    if (FILL && stats) {
        if (n_f64) atomicAdd(stats + 0, n_f64);
        if (n_boundary) atomicAdd(stats + 1, n_boundary);
    }
}

struct RadiusArgs {
    const float4* pts;
    const int* cell_start;
    const float2* ref_latlon;
    int cells;
    const float2* q_latlon;
    const int32_t* qperm;
    int64_t nq;
    float t_in, t_out;
    double rdist_thr;
    int32_t* counts;
    const int64_t* offsets;
    int32_t* out_src;
    int32_t* out_dst;
    int64_t dst_base;
    unsigned long long* stats;
    const int64_t* src_map;  // output label maps (undo_masking fused into the write), NULL: identity
    const int64_t* dst_map;
};

template <bool FILL>
__global__ void __launch_bounds__(AGX_TILE_WARPS * 32) k_radius_tile(RadiusArgs a) {
    __shared__ __align__(128) float4 stage_all[AGX_TILE_WARPS][AGX_TILE_STAGE];
    __shared__ __align__(8) uint64_t bars[AGX_TILE_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4* stage = stage_all[warp];
    uint64_t* bar = &bars[warp];
    if (lane == 0) mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    uint32_t phase = 0;
    const AgxCap cap = agx_make_cap(a.t_out);
    unsigned long long n_f64 = 0, n_boundary = 0;
    const int64_t n_tiles = (a.nq + 31) >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * AGX_TILE_WARPS;
    for (int64_t tile = (int64_t)blockIdx.x * AGX_TILE_WARPS + warp; tile < n_tiles; tile += warps_total) {
        const int64_t slot = tile * 32 + lane;
        const bool active = slot < a.nq;
        const int64_t qs = active ? slot : a.nq - 1;
        const int64_t q = a.qperm ? (int64_t)__ldg(a.qperm + qs) : qs;
        const float2 ql = a.q_latlon[q];
        const float3 qv = agx_search_xyz(ql);
        int s = 0, cnt = 0, incl = 0, m_total = 0;
        const bool fits = agx_tile_plan(a.cell_start, a.cells, qv, cap, lane, s, cnt, incl, m_total);
        if (fits && m_total > 0) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)m_total * 16u);
            if (cnt > 0) bulk_copy_g2s(stage + (incl - cnt), a.pts + s, (uint32_t)cnt * 16u, bar);
            mbar_wait(bar, phase);
            phase ^= 1;
        }
        int found = 0;
        int64_t out_pos = (FILL && active) ? a.offsets[q] : 0;
        const int32_t dst = a.dst_map ? (int32_t)a.dst_map[q] : (int32_t)(a.dst_base + q);
        auto visit = [&](const float4 c) {
            float dx = qv.x - c.x, dy = qv.y - c.y, dz = qv.z - c.z;
            float d = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
            if (d > a.t_out) return;
            int ci = __float_as_int(c.w);
            if (d > a.t_in) {
                double r = agx_rdist64(ql, a.ref_latlon[ci]);
                if (FILL && active) {
                    ++n_f64;
                    if (fabs(r - a.rdist_thr) <= AGX_TIE_TAU * a.rdist_thr) ++n_boundary;
                }
                if (!(r <= a.rdist_thr)) return;
            }
            if (FILL) {
                if (active) {
                    a.out_src[out_pos] = a.src_map ? (int32_t)a.src_map[ci] : ci;
                    a.out_dst[out_pos] = dst;
                    ++out_pos;
                }
            } else {
                ++found;
            }
        };
        if (fits) {
#pragma unroll 4
            for (int p = 0; p < m_total; ++p) visit(stage[p]);
        } else {
            // queries far apart (or a cap too wide to stage): every lane walks its own window in global memory
            for (int face = 0; face < 6; ++face) {
                int i0, i1, j0, j1;
                if (!agx_face_window(face, qv, cap, a.cells, i0, i1, j0, j1)) continue;
                for (int i = i0; i <= i1; ++i) {
                    int row = (face * a.cells + i) * a.cells;
                    int ps = __ldg(a.cell_start + row + j0), pe = __ldg(a.cell_start + row + j1 + 1);
                    for (int p = ps; p < pe; ++p) visit(__ldg(a.pts + p));
                }
            }
        }
        if (!FILL && active) a.counts[q] = found;
        __syncwarp();  // every lane is done with the stage before the next tile overwrites it
    }
    if (FILL && a.stats) {
        if (n_f64) atomicAdd(a.stats + 0, n_f64);
        if (n_boundary) atomicAdd(a.stats + 1, n_boundary);
    }
}

// Tile form when the 3 x 3 cell neighbourhood of a query is expected to hold at most two warps' worth of
// candidates (uniform-density estimate); AGX_RADIUS_TILE=0 / 1 forces the choice.
static bool radius_use_tiles(const agx_index_t* ix) {
    if (const char* env = getenv("AGX_RADIUS_TILE")) return atoi(env) != 0;
    double w = 1.5707963267948966 / (double)ix->cells;
    double expected = (double)ix->n * 9.0 * w * w / 12.566370614359172;
    return expected <= 64.0;
}

// the processing order of the queries: computed by the count pass, reused by the fill pass of the same queries
static int radius_query_order(const agx_index_t* ix_, const float* q_latlon, int64_t nq, float t_out, bool reuse_only,
                              const int32_t** perm, cudaStream_t stream) {
    agx_index* ix = const_cast<agx_index*>(ix_);
    // only a fill pass may reuse the order (its count pass has just seen the same array); a count pass always decides
    // afresh - the address could belong to a new array by now
    if (reuse_only && ix->order_q == (const void*)q_latlon && ix->order_nq == nq) {
        *perm = ix->order_perm;
        return AGX_OK;
    }
    if (ix->order_perm) {
        AGX_CUDA_OK(cudaFreeAsync(ix->order_perm, stream));
        ix->order_perm = nullptr;
    }
    ix->order_q = nullptr;
    int32_t* fresh = nullptr;
    int rc = agx_query_order(ix, (const float2*)q_latlon, nq, t_out, "AGX_RADIUS_BIN", &fresh, stream);
    if (rc != AGX_OK) return rc;
    ix->order_q = (const void*)q_latlon;
    ix->order_nq = nq;
    ix->order_perm = fresh;
    *perm = fresh;
    return AGX_OK;
}

template <bool FILL>
static int launch_radius_tile(const agx_index_t* ix, const float* q_latlon, int64_t nq, float c2, float m, double thr,
                              int32_t* counts, const int64_t* offsets, int32_t* out_src, int32_t* out_dst, int64_t dst_base,
                              int64_t* stats, cudaStream_t stream) {
    RadiusArgs a;
    a.pts = ix->pts;
    a.cell_start = ix->cell_start;
    a.ref_latlon = ix->latlon;
    a.cells = ix->cells;
    a.q_latlon = (const float2*)q_latlon;
    a.nq = nq;
    a.t_in = c2 - m;
    a.t_out = c2 + m;
    a.rdist_thr = thr;
    a.counts = counts;
    a.offsets = offsets;
    a.out_src = out_src;
    a.out_dst = out_dst;
    a.dst_base = dst_base;
    a.stats = (unsigned long long*)stats;
    agx_output_maps(&a.src_map, &a.dst_map);
    const int32_t* perm = nullptr;
    int rc = radius_query_order(ix, q_latlon, nq, a.t_out, FILL, &perm, stream);
    if (rc != AGX_OK) return rc;
    a.qperm = perm;
    int64_t tiles = (nq + 31) / 32;
    int64_t blocks = (tiles + AGX_TILE_WARPS - 1) / AGX_TILE_WARPS;
    int64_t cap = (int64_t)agx_sm_count() * 16;
    k_radius_tile<FILL><<<(int)(blocks < cap ? blocks : cap), AGX_TILE_WARPS * 32, 0, stream>>>(a);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

extern "C" int agx_radius_count(const agx_index_t* ix, const float* q_latlon, int64_t nq, double radius,
                                int32_t* counts, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(ix != nullptr, AGX_ERR_ARG, "agx_radius_count: NULL index");
    AGX_REQUIRE(nq >= 0, AGX_ERR_ARG, "agx_radius_count: nq < 0");
    float c2, m;
    double thr;
    int rc = agx_radius_params(radius, &c2, &m, &thr);
    if (rc) return rc;
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(q_latlon && counts, AGX_ERR_ARG, "agx_radius_count: NULL buffer");
    if (radius_use_tiles(ix))
        return launch_radius_tile<false>(ix, q_latlon, nq, c2, m, thr, counts, nullptr, nullptr, nullptr, 0, nullptr, stream);
    int grid = agx_grid(nq * 32, 256, 8);
    k_radius<false><<<grid, 256, 0, stream>>>(ix->pts, ix->cell_start, ix->latlon, ix->cells, (const float2*)q_latlon,
                                             nq, c2, m, thr, counts, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

extern "C" int agx_radius_fill(const agx_index_t* ix, const float* q_latlon, int64_t nq, double radius,
                               const int64_t* offsets, int32_t* out_src, int32_t* out_dst, int64_t dst_base,
                               int64_t* stats, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(ix != nullptr, AGX_ERR_ARG, "agx_radius_fill: NULL index");
    AGX_REQUIRE(nq >= 0, AGX_ERR_ARG, "agx_radius_fill: nq < 0");
    AGX_REQUIRE(dst_base + nq < (int64_t)2147483647, AGX_ERR_ARG, "agx_radius_fill: target index exceeds int32");
    float c2, m;
    double thr;
    int rc = agx_radius_params(radius, &c2, &m, &thr);
    if (rc) return rc;
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(q_latlon && offsets && out_src && out_dst, AGX_ERR_ARG, "agx_radius_fill: NULL buffer");
    if (radius_use_tiles(ix))
        return launch_radius_tile<true>(ix, q_latlon, nq, c2, m, thr, nullptr, offsets, out_src, out_dst, dst_base, stats, stream);
    int grid = agx_grid(nq * 32, 256, 8);
    const int64_t *src_map = nullptr, *dst_map = nullptr;
    agx_output_maps(&src_map, &dst_map);
    k_radius<true><<<grid, 256, 0, stream>>>(ix->pts, ix->cell_start, ix->latlon, ix->cells, (const float2*)q_latlon, nq,
                                            c2, m, thr, nullptr, offsets, out_src, out_dst, dst_base,
                                            (unsigned long long*)stats, src_map, dst_map);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}
