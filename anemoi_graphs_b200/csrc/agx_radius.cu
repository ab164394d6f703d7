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

// Warp-cooperative walk of the cell window around one query: every lane calls `visit(hit, ci, refined, r)` once per
// 32-record chunk, in window-row / record order (ci is the record's index where it is a candidate; r its float64 rdist
// where `refined`, i.e. the FP32 filter could not decide and the reference's haversine did).
template <typename Visit>
__device__ __forceinline__ void radius_warp_walk(const float4* __restrict__ pts, const int* __restrict__ cell_start,
                                                 const float2* __restrict__ ref_latlon, int cells, float2 ql, float3 qv,
                                                 const AgxCap& cap, float t_in, float t_out, double rdist_thr, int lane,
                                                 Visit&& visit) {
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
                bool hit = false, refined = false;
                int ci = 0;
                double r = 0.0;
                if (p < e) {
                    float4 c = __ldg(pts + p);
                    ci = __float_as_int(c.w);
                    float dx = qv.x - c.x, dy = qv.y - c.y, dz = qv.z - c.z;
                    float d = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
                    if (d <= t_in) {
                        hit = true;
                    } else if (d <= t_out) {
                        r = agx_rdist64(ql, ref_latlon[ci]);
                        hit = r <= rdist_thr;
                        refined = true;
                    }
                }
                visit(hit, ci, refined, r);
            }
        }
    }
}

// FILL with cap_counts: the queries with cap_counts[q] > cap_m are skipped (k_radius_select writes them).
template <bool FILL>
__global__ void __launch_bounds__(256) k_radius(const float4* __restrict__ pts, const int* __restrict__ cell_start,
                                                const float2* __restrict__ ref_latlon, int cells,
                                                const float2* __restrict__ q_latlon, int64_t nq, float chord2_thr,
                                                float chord2_margin, double rdist_thr, int32_t* __restrict__ counts,
                                                const int64_t* __restrict__ offsets, int32_t* __restrict__ out_src,
                                                int32_t* __restrict__ out_dst, int64_t dst_base,
                                                unsigned long long* __restrict__ stats, const int64_t* __restrict__ src_map,
                                                const int64_t* __restrict__ dst_map, const int32_t* __restrict__ cap_counts,
                                                int cap_m) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float t_in = chord2_thr - chord2_margin, t_out = chord2_thr + chord2_margin;
    const AgxCap cap = agx_make_cap(t_out);
    unsigned long long n_f64 = 0, n_boundary = 0;
    for (int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < nq; q += warps) {
        if (FILL && cap_counts && cap_counts[q] > cap_m) continue;
        const float2 ql = q_latlon[q];
        const float3 qv = agx_search_xyz(ql);
        int64_t out_pos = FILL ? offsets[q] : 0;
        const int32_t dst = dst_map ? (int32_t)dst_map[q] : (int32_t)(dst_base + q);
        int found = 0;
        radius_warp_walk(pts, cell_start, ref_latlon, cells, ql, qv, cap, t_in, t_out, rdist_thr, lane,
                         [&](bool hit, int ci, bool refined, double r) {
                             if (FILL && refined) {
                                 ++n_f64;
                                 if (fabs(r - rdist_thr) <= AGX_TIE_TAU * rdist_thr) ++n_boundary;
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
                         });
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
    const int32_t* cap_counts;  // FILL: skip the queries with cap_counts[q] > cap_m (NULL: no cap)
    int cap_m;
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
        const bool writes = FILL && active && !(a.cap_counts && a.cap_counts[q] > a.cap_m);
        int64_t out_pos = writes ? a.offsets[q] : 0;
        const int32_t dst = a.dst_map ? (int32_t)a.dst_map[q] : (int32_t)(a.dst_base + q);
        auto visit = [&](const float4 c) {
            float dx = qv.x - c.x, dy = qv.y - c.y, dz = qv.z - c.z;
            float d = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
            if (d > a.t_out) return;
            int ci = __float_as_int(c.w);
            if (d > a.t_in) {
                double r = agx_rdist64(ql, a.ref_latlon[ci]);
                if (writes) {
                    ++n_f64;
                    if (fabs(r - a.rdist_thr) <= AGX_TIE_TAU * a.rdist_thr) ++n_boundary;
                }
                if (!(r <= a.rdist_thr)) return;
            }
            if (FILL) {
                if (writes) {
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
                              int64_t* stats, const int32_t* cap_counts, int cap_m, cudaStream_t stream) {
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
    a.cap_counts = cap_counts;
    a.cap_m = cap_m;
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
        return launch_radius_tile<false>(ix, q_latlon, nq, c2, m, thr, counts, nullptr, nullptr, nullptr, 0, nullptr,
                                         nullptr, 0, stream);
    int grid = agx_grid(nq * 32, 256, 8);
    k_radius<false><<<grid, 256, 0, stream>>>(ix->pts, ix->cell_start, ix->latlon, ix->cells, (const float2*)q_latlon,
                                             nq, c2, m, thr, counts, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr,
                                             nullptr, 0);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

static int radius_fill_impl(const char* fn, const agx_index_t* ix, const float* q_latlon, int64_t nq, double radius,
                            const int32_t* cap_counts, int cap_m, const int64_t* offsets, int32_t* out_src,
                            int32_t* out_dst, int64_t dst_base, int64_t* stats, cudaStream_t stream) {
    AGX_REQUIRE(ix != nullptr, AGX_ERR_ARG, "%s: NULL index", fn);
    AGX_REQUIRE(nq >= 0, AGX_ERR_ARG, "%s: nq < 0", fn);
    AGX_REQUIRE(dst_base + nq < (int64_t)2147483647, AGX_ERR_ARG, "%s: target index exceeds int32", fn);
    float c2, m;
    double thr;
    int rc = agx_radius_params(radius, &c2, &m, &thr);
    if (rc) return rc;
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(q_latlon && offsets && out_src && out_dst, AGX_ERR_ARG, "%s: NULL buffer", fn);
    if (radius_use_tiles(ix))
        return launch_radius_tile<true>(ix, q_latlon, nq, c2, m, thr, nullptr, offsets, out_src, out_dst, dst_base, stats,
                                        cap_counts, cap_m, stream);
    int grid = agx_grid(nq * 32, 256, 8);
    const int64_t *src_map = nullptr, *dst_map = nullptr;
    agx_output_maps(&src_map, &dst_map);
    k_radius<true><<<grid, 256, 0, stream>>>(ix->pts, ix->cell_start, ix->latlon, ix->cells, (const float2*)q_latlon, nq,
                                            c2, m, thr, nullptr, offsets, out_src, out_dst, dst_base,
                                            (unsigned long long*)stats, src_map, dst_map, cap_counts, cap_m);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

extern "C" int agx_radius_fill(const agx_index_t* ix, const float* q_latlon, int64_t nq, double radius,
                               const int64_t* offsets, int32_t* out_src, int32_t* out_dst, int64_t dst_base,
                               int64_t* stats, void* stream_) {
    return radius_fill_impl("agx_radius_fill", ix, q_latlon, nq, radius, nullptr, 0, offsets, out_src, out_dst, dst_base,
                            stats, (cudaStream_t)stream_);
}

// ------------------------------------------------------------------------------------------------
// Capped cut-off search (CutOffEdges(max_num_neighbours = M)).  The queries with at most M candidates are written by
// the fill as they are; every other query keeps its M nearest candidates under the KNN tie rule (k_radius_select).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_radius_cap(const int32_t* __restrict__ counts, int64_t nq, int cap_m,
                                                    int32_t* __restrict__ capped, uint8_t* __restrict__ over,
                                                    int32_t* __restrict__ seg) {
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        const int32_t c = counts[q];
        if (capped) capped[q] = c < cap_m ? c : cap_m;
        if (over) over[q] = c > cap_m;
        if (seg) seg[q] = c > cap_m ? c : 0;
    }
}

extern "C" int agx_radius_cap_counts(const int32_t* counts, int64_t nq, int max_neighbours, int32_t* capped,
                                     void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(nq >= 0, AGX_ERR_ARG, "agx_radius_cap_counts: nq < 0");
    AGX_REQUIRE(max_neighbours >= 1, AGX_ERR_ARG, "agx_radius_cap_counts: max_neighbours < 1 (got %d)", max_neighbours);
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(counts && capped, AGX_ERR_ARG, "agx_radius_cap_counts: NULL buffer");
    k_radius_cap<<<agx_grid(nq, 256, 8), 256, 0, stream>>>(counts, nq, max_neighbours, capped, nullptr, nullptr);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

extern "C" int agx_radius_fill_capped(const agx_index_t* ix, const float* q_latlon, int64_t nq, double radius,
                                      const int32_t* counts, int max_neighbours, const int64_t* offsets, int32_t* out_src,
                                      int32_t* out_dst, int64_t dst_base, int64_t* stats, void* stream_) {
    AGX_REQUIRE(max_neighbours >= 1, AGX_ERR_ARG, "agx_radius_fill_capped: max_neighbours < 1 (got %d)", max_neighbours);
    AGX_REQUIRE(nq == 0 || counts, AGX_ERR_ARG, "agx_radius_fill_capped: NULL buffer");
    return radius_fill_impl("agx_radius_fill_capped", ix, q_latlon, nq, radius, counts, max_neighbours, offsets, out_src,
                            out_dst, dst_base, stats, (cudaStream_t)stream_);
}

#define SEL_WARPS 8

// Warp-cooperative step of a radix select: the digit (0..255) that holds the rank-th smallest (1-based) of the keys
// counted into hist[256]; rank becomes the rank inside that digit.  hist is zeroed again for the next pass.
__device__ __forceinline__ int sel_pick_digit(unsigned* hist, unsigned& rank, int lane) {
    __syncwarp();
    unsigned c[8], s = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        c[b] = hist[lane * 8 + b];
        hist[lane * 8 + b] = 0;
        s += c[b];
    }
    unsigned incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const unsigned excl = incl - s;
    const int owner = __ffs(__ballot_sync(0xffffffffu, excl < rank && rank <= incl)) - 1;
    unsigned r = rank - excl;
    int digit = -1;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        if (digit < 0) {
            if (r <= c[b]) digit = lane * 8 + b;
            else r -= c[b];
        }
    }
    digit = __shfl_sync(0xffffffffu, digit, owner);
    rank = __shfl_sync(0xffffffffu, r, owner);
    __syncwarp();
    return digit;
}

// The rank-th smallest (1-based) of the keys key(p, k) yields for p in [0, n) (key returns false: p does not take part),
// bits [0, top_shift + 8) of them; 8 bits per pass.
template <typename Key>
__device__ __forceinline__ unsigned long long sel_radix(unsigned* hist, int64_t n, int top_shift, unsigned rank, int lane,
                                                        Key&& key) {
    unsigned long long prefix = 0, mask = 0;
    for (int shift = top_shift; shift >= 0; shift -= 8) {
        for (int64_t p = lane; p < n; p += 32) {
            unsigned long long k;
            if (key(p, k) && (k & mask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1u);
        }
        const int d = sel_pick_digit(hist, rank, lane);
        prefix |= (unsigned long long)d << shift;
        mask |= 0xffull << shift;
    }
    return prefix;
}

struct SelectArgs {
    const float4* pts;
    const int* cell_start;
    const float2* ref_latlon;
    int cells;
    const float2* q_latlon;
    float t_in, t_out;
    double rdist_thr;
    int m;
    const int32_t* list;       // the over-cap queries, ascending ...
    const int64_t* list_count; // ... and how many (device memory)
    const int64_t* seg_off;    // scratch segment of query q: [seg_off[q], seg_off[q + 1])
    unsigned long long* seg_r; // float64 rdist bits (non-negative: ordered as integers)
    int32_t* seg_i;            // reference index
    const int64_t* offsets;    // the query's M output slots start here
    int32_t* out_src;
    int32_t* out_dst;
    int64_t dst_base;
    unsigned long long* stats;
    const int64_t* src_map;
    const int64_t* dst_map;
};

// One warp per over-cap query: stage every candidate of K3's window with its float64 rdist, radix-select the M-th
// smallest rdist v, and keep the candidates below v's tie group (|r - v| <= 2^-40 v) plus the lowest indices of the
// group (the KNN rule, oracle/exact_search.knn_tie_groups).  Output: ascending (rdist, index), the kept group members
// last, by index.
__global__ void __launch_bounds__(SEL_WARPS * 32) k_radius_select(SelectArgs a) {
    __shared__ unsigned hist_all[SEL_WARPS][256];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned* hist = hist_all[warp];
#pragma unroll
    for (int b = 0; b < 8; ++b) hist[lane * 8 + b] = 0;
    __syncwarp();
    const AgxCap cap = agx_make_cap(a.t_out);
    const int64_t n_list = *a.list_count;
    const int64_t warps = (int64_t)gridDim.x * SEL_WARPS;
    unsigned long long n_f64 = 0, n_boundary = 0, n_capped = 0, n_tied = 0;
    for (int64_t li = (int64_t)blockIdx.x * SEL_WARPS + warp; li < n_list; li += warps) {
        const int64_t q = a.list[li];
        const float2 ql = a.q_latlon[q];
        const float3 qv = agx_search_xyz(ql);
        const int64_t sb = a.seg_off[q], n = a.seg_off[q + 1] - sb;
        unsigned long long* kr = a.seg_r + sb;
        int32_t* ki = a.seg_i + sb;
        int64_t pos = 0;
        radius_warp_walk(a.pts, a.cell_start, a.ref_latlon, a.cells, ql, qv, cap, a.t_in, a.t_out, a.rdist_thr, lane,
                         [&](bool hit, int ci, bool refined, double r) {
                             if (refined) {
                                 ++n_f64;
                                 if (fabs(r - a.rdist_thr) <= AGX_TIE_TAU * a.rdist_thr) ++n_boundary;
                             }
                             if (hit && !refined) r = agx_rdist64(ql, a.ref_latlon[ci]);
                             unsigned m = __ballot_sync(0xffffffffu, hit);
                             if (hit) {
                                 int64_t w = pos + __popc(m & ((1u << lane) - 1u));
                                 kr[w] = (unsigned long long)__double_as_longlong(r);
                                 ki[w] = ci;
                             }
                             pos += __popc(m);
                         });
        __syncwarp();
        // the M-th smallest rdist and its tie group
        const unsigned long long vb = sel_radix(hist, n, 56, (unsigned)a.m, lane, [&](int64_t p, unsigned long long& k) {
            k = kr[p];
            return true;
        });
        const double v = __longlong_as_double((long long)vb), tol = AGX_TIE_TAU * v;
        unsigned nb = 0, ng = 0;
        for (int64_t p = lane; p < n; p += 32) {
            const double r = __longlong_as_double((long long)kr[p]);
            const bool g = fabs(r - v) <= tol;
            nb += !g && r < v;
            ng += g;
        }
        nb = (unsigned)agx_warp_sum((int)nb);
        ng = (unsigned)agx_warp_sum((int)ng);
        const unsigned slots = (unsigned)a.m - nb;  // >= 1: fewer than M candidates lie strictly below v
        unsigned long long last = 0xffffffffull;    // the highest index of the group that is kept
        if (ng > slots) {
            last = sel_radix(hist, n, 24, slots, lane, [&](int64_t p, unsigned long long& k) {
                k = (unsigned)ki[p];
                return fabs(__longlong_as_double((long long)kr[p]) - v) <= tol;
            });
            ++n_tied;
        }
        ++n_capped;
        // compact the M kept candidates to the front of the segment (writes never pass the reads), keyed
        // (rdist bits, index) with the group members at v's bits, so that they follow the rest by index
        int64_t kept = 0;
        for (int64_t base = 0; base < n; base += 32) {
            const int64_t p = base + lane;
            bool keep = false;
            unsigned long long key = 0;
            int32_t id = 0;
            if (p < n) {
                key = kr[p];
                id = ki[p];
                const double r = __longlong_as_double((long long)key);
                const bool g = fabs(r - v) <= tol;
                keep = g ? (unsigned long long)(unsigned)id <= last : r < v;
                if (g) key = vb;
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int64_t w = kept + __popc(m & ((1u << lane) - 1u));
                kr[w] = key;
                ki[w] = id;
            }
            kept += __popc(m);
        }
        __syncwarp();
        // emit: the position of a kept candidate is the number of kept candidates before it
        const int64_t ob = a.offsets[q];
        const int32_t dst = a.dst_map ? (int32_t)a.dst_map[q] : (int32_t)(a.dst_base + q);
        for (int i = lane; i < a.m; i += 32) {
            const unsigned long long ka = kr[i];
            const int32_t ia = ki[i];
            int rank = 0;
            for (int j = 0; j < a.m; ++j) {
                const unsigned long long kb = kr[j];
                rank += kb < ka || (kb == ka && ki[j] < ia);
            }
            a.out_src[ob + rank] = a.src_map ? (int32_t)a.src_map[ia] : ia;
            a.out_dst[ob + rank] = dst;
        }
    }
    if (a.stats) {
        if (n_f64) atomicAdd(a.stats + 0, n_f64);
        if (n_boundary) atomicAdd(a.stats + 1, n_boundary);
        if (lane == 0 && n_capped) atomicAdd(a.stats + 2, n_capped);  // per warp, not per lane
        if (lane == 0 && n_tied) atomicAdd(a.stats + 3, n_tied);
    }
}

extern "C" int agx_radius_select(const agx_index_t* ix, const float* q_latlon, int64_t nq, double radius,
                                 const int32_t* counts, int max_neighbours, const int64_t* offsets, int32_t* out_src,
                                 int32_t* out_dst, int64_t dst_base, int64_t* stats, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(ix != nullptr, AGX_ERR_ARG, "agx_radius_select: NULL index");
    AGX_REQUIRE(nq >= 0, AGX_ERR_ARG, "agx_radius_select: nq < 0");
    AGX_REQUIRE(max_neighbours >= 1, AGX_ERR_ARG, "agx_radius_select: max_neighbours < 1 (got %d)", max_neighbours);
    AGX_REQUIRE(dst_base + nq < (int64_t)2147483647, AGX_ERR_ARG, "agx_radius_select: target index exceeds int32");
    float c2, m;
    double thr;
    int rc = agx_radius_params(radius, &c2, &m, &thr);
    if (rc) return rc;
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(q_latlon && counts && offsets && out_src && out_dst, AGX_ERR_ARG, "agx_radius_select: NULL buffer");
    AGX_REQUIRE(nq < (int64_t)2147483647, AGX_ERR_ARG, "agx_radius_select: nq exceeds int32");
    // the over-cap queries (list, count on the device) and their scratch segments: sum of their counts
    uint8_t* over = nullptr;
    int32_t *seg = nullptr, *list = nullptr;
    int64_t *seg_off = nullptr, *list_count = nullptr, seg_total = 0;
    agx_pool_keep_warm();
    AGX_CUDA_OK(cudaMallocAsync(&over, (size_t)((nq + 3) & ~3ll), stream));
    AGX_CUDA_OK(cudaMallocAsync(&seg, nq * sizeof(int32_t), stream));
    AGX_CUDA_OK(cudaMallocAsync(&list, nq * sizeof(int32_t), stream));
    AGX_CUDA_OK(cudaMallocAsync(&seg_off, (nq + 1) * sizeof(int64_t), stream));
    AGX_CUDA_OK(cudaMallocAsync(&list_count, sizeof(int64_t), stream));
    k_radius_cap<<<agx_grid(nq, 256, 8), 256, 0, stream>>>(counts, nq, max_neighbours, nullptr, over, seg);
    agx_note_launch(1);
    rc = agx_compact_flags(over, nq, list, list_count, stream);
    if (rc == AGX_OK) rc = agx_exclusive_scan(seg, nq, seg_off, &seg_total, stream);  // reads the total back
    unsigned long long* seg_r = nullptr;
    int32_t* seg_i = nullptr;
    if (rc == AGX_OK && seg_total > 0) {
        if (cudaMallocAsync(&seg_r, seg_total * sizeof(unsigned long long), stream) != cudaSuccess ||
            cudaMallocAsync(&seg_i, seg_total * sizeof(int32_t), stream) != cudaSuccess) {
            agx_set_error("agx_radius_select: cannot allocate %lld scratch candidates", (long long)seg_total);
            rc = AGX_ERR_CUDA;
        }
    }
    if (rc == AGX_OK && seg_total > 0) {
        SelectArgs a;
        a.pts = ix->pts;
        a.cell_start = ix->cell_start;
        a.ref_latlon = ix->latlon;
        a.cells = ix->cells;
        a.q_latlon = (const float2*)q_latlon;
        a.t_in = c2 - m;
        a.t_out = c2 + m;
        a.rdist_thr = thr;
        a.m = max_neighbours;
        a.list = list;
        a.list_count = list_count;
        a.seg_off = seg_off;
        a.seg_r = seg_r;
        a.seg_i = seg_i;
        a.offsets = offsets;
        a.out_src = out_src;
        a.out_dst = out_dst;
        a.dst_base = dst_base;
        a.stats = (unsigned long long*)stats;
        agx_output_maps(&a.src_map, &a.dst_map);
        k_radius_select<<<agx_grid(nq * 32, SEL_WARPS * 32, 8), SEL_WARPS * 32, 0, stream>>>(a);
        agx_note_launch(1);
        if (cudaGetLastError() != cudaSuccess) {
            agx_set_error("agx_radius_select: launch failed");
            rc = AGX_ERR_CUDA;
        }
    }
    if (seg_r) cudaFreeAsync(seg_r, stream);
    if (seg_i) cudaFreeAsync(seg_i, stream);
    cudaFreeAsync(over, stream);
    cudaFreeAsync(seg, stream);
    cudaFreeAsync(list, stream);
    cudaFreeAsync(seg_off, stream);
    cudaFreeAsync(list_count, stream);
    return rc;
}
