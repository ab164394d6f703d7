// GaussianDistanceWeights (edges/attributes.py): w = exp(-d^2 / (2 sigma^2)) per edge, in float64 from the float32
// EdgeLength d, normalised within each TARGET node's edges (a "group") and rounded to float32 once.
//
// Invariance: permuting the columns of edge_index permutes the output the same way, bit for bit.  So the statistics of
// a group are reduced in an order fixed by the group's contents: its edges in ascending (target, source) order - the
// permutation agx_sort_edges gives - and one fixed tree over that order (below).  Equal columns carry equal weights.
//
// The tree.  The group's n weights in canonical order are cut into chunks of 1024.  A chunk is reduced as one warp
// would: lane l adds the positions l, l + 32, ... of the chunk in order, then a shfl_down tree (16, 8, 4, 2, 1) leaves
// the chunk's value in lane 0.  The chunk values are reduced by the same rule once more (lane l adds chunks l, l + 32,
// ... in order, then the tree).  Lanes without elements carry the identity, and adding +0 (or min / max with +-inf)
// is exact, so a shorter tree over fewer lanes gives the same bits: three paths, one result -
//   n <= 8      one thread per group, the last three levels of the tree in registers;
//   n <= 1024   one warp per group (one chunk: the second level is the identity);
//   n > 1024    every warp of the grid over the chunks of every such group, then one warp per group over its chunks.
// unit-std takes two passes, mean first, then sum (w - mean)^2.
//
// The per-target table holds (shift, div); the scaling pass runs in the original column order:
// out[e] = float32((w[e] - shift[t]) / div[t]).  A division rather than a product with a reciprocal: the reciprocal of
// a subnormal sum overflows, where the reference's w / sum is finite.  The weight is ONE non-inlined function, so the
// reduction and the scaling pass run the same instructions and see the same float64 bits.
#include "agx_common.cuh"

#define GW_CHUNK 1024
#define GW_SMALL 8
#define GW_THREADS 256

__device__ __noinline__ double gw_weight(float len, double two_sigma2) {
    const double d = (double)len;
    return exp(-__ddiv_rn(__dmul_rn(d, d), two_sigma2));
}

struct GwStat {
    double sum, sq, mn, mx;  // pass 1: sum w, sum w^2, min, max; pass 2: sq = sum (w - mean)^2
};

__device__ __forceinline__ GwStat gw_identity() {
    GwStat s = {0.0, 0.0, __longlong_as_double(0x7ff0000000000000ll), __longlong_as_double(0xfff0000000000000ll)};
    return s;
}

__device__ __forceinline__ void gw_merge(GwStat& s, const GwStat& o) {
    s.sum = __dadd_rn(s.sum, o.sum);
    s.sq = __dadd_rn(s.sq, o.sq);
    s.mn = fmin(s.mn, o.mn);
    s.mx = fmax(s.mx, o.mx);
}

// one element into a lane's running value
__device__ __forceinline__ void gw_add(GwStat& s, double w, int pass, double mean) {
    if (pass == 1) {
        s.sum = __dadd_rn(s.sum, w);
        s.sq = __fma_rn(w, w, s.sq);
        s.mn = fmin(s.mn, w);
        s.mx = fmax(s.mx, w);
    } else {
        const double d = __dsub_rn(w, mean);
        s.sq = __fma_rn(d, d, s.sq);
    }
}

__device__ __forceinline__ GwStat gw_warp_tree(GwStat s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        GwStat t;
        t.sum = __shfl_down_sync(0xffffffffu, s.sum, o);
        t.sq = __shfl_down_sync(0xffffffffu, s.sq, o);
        t.mn = __shfl_down_sync(0xffffffffu, s.mn, o);
        t.mx = __shfl_down_sync(0xffffffffu, s.mx, o);
        gw_merge(s, t);
    }
    return s;
}

// one chunk [base, base + cnt), cnt <= GW_CHUNK, of sorted positions; the result is in lane 0
__device__ __forceinline__ GwStat gw_chunk(const int32_t* __restrict__ perm, int64_t base, int cnt, const float* __restrict__ len,
                                           double two_s2, int pass, double mean, int lane) {
    GwStat s = gw_identity();
    for (int j = lane; j < cnt; j += 32) gw_add(s, gw_weight(__ldg(len + __ldg(perm + base + j)), two_s2), pass, mean);
    return gw_warp_tree(s);
}

// (shift, div) of a group from its pass-1 statistics s and (unit-std) the pass-2 sum of squared deviations
__device__ __forceinline__ double2 gw_params(int norm, const GwStat& s, double ssd, int64_t n) {
    double shift = 0.0, div = 1.0;
    if (norm == AGX_NORM_L1) div = s.sum;
    else if (norm == AGX_NORM_L2) div = sqrt(s.sq);
    else if (norm == AGX_NORM_UNIT_MAX) div = s.mx;
    else if (norm == AGX_NORM_UNIT_RANGE) { shift = s.mn; div = __dsub_rn(s.mx, s.mn); }
    else if (norm == AGX_NORM_UNIT_STD) {
        const double sd = sqrt(__ddiv_rn(ssd, (double)n));
        // normalise.py skips std == 0; bit-equal weights (max == min) are that case exactly
        div = (s.mx == s.mn || sd == 0.0) ? 1.0 : sd;
    }
    // a NaN weight (an antipodal pair's length) makes numpy's sum, max, min and std of its group NaN
    if (isnan(s.sum)) { shift = 0.0; div = __longlong_as_double(0x7ff8000000000000ll); }
    return make_double2(shift, div);
}

// first[t] / end[t]: the sorted positions of target t's group (both 0 for a target without edges)
__global__ void __launch_bounds__(GW_THREADS) k_gw_bounds(const int32_t* __restrict__ edst, const int32_t* __restrict__ perm,
                                                          int64_t n, int64_t n_dst, int32_t* __restrict__ first,
                                                          int32_t* __restrict__ end) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t t = __ldg(edst + __ldg(perm + i));
        if (t < 0 || t >= n_dst) continue;  // the caller has checked the endpoints (agx_sort_edges): never taken
        if (i == 0 || __ldg(edst + __ldg(perm + i - 1)) != t) first[t] = (int32_t)i;
        if (i == n - 1 || __ldg(edst + __ldg(perm + i + 1)) != t) end[t] = (int32_t)(i + 1);
    }
}

// counters[0]: groups of (GW_SMALL, GW_CHUNK] edges, listed in warp_list; counters[1]: larger groups, listed in big
// (target, first chunk slot, chunks); counters[2]: chunk slots handed out
struct GwBig {
    int32_t t, slot, chunks, pad;
};

__global__ void __launch_bounds__(GW_THREADS) k_gw_small(const int32_t* __restrict__ perm, const float* __restrict__ len,
                                                         int64_t n_dst, const int32_t* __restrict__ first,
                                                         const int32_t* __restrict__ end, double two_s2, int norm,
                                                         double2* __restrict__ table, int32_t* __restrict__ counters,
                                                         int32_t* __restrict__ warp_list, GwBig* __restrict__ big) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_dst; t += (int64_t)gridDim.x * blockDim.x) {
        const int32_t b = first[t], n = end[t] - b;
        if (n <= 0) continue;
        if (n > GW_CHUNK) {
            const int32_t chunks = (n + GW_CHUNK - 1) / GW_CHUNK;
            GwBig g = {(int32_t)t, atomicAdd(counters + 2, chunks), chunks, 0};
            big[atomicAdd(counters + 1, 1)] = g;
            continue;
        }
        if (n > GW_SMALL) {
            warp_list[atomicAdd(counters, 1)] = (int32_t)t;
            continue;
        }
        // lanes 0..7 of the chunk tree hold one element each; levels 16 and 8 add +0
        double w[GW_SMALL];
#pragma unroll
        for (int j = 0; j < GW_SMALL; ++j) w[j] = j < n ? gw_weight(__ldg(len + __ldg(perm + b + j)), two_s2) : 0.0;
        GwStat s = gw_identity();
        double sum[GW_SMALL], sq[GW_SMALL];
#pragma unroll
        for (int j = 0; j < GW_SMALL; ++j) {
            sum[j] = w[j];
            sq[j] = __dmul_rn(w[j], w[j]);
            if (j < n) {
                s.mn = fmin(s.mn, w[j]);
                s.mx = fmax(s.mx, w[j]);
            }
        }
#pragma unroll
        for (int o = GW_SMALL / 2; o > 0; o >>= 1)
#pragma unroll
            for (int l = 0; l < o; ++l) {
                sum[l] = __dadd_rn(sum[l], sum[l + o]);
                sq[l] = __dadd_rn(sq[l], sq[l + o]);
            }
        s.sum = sum[0];
        s.sq = sq[0];
        double ssd = 0.0;
        if (norm == AGX_NORM_UNIT_STD) {
            const double mean = __ddiv_rn(s.sum, (double)n);
#pragma unroll
            for (int j = 0; j < GW_SMALL; ++j) {
                const double d = __dsub_rn(w[j], mean);
                sq[j] = j < n ? __dmul_rn(d, d) : 0.0;
            }
#pragma unroll
            for (int o = GW_SMALL / 2; o > 0; o >>= 1)
#pragma unroll
                for (int l = 0; l < o; ++l) sq[l] = __dadd_rn(sq[l], sq[l + o]);
            ssd = sq[0];
        }
        table[t] = gw_params(norm, s, ssd, n);
    }
}

__global__ void __launch_bounds__(GW_THREADS) k_gw_warp(const int32_t* __restrict__ perm, const float* __restrict__ len,
                                                        const int32_t* __restrict__ first, const int32_t* __restrict__ end,
                                                        double two_s2, int norm, double2* __restrict__ table,
                                                        const int32_t* __restrict__ counters,
                                                        const int32_t* __restrict__ warp_list) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5, n_items = counters[0];
    for (int64_t q = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < n_items; q += n_warps) {
        const int32_t t = warp_list[q], b = first[t], n = end[t] - b;
        const GwStat s = gw_chunk(perm, b, n, len, two_s2, 1, 0.0, lane);
        double ssd = 0.0;
        if (norm == AGX_NORM_UNIT_STD) {
            const double mean = __ddiv_rn(__shfl_sync(0xffffffffu, s.sum, 0), (double)n);
            ssd = gw_chunk(perm, b, n, len, two_s2, 2, mean, lane).sq;
        }
        if (lane == 0) table[t] = gw_params(norm, s, ssd, n);
    }
}

// large groups, level 1: every warp of the grid takes chunks of every listed group; pass 2 reads the group's mean
// from its pass-1 statistics
__global__ void __launch_bounds__(GW_THREADS) k_gw_big_chunks(const int32_t* __restrict__ perm, const float* __restrict__ len,
                                                              const int32_t* __restrict__ first, const int32_t* __restrict__ end,
                                                              double two_s2, int pass, const int32_t* __restrict__ counters,
                                                              const GwBig* __restrict__ big, const GwStat* __restrict__ big_stat,
                                                              GwStat* __restrict__ partial) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5, gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int n_big = counters[1];
    for (int g = 0; g < n_big; ++g) {
        const GwBig e = big[g];
        const int32_t b = first[e.t], n = end[e.t] - b;
        const double mean = pass == 2 ? __ddiv_rn(big_stat[g].sum, (double)n) : 0.0;
        for (int64_t c = gw; c < e.chunks; c += n_warps) {
            const int64_t base = (int64_t)b + c * GW_CHUNK;
            const int cnt = (int)min((int64_t)GW_CHUNK, (int64_t)b + n - base);
            const GwStat s = gw_chunk(perm, base, cnt, len, two_s2, pass, mean, lane);
            if (lane == 0) partial[e.slot + c] = s;
        }
    }
}

// large groups, level 2: one warp per group over its chunk values
__global__ void __launch_bounds__(GW_THREADS) k_gw_big_groups(const int32_t* __restrict__ first, const int32_t* __restrict__ end,
                                                              int norm, int pass, const int32_t* __restrict__ counters,
                                                              const GwBig* __restrict__ big, GwStat* __restrict__ big_stat,
                                                              const GwStat* __restrict__ partial, double2* __restrict__ table) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5, n_big = counters[1];
    for (int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < n_big; g += n_warps) {
        const GwBig e = big[g];
        GwStat s = gw_identity();
        for (int c = lane; c < e.chunks; c += 32) gw_merge(s, partial[e.slot + c]);
        s = gw_warp_tree(s);
        if (lane != 0) continue;
        const int64_t n = end[e.t] - first[e.t];
        if (pass == 1) big_stat[g] = s;
        if (pass == 2 || norm != AGX_NORM_UNIT_STD) table[e.t] = pass == 2 ? gw_params(norm, big_stat[g], s.sq, n) : gw_params(norm, s, 0.0, n);
    }
}

// the scaling pass, in the original column order (norm None: no table, the weights themselves)
__global__ void __launch_bounds__(GW_THREADS) k_gw_apply(const int32_t* __restrict__ edst, int64_t n, int64_t n_dst,
                                                         const float* __restrict__ len, double two_s2,
                                                         const double2* __restrict__ table, float* __restrict__ out) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const double w = gw_weight(__ldg(len + e), two_s2);
        if (table == nullptr) {
            out[e] = (float)w;
            continue;
        }
        const int32_t t = __ldg(edst + e);
        if (t < 0 || t >= n_dst) continue;  // checked by the caller: never taken
        const double2 p = __ldg(table + t);
        out[e] = (float)__ddiv_rn(__dsub_rn(w, p.x), p.y);
    }
}

static inline int64_t gw_max_big(int64_t n_edges) { return n_edges / GW_CHUNK + 1; }
static inline int64_t gw_max_chunks(int64_t n_edges) { return 2 * (n_edges / GW_CHUNK) + 2; }

extern "C" int agx_gaussian_weights(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, int64_t n_src_nodes,
                                    int64_t n_dst_nodes, const float* lengths, double sigma, int norm, const int32_t* perm,
                                    float* out, void* scratch, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_edges >= 0 && n_edges < (int64_t)2147483647 && n_dst_nodes >= 0 && n_dst_nodes <= 2147483647ll,
                AGX_ERR_ARG, "agx_gaussian_weights: size out of range");
    AGX_REQUIRE(sigma > 0.0 && isfinite(sigma), AGX_ERR_ARG, "agx_gaussian_weights: sigma must be positive");
    AGX_REQUIRE(norm >= 0 && norm <= AGX_NORM_UNIT_STD, AGX_ERR_ARG, "agx_gaussian_weights: unknown norm code");
    if (n_edges == 0) return AGX_OK;
    AGX_REQUIRE(lengths && out, AGX_ERR_ARG, "agx_gaussian_weights: NULL buffer");
    const double two_s2 = 2.0 * (sigma * sigma);
    const int64_t n = n_edges;
    if (norm == 0) {
        k_gw_apply<<<agx_grid(n, GW_THREADS, 8), GW_THREADS, 0, stream>>>(edge_dst, n, n_dst_nodes, lengths, two_s2, nullptr, out);
        AGX_LAUNCH_OK();
        agx_note_launch(1);
        return AGX_OK;
    }
    AGX_REQUIRE(edge_dst && perm && scratch, AGX_ERR_ARG, "agx_gaussian_weights: a norm needs edge_dst, perm and scratch");
    AGX_REQUIRE(((uintptr_t)scratch & 15) == 0, AGX_ERR_ARG, "agx_gaussian_weights: scratch must be 16-byte aligned");
    // scratch layout (agx_b200.h): table | first | end | warp_list | counters | big | big_stat | partial
    char* p = (char*)scratch;
    double2* table = (double2*)p;
    int32_t* first = (int32_t*)(p + 16 * n_dst_nodes);
    int32_t* end = first + n_dst_nodes;
    int32_t* warp_list = end + n_dst_nodes;
    int32_t* counters = (int32_t*)(p + 32 * n_dst_nodes);
    GwBig* big = (GwBig*)(p + 32 * n_dst_nodes + 64);
    GwStat* big_stat = (GwStat*)(big + gw_max_big(n));
    GwStat* partial = big_stat + gw_max_big(n);
    AGX_CUDA_OK(cudaMemsetAsync(first, 0, 8 * n_dst_nodes, stream));
    AGX_CUDA_OK(cudaMemsetAsync(counters, 0, 64, stream));
    const int cap = agx_sm_count() * 8;
    k_gw_bounds<<<agx_grid(n, GW_THREADS, 8), GW_THREADS, 0, stream>>>(edge_dst, perm, n, n_dst_nodes, first, end);
    k_gw_small<<<agx_grid(n_dst_nodes, GW_THREADS, 8), GW_THREADS, 0, stream>>>(perm, lengths, n_dst_nodes, first, end, two_s2,
                                                                               norm, table, counters, warp_list, big);
    k_gw_warp<<<cap, GW_THREADS, 0, stream>>>(perm, lengths, first, end, two_s2, norm, table, counters, warp_list);
    int launches = 3;
    for (int pass = 1; pass <= (norm == AGX_NORM_UNIT_STD ? 2 : 1); ++pass) {
        k_gw_big_chunks<<<cap, GW_THREADS, 0, stream>>>(perm, lengths, first, end, two_s2, pass, counters, big, big_stat, partial);
        k_gw_big_groups<<<agx_sm_count(), GW_THREADS, 0, stream>>>(first, end, norm, pass, counters, big, big_stat, partial, table);
        launches += 2;
    }
    k_gw_apply<<<agx_grid(n, GW_THREADS, 8), GW_THREADS, 0, stream>>>(edge_dst, n, n_dst_nodes, lengths, two_s2, table, out);
    AGX_LAUNCH_OK();
    agx_note_launch(launches + 1);
    return AGX_OK;
}

extern "C" int64_t agx_gaussian_weights_scratch_bytes(int64_t n_edges, int64_t n_dst_nodes) {
    return 32 * n_dst_nodes + 64 + 16 * gw_max_big(n_edges) + 32 * gw_max_big(n_edges) + 32 * gw_max_chunks(n_edges);
}
