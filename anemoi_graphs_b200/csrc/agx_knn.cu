// K2: k-nearest-neighbour search over the cell-binned index.
//
// Replaces sklearn's BallTree.query as driven by KNNEdges.get_adjacency_matrix
// (/root/reference/src/anemoi/graphs/edges/builder.py:259-265), utils.get_grid_reference_distance
// (utils.py:62) and KNNAreaMaskBuilder.get_mask (generate/masks.py:97).
//
// Main path - one WARP per tile of 32 consecutive queries (grids store neighbouring points next to
// each other, so a tile's search caps overlap almost completely):
//   1. every lane turns its query into a unit vector and a per-face cell window for the first search cap;
//      the warp takes the union window per cube face (REDUX min / max);
//   2. each window row is ONE contiguous run of 16-byte records in the cell-sorted array; one lane per row
//      issues a 1-D bulk async copy (TMA, cp.async.bulk -> UBLKCP) of the run into the warp's shared-memory
//      stage, completion tracked by an mbarrier (expect_tx / complete_tx);
//   3. every lane scans the staged candidates with broadcast LDS.128: squared chord on the FP32 FMA pipe,
//      top-(k+1) kept in registers as ONE 32-bit key per entry - the float bits of chord^2 with the low 9 bits
//      replaced by the candidate's stage position - so an insertion is a min/max network (2 integer ops per
//      entry, no compares, no selects).  The 2^-14 relative truncation is added to the ambiguity band; exact
//      FP32 distances and indices of the k+1 survivors are recovered from the stage afterwards;
//   4. a lane whose k-th distance (+ margins) does not fit inside the first cap, and tiles whose window does
//      not fit the stage, fall back to the per-thread search (cap growth until it provably holds the k-th
//      neighbour);
//   5. if the (k+1)-th candidate is within the FP32 error margin of the k-th, the set is decided in float64
//      with the reference's own haversine formula (tie rule: lower index within 2^-40).
// The edge SET is what parity is judged on, so the filter only has to isolate the k members; their float64
// distances are evaluated only on request (out_rdist).
#include <stdlib.h>
#include <string.h>

#include "agx_tile.cuh"

#define KNN_WARPS AGX_TILE_WARPS
#define KNN_STAGE AGX_TILE_STAGE

template <int CAP>
struct TopF {  // ascending d, CAP entries in registers (ties in arbitrary but deterministic scan order)
    float d[CAP];
    int id[CAP];
    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int s = 0; s < CAP; ++s) {
            d[s] = __int_as_float(0x7f800000);
            id[s] = 0x7fffffff;
        }
    }
    // register-resident reads at a runtime position (a dynamic subscript would demote the arrays to local memory)
    __device__ __forceinline__ float d_at(int i) const {
        float r = d[0];
#pragma unroll
        for (int s = 1; s < CAP; ++s) r = (i == s) ? d[s] : r;
        return r;
    }
    __device__ __forceinline__ int id_at(int i) const {
        int r = id[0];
#pragma unroll
        for (int s = 1; s < CAP; ++s) r = (i == s) ? id[s] : r;
        return r;
    }
    // exact FP32 ties at the k / k+1 boundary are always inside the error margin and are re-decided in float64,
    // so the filter does not need an index tie-break
    __device__ __forceinline__ void insert(float cd, int ci) {
#pragma unroll
        for (int s = 0; s < CAP; ++s) {
            bool lt = cd < d[s];
            float td = d[s];
            int ti = id[s];
            d[s] = lt ? cd : td;
            id[s] = lt ? ci : ti;
            cd = lt ? td : cd;
            ci = lt ? ti : ci;
        }
    }
    __device__ __forceinline__ void offer(float cd, int ci) {
        if (cd < d[CAP - 1]) insert(cd, ci);
    }
    // compare-exchange of entries i < j (no-op for positions the list does not have)
    __device__ __forceinline__ void order(int i, int j) {
        if (j >= CAP) return;
        bool sw = d[j] < d[i];
        float td = d[i];
        int ti = id[i];
        d[i] = sw ? d[j] : td;
        id[i] = sw ? id[j] : ti;
        d[j] = sw ? td : d[j];
        id[j] = sw ? ti : id[j];
    }
};

// Packed top list for the staged scan: key = (bits(chord^2) & ~KEY_POS_MASK) | stage position.  chord^2 >= +0 and
// finite, so unsigned integer order is float order; truncation lowers a value by < 2^-14 relative.
#define KEY_POS_BITS 9
#define KEY_POS_MASK ((1u << KEY_POS_BITS) - 1u)
#define KEY_EMPTY 0x7f800000u  // +inf, position 0: above every real key
static_assert(KNN_STAGE <= (1 << KEY_POS_BITS), "stage positions must fit the key's position field");

template <int CAP>
struct TopKey {
    unsigned key[CAP];
    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int s = 0; s < CAP; ++s) key[s] = KEY_EMPTY;
    }
    __device__ __forceinline__ void insert(unsigned c) {
#pragma unroll
        for (int s = 0; s < CAP; ++s) {
            unsigned lo = min(key[s], c);
            c = max(key[s], c);
            key[s] = lo;
        }
    }
    __device__ __forceinline__ void offer(unsigned c) {
        if (CAP <= 4)
            insert(c);  // 2*CAP integer ops: cheaper than a divergent branch around them
        else if (c < key[CAP - 1])
            insert(c);
    }
    __device__ __forceinline__ unsigned key_at(int i) const {
        unsigned r = key[0];
#pragma unroll
        for (int s = 1; s < CAP; ++s) r = (i == s) ? key[s] : r;
        return r;
    }
};

template <int CAP>
struct TopD {  // ascending under agx_tie_less
    double r[CAP];
    int id[CAP];
    __device__ __forceinline__ void reset() {
#pragma unroll
        for (int s = 0; s < CAP; ++s) {
            r[s] = 1e300;
            id[s] = 0x7fffffff;
        }
    }
    __device__ __forceinline__ double r_at(int i) const {
        double v = r[0];
#pragma unroll
        for (int s = 1; s < CAP; ++s) v = (i == s) ? r[s] : v;
        return v;
    }
    __device__ __forceinline__ int id_at(int i) const {
        int v = id[0];
#pragma unroll
        for (int s = 1; s < CAP; ++s) v = (i == s) ? id[s] : v;
        return v;
    }
    __device__ __forceinline__ void insert(double cr, int ci) {
#pragma unroll
        for (int s = 0; s < CAP; ++s) {
            bool lt = agx_tie_less(cr, ci, r[s], id[s]);
            double tr = r[s];
            int ti = id[s];
            r[s] = lt ? cr : tr;
            id[s] = lt ? ci : ti;
            cr = lt ? tr : cr;
            ci = lt ? ti : ci;
        }
    }
    __device__ __forceinline__ void offer(double cr, int ci) {
        if (agx_tie_less(cr, ci, r[CAP - 1], id[CAP - 1])) insert(cr, ci);
    }
};

struct KnnArgs {
    const float4* pts;
    const int* cell_start;
    const float2* ref_latlon;
    int cells;
    float chord2_init;
    float chord2_limit;  // search limit (max_radius, inflated by the margins), +inf when there is none
    const float2* q_latlon;
    const int32_t* qperm;  // optional processing order of the queries (spatially binned), or NULL
    int64_t nq;
    int k;
    int32_t* out_src;
    int32_t* out_dst;
    int64_t dst_base;
    double* out_rdist;
    unsigned long long* stats;
    uint8_t* tie_flags;  // optional: 1 for every query whose k-th boundary is a tie (the result depends on the index order)
    int only_flagged;    // 1: tie_flags is an INPUT - only queries whose flag is set are searched and written
    const int32_t* tile_list;  // only_flagged: the tiles (of 32 consecutive queries) that hold a flagged query ...
    const int* tile_count;     // ... and how many there are (device memory: no read-back)
    // Re-decision against an index whose points still carry PROVISIONAL labels: ties go to the lower FINAL label
    // tie_rank[label]; what is written is again the provisional label tie_order[final label] (the caller relabels
    // the whole row afterwards).  Both NULL: the index labels are final.
    const int64_t* tie_rank;
    const int64_t* tie_order;
    // output label maps (NodeMaskingMixin.undo_masking fused into the write): what is stored is src_map[reference index]
    // / dst_map[query index] instead of the index / dst_base + query (NULL: identity)
    const int64_t* src_map;
    const int64_t* dst_map;
};

// the label the tie rule compares: the final position of a provisionally labelled point
__device__ __forceinline__ int knn_tie_label(const KnnArgs& a, int ci) { return a.tie_rank ? (int)a.tie_rank[ci] : ci; }
__device__ __forceinline__ int knn_out_label(const KnnArgs& a, int id) {
    if (a.tie_order) id = (int)a.tie_order[id];
    return (a.src_map && id >= 0) ? (int)a.src_map[id] : id;
}
__device__ __forceinline__ int knn_dst_label(const KnnArgs& a, int64_t q) {
    return a.dst_map ? (int)a.dst_map[q] : (int32_t)(a.dst_base + q);
}

// the tiles that hold at least one flagged query, appended in arbitrary order (the results do not depend on it)
__global__ void __launch_bounds__(256) k_flagged_tiles(const uint8_t* __restrict__ flags, int64_t nq, int64_t n_tiles,
                                                       int32_t* __restrict__ tile_list, int* __restrict__ tile_count) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_tiles; t += (int64_t)gridDim.x * blockDim.x) {
        bool any = false;
        if (t * 32 + 32 <= nq) {
            const uint4* w = (const uint4*)(flags + t * 32);  // 16-byte aligned: base checked by the entry points, t * 32
            uint4 a = w[0], b = w[1];
            any = (a.x | a.y | a.z | a.w | b.x | b.y | b.z | b.w) != 0u;
        } else {
            for (int64_t q = t * 32; q < nq; ++q) any |= flags[q] != 0;
        }
        if (any) tile_list[atomicAdd(tile_count, 1)] = (int32_t)t;
    }
}

__device__ __forceinline__ float chord2(float3 q, float4 c) {
    float dx = q.x - c.x, dy = q.y - c.y, dz = q.z - c.z;
    return fmaf(dx, dx, fmaf(dy, dy, dz * dz));
}

// true if k candidates within FP32 chord^2 dk prove that the cap of squared chord t2 contains the k nearest
// neighbours (dk = +inf: fewer than k candidates found)
__device__ __forceinline__ bool knn_cap_sufficient(float dk, float t2, float& need) {
    need = dk + 3.75f * agx_chord2_margin(dk);  // d_k + 3 margins (margin taken 1.25x)
    return dk < __int_as_float(0x7f800000) && need <= t2;
}

// Per-thread search straight from global memory: grow the cap until it provably holds the k-th neighbour - or until
// it reaches the caller's search limit (returns true: the list holds what lies inside the limit and nothing is
// proven about the rest).
template <int CAP>
__device__ __forceinline__ bool knn_thread_search(const KnnArgs& a, float3 qv, float t2, TopF<CAP>& top, AgxCap& cap) {
    while (true) {
        top.reset();
        cap = agx_make_cap(t2);
        for (int face = 0; face < 6; ++face) {
            int i0, i1, j0, j1;
            if (!agx_face_window(face, qv, cap, a.cells, i0, i1, j0, j1)) continue;
            for (int i = i0; i <= i1; ++i) {
                int row = (face * a.cells + i) * a.cells;
                int s = __ldg(a.cell_start + row + j0), e = __ldg(a.cell_start + row + j1 + 1);
                for (int p = s; p < e; ++p) {
                    float4 c = __ldg(a.pts + p);
                    top.offer(chord2(qv, c), __float_as_int(c.w));
                }
            }
        }
        if (cap.everything) return false;
        float need;
        float dk = top.d_at(a.k - 1);
        if (knn_cap_sufficient(dk, t2, need)) return false;
        if (t2 >= a.chord2_limit) return true;
        bool have_k = dk < __int_as_float(0x7f800000);
        t2 = fminf(have_k ? fmaxf(need * 1.0001f, t2 * 1.5f) : t2 * 4.0f, a.chord2_limit);
    }
}

// float64 re-decision over every candidate the filter could not separate (d <= amb), candidates from global memory
template <int CAP>
__device__ __forceinline__ void knn_redecide_global(const KnnArgs& a, float2 ql, float3 qv, const AgxCap& cap, float amb,
                                                 TopD<CAP>& fin) {
    for (int face = 0; face < 6; ++face) {
        int i0, i1, j0, j1;
        if (!agx_face_window(face, qv, cap, a.cells, i0, i1, j0, j1)) continue;
        for (int i = i0; i <= i1; ++i) {
            int row = (face * a.cells + i) * a.cells;
            int s = __ldg(a.cell_start + row + j0), e = __ldg(a.cell_start + row + j1 + 1);
            for (int p = s; p < e; ++p) {
                float4 c = __ldg(a.pts + p);
                if (chord2(qv, c) <= amb) {
                    int ci = __float_as_int(c.w);
                    fin.offer(agx_rdist64(ql, a.ref_latlon[ci]), knn_tie_label(a, ci));
                }
            }
        }
    }
}

// ... candidates from the warp's shared-memory stage (a superset of the lane's cap)
template <int CAP>
__device__ __forceinline__ void knn_redecide_stage(const KnnArgs& a, float2 ql, float3 qv, const float4* stage, int m,
                                                float amb, TopD<CAP>& fin) {
    for (int p = 0; p < m; ++p) {
        float4 c = stage[p];
        if (chord2(qv, c) <= amb) {
            int ci = __float_as_int(c.w);
            fin.offer(agx_rdist64(ql, a.ref_latlon[ci]), knn_tie_label(a, ci));
        }
    }
}

// CAP >= k + 1.  Entries beyond k + 1 are carried but never read.
template <int CAP>
__global__ void __launch_bounds__(KNN_WARPS * 32) k_knn(KnnArgs a) {
    __shared__ __align__(128) float4 stage_all[KNN_WARPS][KNN_STAGE];
    __shared__ __align__(8) uint64_t bars[KNN_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float4* stage = stage_all[warp];
    uint64_t* bar = &bars[warp];
    if (lane == 0) mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    uint32_t phase = 0;
    const int k = a.k;
    const int64_t n_tiles = (a.nq + 31) >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * KNN_WARPS;
    const int64_t n_work = a.only_flagged ? (int64_t)*a.tile_count : n_tiles;
    for (int64_t work = (int64_t)blockIdx.x * KNN_WARPS + warp; work < n_work; work += warps_total) {
        const int64_t tile = a.only_flagged ? (int64_t)a.tile_list[work] : work;
        const int64_t slot = tile * 32 + lane;
        bool active = slot < a.nq;
        const int64_t qs = active ? slot : a.nq - 1;
        const int64_t q = a.qperm ? (int64_t)__ldg(a.qperm + qs) : qs;  // binned order, results at the query's own place
        if (a.only_flagged) active = active && a.tie_flags[q] != 0;  // re-decision pass: the other lanes only help
        const float2 ql = a.q_latlon[q];
        const float3 qv = agx_search_xyz(ql);
        const float t2 = a.chord2_init;
        AgxCap cap = agx_make_cap(t2);
        // ---- union window of the tile, one window row per lane ---------------------------------------
        int s = 0, cnt = 0, incl = 0, m_total = 0;
        bool fits = agx_tile_plan(a.cell_start, a.cells, qv, cap, lane, s, cnt, incl, m_total);
        if (fits) {
            if (m_total > 0) {
                // previous tile's generic-proxy reads of the stage are complete (program order + __syncwarp below);
                // order them before the async-proxy writes of this tile
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)m_total * 16u);
                if (cnt > 0) bulk_copy_g2s(stage + (incl - cnt), a.pts + s, (uint32_t)cnt * 16u, bar);
                mbar_wait(bar, phase);
                phase ^= 1;
            }
            if (a.stats && lane == 0) atomicAdd(a.stats + 3, (unsigned long long)m_total * 32ull);  // (query, candidate) pairs
        }
        // ---- scan ------------------------------------------------------------------------------------
        TopF<CAP> top;
        bool staged = fits;
        bool limited = false;
        float t2_thread = t2;
        float dk = __int_as_float(0x7f800000);       // largest FP32 chord^2 among the k chosen candidates
        float rest_lb = __int_as_float(0x7f800000);  // lower bound of the FP32 chord^2 of every other candidate
        if (fits) {
            TopKey<CAP> tk;
            tk.reset();
#pragma unroll 4
            for (int p = 0; p < m_total; ++p) {
                float4 c = stage[p];
                tk.offer((__float_as_uint(chord2(qv, c)) & ~KEY_POS_MASK) | (unsigned)p);
            }
            // exact FP32 distance and index of the k survivors, from the stage
            top.reset();
            float dmax = 0.0f;
#pragma unroll
            for (int s = 0; s < CAP - 1; ++s)
                if (s < k) {
                    unsigned key = tk.key[s];
                    if (key < KEY_EMPTY) {
                        float4 c = stage[key & KEY_POS_MASK];
                        top.d[s] = chord2(qv, c);
                        top.id[s] = __float_as_int(c.w);
                    }
                    dmax = fmaxf(dmax, top.d[s]);
                }
            dk = dmax;
            rest_lb = __uint_as_float(tk.key_at(k) & ~KEY_POS_MASK);
            if (CAP <= 4) {  // ascending exact FP32 distance among the chosen (keys order them only to 2^-14)
                top.order(0, 1);
                top.order(1, 2);
                top.order(0, 1);
            }
            float need;
            if (!knn_cap_sufficient(dk, t2, need)) {
                if (t2 >= a.chord2_limit) {
                    limited = true;  // the tile's cap already is the search limit
                } else {
                    // this lane needs a wider cap than the tile staged: finish it on its own
                    t2_thread = dk < __int_as_float(0x7f800000) ? fmaxf(need * 1.0001f, t2 * 1.5f) : t2 * 4.0f;
                    t2_thread = fminf(t2_thread, a.chord2_limit);
                    staged = false;
                    if (a.stats && active) atomicAdd(a.stats + 2, 1ull);
                }
            }
        }
        if (!staged) {
            limited = knn_thread_search<CAP>(a, qv, t2_thread, top, cap);
            dk = top.d_at(k - 1);
            rest_lb = top.d_at(k);  // +inf when there is no (k+1)-th candidate
        }
        // ---- decide the set --------------------------------------------------------------------------
        // A `limited` lane found fewer than k provable neighbours inside the search limit: it reports what it found
        // there, every point within max_radius among them, and -1 / +inf for the missing slots (see agx_b200.h).
        float amb = dk + 2.5f * agx_chord2_margin(dk);  // d_k + 2 margins
        bool ambiguous = !limited && (CAP > 1) && (rest_lb <= amb);
        if (active) {
            int32_t* os = a.out_src + q * k;
            if (!ambiguous) {
                if (a.out_rdist == nullptr) {
#pragma unroll
                    for (int s = 0; s < CAP - 1; ++s)
                        if (s < k) os[s] = top.id[s] != 0x7fffffff ? knn_out_label(a, top.id[s]) : -1;
                } else {  // ascending (rdist, index), the missing slots last
                    TopD<CAP> fin;
                    fin.reset();
#pragma unroll
                    for (int s = 0; s < CAP - 1; ++s)
                        if (s < k && top.id[s] != 0x7fffffff) fin.insert(agx_rdist64(ql, a.ref_latlon[top.id[s]]), top.id[s]);
#pragma unroll
                    for (int s = 0; s < CAP - 1; ++s)
                        if (s < k) {
                            bool have = fin.id[s] != 0x7fffffff;
                            os[s] = have ? knn_out_label(a, fin.id[s]) : -1;
                            a.out_rdist[q * k + s] = have ? fin.r[s] : __longlong_as_double(0x7ff0000000000000ll);
                        }
                }
            } else {
                TopD<CAP> fin;
                fin.reset();
                if (staged)
                    knn_redecide_stage<CAP>(a, ql, qv, stage, m_total, amb, fin);
                else
                    knn_redecide_global<CAP>(a, ql, qv, cap, amb, fin);
#pragma unroll
                for (int s = 0; s < CAP - 1; ++s)
                    if (s < k) {
                        os[s] = knn_out_label(a, fin.id[s]);
                        if (a.out_rdist) a.out_rdist[q * k + s] = fin.r[s];
                    }
                if (a.stats || a.tie_flags) {
                    double rk = fin.r_at(k - 1), rn = fin.r_at(k);
                    bool tie = fin.id_at(k) != 0x7fffffff && fabs(rn - rk) <= AGX_TIE_TAU * fmax(rn, rk);
                    if (a.stats) {
                        atomicAdd(a.stats + 0, 1ull);
                        if (tie) atomicAdd(a.stats + 1, 1ull);
                    }
                    if (a.tie_flags && tie && !a.only_flagged) a.tie_flags[q] = 1;
                }
            }
            if (a.out_dst) {
                int32_t* od = a.out_dst + q * k;
                int32_t t = knn_dst_label(a, q);
                for (int s = 0; s < k; ++s) od[s] = t;
            }
        }
        __syncwarp();  // every lane is done with the stage before the next tile overwrites it
    }
}


// Re-decision of an explicit LIST of queries (ascending query ids, count in device memory): one thread per listed
// query searches the index from global memory and decides the set in float64 under the (ranked) tie rule.  A handful
// of queries: no staging, no tile plan, no read-back.
template <int CAP>
__global__ void __launch_bounds__(128) k_knn_redecide_list(KnnArgs a, const int32_t* __restrict__ list,
                                                           const int64_t* __restrict__ count) {
    const int k = a.k;
    const int64_t n = *count;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n; w += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = list[w];
        const float2 ql = a.q_latlon[q];
        const float3 qv = agx_search_xyz(ql);
        TopF<CAP> top;
        AgxCap cap;
        if (knn_thread_search<CAP>(a, qv, a.chord2_init, top, cap)) continue;  // beyond the search limit: left as it is
        const float dk = top.d_at(k - 1);
        const float amb = dk + 2.5f * agx_chord2_margin(dk);
        TopD<CAP> fin;
        fin.reset();
        knn_redecide_global<CAP>(a, ql, qv, cap, amb, fin);
        int32_t* os = a.out_src + q * k;
#pragma unroll
        for (int s = 0; s < CAP - 1; ++s)
            if (s < k) os[s] = knn_out_label(a, fin.id[s]);
    }
}

extern "C" int agx_knn_redecide_list(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius,
                                     int32_t* out_src, const int32_t* list, const int64_t* count, const int64_t* rank,
                                     const int64_t* order, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(ix != nullptr, AGX_ERR_ARG, "agx_knn_redecide_list: NULL index");
    AGX_REQUIRE(k > 0 && (int64_t)k <= ix->n && k <= 64, AGX_ERR_ARG, "agx_knn_redecide_list: k out of range");
    AGX_REQUIRE((rank == nullptr) == (order == nullptr), AGX_ERR_ARG, "agx_knn_redecide_list: give rank and order, or neither");
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(q_latlon && out_src && list && count, AGX_ERR_ARG, "agx_knn_redecide_list: NULL buffer");
    KnnArgs a;
    memset(&a, 0, sizeof(a));
    a.pts = ix->pts;
    a.cell_start = ix->cell_start;
    a.ref_latlon = ix->latlon;
    a.cells = ix->cells;
    double t2 = 6.0 * (double)(k + 1) / (double)ix->n;
    if (t2 > 4.0) t2 = 4.0;
    a.chord2_limit = __builtin_inff();
    if (max_radius > 0.0 && max_radius < 3.141592653589793) {
        double sh = sin(0.5 * max_radius), c2 = 4.0 * sh * sh;
        double lim = c2 + 5.0 * (4.2e-7 * sqrt(c2) + 1.0e-6 * c2 + 1.0e-13);
        a.chord2_limit = (float)(lim * 1.000001);
        if (t2 > lim) t2 = lim;
    }
    a.chord2_init = (float)t2;
    a.q_latlon = (const float2*)q_latlon;
    a.nq = nq;
    a.k = k;
    a.out_src = out_src;
    a.tie_rank = rank;
    a.tie_order = order;
    const int grid = 32;  // a few thousand queries at most; grid-stride over the device-side count
    if (k <= 3)
        k_knn_redecide_list<4><<<grid, 128, 0, stream>>>(a, list, count);
    else if (k <= 7)
        k_knn_redecide_list<8><<<grid, 128, 0, stream>>>(a, list, count);
    else if (k <= 16)
        k_knn_redecide_list<17><<<grid, 128, 0, stream>>>(a, list, count);
    else if (k <= 32)
        k_knn_redecide_list<33><<<grid, 128, 0, stream>>>(a, list, count);
    else
        k_knn_redecide_list<65><<<grid, 128, 0, stream>>>(a, list, count);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

template <int CAP>
static void launch_knn(const KnnArgs& a, cudaStream_t stream) {
    int64_t tiles = (a.nq + 31) / 32;
    int64_t blocks = (tiles + KNN_WARPS - 1) / KNN_WARPS;
    int64_t cap = (int64_t)agx_sm_count() * 16;
    int grid = (int)(blocks < cap ? blocks : cap);
    k_knn<CAP><<<grid, KNN_WARPS * 32, 0, stream>>>(a);
}

int agx_knn_ex(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius, int32_t* out_src,
               int32_t* out_dst, int64_t dst_base, double* out_rdist, int64_t* stats, uint8_t* tie_flags, int only_flagged,
               const int64_t* tie_rank, const int64_t* tie_order, void* stream_);

extern "C" int agx_knn(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius, int32_t* out_src,
                       int32_t* out_dst, int64_t dst_base, double* out_rdist, int64_t* stats, void* stream_) {
    return agx_knn_flagged(ix, q_latlon, nq, k, max_radius, out_src, out_dst, dst_base, out_rdist, stats, nullptr, stream_);
}

extern "C" int agx_knn_flagged(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius,
                               int32_t* out_src, int32_t* out_dst, int64_t dst_base, double* out_rdist, int64_t* stats,
                               uint8_t* tie_flags, void* stream_) {
    return agx_knn_ex(ix, q_latlon, nq, k, max_radius, out_src, out_dst, dst_base, out_rdist, stats, tie_flags, 0, nullptr,
                      nullptr, stream_);
}

extern "C" int agx_knn_redecide(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius,
                                int32_t* out_src, const uint8_t* tie_flags, void* stream_) {
    AGX_REQUIRE(tie_flags != nullptr, AGX_ERR_ARG, "agx_knn_redecide: tie_flags is NULL");
    AGX_REQUIRE(((uintptr_t)tie_flags & 15) == 0, AGX_ERR_ARG, "agx_knn_redecide: tie_flags must be 16-byte aligned");
    return agx_knn_ex(ix, q_latlon, nq, k, max_radius, out_src, nullptr, 0, nullptr, nullptr, (uint8_t*)tie_flags, 1, nullptr,
                      nullptr, stream_);
}

extern "C" int agx_knn_redecide_ranked(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius,
                                       int32_t* out_src, const uint8_t* tie_flags, const int64_t* rank,
                                       const int64_t* order, void* stream_) {
    AGX_REQUIRE(tie_flags != nullptr, AGX_ERR_ARG, "agx_knn_redecide_ranked: tie_flags is NULL");
    AGX_REQUIRE(((uintptr_t)tie_flags & 15) == 0, AGX_ERR_ARG, "agx_knn_redecide_ranked: tie_flags must be 16-byte aligned");
    AGX_REQUIRE(rank != nullptr && order != nullptr, AGX_ERR_ARG, "agx_knn_redecide_ranked: rank / order is NULL");
    return agx_knn_ex(ix, q_latlon, nq, k, max_radius, out_src, nullptr, 0, nullptr, nullptr, (uint8_t*)tie_flags, 1, rank,
                      order, stream_);
}

int agx_knn_ex(const agx_index_t* ix, const float* q_latlon, int64_t nq, int k, double max_radius, int32_t* out_src,
               int32_t* out_dst, int64_t dst_base, double* out_rdist, int64_t* stats, uint8_t* tie_flags, int only_flagged,
               const int64_t* tie_rank, const int64_t* tie_order, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(ix != nullptr, AGX_ERR_ARG, "agx_knn: NULL index");
    AGX_REQUIRE(nq >= 0, AGX_ERR_ARG, "agx_knn: nq < 0");
    AGX_REQUIRE(k > 0, AGX_ERR_ARG, "agx_knn: k must be positive (got %d)", k);
    AGX_REQUIRE(max_radius >= 0.0, AGX_ERR_ARG, "agx_knn: max_radius must be >= 0 (0 = unlimited)");
    // sklearn raises "Expected n_neighbors <= n_samples_fit" (neighbors/_base.py kneighbors)
    AGX_REQUIRE((int64_t)k <= ix->n, AGX_ERR_ARG, "Expected n_neighbors <= n_samples_fit, but n_neighbors = %d, n_samples_fit = %lld",
                k, (long long)ix->n);
    AGX_REQUIRE(k <= 64, AGX_ERR_UNSUPPORTED, "agx_knn: k = %d > 64 is not built yet", k);
    AGX_REQUIRE(dst_base + nq < (int64_t)2147483647, AGX_ERR_ARG, "agx_knn: target index exceeds int32");
    if (nq == 0) return AGX_OK;
    AGX_REQUIRE(q_latlon && out_src, AGX_ERR_ARG, "agx_knn: NULL buffer");
    // first cap: chord^2 = 6 (k+1) / n, i.e. 1.5 (k+1) expected points at mean density - 1.7x the k-th
    // neighbour's squared distance on a triangular mesh (measured on O1280 -> res 7: no query needs widening)
    double cap_scale = 6.0;
    if (const char* env = getenv("AGX_KNN_CAP_SCALE")) cap_scale = atof(env);  // tuning knob
    double t2 = cap_scale * (double)(k + 1) / (double)ix->n;
    if (t2 > 4.0) t2 = 4.0;
    KnnArgs a;
    a.pts = ix->pts;
    a.cell_start = ix->cell_start;
    a.ref_latlon = ix->latlon;
    a.cells = ix->cells;
    // search limit: chord^2 of max_radius plus the four margins the sufficiency test needs, so that every query whose
    // k-th neighbour lies within max_radius is still answered exactly
    a.chord2_limit = __builtin_inff();
    if (max_radius > 0.0 && max_radius < 3.141592653589793) {
        double sh = sin(0.5 * max_radius), c2 = 4.0 * sh * sh;
        double lim = c2 + 5.0 * (4.2e-7 * sqrt(c2) + 1.0e-6 * c2 + 1.0e-13);
        a.chord2_limit = (float)(lim * 1.000001);
        if (t2 > lim) t2 = lim;
    }
    a.chord2_init = (float)t2;
    a.q_latlon = (const float2*)q_latlon;
    a.qperm = nullptr;
    a.nq = nq;
    a.k = k;
    a.out_src = out_src;
    a.out_dst = out_dst;
    a.dst_base = dst_base;
    a.out_rdist = out_rdist;
    a.stats = (unsigned long long*)stats;
    a.tie_flags = tie_flags;
    a.only_flagged = only_flagged;
    a.tie_rank = tie_rank;
    a.tie_order = tie_order;
    agx_output_maps(&a.src_map, &a.dst_map);
    AGX_REQUIRE(!(a.src_map && tie_order), AGX_ERR_ARG, "agx_knn: output maps and a ranked re-decision exclude each other");
    int32_t* perm = nullptr;
    int32_t* tile_list = nullptr;
    a.tile_list = nullptr;
    a.tile_count = nullptr;
    if (only_flagged) {
        // the re-decision pass touches a handful of queries: list the tiles that hold one (no read-back), search those
        const int64_t n_tiles = (nq + 31) / 32;
        agx_pool_keep_warm();
        AGX_CUDA_OK(cudaMallocAsync(&tile_list, (n_tiles + 1) * sizeof(int32_t), stream));
        int* count = (int*)(tile_list + n_tiles);
        AGX_CUDA_OK(cudaMemsetAsync(count, 0, sizeof(int), stream));
        k_flagged_tiles<<<agx_grid(n_tiles, 256, 8), 256, 0, stream>>>(tie_flags, nq, n_tiles, tile_list, count);
        agx_note_launch(1);
        a.tile_list = tile_list;
        a.tile_count = count;
    } else {
        int rc = agx_query_order(ix, a.q_latlon, nq, a.chord2_init, "AGX_KNN_BIN", &perm, stream);
        if (rc != AGX_OK) return rc;
        a.qperm = perm;
    }
    if (k <= 3)
        launch_knn<4>(a, stream);
    else if (k <= 7)
        launch_knn<8>(a, stream);
    else if (k <= 16)
        launch_knn<17>(a, stream);
    else if (k <= 32)
        launch_knn<33>(a, stream);
    else
        launch_knn<65>(a, stream);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    if (perm) AGX_CUDA_OK(cudaFreeAsync(perm, stream));
    if (tile_list) AGX_CUDA_OK(cudaFreeAsync(tile_list, stream));
    return AGX_OK;
}
