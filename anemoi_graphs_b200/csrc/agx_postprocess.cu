// Edge post-processors (processors/post_process.py: RestrictEdgeLength, SortEdgeIndexBySourceNodes /
// SortEdgeIndexByTargetNodes).  Each one ends in the same operation: ONE int32 index list applied to edge_index and
// every per-edge array of an edge set.
//   agx_restrict_flags       one keep byte per edge with CutOffEdges' predicate (agx_radius_params: rdist <= sin^2(r/2)),
//                            the optional per-node masks and the endpoint bounds; agx_compact_flags turns it into the list
//   agx_sort_edges           the stable lexicographic permutation: packed (key, other) 64-bit keys over the bits the node
//                            counts can set (agx_pack_keys / agx_key_passes, shared with agx_concat_edges), CUB radix
//                            SortPairs / SortPairsDescending with the positions as values
//   agx_gather_edge_columns  up to 8 arrays gathered through the list in one launch, rows moved as the widest word the
//                            row size and both pointers are aligned to
#include <cub/device/device_radix_sort.cuh>

#include "agx_common.cuh"

__global__ void __launch_bounds__(256) k_restrict_flags(const int32_t* __restrict__ edge_src, const int32_t* __restrict__ edge_dst,
                                                        int64_t n, const float2* __restrict__ src_ll, int64_t n_src,
                                                        const float2* __restrict__ dst_ll, int64_t n_dst,
                                                        const uint8_t* __restrict__ src_mask, const uint8_t* __restrict__ dst_mask,
                                                        double rdist_thr, uint8_t* __restrict__ keep, int* __restrict__ bad) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t s = edge_src[i], d = edge_dst[i];
        uint8_t k = 1;
        if (s < 0 || s >= n_src || d < 0 || d >= n_dst) {
            *bad = 1;
            k = 0;
        } else if ((src_mask == nullptr || src_mask[s]) && (dst_mask == nullptr || dst_mask[d])) {
            k = agx_rdist64(dst_ll[d], src_ll[s]) <= rdist_thr;  // x1 = target (the query of CutOffEdges), x2 = source
        }
        keep[i] = k;
    }
}

extern "C" int agx_restrict_flags(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, const float* src_latlon,
                                  int64_t n_src_nodes, const float* dst_latlon, int64_t n_dst_nodes, const uint8_t* src_mask,
                                  const uint8_t* dst_mask, double max_radius, uint8_t* keep, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_edges >= 0 && n_src_nodes >= 0 && n_dst_nodes >= 0, AGX_ERR_ARG, "agx_restrict_flags: negative size");
    float c2, m;
    double thr;
    int rc = agx_radius_params(max_radius, &c2, &m, &thr);
    if (rc) return rc;
    if (n_edges == 0) return AGX_OK;
    AGX_REQUIRE(edge_src && edge_dst && keep, AGX_ERR_ARG, "agx_restrict_flags: NULL buffer");
    AGX_REQUIRE((n_src_nodes == 0 || src_latlon) && (n_dst_nodes == 0 || dst_latlon), AGX_ERR_ARG,
                "agx_restrict_flags: NULL coordinates");
    int* bad = nullptr;
    rc = agx_bad_flag_alloc(&bad, stream);
    if (rc) return rc;
    k_restrict_flags<<<agx_grid(n_edges, 256, 8), 256, 0, stream>>>(edge_src, edge_dst, n_edges, (const float2*)src_latlon,
                                                                    n_src_nodes, (const float2*)dst_latlon, n_dst_nodes,
                                                                    src_mask, dst_mask, thr, keep, bad);
    agx_note_launch(1);
    if (cudaGetLastError() != cudaSuccess) {
        cudaFreeAsync(bad, stream);
        agx_set_error("agx_restrict_flags: kernel launch failed");
        return AGX_ERR_CUDA;
    }
    return agx_bad_flag_read(bad, "agx_restrict_flags: an edge endpoint is outside [0, num_nodes) of its node set", nullptr,
                             stream);
}

__global__ void __launch_bounds__(256) k_iota(int32_t* __restrict__ out, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (int32_t)i;
}

extern "C" int agx_sort_edges(const int32_t* key_row, const int32_t* other_row, int64_t n_edges, int64_t n_key_nodes,
                              int64_t n_other_nodes, int descending, int32_t* perm, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_edges >= 0 && n_edges < (int64_t)2147483647, AGX_ERR_ARG, "agx_sort_edges: n_edges out of [0, 2^31)");
    if (n_edges == 0) return AGX_OK;
    AGX_REQUIRE(key_row && other_row && perm, AGX_ERR_ARG, "agx_sort_edges: NULL buffer");
    AGX_REQUIRE(n_key_nodes > 0 && n_other_nodes > 0 && n_key_nodes <= 2147483647ll && n_other_nodes <= 2147483647ll,
                AGX_ERR_ARG, "agx_sort_edges: an edge endpoint is outside [0, num_nodes) of its node set (node counts %lld, %lld)",
                (long long)n_key_nodes, (long long)n_other_nodes);
    const int64_t n = n_edges;
    int* bad = nullptr;
    int rc = agx_bad_flag_alloc(&bad, stream);
    if (rc) return rc;
    unsigned long long* keys = nullptr;  // both key buffers, back to back
    int32_t* vals_alt = nullptr;
    void* temp = nullptr;
    cudaError_t e;
#define SE_TRY(expr)                                                                                       \
    if ((e = (expr)) != cudaSuccess) {                                                                     \
        agx_set_error("%s failed: %s", #expr, cudaGetErrorString(e));                                      \
        cudaFreeAsync(keys, stream); cudaFreeAsync(vals_alt, stream); cudaFreeAsync(temp, stream);         \
        cudaFreeAsync(bad, stream);                                                                        \
        return AGX_ERR_CUDA;                                                                               \
    }
    SE_TRY(cudaMallocAsync(&keys, 2 * n * sizeof(unsigned long long), stream));
    SE_TRY(cudaMallocAsync(&vals_alt, n * sizeof(int32_t), stream));
    k_iota<<<agx_grid(n, 256, 8), 256, 0, stream>>>(perm, n);
    agx_note_launch(1);
    SE_TRY(cudaGetLastError());
    rc = agx_pack_keys(key_row, other_row, n, nullptr, nullptr, 0, n_key_nodes, n_other_nodes, keys, bad, stream);
    if (rc) {
        cudaFreeAsync(keys, stream);
        cudaFreeAsync(vals_alt, stream);
        cudaFreeAsync(bad, stream);
        return rc;
    }
    cub::DoubleBuffer<unsigned long long> kbuf(keys, keys + n);
    cub::DoubleBuffer<int32_t> vbuf(perm, vals_alt);
    const AgxKeyPasses passes = agx_key_passes(n_key_nodes, n_other_nodes);
    size_t temp_bytes = 0;
    SE_TRY(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, kbuf, vbuf, (long long)n, 0, passes.end_bit, stream));
    SE_TRY(cudaMallocAsync(&temp, temp_bytes > 0 ? temp_bytes : 16, stream));
    // both sorts are stable: columns equal in both rows keep their input order
    for (int p = 0; p < passes.count; ++p) {
        if (descending) {
            SE_TRY(cub::DeviceRadixSort::SortPairsDescending(temp, temp_bytes, kbuf, vbuf, (long long)n, passes.begin[p],
                                                             passes.end[p], stream));
        } else {
            SE_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, kbuf, vbuf, (long long)n, passes.begin[p], passes.end[p],
                                                   stream));
        }
    }
    agx_note_launch(2 * passes.count);
    if (vbuf.Current() != perm) SE_TRY(cudaMemcpyAsync(perm, vbuf.Current(), n * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));
#undef SE_TRY
    cudaFreeAsync(keys, stream);
    cudaFreeAsync(vals_alt, stream);
    cudaFreeAsync(temp, stream);
    return agx_bad_flag_read(bad, "agx_sort_edges: an edge endpoint is outside [0, num_nodes) of its node set", nullptr, stream);
}

// ------------------------------------------------------------------------------------------------
// gather: dst[a] row j = src[a] row index[j], for up to GATHER_MAX_ARRAYS arrays.  A block owns GATHER_ROWS
// consecutive output rows: it stages their index entries in shared memory once, then walks the arrays one after
// another, every thread moving one word of one row per step (consecutive threads: consecutive words of the output).
// ------------------------------------------------------------------------------------------------
#define GATHER_MAX_ARRAYS 8
#define GATHER_ROWS 1024
#define GATHER_MAX_ROW_BYTES (1 << 20)  // words per tile (GATHER_ROWS x words per row) stay below 2^31

struct GatherArrays {
    const char* src[GATHER_MAX_ARRAYS];
    char* dst[GATHER_MAX_ARRAYS];
    int word[GATHER_MAX_ARRAYS];           // bytes per word: 16, 8, 4, 2 or 1
    int words_per_row[GATHER_MAX_ARRAYS];  // row bytes / word
    int n;
};

template <typename W>
__device__ __forceinline__ void gather_rows(const char* __restrict__ src_, char* __restrict__ dst_, int wpr,
                                            const int32_t* rows, int64_t base, int cnt) {
    const W* __restrict__ src = reinterpret_cast<const W*>(src_);
    W* __restrict__ dst = reinterpret_cast<W*>(dst_);
    const int words = cnt * wpr;
    if (wpr == 1) {
        for (int u = threadIdx.x; u < words; u += blockDim.x) dst[base + u] = src[rows[u]];
        return;
    }
    for (int u = threadIdx.x; u < words; u += blockDim.x) {
        const int j = u / wpr, k = u - j * wpr;
        dst[(base + j) * wpr + k] = src[(int64_t)rows[j] * wpr + k];
    }
}

__global__ void __launch_bounds__(256) k_gather_columns(GatherArrays g, const int32_t* __restrict__ index, int64_t n) {
    __shared__ int32_t rows[GATHER_ROWS];
    for (int64_t base = (int64_t)blockIdx.x * GATHER_ROWS; base < n; base += (int64_t)gridDim.x * GATHER_ROWS) {
        const int cnt = (int)(n - base < GATHER_ROWS ? n - base : GATHER_ROWS);
        __syncthreads();  // the previous tile is done with `rows`
        for (int t = threadIdx.x; t < cnt; t += blockDim.x) rows[t] = index[base + t];
        __syncthreads();
        for (int a = 0; a < g.n; ++a) {
            const int wpr = g.words_per_row[a];
            switch (g.word[a]) {
                case 16: gather_rows<int4>(g.src[a], g.dst[a], wpr, rows, base, cnt); break;
                case 8: gather_rows<unsigned long long>(g.src[a], g.dst[a], wpr, rows, base, cnt); break;
                case 4: gather_rows<unsigned>(g.src[a], g.dst[a], wpr, rows, base, cnt); break;
                case 2: gather_rows<unsigned short>(g.src[a], g.dst[a], wpr, rows, base, cnt); break;
                default: gather_rows<unsigned char>(g.src[a], g.dst[a], wpr, rows, base, cnt); break;
            }
        }
    }
}

extern "C" int agx_gather_edge_columns(int n_arrays, const void* const* src, void* const* dst, const int64_t* row_bytes,
                                       const int32_t* index, int64_t n_index, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_arrays >= 0 && n_arrays <= GATHER_MAX_ARRAYS, AGX_ERR_ARG, "agx_gather_edge_columns: n_arrays out of [0, 8]");
    AGX_REQUIRE(n_index >= 0, AGX_ERR_ARG, "agx_gather_edge_columns: n_index < 0");
    GatherArrays g;
    g.n = 0;
    for (int a = 0; a < n_arrays; ++a) {
        const int64_t rb = row_bytes[a];
        AGX_REQUIRE(rb >= 0 && rb <= GATHER_MAX_ROW_BYTES, AGX_ERR_ARG,
                    "agx_gather_edge_columns: row bytes of array %d out of [0, 2^20]", a);
        if (rb == 0 || n_index == 0) continue;
        AGX_REQUIRE(src[a] && dst[a], AGX_ERR_ARG, "agx_gather_edge_columns: NULL array %d", a);
        const uintptr_t align = (uintptr_t)src[a] | (uintptr_t)dst[a] | (uintptr_t)rb;
        int w = 16;
        while (w > 1 && (align & (uintptr_t)(w - 1))) w >>= 1;
        g.src[g.n] = (const char*)src[a];
        g.dst[g.n] = (char*)dst[a];
        g.word[g.n] = w;
        g.words_per_row[g.n] = (int)(rb / w);
        g.n++;
    }
    if (g.n == 0) return AGX_OK;
    AGX_REQUIRE(index != nullptr, AGX_ERR_ARG, "agx_gather_edge_columns: index is NULL");
    for (int a = g.n; a < GATHER_MAX_ARRAYS; ++a) {
        g.src[a] = nullptr;
        g.dst[a] = nullptr;
        g.word[a] = 1;
        g.words_per_row[a] = 0;
    }
    const int64_t tiles = (n_index + GATHER_ROWS - 1) / GATHER_ROWS;
    const int64_t cap = (int64_t)agx_sm_count() * 8;
    k_gather_columns<<<(unsigned)(tiles < cap ? tiles : cap), 256, 0, stream>>>(g, index, n_index);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}
