// Edge set -> CSR sparse matrix (export.edge_set_to_sparse, `python -m anemoi_graphs_b200 export_to_sparse`).  Rows are
// targets, columns sources: M[dst, src] is the sum of the values of the columns (src, dst), in column order.
//   agx_sort_edges(key = dst, other = src, ascending)  the stable (dst, src) order and the endpoint check - by the caller
//   k_csr_heads        one flag byte per sorted position: 1 where a run of equal (dst, src) starts
//   agx_compact_flags  the run starts, ascending; their number stays on the device
//   k_csr_fill         one thread per run: its source (indices), its target (row scratch), its values summed in order
//   k_csr_indptr       one thread per target row r <= n_dst: the first run whose target is >= r (binary search)
// One read-back, at the end: the number of runs (nnz).
#include "agx_common.cuh"

#define CSR_VALUES_ONES 0
#define CSR_VALUES_FLOAT32 1
#define CSR_VALUES_BOOL 2

__device__ __forceinline__ unsigned long long csr_key(const int32_t* __restrict__ src, const int32_t* __restrict__ dst, int32_t p) {
    return ((unsigned long long)(uint32_t)dst[p] << 32) | (uint32_t)src[p];
}

// The loop runs while the warp's first position is inside the list, so every lane takes part in the shuffle; lane 0
// gathers its left neighbour itself.
__global__ void __launch_bounds__(256) k_csr_heads(const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                                                   const int32_t* __restrict__ perm, int64_t n, uint8_t* __restrict__ head) {
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i - lane < n; i += stride) {
        const bool in = i < n;
        const unsigned long long key = in ? csr_key(src, dst, perm[i]) : 0ull;
        unsigned long long prev = __shfl_up_sync(0xffffffffu, key, 1);
        if (in) {
            if (lane == 0 && i > 0) prev = csr_key(src, dst, perm[i - 1]);
            head[i] = (i == 0 || key != prev) ? 1 : 0;
        }
    }
}

// Run j covers sorted positions [starts[j], starts[j + 1]).  float32 is summed left to right from the first value with
// round-to-nearest adds (scipy's csr_sum_duplicates: x = Ax[jj]; x += Ax[jj + 1] ...), bool is OR.
template <int KIND>
__global__ void __launch_bounds__(256) k_csr_fill(const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                                                  const int32_t* __restrict__ perm, int64_t n, const int32_t* __restrict__ starts,
                                                  const int64_t* __restrict__ count, const void* __restrict__ values,
                                                  int32_t* __restrict__ indices, int32_t* __restrict__ rows, void* __restrict__ data) {
    const int64_t m = *count;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = starts[j], e = j + 1 < m ? starts[j + 1] : n;
        const int32_t p = perm[b];
        indices[j] = src[p];
        rows[j] = dst[p];
        if (KIND == CSR_VALUES_BOOL) {
            const uint8_t* v = (const uint8_t*)values;
            uint8_t s = v[p] != 0;
            for (int64_t k = b + 1; k < e; ++k) s |= v[perm[k]] != 0;
            ((uint8_t*)data)[j] = s;
        } else {
            const float* v = (const float*)values;
            float s = KIND == CSR_VALUES_ONES ? 1.0f : v[p];
            for (int64_t k = b + 1; k < e; ++k) s = __fadd_rn(s, KIND == CSR_VALUES_ONES ? 1.0f : v[perm[k]]);
            ((float*)data)[j] = s;
        }
    }
}

__global__ void __launch_bounds__(256) k_csr_indptr(const int32_t* __restrict__ rows, const int64_t* __restrict__ count,
                                                    int64_t n_rows, int64_t* __restrict__ indptr) {
    const int64_t m = *count;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r <= n_rows; r += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = m;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (rows[mid] < r) lo = mid + 1;
            else hi = mid;
        }
        indptr[r] = lo;
    }
}

extern "C" int agx_edges_to_csr(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, int64_t n_dst_nodes,
                                const int32_t* perm, const void* values, int value_kind, int64_t* indptr, int32_t* indices,
                                void* data, int64_t* nnz, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_edges >= 0 && n_edges < 2147483648ll, AGX_ERR_ARG, "agx_edges_to_csr: n_edges = %lld out of [0, 2^31)",
                (long long)n_edges);
    AGX_REQUIRE(n_dst_nodes >= 0 && n_dst_nodes <= 2147483647ll, AGX_ERR_ARG,
                "agx_edges_to_csr: n_dst_nodes = %lld out of [0, 2^31)", (long long)n_dst_nodes);
    AGX_REQUIRE(value_kind >= CSR_VALUES_ONES && value_kind <= CSR_VALUES_BOOL, AGX_ERR_ARG,
                "agx_edges_to_csr: value_kind %d is not 0 (ones), 1 (float32) or 2 (bool)", value_kind);
    AGX_REQUIRE(indptr && nnz, AGX_ERR_ARG, "agx_edges_to_csr: NULL indptr or nnz");
    if (n_edges == 0) {
        AGX_CUDA_OK(cudaMemsetAsync(indptr, 0, (n_dst_nodes + 1) * sizeof(int64_t), stream));
        *nnz = 0;
        return AGX_OK;
    }
    AGX_REQUIRE(edge_src && edge_dst && perm && indices && data && (value_kind == CSR_VALUES_ONES || values), AGX_ERR_ARG,
                "agx_edges_to_csr: NULL buffer");
    AGX_REQUIRE(n_dst_nodes > 0, AGX_ERR_ARG, "agx_edges_to_csr: edges into an empty target node set");
    const int64_t n = n_edges;
    // scratch, one allocation: the run count, the run starts, the run targets, the head flags (4-byte aligned)
    char* scratch = nullptr;
    agx_pool_keep_warm();
    AGX_CUDA_OK(cudaMallocAsync(&scratch, 8 + 9 * n, stream));
    int64_t* count = (int64_t*)scratch;
    int32_t* starts = (int32_t*)(scratch + 8);
    int32_t* rows = starts + n;
    uint8_t* head = (uint8_t*)(rows + n);
    const int grid = agx_grid(n, 256, 8);
    int rc = AGX_OK;
    k_csr_heads<<<grid, 256, 0, stream>>>(edge_src, edge_dst, perm, n, head);
    agx_note_launch(1);
    if (cudaGetLastError() != cudaSuccess) {
        agx_set_error("agx_edges_to_csr: kernel launch failed");
        rc = AGX_ERR_CUDA;
    }
    if (rc == AGX_OK) rc = agx_compact_flags(head, n, starts, count, stream);
    if (rc == AGX_OK) {
        if (value_kind == CSR_VALUES_ONES)
            k_csr_fill<CSR_VALUES_ONES><<<grid, 256, 0, stream>>>(edge_src, edge_dst, perm, n, starts, count, values, indices, rows, data);
        else if (value_kind == CSR_VALUES_FLOAT32)
            k_csr_fill<CSR_VALUES_FLOAT32><<<grid, 256, 0, stream>>>(edge_src, edge_dst, perm, n, starts, count, values, indices, rows, data);
        else
            k_csr_fill<CSR_VALUES_BOOL><<<grid, 256, 0, stream>>>(edge_src, edge_dst, perm, n, starts, count, values, indices, rows, data);
        k_csr_indptr<<<agx_grid(n_dst_nodes + 1, 256, 8), 256, 0, stream>>>(rows, count, n_dst_nodes, indptr);
        agx_note_launch(2);
        if (cudaGetLastError() != cudaSuccess) {
            agx_set_error("agx_edges_to_csr: kernel launch failed");
            rc = AGX_ERR_CUDA;
        }
    }
    if (rc == AGX_OK) rc = agx_readback(nnz, count, 1, stream);
    cudaFreeAsync(scratch, stream);
    return rc;
}
