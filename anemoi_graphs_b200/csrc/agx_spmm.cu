// Edge set as an operator: y = M x for the canonical CSR of agx_edges_to_csr (export.EdgeSetOperator, ops.csr_spmm).
//   y[t, f] = sum over the entries j of row t, in CSR order (ascending source), of data[j] * x[indices[j], f]
// One thread owns (row t, V consecutive features) and accumulates acc = fmaf(data[j], x_j, acc) from +0 in float32,
// left to right; bf16 x is widened exactly and the sum rounded once (to nearest even).  No atomics and no sums across
// threads, so the bits depend on nothing but the inputs.
//   k_csr_spmm  a group of G lanes per row (G a power of two <= 32, enough groups of V features to cover F, so that
//               F = 1 puts 32 rows in a warp and F >= 32 V one); the lanes of a group read each (index, value) pair at
//               the same address - one transaction broadcast to the group - four pairs at a time: four gathers of x
//               in flight, then their FMAs in order; the next row's indptr pair is loaded before this row's work.  V is the widest vector (16 B, 8 B or one element) that the
//               alignment of x and out and the row length F allow.  Output rows are written with streaming stores,
//               so that a gathered x that fits the L2 stays there while y streams past it.
// An index outside [0, n_cols) raises a flag instead of being read; one read-back at the end reports it.
#include <cuda_bf16.h>

#include "agx_common.cuh"

#define SPMM_UNROLL 4

// The BYTES bytes at p as 32-bit words (BYTES = 2: one 16-bit word in w[0]).
template <int BYTES>
__device__ __forceinline__ void spmm_load(const char* p, uint32_t* w) {
    if constexpr (BYTES == 16) {
        const uint4 r = __ldg((const uint4*)p);
        w[0] = r.x, w[1] = r.y, w[2] = r.z, w[3] = r.w;
    } else if constexpr (BYTES == 8) {
        const uint2 r = __ldg((const uint2*)p);
        w[0] = r.x, w[1] = r.y;
    } else if constexpr (BYTES == 4) {
        w[0] = __ldg((const unsigned int*)p);
    } else {
        w[0] = __ldg((const unsigned short*)p);
    }
}

template <int BYTES>
__device__ __forceinline__ void spmm_store(char* p, const uint32_t* w) {
    if constexpr (BYTES == 16) __stcs((uint4*)p, make_uint4(w[0], w[1], w[2], w[3]));
    else if constexpr (BYTES == 8) __stcs((uint2*)p, make_uint2(w[0], w[1]));
    else if constexpr (BYTES == 4) __stcs((unsigned int*)p, w[0]);
    else __stcs((unsigned short*)p, (unsigned short)w[0]);
}

// Element q of the V loaded elements as float32 (bf16: the 16 bits are the top half of the float32, exactly).
template <bool BF16, int V>
__device__ __forceinline__ float spmm_elem(const uint32_t* w, int q) {
    if constexpr (!BF16) return __uint_as_float(w[q]);
    else if constexpr (V == 1) return __uint_as_float(w[0] << 16);
    else return __uint_as_float((q & 1) ? (w[q >> 1] & 0xffff0000u) : (w[q >> 1] << 16));
}

template <bool BF16, int V>
__device__ __forceinline__ void spmm_pack(const float* acc, uint32_t* w) {
    if constexpr (!BF16) {
#pragma unroll
        for (int q = 0; q < V; ++q) w[q] = __float_as_uint(acc[q]);
    } else if constexpr (V == 1) {
        w[0] = __bfloat16_as_ushort(__float2bfloat16_rn(acc[0]));
    } else {
#pragma unroll
        for (int q = 0; q < V; q += 2)
            w[q >> 1] = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(acc[q])) |
                        ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(acc[q + 1])) << 16);
    }
}

// n_vec = F / V vectors per row of x and of out; row t's vector k is at byte (t * n_vec + k) * V * elem.
template <bool BF16, int V>
__global__ void __launch_bounds__(256) k_csr_spmm(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                                                  const float* __restrict__ data, int64_t n_rows, int64_t n_cols,
                                                  const char* __restrict__ x, int64_t n_vec, char* __restrict__ out,
                                                  int log_g, int* __restrict__ bad) {
    constexpr int BYTES = V * (BF16 ? 2 : 4);
    constexpr int WORDS = BYTES >= 4 ? BYTES / 4 : 1;
    const int g = 1 << log_g;
    const int sub = threadIdx.x & (g - 1);
    const int64_t row_bytes = n_vec * BYTES;
    const int64_t step = ((int64_t)gridDim.x * blockDim.x) >> log_g;
    int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> log_g;
    int64_t next_b = 0, next_e = 0;
    if (row < n_rows) next_b = indptr[row], next_e = indptr[row + 1];
    for (; row < n_rows; row += step) {
        const int64_t b = next_b, e = next_e;
        {  // the next row's pair, loaded before this row's work: one level off the chain of dependent loads
            const int64_t ahead = row + step < n_rows ? row + step : row;
            next_b = indptr[ahead], next_e = indptr[ahead + 1];
        }
        for (int64_t k = sub; k < n_vec; k += g) {
            const char* xk = x + k * BYTES;
            float acc[V];
#pragma unroll
            for (int q = 0; q < V; ++q) acc[q] = 0.0f;
            for (int64_t j = b; j < e; j += SPMM_UNROLL) {
                float wt[SPMM_UNROLL];
                bool ok[SPMM_UNROLL];
                uint32_t xw[SPMM_UNROLL][WORDS];
#pragma unroll
                for (int u = 0; u < SPMM_UNROLL; ++u) {
                    ok[u] = j + u < e;
                    const int32_t c = ok[u] ? __ldg(indices + j + u) : 0;
                    wt[u] = ok[u] ? __ldg(data + j + u) : 0.0f;
                    if (ok[u] && (int64_t)(uint32_t)c >= n_cols) {  // negative entries are >= 2^31 here
                        *bad = 1;
                        ok[u] = false;
                    }
                    if (ok[u]) spmm_load<BYTES>(xk + (int64_t)c * row_bytes, xw[u]);
                }
#pragma unroll
                for (int u = 0; u < SPMM_UNROLL; ++u) {
                    if (ok[u]) {
#pragma unroll
                        for (int q = 0; q < V; ++q) acc[q] = fmaf(wt[u], spmm_elem<BF16, V>(xw[u], q), acc[q]);
                    }
                }
            }
            uint32_t ow[WORDS];
            spmm_pack<BF16, V>(acc, ow);
            spmm_store<BYTES>(out + row * row_bytes + k * BYTES, ow);
        }
    }
}

template <bool BF16, int V>
static void launch_spmm(const int64_t* indptr, const int32_t* indices, const float* data, int64_t n_rows, int64_t n_cols,
                        const void* x, int64_t n_features, void* out, int* bad, cudaStream_t stream) {
    const int64_t n_vec = n_features / V;
    int log_g = 0;
    while (log_g < 5 && (1ll << log_g) < n_vec) ++log_g;
    static int resident = 0;  // blocks per SM at this kernel's register count: the grid fills the GPU in one wave
    if (resident == 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, k_csr_spmm<BF16, V>, 256, 0) != cudaSuccess)
        resident = 4;
    const int grid = agx_grid(n_rows << log_g, 256, resident > 0 ? resident : 1);
    k_csr_spmm<BF16, V><<<grid, 256, 0, stream>>>(indptr, indices, data, n_rows, n_cols, (const char*)x, n_vec, (char*)out,
                                                   log_g, bad);
}

extern "C" int agx_csr_spmm(const int64_t* indptr, const int32_t* indices, const float* data, int64_t n_rows, int64_t n_cols,
                            const void* x, int64_t n_features, int dtype, void* out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(dtype == AGX_SPMM_FLOAT32 || dtype == AGX_SPMM_BFLOAT16, AGX_ERR_ARG,
                "agx_csr_spmm: dtype %d is not %d (float32) or %d (bfloat16)", dtype, AGX_SPMM_FLOAT32, AGX_SPMM_BFLOAT16);
    AGX_REQUIRE(n_rows >= 0 && n_cols >= 0 && n_features >= 0, AGX_ERR_ARG,
                "agx_csr_spmm: negative size (n_rows = %lld, n_cols = %lld, n_features = %lld)", (long long)n_rows,
                (long long)n_cols, (long long)n_features);
    AGX_REQUIRE(n_cols <= 2147483647ll, AGX_ERR_ARG, "agx_csr_spmm: n_cols = %lld does not fit the int32 indices",
                (long long)n_cols);
    AGX_REQUIRE(indptr && indices && data && x && out, AGX_ERR_ARG, "agx_csr_spmm: NULL buffer");
    const int elem = dtype == AGX_SPMM_BFLOAT16 ? 2 : 4;
    const uintptr_t addr = (uintptr_t)x | (uintptr_t)out;
    AGX_REQUIRE(addr % elem == 0, AGX_ERR_ARG, "agx_csr_spmm: x or out is not aligned to its %d-byte elements", elem);
    if (n_rows == 0 || n_features == 0) return AGX_OK;
    const int64_t row_bytes = n_features * elem;
    const int vec_bytes = (row_bytes % 16 == 0 && addr % 16 == 0) ? 16 : (row_bytes % 8 == 0 && addr % 8 == 0) ? 8 : elem;
    int* bad = nullptr;
    int rc = agx_bad_flag_alloc(&bad, stream);
    if (rc) return rc;
    if (dtype == AGX_SPMM_FLOAT32) {
        if (vec_bytes == 16) launch_spmm<false, 4>(indptr, indices, data, n_rows, n_cols, x, n_features, out, bad, stream);
        else if (vec_bytes == 8) launch_spmm<false, 2>(indptr, indices, data, n_rows, n_cols, x, n_features, out, bad, stream);
        else launch_spmm<false, 1>(indptr, indices, data, n_rows, n_cols, x, n_features, out, bad, stream);
    } else {
        if (vec_bytes == 16) launch_spmm<true, 8>(indptr, indices, data, n_rows, n_cols, x, n_features, out, bad, stream);
        else if (vec_bytes == 8) launch_spmm<true, 4>(indptr, indices, data, n_rows, n_cols, x, n_features, out, bad, stream);
        else launch_spmm<true, 1>(indptr, indices, data, n_rows, n_cols, x, n_features, out, bad, stream);
    }
    agx_note_launch(1);
    if (cudaGetLastError() != cudaSuccess) {
        cudaFreeAsync(bad, stream);
        agx_set_error("agx_csr_spmm: kernel launch failed");
        return AGX_ERR_CUDA;
    }
    char msg[128];
    snprintf(msg, sizeof msg, "agx_csr_spmm: an index is outside [0, n_cols = %lld)", (long long)n_cols);
    return agx_bad_flag_read(bad, msg, nullptr, stream);
}
