// N1: utils.concat_edges on the device (/root/reference/src/anemoi/graphs/utils.py:66-81: `torch.unique(torch.cat([e1, e2],
// dim=1), dim=1)` - the columns of both lists sorted lexicographically by (source, target), duplicates removed) - without
// materialising the concatenated int64 list and torch.unique's temporaries:
//   k_pack_keys        both (2, E) int32 lists -> ONE array of packed 64-bit keys (source << 32 | target); indices are
//                      non-negative, so unsigned key order = lexicographic column order
//   cub::DeviceRadixSort::SortKeys on a double buffer, only the key bits the node counts can set (plain library sort)
//   k_concat_heads     number of distinct keys per tile of 1024 (a key is a head if it differs from its predecessor)
//   agx_exclusive_scan tile offsets (+ the total, read back: the caller allocates the result)
//   k_concat_fill      heads unpacked straight into the two rows of the result
// The result allocation (sized for na + nb columns) doubles as the sort's alternate buffer, so the scratch besides the
// result is ONE key buffer: 8 bytes per input edge (plus CUB's histograms).
#include <cub/device/device_radix_sort.cuh>

#include "agx_common.cuh"

#define CONCAT_TILE 1024

__global__ void __launch_bounds__(256) k_pack_keys(const int32_t* __restrict__ a_hi, const int32_t* __restrict__ a_lo, int64_t na,
                                                   const int32_t* __restrict__ b_hi, const int32_t* __restrict__ b_lo, int64_t nb,
                                                   int64_t n_hi_nodes, int64_t n_lo_nodes, unsigned long long* __restrict__ keys,
                                                   int* __restrict__ bad) {
    const int64_t n = na + nb;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const bool first = i < na;
        const int64_t j = first ? i : i - na;
        const unsigned s = (unsigned)(first ? a_hi[j] : b_hi[j]), d = (unsigned)(first ? a_lo[j] : b_lo[j]);
        if (bad && ((int64_t)s >= n_hi_nodes || (int64_t)d >= n_lo_nodes)) *bad = 1;  // negative entries are >= 2^31 here
        keys[i] = ((unsigned long long)s << 32) | (unsigned long long)d;
    }
}

int agx_pack_keys(const int32_t* a_hi, const int32_t* a_lo, int64_t na, const int32_t* b_hi, const int32_t* b_lo,
                  int64_t nb, int64_t n_hi_nodes, int64_t n_lo_nodes, unsigned long long* keys, int* bad,
                  cudaStream_t stream) {
    if (na + nb == 0) return AGX_OK;
    k_pack_keys<<<agx_grid(na + nb, 256, 8), 256, 0, stream>>>(a_hi, a_lo, na, b_hi, b_lo, nb, n_hi_nodes, n_lo_nodes,
                                                               keys, bad);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

__device__ __forceinline__ bool concat_is_head(const unsigned long long* __restrict__ keys, int64_t i) {
    return i == 0 || keys[i] != keys[i - 1];
}

__global__ void __launch_bounds__(256) k_concat_heads(const unsigned long long* __restrict__ keys, int64_t n, int32_t* __restrict__ counts) {
    const int64_t base = (int64_t)blockIdx.x * CONCAT_TILE;
    int c = 0;
    for (int t = threadIdx.x; t < CONCAT_TILE; t += 256) {
        const int64_t i = base + t;
        c += (i < n && concat_is_head(keys, i)) ? 1 : 0;
    }
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ int warp_c[8];
    if ((threadIdx.x & 31) == 0) warp_c[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < 8; ++w) t += warp_c[w];
        counts[blockIdx.x] = t;
    }
}

// thread t of a tile owns the 4 consecutive keys [4t, 4t + 4): block-wide exclusive scan of the head counts, then writes
__global__ void __launch_bounds__(256) k_concat_fill(const unsigned long long* __restrict__ keys, int64_t n, const int64_t* __restrict__ offsets,
                                                     int32_t* __restrict__ out_src, int32_t* __restrict__ out_dst) {
    const int64_t i0 = (int64_t)blockIdx.x * CONCAT_TILE + (int64_t)threadIdx.x * 4;
    bool head[4];
    int c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        head[j] = (i0 + j < n) && concat_is_head(keys, i0 + j);
        c += head[j] ? 1 : 0;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __shared__ int warp_tot[8];
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    int64_t pos = offsets[blockIdx.x] + before + incl - c;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (head[j]) {
            const unsigned long long k = keys[i0 + j];
            out_src[pos] = (int32_t)(k >> 32);
            out_dst[pos] = (int32_t)(k & 0xffffffffull);
            ++pos;
        }
}

static int bits_for(int64_t max_value) {
    int b = 1;
    while (b < 32 && ((int64_t)1 << b) <= max_value) ++b;
    return b;
}

AgxKeyPasses agx_key_passes(int64_t n_hi_nodes, int64_t n_lo_nodes) {
    AgxKeyPasses p;
    p.end_bit = 32 + bits_for(n_hi_nodes - 1);
    const int lo_bits = bits_for(n_lo_nodes - 1);
    if ((32 - lo_bits) >= 8) {
        p.count = 2;
        p.begin[0] = 0, p.end[0] = lo_bits;
        p.begin[1] = 32, p.end[1] = p.end_bit;
    } else {
        p.count = 1;
        p.begin[0] = 0, p.end[0] = p.end_bit;
    }
    return p;
}

// `out` is the RESULT allocation, sized for the worst case (2 * (na + nb) int32 = as many bytes as one key buffer): it
// doubles as the radix sort's alternate buffer, so the only scratch besides it is ONE key buffer (8 bytes per input
// edge) + CUB's histograms.  On return the first 2 * n_unique int32 of `out` are the result, row-major (2, n_unique).
extern "C" int agx_concat_edges(const int32_t* a_src, const int32_t* a_dst, int64_t na, const int32_t* b_src,
                                const int32_t* b_dst, int64_t nb, int64_t n_src_nodes, int64_t n_dst_nodes, int32_t* out,
                                int64_t* n_unique, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_unique != nullptr, AGX_ERR_ARG, "agx_concat_edges: n_unique is NULL");
    *n_unique = 0;
    AGX_REQUIRE(na >= 0 && nb >= 0, AGX_ERR_ARG, "agx_concat_edges: negative length");
    AGX_REQUIRE(n_src_nodes > 0 && n_dst_nodes > 0 && n_src_nodes <= 2147483647ll && n_dst_nodes <= 2147483647ll, AGX_ERR_ARG,
                "agx_concat_edges: node counts must be in [1, 2^31)");
    const int64_t n = na + nb;
    if (n == 0) return AGX_OK;
    AGX_REQUIRE((na == 0 || (a_src && a_dst)) && (nb == 0 || (b_src && b_dst)) && out, AGX_ERR_ARG, "agx_concat_edges: NULL buffer");
    AGX_REQUIRE(((uintptr_t)out & 7) == 0, AGX_ERR_ARG, "agx_concat_edges: out must be 8-byte aligned");
    agx_pool_keep_warm();
    unsigned long long* keys = nullptr;
    unsigned long long* alt = reinterpret_cast<unsigned long long*>(out);
    void* temp = nullptr;
    int32_t* counts = nullptr;
    int64_t* offsets = nullptr;
    const int64_t n_tiles = (n + CONCAT_TILE - 1) / CONCAT_TILE;
    cudaError_t e;
#define CC_TRY(expr)                                                                                       \
    if ((e = (expr)) != cudaSuccess) {                                                                     \
        agx_set_error("%s failed: %s", #expr, cudaGetErrorString(e));                                      \
        cudaFreeAsync(keys, stream); cudaFreeAsync(temp, stream); cudaFreeAsync(counts, stream);           \
        cudaFreeAsync(offsets, stream);                                                                    \
        return AGX_ERR_CUDA;                                                                               \
    }
    CC_TRY(cudaMallocAsync(&keys, n * sizeof(unsigned long long), stream));
    int rc = agx_pack_keys(a_src, a_dst, na, b_src, b_dst, nb, n_src_nodes, n_dst_nodes, keys, nullptr, stream);
    if (rc) {
        cudaFreeAsync(keys, stream);
        return rc;
    }
    cub::DoubleBuffer<unsigned long long> buf(keys, alt);
    const AgxKeyPasses passes = agx_key_passes(n_src_nodes, n_dst_nodes);
    size_t temp_bytes = 0;
    CC_TRY(cub::DeviceRadixSort::SortKeys(nullptr, temp_bytes, buf, (long long)n, 0, passes.end_bit, stream));
    CC_TRY(cudaMallocAsync(&temp, temp_bytes > 0 ? temp_bytes : 16, stream));
    for (int p = 0; p < passes.count; ++p)
        CC_TRY(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, buf, (long long)n, passes.begin[p], passes.end[p], stream));
    agx_note_launch(2);
    if (buf.Current() != keys)  // the sorted keys must not live in the buffer the result is unpacked into
        CC_TRY(cudaMemcpyAsync(keys, alt, n * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, stream));
    CC_TRY(cudaMallocAsync(&counts, n_tiles * sizeof(int32_t), stream));
    CC_TRY(cudaMallocAsync(&offsets, (n_tiles + 1) * sizeof(int64_t), stream));
    k_concat_heads<<<(unsigned)n_tiles, 256, 0, stream>>>(keys, n, counts);
    agx_note_launch(1);
    rc = agx_exclusive_scan(counts, n_tiles, offsets, n_unique, stream);  // reads the total back (one sync)
    if (rc == AGX_OK) {
        k_concat_fill<<<(unsigned)n_tiles, 256, 0, stream>>>(keys, n, offsets, out, out + *n_unique);
        agx_note_launch(1);
        if (cudaGetLastError() != cudaSuccess) {
            agx_set_error("agx_concat_edges: kernel launch failed");
            rc = AGX_ERR_CUDA;
        }
    }
#undef CC_TRY
    cudaFreeAsync(keys, stream);
    cudaFreeAsync(temp, stream);
    cudaFreeAsync(counts, stream);
    cudaFreeAsync(offsets, stream);
    return rc;
}
