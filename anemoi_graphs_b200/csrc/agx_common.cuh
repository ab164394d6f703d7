// Shared device/host helpers for the agx_b200 kernels (sm_100a only).
//
// Coordinate conventions follow the reference: node coordinates are float32 (lat, lon) in radians
// (/root/reference/src/anemoi/graphs/nodes/builders/base.py:54,84-101).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/agx_b200.h"

// ------------------------------------------------------------------------------------------------
// error plumbing: every entry point returns 0 or a negative code, message in a thread-local buffer
// ------------------------------------------------------------------------------------------------
void agx_set_error(const char* fmt, ...);
void agx_note_launch(int n);  // bench.py "gpu_launches" accounting
void agx_pool_keep_warm(void);
// copy `words` 8-byte words from device memory to host memory WITHOUT the copy engine, then sync the stream
int agx_readback(void* host_dst, const void* dev_src, int words, cudaStream_t stream);
void agx_output_maps(const int64_t** src_map, const int64_t** dst_map);  // set by agx_set_output_maps (thread-local)
int agx_order_mode(void);         // thread-local override of the query-order decision: -1 auto, 0 as given, 1 binned
void agx_note_order(int binned);  // what the last decision was  // raise the release threshold of the device's cudaMallocAsync pool (once)

#define AGX_CUDA_OK(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            agx_set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,              \
                          cudaGetErrorString(_e));                                          \
            return AGX_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

#define AGX_REQUIRE(cond, code, ...)  \
    do {                              \
        if (!(cond)) {                \
            agx_set_error(__VA_ARGS__); \
            return (code);            \
        }                             \
    } while (0)

#define AGX_LAUNCH_OK()                                                                      \
    do {                                                                                    \
        cudaError_t _e = cudaGetLastError();                                                \
        if (_e != cudaSuccess) {                                                            \
            agx_set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__,          \
                          cudaGetErrorString(_e));                                          \
            return AGX_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

// One pair of ints per call, zeroed: [0] is the flag a kernel raises on bad input, [1] is free for a count a kernel
// leaves on the device.  agx_bad_flag_read reads both back with one synchronisation (the agx_mark_nodes pattern), frees
// them, stores [1] in *second (may be NULL) and returns AGX_ERR_ARG with `msg` if the flag was raised.
static inline int agx_bad_flag_alloc(int** bad, cudaStream_t stream) {
    agx_pool_keep_warm();
    AGX_CUDA_OK(cudaMallocAsync(bad, 2 * sizeof(int), stream));
    AGX_CUDA_OK(cudaMemsetAsync(*bad, 0, 2 * sizeof(int), stream));
    return AGX_OK;
}

static inline int agx_bad_flag_read(int* bad, const char* msg, int* second, cudaStream_t stream) {
    int host2[2] = {0, 0};
    int rc = agx_readback(host2, bad, 1, stream);
    cudaFreeAsync(bad, stream);
    if (rc) return rc;
    if (second) *second = host2[1];
    AGX_REQUIRE(host2[0] == 0, AGX_ERR_ARG, "%s", msg);
    return AGX_OK;
}

// The cut-off test of a radius (radians): a pair is inside iff rdist <= rdist_thr = sin^2(radius / 2) (sklearn
// HaversineDistance64._dist_to_rdist, inclusive).  chord2_thr / margin are the FP32 pre-filter of the searches.  One
// definition for CutOffEdges (agx_radius_*) and RestrictEdgeLength (agx_restrict_flags): the two agree bit for bit.
static inline int agx_radius_params(double radius, float* chord2_thr, float* margin, double* rdist_thr) {
    AGX_REQUIRE(radius >= 0.0, AGX_ERR_ARG, "radius must be non-negative (got %g)", radius);
    double s = sin(0.5 * (radius < 3.141592653589793 ? radius : 3.141592653589793));
    *rdist_thr = s * s;
    double c2 = 4.0 * (*rdist_thr);
    *chord2_thr = (float)c2;
    // same bound as agx_chord2_margin plus the rounding of the threshold itself
    *margin = (float)(4.2e-7 * sqrt(c2) + 1.2e-6 * c2 + 1.0e-13);
    return AGX_OK;
}

// Packed 64-bit sort keys of edge columns, (hi << 32) | lo with non-negative int32 (hi, lo), so that unsigned key order
// is lexicographic (hi, lo) column order (agx_concat.cu; shared by agx_concat_edges and agx_sort_edges).
// agx_pack_keys writes the keys of list a followed by list b; with `bad` (DEV int, zeroed) it also sets *bad = 1 if
// an entry is outside [0, n_hi_nodes) / [0, n_lo_nodes).  agx_key_passes: the radix passes over only the key bits the
// node counts can set - one pass over [0, 32 + hi bits), or, when the lo field leaves >= 8 bits unused, the used lo
// bits then the hi bits (LSD order: stable passes from the least significant field).
int agx_pack_keys(const int32_t* a_hi, const int32_t* a_lo, int64_t na, const int32_t* b_hi, const int32_t* b_lo,
                  int64_t nb, int64_t n_hi_nodes, int64_t n_lo_nodes, unsigned long long* keys, int* bad,
                  cudaStream_t stream);
struct AgxKeyPasses {
    int count;
    int begin[2], end[2];
    int end_bit;  // the widest pass, [0, end_bit): what the CUB temporary storage is sized for
};
AgxKeyPasses agx_key_passes(int64_t n_hi_nodes, int64_t n_lo_nodes);

static inline int agx_sm_count() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

// Grid sized as a multiple of the SM count: `waves` resident CTAs per SM, capped by the work.
static inline int agx_grid(int64_t work_items, int block, int ctas_per_sm) {
    int64_t need = (work_items + block - 1) / block;
    int64_t cap = (int64_t)agx_sm_count() * ctas_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// ------------------------------------------------------------------------------------------------
// the cell-binned index over a reference point set (cube-sphere, equi-angular cells)
// ------------------------------------------------------------------------------------------------
struct agx_index {
    int64_t n;            // reference points
    int cells;            // C: cells per face edge; 6*C*C cells
    int device;
    const float2* latlon; // caller-owned device array (n): float32 (lat, lon), must outlive the index
    float4* pts;          // (n) cell-sorted (x, y, z, __int_as_float(original index)); in-cell order = index
    int* cell_start;      // (6*C*C + 1) offsets into pts
    float chord2_typ;     // typical squared chord between neighbouring points (4*pi/n), for initial radii
    // processing order chosen by agx_radius_count for a query set, kept for the agx_radius_fill that follows
    const void* order_q;  // the query array it belongs to (NULL: none cached)
    int64_t order_nq;
    int32_t* order_perm;  // NULL: as given
};

#define AGX_PI_F 3.14159265358979323846f
#define AGX_QUARTER_PI_F 0.78539816339744830962f

// Face numbering: 0:+x 1:-x 2:+y 3:-y 4:+z 5:-z.  (a, b) are the in-face axes, c the outward normal
// component (c > 0 on the face).
__device__ __forceinline__ void agx_face_frame(int face, float x, float y, float z, float& a, float& b, float& c) {
    switch (face) {
        case 0: a = y; b = z; c = x; break;
        case 1: a = z; b = y; c = -x; break;
        case 2: a = z; b = x; c = y; break;
        case 3: a = x; b = z; c = -y; break;
        case 4: a = x; b = y; c = z; break;
        default: a = y; b = x; c = -z; break;
    }
}

__device__ __forceinline__ int agx_major_face(float x, float y, float z) {
    float ax = fabsf(x), ay = fabsf(y), az = fabsf(z);
    if (ax >= ay && ax >= az) return x >= 0.f ? 0 : 1;
    if (ay >= az) return y >= 0.f ? 2 : 3;
    return z >= 0.f ? 4 : 5;
}

// angle in [-pi/4, pi/4] -> cell coordinate in [0, C)
__device__ __forceinline__ int agx_angle_to_cell(float ang, int cells) {
    int i = (int)floorf((ang + AGX_QUARTER_PI_F) * ((float)cells * (2.0f / AGX_PI_F)));
    return min(max(i, 0), cells - 1);
}

__device__ __forceinline__ int agx_cell_of(float x, float y, float z, int cells) {
    int face = agx_major_face(x, y, z);
    float a, b, c;
    agx_face_frame(face, x, y, z, a, b, c);
    int i = agx_angle_to_cell(atanf(a / c), cells);
    int j = agx_angle_to_cell(atanf(b / c), cells);
    return (face * cells + i) * cells + j;
}

// sin / cos in float64 to <= 1e-11 absolute (Cody-Waite reduction by pi/2 in two parts, Taylor to r^11 / r^12 on
// |r| <= pi/4: truncation 7e-12) - a third of the instructions of the correctly rounded library sincos, and 2^-25
// (the float32 rounding of the result) is all the search needs.
__device__ __forceinline__ void agx_sincos_search(double x, double& s, double& c) {
    double k = rint(x * 0.6366197723675814);
    double r = fma(-k, 1.5707963267948966, x);
    r = fma(-k, 6.123233995736766e-17, r);
    double r2 = r * r;
    double ps = fma(r2, -2.505210838544172e-8, 2.7557319223985893e-6);
    ps = fma(ps, r2, -1.984126984126984e-4);
    ps = fma(ps, r2, 8.333333333333333e-3);
    ps = fma(ps, r2, -1.6666666666666666e-1);
    double sr = fma(ps * r2, r, r);
    double pc = fma(r2, 2.08767569878681e-9, -2.755731922398589e-7);
    pc = fma(pc, r2, 2.48015873015873e-5);
    pc = fma(pc, r2, -1.388888888888889e-3);
    pc = fma(pc, r2, 4.1666666666666664e-2);
    pc = fma(pc, r2, -0.5);
    double cr = fma(pc, r2, 1.0);
    int q = (int)k;
    s = (q & 1) ? cr : sr;
    c = (q & 1) ? sr : cr;
    if (q & 2) s = -s;
    if ((q + 1) & 2) c = -c;
}

// float32 unit vector for the SEARCH: float64 trig (<= 1e-11), products, rounded once - every component is within
// 2^-25 + 3e-11 of the exact value.
__device__ __forceinline__ float3 agx_search_xyz(float2 latlon) {
    double sl, cl, so, co;
    agx_sincos_search((double)latlon.x, sl, cl);
    agx_sincos_search((double)latlon.y, so, co);
    return make_float3((float)(cl * co), (float)(cl * so), (float)sl);
}

// Bound on |fp32 chord^2 - exact chord^2| for two search vectors (see DESIGN.md "FP32 filter margin"):
// each component carries <= 2^-25 (+ 3e-11) absolute error, the differences <= 2^-24 (+ one rounding), so
// |err| <= 2*sqrt(3)*2^-24*chord + fp32 evaluation error (<= 4 ulp of chord^2) + 3*2^-48.
// 4.2e-7*chord + 1e-6*chord^2 + 1e-13 covers it with >2x slack.
__device__ __forceinline__ float agx_chord2_margin(float d2) {
    return 4.2e-7f * sqrtf(d2) + 1.0e-6f * d2 + 1.0e-13f;
}

// sklearn HaversineDistance64.rdist (sklearn/metrics/_dist_metrics.pyx.tp:2639-2648), float64 on the
// float32 inputs: x1 = query, x2 = tree point.  __dmul_rn/__dadd_rn keep ptxas from contracting
// into FMAs so the operation order is the reference's.
__device__ __forceinline__ double agx_rdist64(float2 q, float2 p) {
    double lat1 = (double)q.x, lon1 = (double)q.y, lat2 = (double)p.x, lon2 = (double)p.y;
    double sin_0 = sin(0.5 * (lat1 - lat2));
    double sin_1 = sin(0.5 * (lon1 - lon2));
    double cc = __dmul_rn(cos(lat1), cos(lat2));
    return __dadd_rn(__dmul_rn(sin_0, sin_0), __dmul_rn(__dmul_rn(cc, sin_1), sin_1));
}

// relative width of an ulp-level tie in float64 rdist (DESIGN.md parity rules; oracle/ref_path.py TIE_TAU)
#define AGX_TIE_TAU 9.094947017729282e-13 /* 2^-40 */

// (rdist, index) ordering with the tie rule: values within TAU (relative) compare by index.
__device__ __forceinline__ bool agx_tie_less(double ra, int ia, double rb, int ib) {
    double big = fmax(ra, rb);
    if (fabs(ra - rb) <= AGX_TIE_TAU * big) return ia < ib;
    return ra < rb;
}

// ------------------------------------------------------------------------------------------------
// numpy's float32 sin/cos, bit for bit (Cody-Waite reduction + minimax polynomials evaluated with
// FMAs; numpy/_core/src/umath/loops_trigonometric.dispatch.*).  Verified against numpy 2.3.5 on
// EVERY float32 in [-2pi, 2pi] (tests/test_numpy_sincos.py documents the check).  Needed because
// the reference evaluates latlon -> xyz in float32 (generate/transforms.py:106-110) and
// EdgeDirection is ill-conditioned in those bits (SURVEY.md H3).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void agx_np_sincosf(float x, float& s_out, float& c_out) {
    float q = __fmaf_rn(x, 0x1.45f306p-1f, 0x1.8p+23f);  // numpy's build contracts x*(2/pi) + magic
    q = __fsub_rn(q, 0x1.8p+23f);
    float r = __fmaf_rn(q, -0x1.921fb0p+00f, x);
    r = __fmaf_rn(q, -0x1.5110b4p-22f, r);
    r = __fmaf_rn(q, -0x1.846988p-48f, r);
    float r2 = __fmul_rn(r, r);
    float c = __fmaf_rn(0x1.98e616p-16f, r2, -0x1.6c06dcp-10f);
    c = __fmaf_rn(c, r2, 0x1.55553cp-05f);
    c = __fmaf_rn(c, r2, -0x1p-1f);
    c = __fmaf_rn(c, r2, 0x1p0f);
    float s = __fmaf_rn(0x1.7d3bbcp-19f, r2, -0x1.a06bbap-13f);
    s = __fmaf_rn(s, r2, 0x1.11119ap-07f);
    s = __fmaf_rn(s, r2, -0x1.555556p-03f);
    s = __fmaf_rn(s, r2, 0.0f);
    s = __fmaf_rn(s, r, r);
    int iq = (int)q;
    // sine: quadrant iq; cosine: quadrant iq + 1
    float vs = (iq & 1) ? c : s;
    if (iq & 2) vs = __fsub_rn(0.0f, vs);
    int ic = iq + 1;
    float vc = (ic & 1) ? c : s;
    if (ic & 2) vc = __fsub_rn(0.0f, vc);
    s_out = vs;
    c_out = vc;
}

// numpy's float32 sin(x), bit for bit, with a short cut for |x| < ~pi/4 (quadrant 0: the argument reduction is the
// identity and only the sine polynomial is needed) - the half-differences of an edge's endpoints.
__device__ __forceinline__ float agx_np_sinf_short(float x) {
    float q = __fsub_rn(__fmaf_rn(x, 0x1.45f306p-1f, 0x1.8p+23f), 0x1.8p+23f);
    if (q == 0.0f) {
        float r2 = __fmul_rn(x, x);
        float s = __fmaf_rn(0x1.7d3bbcp-19f, r2, -0x1.a06bbap-13f);
        s = __fmaf_rn(s, r2, 0x1.11119ap-07f);
        s = __fmaf_rn(s, r2, -0x1.555556p-03f);
        s = __fmaf_rn(s, r2, 0.0f);
        return __fmaf_rn(s, x, x);
    }
    float s, c;
    agx_np_sincosf(x, s, c);
    return s;
}

// warp helpers
__device__ __forceinline__ int agx_warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
