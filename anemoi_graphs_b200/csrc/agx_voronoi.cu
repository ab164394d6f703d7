// Spherical Voronoi cell areas - SphericalAreaWeights.get_raw_values
// (/root/reference/src/anemoi/graphs/nodes/attributes.py:165-221): scipy.spatial.SphericalVoronoi(points).calculate_areas()
// on points = latlon_rad_to_cartesian(x) evaluated in float32 (generate/transforms.py:106-110).
//
// scipy builds the diagram from the convex hull of the generators: a Voronoi vertex is the unit normal of a hull
// facet, and the region of generator p is the set of directions x whose support point is p, i.e.
//     region(p) = { x on the sphere : x . (q - p) <= 0 for every other generator q }
// with the generators AS GIVEN - float32-rounded, so up to 6e-8 off the unit sphere, which tilts a bisector between
// neighbours 1e-3 rad apart by up to 1e-4 rad.  (The areas of a fine grid therefore carry percent-level noise in the
// reference; parity means reproducing it, so the half-spaces below use q - p un-normalised.)
//
// One thread per generator: its k nearest neighbours (agx_knn self query, ascending distance) cut a convex polygon in
// the gnomonic plane at p (planes through the origin are straight lines there); the loop stops once no farther
// generator can reach the polygon ("security radius").  The polygon's vertices are then re-evaluated in 3-D as
// normalised cross products of adjacent half-space normals - scipy's facet normals - and the area is scipy's sum of
// |2 atan2(det[p, v_i, v_i+1], 1 + p.v_i + v_i.v_i+1 + v_i+1.p)| (Van Oosterom - Strackee, _voronoi.pyx).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>

#include "agx_common.cuh"

#include <math.h>

#define VOR_MAXV 32
#define VOR_BOX 1.0e3               /* initial square in the gnomonic plane: 89.94 degrees, i.e. the open hemisphere */
#define VOR_NORM_SLACK 2.5e-7       /* bisector tilt budget: (|q| - |p|) / angle, float32 generators */

#define VOR_OK 0
#define VOR_MORE 1       /* neighbours exhausted before the security radius was reached */
#define VOR_UNBOUNDED 2  /* ... and the cell still touches the initial square */
#define VOR_DUPLICATE 3  /* two generators coincide (scipy: "Duplicate generators present") */
#define VOR_OVERFLOW 4   /* more than VOR_MAXV edges */

struct VorPoly {
    double a[VOR_MAXV], b[VOR_MAXV], c[VOR_MAXV];  // edge j: a u + b v + c <= 0
    double u[VOR_MAXV], v[VOR_MAXV];               // vertex j: end of edge j = its meeting point with edge j+1
    int id[VOR_MAXV];                              // generator behind edge j (-1: initial square)
    int m;
};

__device__ __forceinline__ double3 vor_xyz(float2 ll) {
    float sl, cl, so, co;
    agx_np_sincosf(ll.x, sl, cl);
    agx_np_sincosf(ll.y, so, co);
    return make_double3((double)__fmul_rn(cl, co), (double)__fmul_rn(cl, so), (double)sl);
}

__device__ __forceinline__ double dot3(double3 a, double3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ double3 cross3(double3 a, double3 b) {
    return make_double3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ double3 scale3(double3 a, double s) { return make_double3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ double3 sub3(double3 a, double3 b) { return make_double3(a.x - b.x, a.y - b.y, a.z - b.z); }

__device__ __forceinline__ void vor_meet(double a1, double b1, double c1, double a2, double b2, double c2, double& u, double& v) {
    double det = a1 * b2 - a2 * b1;
    u = (b1 * c2 - b2 * c1) / det;
    v = (a2 * c1 - a1 * c2) / det;
}

// clip the polygon by a u + b v + c <= 0; returns false on overflow
__device__ bool vor_clip(VorPoly& P, double a, double b, double c, int id) {
    double s[VOR_MAXV];
    int first_in = -1, n_out = 0;
    for (int j = 0; j < P.m; ++j) {
        s[j] = a * P.u[j] + b * P.v[j] + c;
        if (s[j] > 0.0) ++n_out;
        else if (first_in < 0) first_in = j;
    }
    if (n_out == 0) return true;
    if (first_in < 0) {  // cannot happen for a generator inside its own cell; keep the polygon
        return true;
    }
    VorPoly Q;
    Q.m = 0;
    int open = -1;  // position in Q of the new edge whose end vertex is still unknown
    for (int t = 1; t <= P.m; ++t) {
        int j = (first_in + t) % P.m, jp = (j + P.m - 1) % P.m;  // edge j runs from vertex jp to vertex j
        bool in_prev = s[jp] <= 0.0, in_cur = s[j] <= 0.0;
        if (!in_prev && !in_cur) continue;
        if (Q.m + 2 > VOR_MAXV) return false;
        if (!in_prev && in_cur) {  // re-entering: close the new edge on this one
            vor_meet(a, b, c, P.a[j], P.b[j], P.c[j], Q.u[open], Q.v[open]);
        }
        int o = Q.m++;
        Q.a[o] = P.a[j]; Q.b[o] = P.b[j]; Q.c[o] = P.c[j]; Q.id[o] = P.id[j];
        if (in_cur) {
            Q.u[o] = P.u[j]; Q.v[o] = P.v[j];
        } else {  // leaving: edge j now ends on the new line, which becomes the next edge
            vor_meet(P.a[j], P.b[j], P.c[j], a, b, c, Q.u[o], Q.v[o]);
            open = Q.m++;
            Q.a[open] = a; Q.b[open] = b; Q.c[open] = c; Q.id[open] = id;
        }
    }
    P = Q;
    return true;
}

__global__ void __launch_bounds__(128) k_voronoi_areas(const float2* __restrict__ latlon, int64_t n,
                                                       const int32_t* __restrict__ knn, int k, int exhaustive,
                                                       const int32_t* __restrict__ subset, int64_t m, double radius,
                                                       double* __restrict__ areas, int32_t* __restrict__ status) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = subset ? subset[t] : t;
        const double3 p = vor_xyz(latlon[i]);
        const double pn = sqrt(dot3(p, p));
        const double3 ph = scale3(p, 1.0 / pn);
        // tangent frame
        double3 axis = fabs(ph.x) <= fabs(ph.y) && fabs(ph.x) <= fabs(ph.z) ? make_double3(1, 0, 0)
                       : (fabs(ph.y) <= fabs(ph.z) ? make_double3(0, 1, 0) : make_double3(0, 0, 1));
        double3 e1 = cross3(ph, axis);
        e1 = scale3(e1, 1.0 / sqrt(dot3(e1, e1)));
        const double3 e2 = cross3(ph, e1);
        VorPoly P;
        P.m = 4;
        const double B = VOR_BOX;
        P.a[0] = 1;  P.b[0] = 0;  P.c[0] = -B; P.u[0] = B;  P.v[0] = B;   // u <= B, ends at (B, B)
        P.a[1] = 0;  P.b[1] = 1;  P.c[1] = -B; P.u[1] = -B; P.v[1] = B;
        P.a[2] = -1; P.b[2] = 0;  P.c[2] = -B; P.u[2] = -B; P.v[2] = -B;
        P.a[3] = 0;  P.b[3] = -1; P.c[3] = -B; P.u[3] = B;  P.v[3] = -B;
        P.id[0] = P.id[1] = P.id[2] = P.id[3] = -1;
        int st = VOR_MORE;
        for (int j = 0; j < k; ++j) {
            const int q_idx = knn[t * k + j];
            if (q_idx == (int)i || q_idx < 0) continue;
            const double3 q = vor_xyz(latlon[q_idx]);
            const double3 nrm = sub3(q, p);
            const double d2 = dot3(nrm, nrm);
            if (d2 == 0.0) { st = VOR_DUPLICATE; break; }
            // security radius: every generator from here on is at least this far (the list is ascending up to the
            // search's float32 resolution, hence the 1e-3), its bisector at least `reach` from p in the gnomonic plane
            double rho2 = 0.0;
            for (int e = 0; e < P.m; ++e) rho2 = fmax(rho2, P.u[e] * P.u[e] + P.v[e] * P.v[e]);
            const double theta = 2.0 * asin(fmin(0.5 * sqrt(d2), 1.0));
            const double half = 0.5 * theta - VOR_NORM_SLACK / theta;
            if (half > 0.0 && half < 1.5) {
                const double reach = tan(half) * (1.0 - 1.0e-3);
                if (reach * reach > rho2) {
                    bool boxed = false;
                    for (int e = 0; e < P.m; ++e) boxed |= (P.id[e] < 0);
                    if (!boxed) { st = VOR_OK; break; }
                }
            }
            if (!vor_clip(P, dot3(nrm, e1), dot3(nrm, e2), dot3(nrm, ph), q_idx)) { st = VOR_OVERFLOW; break; }
        }
        if (st == VOR_MORE) {
            bool boxed = false;
            for (int e = 0; e < P.m; ++e) boxed |= (P.id[e] < 0);
            if (boxed) st = VOR_UNBOUNDED;
            else if (exhaustive) st = VOR_OK;  // every other generator has been applied: the cell is what is left
        }
        double area = 0.0;
        if (st == VOR_OK) {
            // 3-D vertices: unit normal of the hull facet (p, q_j, q_j+1), on p's side
            double3 first = make_double3(0, 0, 0), prev = make_double3(0, 0, 0);
            for (int e = 0; e <= P.m; ++e) {
                double3 vtx;
                if (e < P.m) {
                    const int e2i = (e + 1) % P.m;
                    const double3 n1 = sub3(vor_xyz(latlon[P.id[e]]), p);
                    const double3 n2 = sub3(vor_xyz(latlon[P.id[e2i]]), p);
                    double3 w = cross3(n1, n2);
                    double wn = sqrt(dot3(w, w));
                    if (wn > 0.0) {
                        w = scale3(w, (dot3(w, ph) < 0.0 ? -1.0 : 1.0) / wn);
                    } else {  // parallel normals (cannot bound a vertex): fall back to the planar meeting point
                        w = make_double3(ph.x + P.u[e] * e1.x + P.v[e] * e2.x, ph.y + P.u[e] * e1.y + P.v[e] * e2.y,
                                         ph.z + P.u[e] * e1.z + P.v[e] * e2.z);
                        w = scale3(w, 1.0 / sqrt(dot3(w, w)));
                    }
                    vtx = w;
                    if (e == 0) first = vtx;
                } else {
                    vtx = first;
                }
                if (e > 0) {
                    // scipy _voronoi.calculate_solid_angles on the triangle (p, prev, vtx), p as given (not normalised)
                    const double num = dot3(p, cross3(prev, vtx));
                    const double den = 1.0 + dot3(p, prev) + dot3(prev, vtx) + dot3(vtx, p);
                    area += fabs(2.0 * atan2(num, den));
                }
                prev = vtx;
            }
            area *= radius * radius;
        }
        if (st == VOR_OK) areas[i] = area;
        status[t] = st;
    }
}

extern "C" int agx_voronoi_areas(const float* latlon, int64_t n, const int32_t* knn, int k, int exhaustive, const int32_t* subset, int64_t m,
                                 double radius, double* areas, int32_t* status, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n >= 0 && m >= 0 && k > 0, AGX_ERR_ARG, "agx_voronoi_areas: bad sizes");
    if (m == 0) return AGX_OK;
    AGX_REQUIRE(latlon && knn && areas && status, AGX_ERR_ARG, "agx_voronoi_areas: NULL buffer");
    k_voronoi_areas<<<agx_grid(m, 128, 8), 128, 0, stream>>>((const float2*)latlon, n, knn, k, exhaustive ? 1 : 0, subset, m, radius, areas, status);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Very few generators (n <= VOR_SMALL_N): a cell can be wider than a hemisphere, which the gnomonic plane at its
// generator cannot hold.  Exhaustive form on the sphere itself, one thread per generator: every pair of half-space
// normals n_a = q_a - p, n_b = q_b - p meets in the two directions +-(n_a x n_b) / |.|; a direction is a vertex of the
// cell iff it satisfies every other half-space.  The vertices are ordered by azimuth about p (the cell is star-shaped
// about its generator: every half-space contains p) and the area is the same Van Oosterom - Strackee sum.  O(n^3) per
// cell - a few hundred thousand operations at most.
// ------------------------------------------------------------------------------------------------------------------
#define VOR_SMALL_N 64
#define VOR_SMALL_MAXV 128

__global__ void __launch_bounds__(64) k_voronoi_areas_small(const float2* __restrict__ latlon, int n,
                                                            const int32_t* __restrict__ subset, int m, double radius,
                                                            double* __restrict__ areas, int32_t* __restrict__ status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const int i = subset ? subset[t] : t;
    const double3 p = vor_xyz(latlon[i]);
    const double3 ph = scale3(p, 1.0 / sqrt(dot3(p, p)));
    double3 axis = fabs(ph.x) <= fabs(ph.y) && fabs(ph.x) <= fabs(ph.z) ? make_double3(1, 0, 0)
                   : (fabs(ph.y) <= fabs(ph.z) ? make_double3(0, 1, 0) : make_double3(0, 0, 1));
    double3 e1 = cross3(ph, axis);
    e1 = scale3(e1, 1.0 / sqrt(dot3(e1, e1)));
    const double3 e2 = cross3(ph, e1);
    double3 vtx[VOR_SMALL_MAXV];
    double ang[VOR_SMALL_MAXV];
    int nv = 0;
    int st = VOR_OK;
    for (int a = 0; a < n && st == VOR_OK; ++a) {
        if (a == i) continue;
        const double3 na = sub3(vor_xyz(latlon[a]), p);
        if (dot3(na, na) == 0.0) { st = VOR_DUPLICATE; break; }
        for (int b = a + 1; b < n && st == VOR_OK; ++b) {
            if (b == i) continue;
            const double3 nb = sub3(vor_xyz(latlon[b]), p);
            double3 w = cross3(na, nb);
            const double wn = sqrt(dot3(w, w));
            if (wn <= 1e-14 * sqrt(dot3(na, na) * dot3(nb, nb))) continue;  // parallel bisector planes: no vertex
            w = scale3(w, 1.0 / wn);
            for (int sgn = 0; sgn < 2; ++sgn) {
                const double3 v = sgn ? scale3(w, -1.0) : w;
                bool inside = true;
                for (int q = 0; q < n && inside; ++q) {
                    if (q == i || q == a || q == b) continue;
                    const double3 nq = sub3(vor_xyz(latlon[q]), p);
                    inside = dot3(v, nq) <= 1e-13 * sqrt(dot3(nq, nq));
                }
                if (!inside) continue;
                bool dup = false;  // three or more bisectors through one point: keep one copy
                for (int e = 0; e < nv && !dup; ++e) {
                    const double3 d = sub3(vtx[e], v);
                    dup = dot3(d, d) < 1e-24;
                }
                if (dup) continue;
                if (nv == VOR_SMALL_MAXV) { st = VOR_OVERFLOW; break; }
                vtx[nv] = v;
                ang[nv] = atan2(dot3(v, e2), dot3(v, e1));
                ++nv;
            }
        }
    }
    if (st == VOR_OK && nv < 3) st = VOR_UNBOUNDED;  // fewer than 4 generators in general position
    double area = 0.0;
    if (st == VOR_OK) {
        for (int x = 1; x < nv; ++x) {  // insertion sort by azimuth
            const double3 kv = vtx[x];
            const double ka = ang[x];
            int y = x - 1;
            while (y >= 0 && ang[y] > ka) {
                vtx[y + 1] = vtx[y];
                ang[y + 1] = ang[y];
                --y;
            }
            vtx[y + 1] = kv;
            ang[y + 1] = ka;
        }
        for (int x = 0; x < nv; ++x) {
            const double3 v0 = vtx[x], v1 = vtx[(x + 1) % nv];
            const double num = dot3(p, cross3(v0, v1));
            const double den = 1.0 + dot3(p, v0) + dot3(v0, v1) + dot3(v1, p);
            area += fabs(2.0 * atan2(num, den));
        }
        areas[i] = area * radius * radius;
    }
    status[t] = st;
}

extern "C" int agx_voronoi_areas_small(const float* latlon, int64_t n, const int32_t* subset, int64_t m, double radius,
                                       double* areas, int32_t* status, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n >= 4 && n <= VOR_SMALL_N, AGX_ERR_ARG, "agx_voronoi_areas_small: 4 <= n <= 64 generators");
    AGX_REQUIRE(m >= 0 && m <= n, AGX_ERR_ARG, "agx_voronoi_areas_small: bad subset size");
    if (m == 0) return AGX_OK;
    AGX_REQUIRE(latlon && areas && status, AGX_ERR_ARG, "agx_voronoi_areas_small: NULL buffer");
    k_voronoi_areas_small<<<((int)m + 63) / 64, 64, 0, stream>>>((const float2*)latlon, (int)n, subset, (int)m, radius, areas, status);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Isolatitude area weights (IsolatitudeAreaWeights of newer releases; DESIGN section 4).  A row is one float32
// latitude (-0.0 and +0.0 one row); with the distinct latitudes phi_0 > ... > phi_{R-1} in float64, row r is the band
// between b_r = (phi_{r-1} + phi_r) / 2 and b_{r+1}, b_0 = pi/2 and b_R = -pi/2, and each of its c_r nodes weighs
//     4 pi cos((b_r + b_{r+1}) / 2) sin((b_r - b_{r+1}) / 2) / c_r
// (the product form: 2 pi (sin b_r - sin b_{r+1}) cancels near the poles).  Rows come from a radix sort of
// order-preserving latitude keys and a run-length encoding of the sorted keys; every input takes this one path.
// ------------------------------------------------------------------------------------------------------------------
#define ISO_HALF_PI_F_BITS 0x3fc90fdbu  // float32(pi/2) = 1.5707963705 > pi/2: a node at a pole is valid

// uint32 key whose unsigned order is the float order of the latitude; -0.0 and +0.0 give the key of +0.0
__device__ __forceinline__ uint32_t iso_key(float lat) {
    const uint32_t u = __float_as_uint(__fadd_rn(lat, 0.0f));
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ double iso_lat(uint32_t key) {
    return (double)__uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
}

__global__ void __launch_bounds__(256) k_iso_keys(const float2* __restrict__ latlon, int64_t n, uint32_t* __restrict__ keys,
                                                  int* __restrict__ bad) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float lat = latlon[i].x;
        if ((__float_as_uint(lat) & 0x7fffffffu) > ISO_HALF_PI_F_BITS) *bad = 1;  // NaN or beyond +-float32(pi/2)
        keys[i] = iso_key(lat);
    }
}

// one thread per row of the sorted distinct keys (ascending latitude: south to north); R = *n_rows on the device
__global__ void __launch_bounds__(256) k_iso_bands(const uint32_t* __restrict__ row_keys, const int32_t* __restrict__ counts,
                                                   const int* __restrict__ n_rows, double* __restrict__ row_weight) {
    const int R = *n_rows;
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < R; r += gridDim.x * blockDim.x) {
        const double phi = iso_lat(row_keys[r]);
        const double north = r + 1 < R ? (phi + iso_lat(row_keys[r + 1])) * 0.5 : 1.5707963267948966;
        const double south = r > 0 ? (iso_lat(row_keys[r - 1]) + phi) * 0.5 : -1.5707963267948966;
        const double area = __dmul_rn(__dmul_rn(12.566370614359172, cos((north + south) * 0.5)), sin((north - south) * 0.5));
        row_weight[r] = area / (double)counts[r];
    }
}

// one thread per node: its row by binary search among the R distinct keys
__global__ void __launch_bounds__(256) k_iso_weights(const uint32_t* __restrict__ keys, int64_t n,
                                                     const uint32_t* __restrict__ row_keys, const int* __restrict__ n_rows,
                                                     const double* __restrict__ row_weight, double* __restrict__ areas) {
    const int R = *n_rows;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t key = keys[i];
        int lo = 0, hi = R - 1;  // row_keys[lo] <= key <= row_keys[hi]: every key is one of the row keys
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (row_keys[mid] < key) lo = mid + 1;
            else hi = mid;
        }
        areas[i] = row_weight[lo];
    }
}

extern "C" int agx_isolatitude_areas(const float* latlon, int64_t n, double* areas, int32_t* n_rows, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n >= 0 && n < (int64_t)2147483647, AGX_ERR_ARG, "agx_isolatitude_areas: n out of [0, 2^31)");
    if (n_rows) *n_rows = 0;
    if (n == 0) return AGX_OK;
    AGX_REQUIRE(latlon && areas, AGX_ERR_ARG, "agx_isolatitude_areas: NULL buffer");
    int* flag = nullptr;  // [0] bad latitude, [1] R
    int rc = agx_bad_flag_alloc(&flag, stream);
    if (rc) return rc;
    uint32_t* keys = nullptr;  // node keys, sorted keys, row keys: n each
    int32_t* counts = nullptr;
    double* row_weight = nullptr;
    void* temp = nullptr;
    cudaError_t e;
#define ISO_TRY(expr)                                                                                      \
    if ((e = (expr)) != cudaSuccess) {                                                                     \
        agx_set_error("%s failed: %s", #expr, cudaGetErrorString(e));                                      \
        cudaFreeAsync(keys, stream); cudaFreeAsync(counts, stream); cudaFreeAsync(row_weight, stream);     \
        cudaFreeAsync(temp, stream); cudaFreeAsync(flag, stream);                                          \
        return AGX_ERR_CUDA;                                                                               \
    }
    ISO_TRY(cudaMallocAsync(&keys, 3 * n * sizeof(uint32_t), stream));
    ISO_TRY(cudaMallocAsync(&counts, n * sizeof(int32_t), stream));
    ISO_TRY(cudaMallocAsync(&row_weight, n * sizeof(double), stream));
    uint32_t* sorted = keys + n;
    uint32_t* row_keys = keys + 2 * n;
    size_t sort_bytes = 0, rle_bytes = 0;
    ISO_TRY(cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, keys, sorted, (int)n, 0, 32, stream));
    ISO_TRY(cub::DeviceRunLengthEncode::Encode(nullptr, rle_bytes, sorted, row_keys, counts, flag + 1, (int)n, stream));
    size_t temp_bytes = sort_bytes > rle_bytes ? sort_bytes : rle_bytes;
    ISO_TRY(cudaMallocAsync(&temp, temp_bytes > 0 ? temp_bytes : 16, stream));
    const int grid = agx_grid(n, 256, 8);
    k_iso_keys<<<grid, 256, 0, stream>>>((const float2*)latlon, n, keys, flag);
    ISO_TRY(cudaGetLastError());
    ISO_TRY(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys, sorted, (int)n, 0, 32, stream));
    ISO_TRY(cub::DeviceRunLengthEncode::Encode(temp, temp_bytes, sorted, row_keys, counts, flag + 1, (int)n, stream));
    k_iso_bands<<<grid, 256, 0, stream>>>(row_keys, counts, flag + 1, row_weight);
    ISO_TRY(cudaGetLastError());
    k_iso_weights<<<grid, 256, 0, stream>>>(keys, n, row_keys, flag + 1, row_weight, areas);
    ISO_TRY(cudaGetLastError());
#undef ISO_TRY
    agx_note_launch(3 + 5 + 2);  // the three kernels; CUB's histogram and four onesweep passes, and its encoding scan
    cudaFreeAsync(keys, stream);
    cudaFreeAsync(counts, stream);
    cudaFreeAsync(row_weight, stream);
    cudaFreeAsync(temp, stream);
    return agx_bad_flag_read(flag, "agx_isolatitude_areas: a latitude is NaN or its magnitude exceeds float32(pi/2)", n_rows,
                             stream);
}
