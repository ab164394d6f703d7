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
// Wide cells (DESIGN section 4, K9): the cells that k_voronoi_areas leaves open after its 63 nearest neighbours - a
// coarse generator next to a much finer region, whose nearest neighbours all lie on one side of it - or that have
// more than VOR_MAXV edges.  No radius sweep: a polygon built from a candidate set C is the true cell of g exactly
// when no generator h has (h - g) . v > 0 at any of its vertices v (the corners of the initial square included),
// because the polygon is the convex hull of its vertices.  So, in rounds over the cells still open:
//   clip   one warp per cell clips the square with C in ascending (float64 rdist, index) order; the polygon lives in
//          shared memory (VOR_WIDE_CAP edges) and the lanes split each clip's vertices;
//   query  agx_knn of every vertex against the node set's index, VOR_WIDE_K neighbours;
//   check  each (vertex, neighbour) pair in float64; the violators that are not candidates yet join C.
// A cell without a violator whose vertices are certified (below) is final and gets its area as k_voronoi_areas
// computes it; a cell that still touches the square then is not inside its open hemisphere.
//
// Certification of a vertex v: every generator h outside its VOR_WIDE_K nearest is at least as far from v (haversine
// on the float32 (lat, lon)) as the K-th, a_K.  The float32 generator has |h| <= 1 + 2 VOR_NORM_SLACK and its
// direction (and v's float32 query point) is within 2 VOR_NORM_SLACK rad of the exact one, so
//     h . v <= (1 + 2 S) (cos a_K + 2 S sin a_K),   S = VOR_NORM_SLACK;
// once that is below g . v, no generator outside the list can cut the cell at v.
// ------------------------------------------------------------------------------------------------------------------
#define VOR_WIDE_CAP 1024  /* polygon edges a warp holds in shared memory */
#define VOR_WIDE_NEW 64    /* violators a cell takes per round; any others are found again in the next round */
#define VOR_WIDE_K 32      /* neighbours of each vertex */
#define VOR_WIDE_ROUNDS 32
#define VOR_WIDE_OVERFLOW 5  /* more than VOR_WIDE_CAP edges */
#define VOR_UNCERTIFIED 6    /* no violator, but VOR_WIDE_K neighbours do not certify a vertex */

struct VorWideSmem {  // two polygons: each clip reads one and writes the other
    double a[2][VOR_WIDE_CAP], b[2][VOR_WIDE_CAP], c[2][VOR_WIDE_CAP], u[2][VOR_WIDE_CAP], v[2][VOR_WIDE_CAP];
    int id[2][VOR_WIDE_CAP];
    unsigned in[VOR_WIDE_CAP / 32];  // bit j: vertex j is inside the clipping half-plane
};

// generator p (as given, float32-rounded), its unit direction and the tangent frame of k_voronoi_areas
struct VorFrame {
    double3 p, ph, e1, e2;
};

__device__ __forceinline__ VorFrame vor_frame(float2 ll) {
    VorFrame f;
    f.p = vor_xyz(ll);
    f.ph = scale3(f.p, 1.0 / sqrt(dot3(f.p, f.p)));
    const double3 axis = fabs(f.ph.x) <= fabs(f.ph.y) && fabs(f.ph.x) <= fabs(f.ph.z) ? make_double3(1, 0, 0)
                         : (fabs(f.ph.y) <= fabs(f.ph.z) ? make_double3(0, 1, 0) : make_double3(0, 0, 1));
    f.e1 = cross3(f.ph, axis);
    f.e1 = scale3(f.e1, 1.0 / sqrt(dot3(f.e1, f.e1)));
    f.e2 = cross3(f.ph, f.e1);
    return f;
}

// One warp per open cell t (open[w], w < *n_open).  Candidates cand[off[t], off[t+1]) (self and -1 are skipped);
// sorted receives them in clip order, key is scratch.  Vertex slots start at off[t] + 4 t (a polygon has at most
// one edge per candidate plus the four of the square): unit xyz, float32 (lat, lon) to search with, and the
// generator behind the edge that ends there (-1: the square).  nv[t] = vertex count, 0 if the cell failed.
__global__ void __launch_bounds__(32) k_voronoi_wide_clip(const float2* __restrict__ latlon, const int32_t* __restrict__ wide,
                                                          const int32_t* __restrict__ open, const int64_t* __restrict__ n_open,
                                                          const int64_t* __restrict__ off, const int32_t* __restrict__ cand,
                                                          double* __restrict__ key, int32_t* __restrict__ sorted,
                                                          double* __restrict__ vxyz, float2* __restrict__ vll,
                                                          int32_t* __restrict__ vid, int32_t* __restrict__ nv,
                                                          unsigned long long* __restrict__ ctl) {
    extern __shared__ __align__(16) unsigned char vor_smem[];
    VorWideSmem& S = *reinterpret_cast<VorWideSmem*>(vor_smem);
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    const int64_t count = *n_open;
    for (int64_t w = blockIdx.x; w < count; w += gridDim.x) {
        const int t = open[w];
        const int i = wide[t];
        const float2 gll = latlon[i];
        const VorFrame F = vor_frame(gll);
        const int64_t o0 = off[t];
        const int L = (int)(off[t + 1] - o0);
        // clip order: ascending (rdist, index), by rank counting (the lists are a few hundred long)
        for (int j = lane; j < L; j += 32) {
            const int q = cand[o0 + j];
            key[o0 + j] = q >= 0 ? agx_rdist64(gll, latlon[q]) : HUGE_VAL;
        }
        __syncwarp();
        for (int j = lane; j < L; j += 32) {
            const double kj = key[o0 + j];
            const int ij = cand[o0 + j];
            int r = 0;
            for (int x = 0; x < L; ++x) {
                const double kx = key[o0 + x];
                const int ix = cand[o0 + x];
                r += kx < kj || (kx == kj && (ix < ij || (ix == ij && x < j)));
            }
            sorted[o0 + r] = ij;
        }
        __syncwarp();
        const double B = VOR_BOX;
        if (lane < 4) {  // the square of k_voronoi_areas: edge e is u <= B, v <= B, -u <= B, -v <= B
            S.a[0][lane] = lane == 0 ? 1.0 : (lane == 2 ? -1.0 : 0.0);
            S.b[0][lane] = lane == 1 ? 1.0 : (lane == 3 ? -1.0 : 0.0);
            S.c[0][lane] = -B;
            S.u[0][lane] = lane == 0 || lane == 3 ? B : -B;
            S.v[0][lane] = lane < 2 ? B : -B;
            S.id[0][lane] = -1;
        }
        __syncwarp();
        int cur = 0, m = 4, st = VOR_OK;
        for (int x = 0; x < L; ++x) {
            const int q = sorted[o0 + x];
            if (q == i || q < 0) continue;
            const double3 nrm = sub3(vor_xyz(latlon[q]), F.p);
            if (dot3(nrm, nrm) == 0.0) { st = VOR_DUPLICATE; break; }
            const double A = dot3(nrm, F.e1), Bq = dot3(nrm, F.e2), C = dot3(nrm, F.ph);
            int n_out = 0, first_in = -1;
            for (int base = 0; base < m; base += 32) {
                const int j = base + lane;
                const bool out = j < m && A * S.u[cur][j] + Bq * S.v[cur][j] + C > 0.0;
                const unsigned bo = __ballot_sync(full, out), bi = __ballot_sync(full, j < m && !out);
                if (lane == 0) S.in[base >> 5] = bi;
                n_out += __popc(bo);
                if (bi && first_in < 0) first_in = base + __ffs(bi) - 1;
            }
            __syncwarp();
            if (n_out == 0 || first_in < 0) continue;  // no vertex cut, or all of them (as vor_clip: keep the polygon)
            // the edges in the order vor_clip visits them, j = (first_in + s) % m for s = 1..m: an edge inside at both
            // ends is kept, one that leaves is kept up to the new line and followed by it, one that re-enters closes
            // the new line (the output just before it) and is kept
            const int nx = cur ^ 1;
            int total = 0;
            for (int base = 0; base < m; base += 32) {
                const int s = base + lane + 1;
                int cnt = 0, j = 0;
                bool in_prev = false, in_cur = false;
                if (s <= m) {
                    j = (first_in + s) % m;
                    const int jp = (j + m - 1) % m;
                    in_prev = (S.in[jp >> 5] >> (jp & 31)) & 1u;
                    in_cur = (S.in[j >> 5] >> (j & 31)) & 1u;
                    cnt = in_cur ? 1 : (in_prev ? 2 : 0);
                }
                int incl = cnt;
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(full, incl, o);
                    if (lane >= o) incl += y;
                }
                const int pos = total + incl - cnt;
                total += __shfl_sync(full, incl, 31);
                if (cnt && pos + cnt <= VOR_WIDE_CAP) {
                    const double pa = S.a[cur][j], pb = S.b[cur][j], pc = S.c[cur][j];
                    S.a[nx][pos] = pa; S.b[nx][pos] = pb; S.c[nx][pos] = pc; S.id[nx][pos] = S.id[cur][j];
                    if (in_cur) {
                        S.u[nx][pos] = S.u[cur][j]; S.v[nx][pos] = S.v[cur][j];
                        if (!in_prev) vor_meet(A, Bq, C, pa, pb, pc, S.u[nx][pos - 1], S.v[nx][pos - 1]);
                    } else {
                        vor_meet(pa, pb, pc, A, Bq, C, S.u[nx][pos], S.v[nx][pos]);
                        S.a[nx][pos + 1] = A; S.b[nx][pos + 1] = Bq; S.c[nx][pos + 1] = C; S.id[nx][pos + 1] = q;
                    }
                }
            }
            __syncwarp();
            // the polygon must fit shared memory and the cell's L + 4 vertex slots (in exact arithmetic a clip adds at
            // most one edge, and the list holds the generator itself)
            if (total > VOR_WIDE_CAP || total > L + 4) { st = VOR_WIDE_OVERFLOW; break; }
            cur = nx;
            m = total;
        }
        const int64_t vb = o0 + 4 * (int64_t)t;
        if (st == VOR_OK) {
            for (int j = lane; j < m; j += 32) {
                const double u = S.u[cur][j], v = S.v[cur][j];
                double3 w = make_double3(F.ph.x + u * F.e1.x + v * F.e2.x, F.ph.y + u * F.e1.y + v * F.e2.y,
                                         F.ph.z + u * F.e1.z + v * F.e2.z);
                w = scale3(w, 1.0 / sqrt(dot3(w, w)));
                vxyz[3 * (vb + j)] = w.x; vxyz[3 * (vb + j) + 1] = w.y; vxyz[3 * (vb + j) + 2] = w.z;
                vll[vb + j] = make_float2((float)atan2(w.z, hypot(w.x, w.y)), (float)atan2(w.y, w.x));
                vid[vb + j] = S.id[cur][j];
            }
        } else if (lane == 0) {
            atomicOr(ctl, 1ull << st);
        }
        if (lane == 0) nv[t] = st == VOR_OK ? m : 0;
        __syncwarp();
    }
}

// the vertices of the open cells, packed in open-list order for the search: q[voff[t] + j] = vll[off[t] + 4 t + j]
__global__ void __launch_bounds__(32) k_voronoi_wide_pack(const int32_t* __restrict__ open, int64_t n_open,
                                                          const int64_t* __restrict__ off, const int64_t* __restrict__ voff,
                                                          const float2* __restrict__ vll, float2* __restrict__ q) {
    for (int64_t w = blockIdx.x; w < n_open; w += gridDim.x) {
        const int t = open[w];
        const int64_t vb = off[t] + 4 * (int64_t)t;
        for (int64_t j = threadIdx.x; j < voff[t + 1] - voff[t]; j += 32) q[voff[t] + j] = vll[vb + j];
    }
}

// one warp per open cell: every (vertex, neighbour) pair.  A cell with violators stays open - flag[t] = 1,
// grow[t] = its next candidate count, the violators (at most VOR_WIDE_NEW, first found first) in fresh[w * NEW ..] -
// and any other cell is final: its area, or a failure bit in ctl[0].  ctl[1] / ctl[2]: largest / total candidate
// count of the final cells; ctl[6]: cells that stay open and still touch the initial square.  flag, grow and ctl[6]
// are zero on entry.
__global__ void __launch_bounds__(32) k_voronoi_wide_check(const float2* __restrict__ latlon, const int32_t* __restrict__ wide,
                                                           const int32_t* __restrict__ open, int64_t n_open,
                                                           const int64_t* __restrict__ off, const int32_t* __restrict__ cand,
                                                           const int64_t* __restrict__ voff, const double* __restrict__ vxyz,
                                                           const int32_t* __restrict__ vid, const int32_t* __restrict__ nbr,
                                                           const double* __restrict__ nrd, double radius,
                                                           double* __restrict__ areas, uint8_t* __restrict__ flag,
                                                           int32_t* __restrict__ grow, int32_t* __restrict__ fresh,
                                                           unsigned long long* __restrict__ ctl) {
    __shared__ int found[VOR_WIDE_NEW];
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    const double S2 = 2.0 * VOR_NORM_SLACK;
    for (int64_t w = blockIdx.x; w < n_open; w += gridDim.x) {
        const int t = open[w];
        const int nvt = (int)(voff[t + 1] - voff[t]);
        if (nvt == 0) continue;  // failed in the clip
        const int i = wide[t];
        const double3 p = vor_xyz(latlon[i]);
        const int64_t o0 = off[t], vb = o0 + 4 * (int64_t)t, q0 = voff[t];
        const int L = (int)(off[t + 1] - o0);
        bool boxed = false, uncertified = false;
        int n_new = 0;
        for (int base = 0; base < nvt * VOR_WIDE_K; base += 32) {
            const int idx = base + lane;
            bool viol = false;
            int h = -1;
            if (idx < nvt * VOR_WIDE_K) {
                const int j = idx / VOR_WIDE_K, r = idx % VOR_WIDE_K;
                const double3 v = make_double3(vxyz[3 * (vb + j)], vxyz[3 * (vb + j) + 1], vxyz[3 * (vb + j) + 2]);
                const int ja = vid[vb + j], jb = vid[vb + (j + 1) % nvt];
                boxed |= ja < 0;
                h = nbr[(q0 + j) * VOR_WIDE_K + r];
                if (r == VOR_WIDE_K - 1 && h >= 0) {
                    const double ck = 1.0 - 2.0 * nrd[(q0 + j) * VOR_WIDE_K + r];
                    const double sk = sqrt(fmax(0.0, 1.0 - ck * ck));
                    uncertified |= (1.0 + S2) * (ck + S2 * sk) >= dot3(p, v);
                }
                if (h >= 0 && h != i && h != ja && h != jb) {
                    viol = dot3(sub3(vor_xyz(latlon[h]), p), v) > 0.0;
                    for (int x = 0; x < L && viol; ++x) viol = cand[o0 + x] != h;
                    for (int x = 0; x < n_new && viol; ++x) viol = found[x] != h;
                }
            }
            const unsigned vm = __ballot_sync(full, viol);
            if (vm) {
                bool keep = false;
                if (viol) keep = __ffs(__match_any_sync(vm, h)) - 1 == lane;  // one lane per distinct violator
                const unsigned km = __ballot_sync(full, keep);
                const int at = n_new + __popc(km & ((1u << lane) - 1u));
                if (keep && at < VOR_WIDE_NEW) found[at] = h;
                n_new = min(n_new + __popc(km), VOR_WIDE_NEW);
                __syncwarp();
            }
        }
        boxed = __any_sync(full, boxed);
        uncertified = __any_sync(full, uncertified);
        if (n_new > 0) {
            for (int x = lane; x < n_new; x += 32) fresh[w * VOR_WIDE_NEW + x] = found[x];
            if (lane == 0) {
                flag[t] = 1;
                grow[t] = L + n_new;
                if (boxed) atomicAdd(ctl + 6, 1ull);
            }
        } else if (lane == 0) {
            if (boxed) atomicOr(ctl, 1ull << VOR_UNBOUNDED);
            else if (uncertified) atomicOr(ctl, 1ull << VOR_UNCERTIFIED);
            else {
                // k_voronoi_areas' area: 3-D vertices from adjacent half-space normals, Van Oosterom - Strackee sum
                const double3 ph = scale3(p, 1.0 / sqrt(dot3(p, p)));
                double area = 0.0;
                double3 first = make_double3(0, 0, 0), prev = make_double3(0, 0, 0);
                for (int e = 0; e <= nvt; ++e) {
                    double3 vtx;
                    if (e < nvt) {
                        const double3 n1 = sub3(vor_xyz(latlon[vid[vb + e]]), p);
                        const double3 n2 = sub3(vor_xyz(latlon[vid[vb + (e + 1) % nvt]]), p);
                        double3 cw = cross3(n1, n2);
                        const double wn = sqrt(dot3(cw, cw));
                        vtx = wn > 0.0 ? scale3(cw, (dot3(cw, ph) < 0.0 ? -1.0 : 1.0) / wn)
                                       : make_double3(vxyz[3 * (vb + e)], vxyz[3 * (vb + e) + 1], vxyz[3 * (vb + e) + 2]);
                        if (e == 0) first = vtx;
                    } else {
                        vtx = first;
                    }
                    if (e > 0) {
                        const double num = dot3(p, cross3(prev, vtx));
                        const double den = 1.0 + dot3(p, prev) + dot3(prev, vtx) + dot3(vtx, p);
                        area += fabs(2.0 * atan2(num, den));
                    }
                    prev = vtx;
                }
                areas[i] = area * radius * radius;
                atomicMax(ctl + 1, (unsigned long long)L);
                atomicAdd(ctl + 2, (unsigned long long)L);
            }
        }
        __syncwarp();
    }
}

// next candidate lists: cand2[off2[t] ..] = the clip-ordered list, then the violators
__global__ void __launch_bounds__(32) k_voronoi_wide_merge(const int32_t* __restrict__ open, int64_t n_open,
                                                           const int64_t* __restrict__ off, const int32_t* __restrict__ sorted,
                                                           const int32_t* __restrict__ grow, const int32_t* __restrict__ fresh,
                                                           const int64_t* __restrict__ off2, int32_t* __restrict__ cand2) {
    for (int64_t w = blockIdx.x; w < n_open; w += gridDim.x) {
        const int t = open[w];
        if (grow[t] == 0) continue;
        const int L = (int)(off[t + 1] - off[t]);
        for (int j = threadIdx.x; j < grow[t]; j += 32)
            cand2[off2[t] + j] = j < L ? sorted[off[t] + j] : fresh[w * VOR_WIDE_NEW + j - L];
    }
}

__global__ void k_voronoi_wide_seed_off(int64_t* off, int64_t m, int k) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t <= m; t += (int64_t)gridDim.x * blockDim.x) off[t] = t * k;
}

// ctl[3] = open cells, ctl[4] = vertices, ctl[5] = candidates: the one read-back of a round
__global__ void k_voronoi_wide_sizes(const int64_t* n_open, const int64_t* voff, const int64_t* off, int64_t m,
                                     unsigned long long* ctl) {
    ctl[3] = (unsigned long long)*n_open;
    ctl[4] = (unsigned long long)voff[m];
    ctl[5] = (unsigned long long)off[m];
}

extern "C" int agx_voronoi_areas_wide(const agx_index_t* index, const float* latlon, int64_t n, const int32_t* wide,
                                      int64_t m, const int32_t* seeds, int k_seed, double radius, double* areas,
                                      int64_t* stats, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n >= 0 && n < (int64_t)2147483647 && m >= 0 && m <= n && k_seed > 0, AGX_ERR_ARG,
                "agx_voronoi_areas_wide: bad sizes");
    AGX_REQUIRE(index && latlon && areas && stats && (m == 0 || (wide && seeds)), AGX_ERR_ARG,
                "agx_voronoi_areas_wide: NULL buffer");
    for (int s = 0; s < 6; ++s) stats[s] = 0;
    if (m == 0) return AGX_OK;
    AGX_REQUIRE(n > VOR_WIDE_K, AGX_ERR_ARG, "agx_voronoi_areas_wide: needs more than %d generators", VOR_WIDE_K);
    const size_t smem = sizeof(VorWideSmem);
    AGX_CUDA_OK(cudaFuncSetAttribute(k_voronoi_wide_clip, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // per-round buffers are (re)allocated to the sizes the round's read-back gives; everything else lives throughout
    unsigned long long* ctl = nullptr;  // [0] failure bits, [1] max and [2] total candidates of final cells, [3..5] sizes, [6] boxed open cells
    int64_t *off = nullptr, *off2 = nullptr, *voff = nullptr, *n_open = nullptr;
    int32_t *open = nullptr, *nv = nullptr, *grow = nullptr, *cand = nullptr, *cand2 = nullptr, *sorted = nullptr;
    int32_t *fresh = nullptr, *vid = nullptr, *nbr = nullptr;
    uint8_t* flag = nullptr;
    double *key = nullptr, *vxyz = nullptr, *nrd = nullptr;
    float2 *vll = nullptr, *q = nullptr;
    int rc = AGX_OK;
    cudaError_t e;
#define WIDE_TRY(expr)                                                              \
    if ((e = (expr)) != cudaSuccess) {                                              \
        agx_set_error("%s failed: %s", #expr, cudaGetErrorString(e));               \
        rc = AGX_ERR_CUDA;                                                          \
        goto done;                                                                  \
    }
#define WIDE_CALL(expr) \
    if ((rc = (expr)) != AGX_OK) goto done;
#define WIDE_FREE(ptr_)                         \
    do {                                        \
        if (ptr_) cudaFreeAsync(ptr_, stream);  \
        ptr_ = nullptr;                         \
    } while (0)
    {
        agx_pool_keep_warm();
        WIDE_TRY(cudaMallocAsync(&ctl, 8 * sizeof(unsigned long long), stream));
        WIDE_TRY(cudaMemsetAsync(ctl, 0, 8 * sizeof(unsigned long long), stream));
        WIDE_TRY(cudaMallocAsync(&off, (m + 1) * sizeof(int64_t), stream));
        WIDE_TRY(cudaMallocAsync(&voff, (m + 1) * sizeof(int64_t), stream));
        WIDE_TRY(cudaMallocAsync(&off2, (m + 1) * sizeof(int64_t), stream));
        WIDE_TRY(cudaMallocAsync(&n_open, sizeof(int64_t), stream));
        WIDE_TRY(cudaMallocAsync(&open, m * sizeof(int32_t), stream));
        WIDE_TRY(cudaMallocAsync(&nv, m * sizeof(int32_t), stream));
        WIDE_TRY(cudaMallocAsync(&grow, m * sizeof(int32_t), stream));
        WIDE_TRY(cudaMallocAsync(&flag, (m + 3) / 4 * 4, stream));
        // round 0: every cell open, its candidates the k_seed entries of its row of the last agx_knn pass
        WIDE_TRY(cudaMemsetAsync(flag, 1, m, stream));
        WIDE_CALL(agx_compact_flags(flag, m, open, n_open, stream));
        WIDE_TRY(cudaMemsetAsync(nv, 0, m * sizeof(int32_t), stream));
        WIDE_TRY(cudaMemsetAsync(grow, 0, m * sizeof(int32_t), stream));
        WIDE_TRY(cudaMallocAsync(&cand, m * (int64_t)k_seed * sizeof(int32_t), stream));
        WIDE_TRY(cudaMemcpyAsync(cand, seeds, m * (int64_t)k_seed * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));
        k_voronoi_wide_seed_off<<<agx_grid(m + 1, 256, 4), 256, 0, stream>>>(off, m, k_seed);
        WIDE_TRY(cudaGetLastError());
        agx_note_launch(1);
        int64_t n_open_h = m, n_cand_h = m * (int64_t)k_seed;
        int round = 0;
        for (;; ++round) {
            // clip the open cells with their lists
            WIDE_TRY(cudaMallocAsync(&key, n_cand_h * sizeof(double), stream));
            WIDE_TRY(cudaMallocAsync(&sorted, n_cand_h * sizeof(int32_t), stream));
            const int64_t slots = n_cand_h + 4 * m;
            WIDE_TRY(cudaMallocAsync(&vxyz, 3 * slots * sizeof(double), stream));
            WIDE_TRY(cudaMallocAsync(&vll, slots * sizeof(float2), stream));
            WIDE_TRY(cudaMallocAsync(&vid, slots * sizeof(int32_t), stream));
            WIDE_TRY(cudaMemsetAsync(nv, 0, m * sizeof(int32_t), stream));
            if (n_open_h > 0) {
                k_voronoi_wide_clip<<<(unsigned)n_open_h, 32, smem, stream>>>((const float2*)latlon, wide, open, n_open, off,
                                                                              cand, key, sorted, vxyz, vll, vid, nv, ctl);
                WIDE_TRY(cudaGetLastError());
                agx_note_launch(1);
            }
            WIDE_CALL(agx_exclusive_scan(nv, m, voff, nullptr, stream));
            k_voronoi_wide_sizes<<<1, 1, 0, stream>>>(n_open, voff, off, m, ctl);
            WIDE_TRY(cudaGetLastError());
            agx_note_launch(1);
            unsigned long long h[7];
            WIDE_CALL(agx_readback(h, ctl, 7, stream));
            n_open_h = (int64_t)h[3];
            n_cand_h = (int64_t)h[5];
            const int64_t n_vert = (int64_t)h[4];
            stats[0] = round;
            stats[1] = n_open_h;
            stats[2] = (int64_t)h[1];
            stats[3] = (int64_t)h[2];
            stats[4] = (int64_t)h[0];
            stats[5] = (int64_t)h[6];
            if (h[0] != 0 || n_open_h == 0 || round == VOR_WIDE_ROUNDS) break;
            // search the vertices, check every (vertex, neighbour) pair
            WIDE_TRY(cudaMallocAsync(&q, (n_vert > 0 ? n_vert : 1) * sizeof(float2), stream));
            WIDE_TRY(cudaMallocAsync(&nbr, (n_vert > 0 ? n_vert : 1) * VOR_WIDE_K * sizeof(int32_t), stream));
            WIDE_TRY(cudaMallocAsync(&nrd, (n_vert > 0 ? n_vert : 1) * VOR_WIDE_K * sizeof(double), stream));
            WIDE_TRY(cudaMallocAsync(&fresh, n_open_h * VOR_WIDE_NEW * sizeof(int32_t), stream));
            const unsigned grid = (unsigned)n_open_h;
            k_voronoi_wide_pack<<<grid, 32, 0, stream>>>(open, n_open_h, off, voff, vll, q);
            WIDE_TRY(cudaGetLastError());
            agx_note_launch(1);
            if (n_vert > 0)
                WIDE_CALL(agx_knn(index, (const float*)q, n_vert, VOR_WIDE_K, 0.0, nbr, nullptr, 0, nrd, nullptr, stream));
            WIDE_TRY(cudaMemsetAsync(flag, 0, m, stream));
            WIDE_TRY(cudaMemsetAsync(ctl + 6, 0, sizeof(unsigned long long), stream));
            WIDE_TRY(cudaMemsetAsync(grow, 0, m * sizeof(int32_t), stream));
            k_voronoi_wide_check<<<grid, 32, 0, stream>>>((const float2*)latlon, wide, open, n_open_h, off, cand, voff, vxyz,
                                                          vid, nbr, nrd, radius, areas, flag, grow, fresh, ctl);
            WIDE_TRY(cudaGetLastError());
            agx_note_launch(1);
            // the lists of the cells that stay open: count (grow), scan, write
            WIDE_CALL(agx_exclusive_scan(grow, m, off2, nullptr, stream));
            WIDE_TRY(cudaMallocAsync(&cand2, (n_cand_h + n_open_h * VOR_WIDE_NEW) * sizeof(int32_t), stream));
            k_voronoi_wide_merge<<<grid, 32, 0, stream>>>(open, n_open_h, off, sorted, grow, fresh, off2, cand2);
            WIDE_TRY(cudaGetLastError());
            agx_note_launch(1);
            WIDE_CALL(agx_compact_flags(flag, m, open, n_open, stream));
            n_cand_h += n_open_h * VOR_WIDE_NEW;  // a bound; the read-back of the next round gives the size
            int64_t* to = off; off = off2; off2 = to;
            WIDE_FREE(cand);
            cand = cand2;
            cand2 = nullptr;
            WIDE_FREE(key); WIDE_FREE(sorted); WIDE_FREE(vxyz); WIDE_FREE(vll); WIDE_FREE(vid);
            WIDE_FREE(q); WIDE_FREE(nbr); WIDE_FREE(nrd); WIDE_FREE(fresh);
        }
    }
done:
    WIDE_FREE(ctl); WIDE_FREE(off); WIDE_FREE(off2); WIDE_FREE(voff); WIDE_FREE(n_open); WIDE_FREE(open);
    WIDE_FREE(nv); WIDE_FREE(grow); WIDE_FREE(flag); WIDE_FREE(cand); WIDE_FREE(cand2); WIDE_FREE(sorted);
    WIDE_FREE(key); WIDE_FREE(vxyz); WIDE_FREE(vll); WIDE_FREE(vid); WIDE_FREE(q); WIDE_FREE(nbr); WIDE_FREE(nrd);
    WIDE_FREE(fresh);
#undef WIDE_TRY
#undef WIDE_CALL
#undef WIDE_FREE
    return rc;
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
