// Hexagonal (H3) hidden mesh: cell centres of a resolution, cell adjacency, and the multi-scale expansion over
// caller-supplied adjacency tables.  Replaces the h3 calls of
// /root/reference/src/anemoi/graphs/generate/hex_icosahedron.py:47,99,136-154 (h3.uncompact(get_res0_indexes),
// h3_to_geo, k_ring, h3_to_center_child).
//
// H3's published geometry (h3lib faceijk.c / coordijk.c / geoCoord.c, H3 3.7): on each of the 20 icosahedron faces
// the cells of resolution r are the points of a hexagonal lattice in the face's gnomonic plane, unit
// RES0_U_GNOMONIC / sqrt(7)^r, rotated asin(sqrt(3/28)) counter-clockwise at odd resolutions; the face's corners
// are lattice points (the 12 pentagons).  A lattice point is tested against the face triangle in exact integer
// arithmetic; a point on an edge / corner shared by several faces is emitted by the lowest-numbered one, so the
// resolution has exactly 2 + 120 * 7^r cells, in (face, i, j) order.  The centre is H3's _hex2dToGeo of the point.
#include "agx_common.cuh"

#include <math.h>

namespace {

constexpr double M_SQRT7_ = 2.6457513110645905905016157536392604257102;
constexpr double M_SQRT3_2_ = 0.8660254037844386467637231707529361834714;
constexpr double M_AP7_ROT_RADS_ = 0.333473172251832115336090755351601070065900389;
constexpr double RES0_U_GNOMONIC_ = 0.38196601125010500003;
constexpr double H3_EPSILON = 0.0000000000000001;
constexpr double M_PI_ = 3.14159265358979323846;
constexpr double M_PI_2_ = 1.5707963267948966;
constexpr double M_2PI_ = 6.28318530717958647692528676655900576839433;
constexpr double M_180_PI_ = 57.29577951308232087679815481410517033240547;  // h3api radsToDegs
constexpr double NPY_DEG2RAD = M_PI_ / 180.0;                                // numpy deg2rad

// faceijk.c faceCenterGeo: (lat, lon) radians of the icosahedron face centres
const double kFaceCenterGeo[20][2] = {
    {0.803582649718989942, 1.248397419617396099},   {1.307747883455638156, 2.536945009877921159},
    {1.054751253523952054, -1.347517358900396623},  {0.600191595538186799, -0.450603909469755746},
    {0.491715428198773866, 0.401988202911306943},   {0.172745327415618701, 1.678146885280433686},
    {0.605929321571350690, 2.953923329812411617},   {0.427370518328979641, -1.888876200336285401},
    {-0.079066118549212831, -0.733429513380867741}, {-0.230961644455383637, 0.506495587332349035},
    {0.079066118549212831, 2.408163140208925497},   {0.230961644455383637, -2.635097066257444203},
    {-0.172745327415618701, -1.463445768309359553}, {-0.605929321571350690, -0.187669323777381622},
    {-0.427370518328979641, 1.252716453253507838},  {-0.600191595538186799, 2.690988744120037492},
    {-0.491715428198773866, -2.739604450678486295}, {-0.803582649718989942, -1.893195233972397139},
    {-1.307747883455638156, -0.604647643711872080}, {-1.054751253523952054, 1.794075294689396615},
};

// faceijk.c faceAxesAzRadsCII: azimuth of the Class II i, j, k axes at each face centre
const double kFaceAxesAz[20][3] = {
    {5.619958268523939882, 3.525563166130744542, 1.431168063737548730},
    {5.760339081714187279, 3.665943979320991689, 1.571548876927796127},
    {0.780213654393430055, 4.969003859179821079, 2.874608756786625655},
    {0.430469363979999913, 4.619259568766391033, 2.524864466373195467},
    {6.130269123335111400, 4.035874020941915804, 1.941478918548720291},
    {2.692877706530642877, 0.598482604137447119, 4.787272808923838195},
    {2.982963003477243874, 0.888567901084048369, 5.077358105870439581},
    {3.532912002790141181, 1.438516900396945656, 5.627307105183336758},
    {3.494305004259568154, 1.399909901866372864, 5.588700106652763840},
    {3.003214169499538391, 0.908819067106342928, 5.097609271892733906},
    {5.930472956509811562, 3.836077854116615875, 1.741682751723420374},
    {0.138378484090254847, 4.327168688876645809, 2.232773586483450311},
    {0.448714947059150361, 4.637505151845541521, 2.543110049452346120},
    {0.158629650112549365, 4.347419854898940135, 2.253024752505744869},
    {5.891865957979238535, 3.797470855586042958, 1.703075753192847583},
    {2.711123289609793325, 0.616728187216597771, 4.805518392002988683},
    {3.294508837434268316, 1.200113735041072948, 5.388903939827463911},
    {3.804819692245439833, 1.710424589852244509, 5.899214794638635174},
    {3.664438879055192436, 1.570043776661997111, 5.758833981448388027},
    {2.361378999196363184, 0.266983896803167583, 4.455774101589558636},
};

struct HexPlan {
    double clat[20], clon[20], az0[20];
    int corner_owner[20][3];  // lowest face holding corner k of the face
    int edge_owner[20][3];    // lowest face holding edge k (corner k -> corner k+1)
    long long v[3][2];        // lattice coordinates (i, j; k = 0) of the three corners at this resolution
    long long lo[2];          // bounding box of the triangle
    long long w, h;           // box extent along i and j
    int res;
};

__host__ __device__ inline double h3_pos_angle(double a) {
    double t = a < 0.0 ? a + M_2PI_ : a;
    if (a >= M_2PI_) t -= M_2PI_;
    return t;
}

__host__ __device__ inline double h3_constrain_lng(double lng) {
    while (lng > M_PI_) lng = lng - M_2PI_;
    while (lng < -M_PI_) lng = lng + M_2PI_;
    return lng;
}

// geoCoord.c _geoAzDistanceRads
__host__ __device__ inline void h3_geo_az_distance(double lat1, double lon1, double az, double distance, double& lat2,
                                                   double& lon2) {
    if (distance < H3_EPSILON) {
        lat2 = lat1;
        lon2 = lon1;
        return;
    }
    az = h3_pos_angle(az);
    if (az < H3_EPSILON || fabs(az - M_PI_) < H3_EPSILON) {  // due north or south
        lat2 = az < H3_EPSILON ? lat1 + distance : lat1 - distance;
        if (fabs(lat2 - M_PI_2_) < H3_EPSILON) {
            lat2 = M_PI_2_;
            lon2 = 0.0;
        } else if (fabs(lat2 + M_PI_2_) < H3_EPSILON) {
            lat2 = -M_PI_2_;
            lon2 = 0.0;
        } else {
            lon2 = h3_constrain_lng(lon1);
        }
        return;
    }
    double sinlat = sin(lat1) * cos(distance) + cos(lat1) * sin(distance) * cos(az);
    if (sinlat > 1.0) sinlat = 1.0;
    if (sinlat < -1.0) sinlat = -1.0;
    lat2 = asin(sinlat);
    if (fabs(lat2 - M_PI_2_) < H3_EPSILON) {
        lat2 = M_PI_2_;
        lon2 = 0.0;
    } else if (fabs(lat2 + M_PI_2_) < H3_EPSILON) {
        lat2 = -M_PI_2_;
        lon2 = 0.0;
    } else {
        double sinlon = sin(az) * sin(distance) / cos(lat2);
        double coslon = (cos(distance) - sin(lat1) * sin(lat2)) / cos(lat1) / cos(lat2);
        if (sinlon > 1.0) sinlon = 1.0;
        if (sinlon < -1.0) sinlon = -1.0;
        if (coslon > 1.0) coslon = 1.0;
        if (coslon < -1.0) coslon = -1.0;
        lon2 = h3_constrain_lng(lon1 + atan2(sinlon, coslon));
    }
}

// membership of lattice point (a, b) in the cell set of `face`: inside or on the triangle, and owned by this face
__device__ __forceinline__ bool hex_keep(const HexPlan& p, int face, long long a, long long b, bool& pentagon) {
    long long c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int k1 = (k + 1) % 3;
        long long ex = p.v[k1][0] - p.v[k][0], ey = p.v[k1][1] - p.v[k][1];
        c[k] = ex * (b - p.v[k][1]) - ey * (a - p.v[k][0]);
    }
    pentagon = false;
    if (c[0] < 0 || c[1] < 0 || c[2] < 0) return false;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (c[k] == 0 && c[(k + 2) % 3] == 0) {  // corner k: the meeting point of edges k and k-1
            pentagon = true;
            return p.corner_owner[face][k] == face;
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k)
        if (c[k] == 0) return p.edge_owner[face][k] == face;
    return true;
}

__global__ void k_hex_flags(HexPlan p, int64_t n_cand, int32_t* __restrict__ flags) {
    const long long per_face = p.w * p.h;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cand; i += (int64_t)gridDim.x * blockDim.x) {
        int face = (int)(i / per_face);
        long long rem = i - face * per_face;
        long long a = p.lo[0] + rem / p.h, b = p.lo[1] + rem % p.h;
        bool pent;
        flags[i] = hex_keep(p, face, a, b, pent) ? 1 : 0;
    }
}

// faceijk.c _hex2dToGeo (substrate = 0) of the kept lattice points; h3_to_geo's degrees and numpy's deg2rad on top
// (generate/hex_icosahedron.py:47) so the float64 value is the one the reference sorts and rounds to float32.
__global__ void k_hex_centres(HexPlan p, int64_t n_cand, const int32_t* __restrict__ flags,
                              const int64_t* __restrict__ offsets, double2* __restrict__ latlon,
                              uint8_t* __restrict__ pentagon) {
    const long long per_face = p.w * p.h;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cand; i += (int64_t)gridDim.x * blockDim.x) {
        if (!flags[i]) continue;
        int face = (int)(i / per_face);
        long long rem = i - face * per_face;
        long long a = p.lo[0] + rem / p.h, b = p.lo[1] + rem % p.h;
        bool pent;
        hex_keep(p, face, a, b, pent);
        // coordijk.c _ijkToHex2d with k = 0
        double x = (double)a - 0.5 * (double)b;
        double y = (double)b * M_SQRT3_2_;
        double r = sqrt(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)));
        double lat, lon;
        if (r < H3_EPSILON) {
            lat = p.clat[face];
            lon = p.clon[face];
        } else {
            double theta = atan2(y, x);
            for (int l = 0; l < p.res; ++l) r /= M_SQRT7_;
            r *= RES0_U_GNOMONIC_;
            r = atan(r);
            if (p.res & 1) theta = h3_pos_angle(theta + M_AP7_ROT_RADS_);
            theta = h3_pos_angle(p.az0[face] - theta);
            h3_geo_az_distance(p.clat[face], p.clon[face], theta, r, lat, lon);
        }
        int64_t o = offsets[i];
        latlon[o] = make_double2(__dmul_rn(__dmul_rn(lat, M_180_PI_), NPY_DEG2RAD),
                                 __dmul_rn(__dmul_rn(lon, M_180_PI_), NPY_DEG2RAD));
        if (pentagon) pentagon[o] = pent ? 1 : 0;
    }
}

// neighbour table of one level from a k = 7 self query: the 6 nearest other cells (5 for a pentagon)
__global__ void k_hex_adjacency(const int32_t* __restrict__ knn7, const uint8_t* __restrict__ pentagon, int64_t n,
                                int32_t* __restrict__ nb, int* __restrict__ deg) {
    for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < n; u += (int64_t)gridDim.x * blockDim.x) {
        int want = pentagon[u] ? 5 : 6, m = 0;
        for (int j = 0; j < 7; ++j) {
            int v = knn7[7 * u + j];
            if (v == (int)u || v < 0 || m >= want) continue;
            nb[6 * u + m++] = v;
        }
        deg[u] = m;
        for (; m < 6; ++m) nb[6 * u + m] = -1;
    }
}

void xyz_of(double lat, double lon, double* o) {
    o[0] = cos(lat) * cos(lon);
    o[1] = cos(lat) * sin(lon);
    o[2] = sin(lat);
}

// corner / edge ownership from the geometry of the tables (no hand-written adjacency list to get wrong)
void hex_plan(int res, HexPlan& p) {
    double corner_xyz[20][3][3];
    const double dist = atan(2.0 * RES0_U_GNOMONIC_);  // face centre -> corner
    for (int f = 0; f < 20; ++f) {
        p.clat[f] = kFaceCenterGeo[f][0];
        p.clon[f] = kFaceCenterGeo[f][1];
        p.az0[f] = kFaceAxesAz[f][0];
        for (int k = 0; k < 3; ++k) {
            double lat, lon;
            h3_geo_az_distance(p.clat[f], p.clon[f], kFaceAxesAz[f][k], dist, lat, lon);
            xyz_of(lat, lon, corner_xyz[f][k]);
        }
    }
    auto same = [&](int f, int k, int g, int m) {
        double d = 0;
        for (int c = 0; c < 3; ++c) d += (corner_xyz[f][k][c] - corner_xyz[g][m][c]) * (corner_xyz[f][k][c] - corner_xyz[g][m][c]);
        return d < 1e-18;
    };
    auto has = [&](int g, int f, int k) { return same(f, k, g, 0) || same(f, k, g, 1) || same(f, k, g, 2); };
    for (int f = 0; f < 20; ++f)
        for (int k = 0; k < 3; ++k) {
            int co = f, eo = f;
            for (int g = 19; g >= 0; --g) {
                if (has(g, f, k)) co = g;
                if (has(g, f, k) && has(g, f, (k + 1) % 3)) eo = g;
            }
            p.corner_owner[f][k] = co;
            p.edge_owner[f][k] = eo;
        }
    // corners: res 0 has them two units out on the i, j, k axes; every finer level applies coordijk.c _downAp7
    // (odd levels, counter-clockwise: i -> (3,0,1), j -> (1,3,0)) or _downAp7r (even, clockwise: i -> (3,1,0), j -> (0,3,1))
    long long v[3][2] = {{2, 0}, {0, 2}, {-2, -2}};
    for (int level = 1; level <= res; ++level) {
        long long iv[2], jv[2];
        if (level & 1) { iv[0] = 2; iv[1] = -1; jv[0] = 1; jv[1] = 3; }
        else { iv[0] = 3; iv[1] = 1; jv[0] = -1; jv[1] = 2; }
        for (int k = 0; k < 3; ++k) {
            long long a = v[k][0], b = v[k][1];
            v[k][0] = a * iv[0] + b * jv[0];
            v[k][1] = a * iv[1] + b * jv[1];
        }
    }
    long long hi[2];
    for (int c = 0; c < 2; ++c) {
        p.lo[c] = hi[c] = v[0][c];
        for (int k = 0; k < 3; ++k) {
            p.v[k][c] = v[k][c];
            if (v[k][c] < p.lo[c]) p.lo[c] = v[k][c];
            if (v[k][c] > hi[c]) hi[c] = v[k][c];
        }
    }
    p.w = hi[0] - p.lo[0] + 1;
    p.h = hi[1] - p.lo[1] + 1;
    p.res = res;
}

}  // namespace

#define HEX_MAX_RES 8 /* 691 M cells; int32 node indices and the 180 GB of one GPU end here */

extern "C" int64_t agx_hex_num_cells(int res) {
    if (res < 0 || res > 15) return -1;
    int64_t n = 120;
    for (int i = 0; i < res; ++i) n *= 7;
    return n + 2;
}

extern "C" int agx_hex_cells(int res, double* latlon, uint8_t* pentagon, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(res >= 0 && res <= 15, AGX_ERR_ARG, "agx_hex_cells: H3 resolutions are 0..15, got %d", res);
    AGX_REQUIRE(res <= HEX_MAX_RES, AGX_ERR_UNSUPPORTED, "agx_hex_cells: resolution %d > %d is not built (%lld cells)", res,
                HEX_MAX_RES, (long long)agx_hex_num_cells(res));
    AGX_REQUIRE(latlon != nullptr, AGX_ERR_ARG, "agx_hex_cells: latlon is NULL");
    HexPlan plan;
    hex_plan(res, plan);
    const int64_t n_cand = 20 * plan.w * plan.h;
    agx_pool_keep_warm();
    int32_t* flags = nullptr;
    int64_t* offsets = nullptr;
    AGX_CUDA_OK(cudaMallocAsync(&flags, n_cand * sizeof(int32_t), stream));
    AGX_CUDA_OK(cudaMallocAsync(&offsets, (n_cand + 1) * sizeof(int64_t), stream));
    k_hex_flags<<<agx_grid(n_cand, 256, 8), 256, 0, stream>>>(plan, n_cand, flags);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    int64_t total = 0;
    int rc = agx_exclusive_scan(flags, n_cand, offsets, &total, stream);
    if (rc == AGX_OK && total != agx_hex_num_cells(res)) {
        agx_set_error("agx_hex_cells: resolution %d produced %lld cells, H3 has %lld", res, (long long)total,
                      (long long)agx_hex_num_cells(res));
        rc = AGX_ERR_OVERFLOW;
    }
    if (rc == AGX_OK) {
        k_hex_centres<<<agx_grid(n_cand, 256, 8), 256, 0, stream>>>(plan, n_cand, flags, offsets, (double2*)latlon, pentagon);
        if (cudaGetLastError() != cudaSuccess) {
            agx_set_error("agx_hex_cells: kernel launch failed");
            rc = AGX_ERR_CUDA;
        }
        agx_note_launch(1);
    }
    cudaFreeAsync(flags, stream);
    cudaFreeAsync(offsets, stream);
    return rc;
}

extern "C" int agx_hex_adjacency(const int32_t* knn7, const uint8_t* pentagon, int64_t n, int32_t* nb, int32_t* deg,
                                 void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n >= 0, AGX_ERR_ARG, "agx_hex_adjacency: n < 0");
    if (n == 0) return AGX_OK;
    AGX_REQUIRE(knn7 && pentagon && nb && deg, AGX_ERR_ARG, "agx_hex_adjacency: NULL buffer");
    k_hex_adjacency<<<agx_grid(n, 256, 8), 256, 0, stream>>>(knn7, pentagon, n, nb, deg);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

// ------------------------------------------------------------------------------------------------
// HEALPix nodes: hp.pix2ang(nside, range(npix), nest=True, lonlat=True) + reshape_coords
// (/root/reference/src/anemoi/graphs/nodes/builders/from_healpix.py:61-66, nodes/builders/base.py:84-101).
// HEALPix's published pix2loc for the NESTED scheme (healpix_cxx healpix_base.cc): face = pix >> 2*order, (ix, iy) =
// the even / odd bits of the rest, ring jr = jrll[face]*nside - ix - iy - 1, z and phi from the polar-cap or
// equatorial formulas; theta = atan2(sin theta, z) where the library carries sin theta (|z| > 0.99), acos(z) else;
// healpy's degrees (lon = degrees(phi), lat = 90 - degrees(theta)), numpy's deg2rad, one rounding to float32.
// ------------------------------------------------------------------------------------------------
namespace {
__device__ __forceinline__ unsigned hp_compress_bits(unsigned long long v) {
    v &= 0x5555555555555555ull;
    v = (v | (v >> 1)) & 0x3333333333333333ull;
    v = (v | (v >> 2)) & 0x0f0f0f0f0f0f0f0full;
    v = (v | (v >> 4)) & 0x00ff00ff00ff00ffull;
    v = (v | (v >> 8)) & 0x0000ffff0000ffffull;
    v = (v | (v >> 16)) & 0x00000000ffffffffull;
    return (unsigned)v;
}

__global__ void k_healpix_nodes(int order, int64_t npix, float2* __restrict__ latlon) {
    const int jrll[12] = {2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4};
    const int jpll[12] = {1, 3, 5, 7, 0, 2, 4, 6, 1, 3, 5, 7};
    const long long nside = 1ll << order;
    const double halfpi = 1.570796326794896619231321691639751442099;
    const double fact2 = 4.0 / (double)npix;
    const double fact1 = (double)(nside << 1) * fact2;
    for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < npix; pix += (int64_t)gridDim.x * blockDim.x) {
        const int face = (int)(pix >> (2 * order));
        const unsigned long long p = (unsigned long long)pix & (unsigned long long)(nside * nside - 1);
        const long long ix = hp_compress_bits(p), iy = hp_compress_bits(p >> 1);
        const long long jr = ((long long)jrll[face] << order) - ix - iy - 1;
        long long nr;
        double z, sth = 0.0;
        bool have_sth = false;
        if (jr < nside) {
            nr = jr;
            double tmp = (double)(nr * nr) * fact2;
            z = 1.0 - tmp;
            if (z > 0.99) { sth = sqrt(tmp * (2.0 - tmp)); have_sth = true; }
        } else if (jr > 3 * nside) {
            nr = nside * 4 - jr;
            double tmp = (double)(nr * nr) * fact2;
            z = tmp - 1.0;
            if (z < -0.99) { sth = sqrt(tmp * (2.0 - tmp)); have_sth = true; }
        } else {
            nr = nside;
            z = (double)(2 * nside - jr) * fact1;
        }
        long long t = (long long)jpll[face] * nr + ix - iy;
        if (t < 0) t += 8 * nr;
        const double phi = (nr == nside) ? 0.75 * halfpi * (double)t * fact1 : (0.5 * halfpi * (double)t) / (double)nr;
        const double theta = have_sth ? atan2(sth, z) : acos(z);
        // healpy lonlat: np.degrees = x * (180 / pi); reference: np.deg2rad = x * (pi / 180)
        const double lon_deg = __dmul_rn(phi, 180.0 / M_PI_), lat_deg = 90.0 - __dmul_rn(theta, 180.0 / M_PI_);
        latlon[pix] = make_float2((float)__dmul_rn(lat_deg, M_PI_ / 180.0), (float)__dmul_rn(lon_deg, M_PI_ / 180.0));
    }
}
}  // namespace

extern "C" int agx_healpix_nodes(int order, float* latlon, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(order >= 0 && order <= 13, AGX_ERR_ARG, "agx_healpix_nodes: resolution (log2 nside) must be in 0..13, got %d", order);
    AGX_REQUIRE(latlon != nullptr, AGX_ERR_ARG, "agx_healpix_nodes: latlon is NULL");
    const int64_t npix = 12ll << (2 * order);
    k_healpix_nodes<<<agx_grid(npix, 256, 8), 256, 0, stream>>>(order, npix, (float2*)latlon);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

// ------------------------------------------------------------------------------------------------
// Octahedral reduced Gaussian grid O<n> (ReducedGaussianGridNodes of newer releases, grids.octahedral_grid): the 2n
// Gaussian latitudes are the roots of the Legendre polynomial P_2n; row i (1-based from the nearer pole) holds 4i + 16
// points at longitudes j * 360 / (4i + 16).
// ------------------------------------------------------------------------------------------------
namespace {
constexpr double PIO2_HI = 1.5707963267948966;      // fl(pi / 2)
constexpr double PIO2_LO = 6.123233995736766e-17;   // pi / 2 - PIO2_HI
constexpr double RAD2DEG = 180.0 / M_PI_;           // numpy rad2deg

// One thread per northern root k: Newton on f(theta) = P_m(cos theta), m = 2n, from Tricomi's guess
// theta = pi (k + 3/4) / (m + 1/2) (k counted from 0).  P_m is evaluated through y = 1 - cos theta = 2 sin^2(theta/2) and
// the differences D_j = P_j - P_{j-1} (j D_j = (j-1) D_{j-1} - (2j-1) y P_{j-1}): near the pole cos theta rounds away
// most of theta (1 ulp of x is 1e-13 rad at O1280's first row), y keeps it, so the roots are good to 1e-14 degrees at
// every row.  df/dtheta = m (x P_m - P_{m-1}) / sin theta, with x P_m - P_{m-1} = D_m - y P_m.  The loop stops after a
// step below 1e-11: Newton's error after it is cot(theta) / 2 * step^2 < 1e-17.
__global__ void k_gaussian_latitudes(int n, double* __restrict__ lat_deg) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int m = 2 * n;
    double theta = M_PI_ * ((double)k + 0.75) / ((double)m + 0.5);
    for (int it = 0; it < 32; ++it) {
        const double h = sin(0.5 * theta);
        const double y = 2.0 * h * h;
        double p = 1.0 - y, d = -y;  // P_1, D_1
#pragma unroll 4
        for (int j = 2; j <= m; ++j) {
            const double r = __drcp_rn((double)j);
            d = fma(1.0 - r, d, -((2.0 - r) * y) * p);
            p += d;
        }
        const double step = p * sin(theta) / ((double)m * (d - y * p));
        theta -= step;
        if (fabs(step) < 1e-11) break;
    }
    const double lat = __dmul_rn(__dadd_rn(__dsub_rn(PIO2_HI, theta), PIO2_LO), RAD2DEG);
    lat_deg[k] = lat;
    lat_deg[m - 1 - k] = -lat;
}

// One point per thread.  q = the position counted from the nearer pole (from the last point in the southern half);
// row r (0-based from that pole) starts at 2r(r + 9), so r is the largest with (2r + 9)^2 <= 2q + 81: an exact integer
// square root (the double sqrt of an integer < 2^34, corrected by one either way).  Roundings as the oracle's:
// lon = j * fl(360 / count), then numpy's deg2rad and one rounding to float32.
__global__ void k_octahedral_nodes(int n, int64_t half, const double* __restrict__ lat_deg, float2* __restrict__ latlon) {
    const int64_t total = 2 * half;
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
        const bool south = p >= half;
        const int64_t q = south ? total - 1 - p : p;
        const int64_t v = 2 * q + 81;
        int64_t s = (int64_t)sqrt((double)v);
        if (s * s > v) --s;
        if ((s + 1) * (s + 1) <= v) ++s;
        const int64_t r = (s - 9) >> 1;
        const int64_t count = 4 * r + 20;
        int64_t j = q - 2 * r * (r + 9);
        if (south) j = count - 1 - j;
        const double lat = lat_deg[south ? 2 * n - 1 - r : r];
        const double lon = __dmul_rn((double)j, 360.0 / (double)count);
        latlon[p] = make_float2((float)__dmul_rn(lat, NPY_DEG2RAD), (float)__dmul_rn(lon, NPY_DEG2RAD));
    }
}

int octahedral_args(const char* fn, int n) {
    AGX_REQUIRE(n >= 1, AGX_ERR_ARG, "%s: the grid number must be >= 1, got %d", fn, n);
    AGX_REQUIRE(4ll * n * (n + 9ll) <= INT32_MAX, AGX_ERR_ARG, "%s: O%d has %lld points, more than int32 node indices hold",
                fn, n, 4ll * n * (n + 9ll));
    return AGX_OK;
}
}  // namespace

extern "C" int agx_gaussian_latitudes(int n, double* lat_deg, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int rc = octahedral_args("agx_gaussian_latitudes", n);
    if (rc != AGX_OK) return rc;
    AGX_REQUIRE(lat_deg != nullptr, AGX_ERR_ARG, "agx_gaussian_latitudes: lat_deg is NULL");
    k_gaussian_latitudes<<<(n + 31) / 32, 32, 0, stream>>>(n, lat_deg);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

extern "C" int agx_octahedral_nodes(int n, const double* lat_deg, float* latlon, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int rc = octahedral_args("agx_octahedral_nodes", n);
    if (rc != AGX_OK) return rc;
    AGX_REQUIRE(lat_deg != nullptr && latlon != nullptr, AGX_ERR_ARG, "agx_octahedral_nodes: NULL buffer");
    const int64_t half = 2ll * n * (n + 9);
    k_octahedral_nodes<<<agx_grid(2 * half, 256, 8), 256, 0, stream>>>(n, half, lat_deg, (float2*)latlon);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}
