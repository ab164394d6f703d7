// K5: fused edge attributes (EdgeLength + EdgeDirection) with global normalisation.
//
// Replaces EdgeLength.compute / EdgeDirection.compute
// (/root/reference/src/anemoi/graphs/edges/attributes.py:42-157; utils.py:84-103;
// edges/directional.py:19-94; generate/transforms.py:91-140; normalise.py:20-55).
//
// Arithmetic follows the reference stage by stage:
//  * float32 stage (numpy): latlon -> xyz and the haversine `a` term use numpy's float32 sin/cos
//    reproduced bit for bit (agx_np_sincosf) with un-fused float32 multiplies/adds.
//  * float64 stage (numpy/scipy): cross products, arccos, scipy Rotation.from_rotvec (small-angle
//    series for angle <= 1e-3), as_matrix, apply, the two epsilon nudges of direction_vec.
// Everything that depends on ONE node only (xyz, cos lat, the rotation quaternion of a target) is either
//  * tabulated per node in ONE 32-byte record per role (small node sets - the hidden mesh - whose tables stay in L2):
//      source record  float[8]  = (x, y, z, cos lat, lat, lon, 0, 0)
//      target record  double[4] = (quat x, quat y, quat w, bits(lat, lon))   (quat z is exactly 0)
//  * or evaluated per edge from the node's 8-byte (lat, lon) (large node sets - the data grid: a table would cost
//    32 B written + 32 B gathered per node where the coordinates cost 8 B; the quaternion needs no trigonometry).
// The per-edge kernel works on warp tiles of 64 consecutive edges, two ADJACENT edges per lane: 8-byte index loads,
// all node gathers in flight before the arithmetic, one 8-byte (length) and one 128-bit (direction) store per lane.
#include "agx_common.cuh"

#define ATTR_THREADS 256
#define ATTR_MAX_BLOCKS 4096
#define ATTR_STAT_FIELDS 8  // len: sum, sumsq, min, max; dir: sum, sumsq, min, max
#define AGX_ATTR_FLAGS_SKIP 1
#define AGX_ATTR_FLAGS_ONLY 2

extern "C" int64_t agx_edge_attrs_workspace(void) { return (int64_t)ATTR_STAT_FIELDS * (ATTR_MAX_BLOCKS + 2); }

// ------------------------------------------------------------------------------------------------
// per-node quantities: tabulated (small node sets: the tables stay in L2) or evaluated per edge from the 8-byte
// coordinates (large node sets: a table would be written once, 32 bytes per node, and gathered back sector by sector)
// ------------------------------------------------------------------------------------------------
struct SrcNode {  // a node as an edge SOURCE
    float x, y, z, cl;  // latlon_rad_to_cartesian (generate/transforms.py:106-110) in numpy's float32 bits, cos(lat)
    float lat, lon;
};
struct DstNode {  // a node as an edge TARGET
    double qx, qy, qw;  // rotation to the north pole as a unit quaternion (x, y, 0, w)
    float lat, lon;
};

__device__ __forceinline__ SrcNode agx_src_node(float2 ll) {
    SrcNode n;
    float sl, so, co;
    agx_np_sincosf(ll.x, sl, n.cl);
    agx_np_sincosf(ll.y, so, co);
    n.x = __fmul_rn(n.cl, co);
    n.y = __fmul_rn(n.cl, so);
    n.z = sl;
    n.lat = ll.x;
    n.lon = ll.y;
    return n;
}

// get_rotation_from_unit_vecs(points = this node as TARGET, reference = (0, 0, 1)) (edges/directional.py:19-37):
// axis u = direction_vec(p, z^) = (p_y, -p_x, 0) / |.| in float64 from the float32 components - with the float32
// in-place nudge of all three components when |v|^2 < 1e-10 (generate/transforms.py:135-139) -, angle
// theta = arccos(p_z), scipy Rotation.from_rotvec(u theta) = quaternion (u sin(theta/2), cos(theta/2)).  The half-angle
// functions of arccos(p_z) are algebraic: sin(theta/2) = sqrt((1 - p_z)/2), cos(theta/2) = sqrt((1 + p_z)/2) - both
// differences are exact in float64 for a float32 p_z - so no inverse or forward trigonometry is evaluated at all; the
// result agrees with scipy's (arccos, then sin / cos or its small-angle series, _rotation_xp.py:159-179) to ~1e-16
// absolute, four orders below what the float32 attributes resolve.
__device__ __forceinline__ void agx_target_quat(float x, float y, float z, double& qx, double& qy, double& qw) {
    double v0 = (double)y, v1 = -(double)x;
    double vn = __dadd_rn(__dmul_rn(v0, v0), __dmul_rn(v1, v1));
    float pz = z;
    if (vn < 10e-11) {
        const float eps32 = (float)10e-11;
        float xn = __fadd_rn(x, eps32), yn = __fadd_rn(y, eps32);
        pz = __fadd_rn(z, eps32);
        v0 = (double)yn;
        v1 = -(double)xn;
        vn = __dadd_rn(__dmul_rn(v0, v0), __dmul_rn(v1, v1));
    }
    const double inv = rsqrt(vn);
    const double p = fmin(fmax((double)pz, -1.0), 1.0);
    const double sh = sqrt(0.5 * (1.0 - p)), ch = sqrt(0.5 * (1.0 + p));
    qx = v0 * inv * sh;
    qy = v1 * inv * sh;
    qw = ch;
}

__device__ __forceinline__ DstNode agx_dst_node(float2 ll, bool want_quat) {
    DstNode n;
    n.lat = ll.x;
    n.lon = ll.y;
    n.qx = n.qy = 0.0;
    n.qw = 1.0;
    if (want_quat) {
        SrcNode s = agx_src_node(ll);
        agx_target_quat(s.x, s.y, s.z, n.qx, n.qy, n.qw);
    }
    return n;
}

__global__ void __launch_bounds__(256) k_node_tables(const float2* __restrict__ latlon, int64_t n,
                                                      float4* __restrict__ src_rec, double4* __restrict__ dst_rec) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float2 ll = latlon[i];
        const SrcNode sn = agx_src_node(ll);
        if (src_rec != nullptr) {
            src_rec[2 * i] = make_float4(sn.x, sn.y, sn.z, sn.cl);
            src_rec[2 * i + 1] = make_float4(ll.x, ll.y, 0.0f, 0.0f);
        }
        if (dst_rec != nullptr) {
            double qx, qy, qw;
            agx_target_quat(sn.x, sn.y, sn.z, qx, qy, qw);
            long long packed = ((long long)__float_as_int(ll.y) << 32) | (unsigned int)__float_as_int(ll.x);
            dst_rec[i] = make_double4(qx, qy, qw, __longlong_as_double(packed));
        }
    }
}

extern "C" int agx_node_tables(const float* latlon, int64_t n, float* src_rec, double* dst_rec, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n >= 0, AGX_ERR_ARG, "agx_node_tables: n < 0");
    if (n == 0) return AGX_OK;
    AGX_REQUIRE(latlon && (src_rec || dst_rec), AGX_ERR_ARG, "agx_node_tables: NULL buffer");
    AGX_REQUIRE(((uintptr_t)src_rec & 15) == 0 && ((uintptr_t)dst_rec & 31) == 0, AGX_ERR_ARG,
                "agx_node_tables: records must be 16-byte (source) / 32-byte (target) aligned");
    int grid = agx_grid(n, 256, 8);
    k_node_tables<<<grid, 256, 0, stream>>>((const float2*)latlon, n, (float4*)src_rec, (double4*)dst_rec);
    AGX_LAUNCH_OK();
    agx_note_launch(1);
    return AGX_OK;
}

// ------------------------------------------------------------------------------------------------
// per-edge raw values
// ------------------------------------------------------------------------------------------------
// atan2(ra, rb) for ra, rb >= 0 in float64.  Edges are short, so ra/rb = tan(d/2) is tiny: below 1/16 the odd
// Taylor series to t^11 is exact to < 3e-16 relative (next term t^12/13) and costs a handful of DFMAs instead of
// the library's ~150-instruction path.  The quotient uses a float reciprocal seed + two Newton steps (1e-14
// relative); the result is rounded to float32 by the caller, so this cannot be told from the exact quotient.
__device__ __forceinline__ double atan2_short(float ra32, float rb32) {
    double ra = (double)ra32, rb = (double)rb32;
    if (ra <= 0.0625 * rb) {
        float seed;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(seed) : "f"(rb32));  // 2^-23 relative; two Newton steps -> 2^-90
        double r = (double)seed;
        r = r * (2.0 - rb * r);
        r = r * (2.0 - rb * r);
        double t = ra * r, t2 = t * t;
        double p = fma(t2, -1.0 / 11.0, 1.0 / 9.0);
        p = fma(t2, -p, 1.0 / 7.0);
        p = fma(t2, -p, 1.0 / 5.0);
        p = fma(t2, -p, 1.0 / 3.0);
        p = fma(t2, -p, 1.0);
        return t * p;
    }
    return atan2(ra, rb);  // long edges, and NaN (a > 1 in float32: antipodal pairs, as in the reference)
}

// utils.haversine_distance in float32 (numpy), last step in float64 then rounded (see DESIGN.md).
__device__ __forceinline__ float edge_length_raw(float2 s, float cs, float2 t, float ct) {
    float dlat = __fsub_rn(t.x, s.x), dlon = __fsub_rn(t.y, s.y);
    float sh_lat = agx_np_sinf_short(__fmul_rn(dlat, 0.5f));
    float sh_lon = agx_np_sinf_short(__fmul_rn(dlon, 0.5f));
    float a = __fadd_rn(__fmul_rn(sh_lat, sh_lat), __fmul_rn(__fmul_rn(cs, ct), __fmul_rn(sh_lon, sh_lon)));
    float ra = __fsqrt_rn(a), rb = __fsqrt_rn(__fsub_rn(1.0f, a));
    return __fmul_rn(2.0f, (float)atan2_short(ra, rb));
}

// compute_directions (edges/directional.py:40-65) for one edge; q = R(target) * source_xyz.
// For the unit quaternion (x, y, 0, w) scipy's as_matrix rows 0 and 1 are (1 - 2y^2, 2xy, 2yw) and
// (2xy, 1 - 2x^2, -2xw) (it writes them as x^2 - y^2 + w^2 etc., equal to 1e-16), so with
// T = x s_y - y s_x + w s_z:  q_x = s_x + 2 y T,  q_y = s_y - 2 x T  - seven float64 operations.  For nearby
// endpoints q_x, q_y are O(separation) differences of O(1) terms; each rounding is <= 1.1e-16 absolute, i.e.
// <= 1e-12 relative at the shortest edges of an O1280 graph (separation 1e-3).
__device__ __forceinline__ void edge_direction_rotated(float4 sxyz, double x, double y, double w, double& o0, double& o1) {
    double sx = (double)sxyz.x, sy = (double)sxyz.y, sz = (double)sxyz.z;
    double T2 = 2.0 * fma(x, sy, fma(-y, sx, w * sz));
    double qx = fma(y, T2, sx);
    double qy = fma(-x, T2, sy);
    // direction_vec(q, z^): v = (q_y, -q_x, 0); nudge in float64 when |v|^2 < 1e-10
    double vn = fma(qy, qy, qx * qx);
    if (vn < 10e-11) {
        qx += 10e-11;
        qy += 10e-11;
        vn = fma(qy, qy, qx * qx);
    }
    // v / |v|; the reference normalises once more (edges/directional.py:65), which moves a unit vector by at most
    // an ulp of float64 - invisible after the float32 cast.  NaN inputs propagate as they do there.
    double inv = rsqrt(vn);
    o0 = qy * inv;
    o1 = -qx * inv;
}

// Running statistics of one attribute.  Sums are float64 (the reference reduces a float64 array for directions and
// numpy's pairwise float32 sum for lengths - both within 1e-7 of this).  Minimum / maximum are tracked on the
// float32 value that is stored, one FMNMX each: for lengths that IS the reference's value; for rotated directions
// the reference takes them on the float64 array, whose float32 rounding differs by <= 6e-8 relative.
struct Stat4 {
    double sum, sumsq;
    float mn, mx;
    __device__ __forceinline__ void init() {
        sum = 0.0;
        sumsq = 0.0;
        mn = __int_as_float(0x7f800000);
        mx = __int_as_float(0xff800000);
    }
    __device__ __forceinline__ void add(double v, float v32) {
        sum += v;
        sumsq = fma(v, v, sumsq);
        mn = fminf(mn, v32);
        mx = fmaxf(mx, v32);
    }
    __device__ __forceinline__ void merge(const Stat4& o) {
        sum += o.sum;
        sumsq += o.sumsq;
        mn = fminf(mn, o.mn);
        mx = fmaxf(mx, o.mx);
    }
    // the workspace / C-ABI form: {sum, sumsq, min, max} as doubles, +-1e300 for "no value"
    __device__ __forceinline__ void store(double* p) const {
        p[0] = sum;
        p[1] = sumsq;
        p[2] = mn == __int_as_float(0x7f800000) ? 1e300 : (double)mn;
        p[3] = mx == __int_as_float(0xff800000) ? -1e300 : (double)mx;
    }
};

// the same four fields in float64, for folding per-block partials
struct Stat4D {
    double sum, sumsq, mn, mx;
    __device__ __forceinline__ void init() {
        sum = 0.0;
        sumsq = 0.0;
        mn = 1e300;
        mx = -1e300;
    }
    __device__ __forceinline__ void merge(const Stat4D& o) {
        sum += o.sum;
        sumsq += o.sumsq;
        mn = fmin(mn, o.mn);
        mx = fmax(mx, o.mx);
    }
};

template <class S>
__device__ __forceinline__ S warp_reduce(S s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        S t;
        t.sum = __shfl_down_sync(0xffffffffu, s.sum, o);
        t.sumsq = __shfl_down_sync(0xffffffffu, s.sumsq, o);
        t.mn = __shfl_down_sync(0xffffffffu, s.mn, o);
        t.mx = __shfl_down_sync(0xffffffffu, s.mx, o);
        s.merge(t);
    }
    return s;
}

// In-place normalisation of the raw float32 attributes: out = (v - shift) / div (+ optional 1 - v).
// EdgeLength and non-rotated directions are float32 arrays in the reference, so the division is float32
// (normalise.py on a float32 array); rotated directions are float64 there and cast last, so the arithmetic is
// float64 on the stored float32 value (one extra rounding, <= 6e-8 relative).  A flat array of n floats is
// processed as 128-bit vectors between an aligned head and tail.
template <bool F64>
__device__ __forceinline__ float scale_one(float v, float shift32, float div32, double shift, double mul, int invert) {
    float r = F64 ? (float)(((double)v - shift) * mul) : __fdiv_rn(__fsub_rn(v, shift32), div32);
    return invert ? __fsub_rn(1.0f, r) : r;
}

// what one launch of the per-edge kernel reads and writes
struct AttrArgs {
    const int32_t* esrc;
    const int32_t* edst;
    int64_t n_edges;
    const float4* s_rec;   // source records, or NULL: evaluate the source from s_ll
    const float2* s_ll;
    const double2* t_rec;  // target records, or NULL: evaluate the target from t_ll
    const float2* t_ll;
    int want_len, len_invert_now, want_dir, dir_rotated;
    float* out_len;
    float* out_dir;
    double* ws;
    const uint8_t* dst_flags;  // one byte per TARGET node (flag_mode != 0)
    int flag_mode;             // AGX_ATTR_FLAGS_SKIP: flagged targets' edges are written but not counted;
                               // AGX_ATTR_FLAGS_ONLY: only those edges are evaluated at all
    const int32_t* only_list;  // with regular_k: the work items are the edges [t k, (t + 1) k) of the listed targets
    const int64_t* only_count;
    int regular_k;
};

template <bool COORD>
__device__ __forceinline__ SrcNode attr_load_src(const AttrArgs& a, int i) {
    if (COORD) return agx_src_node(__ldg(a.s_ll + i));
    const float4 r0 = __ldg(a.s_rec + 2 * (int64_t)i);
    const float2 r1 = __ldg(reinterpret_cast<const float2*>(a.s_rec + 2 * (int64_t)i + 1));
    SrcNode n = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y};
    return n;
}

template <bool COORD>
__device__ __forceinline__ DstNode attr_load_dst(const AttrArgs& a, int i, bool want_quat) {
    if (COORD) return agx_dst_node(__ldg(a.t_ll + i), want_quat);
    const double2 qa = __ldg(a.t_rec + 2 * (int64_t)i), qb = __ldg(a.t_rec + 2 * (int64_t)i + 1);
    const long long packed = __double_as_longlong(qb.y);
    DstNode n = {qa.x, qa.y, qb.x, __int_as_float((int)(packed & 0xffffffffll)), __int_as_float((int)(packed >> 32))};
    return n;
}

// Stores the raw float32 values; STATS: also reduces them (a shard's statistics, or the first pass) - the
// normalisation follows as an in-place scaling pass (k_attr_scale), so the trigonometry runs ONCE per edge.
// J = 2: every lane owns TWO ADJACENT edges of a 64-edge warp tile: the index rows are read as one 8-byte load per lane
// and row, the lengths leave as one 8-byte store and the directions as ONE 128-bit store (2 edges x 2 floats) - fully
// coalesced 256 / 512-byte warp transactions.  J = 1 (unaligned rows, the list-driven patch pass): scalar accesses.
template <bool STATS, int J, bool SRC_COORD, bool DST_COORD>
__global__ void __launch_bounds__(ATTR_THREADS, 3) k_edge_attrs(AttrArgs a) {
    Stat4 st_len, st_dir;
    st_len.init();
    st_dir.init();
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n_work = a.only_list ? *a.only_count * a.regular_k : a.n_edges;
    const int64_t n_tiles = (n_work + 32 * J - 1) / (32 * J);
    for (int64_t tile = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; tile < n_tiles; tile += n_warps) {
        const int64_t w0 = tile * (32 * J) + (int64_t)lane * J;  // this lane's first work item
        int s[J], t[J];
        int64_t eid[J];
        bool live[J];
        if (J == 2 && a.only_list == nullptr && w0 + 1 < n_work) {
            const int2 sv = __ldg(reinterpret_cast<const int2*>(a.esrc + w0));
            const int2 tv = __ldg(reinterpret_cast<const int2*>(a.edst + w0));
            s[0] = sv.x; s[J - 1] = sv.y;
            t[0] = tv.x; t[J - 1] = tv.y;
            eid[0] = w0; eid[J - 1] = w0 + 1;
            live[0] = live[J - 1] = true;
        } else {
#pragma unroll
            for (int j = 0; j < J; ++j) {
                int64_t w = w0 + j;
                live[j] = w < n_work;
                w = live[j] ? w : n_work - 1;  // dead lanes repeat the last item (never stored, never counted)
                const int64_t e = a.only_list ? (int64_t)a.only_list[w / a.regular_k] * a.regular_k + (w % a.regular_k) : w;
                eid[j] = e;
                s[j] = __ldg(a.esrc + e);
                t[j] = __ldg(a.edst + e);
            }
        }
        bool flagged[J];
#pragma unroll
        for (int j = 0; j < J; ++j) flagged[j] = a.flag_mode != 0 && a.dst_flags[t[j]] != 0;
        if (a.flag_mode == AGX_ATTR_FLAGS_ONLY) {
            bool any = false;
#pragma unroll
            for (int j = 0; j < J; ++j) {
                live[j] = live[j] && flagged[j];
                any |= live[j];
            }
            if (!__any_sync(0xffffffffu, any)) continue;
        }
        SrcNode sn[J];
        DstNode dn[J];
#pragma unroll
        for (int j = 0; j < J; ++j) {  // all gathers in flight before the arithmetic
            sn[j] = attr_load_src<SRC_COORD>(a, s[j]);
            dn[j] = attr_load_dst<DST_COORD>(a, t[j], a.want_dir && a.dir_rotated);
        }
        float vlen[J], d0[J], d1[J];
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const bool counted = live[j] && (a.flag_mode != AGX_ATTR_FLAGS_SKIP || !flagged[j]);
            vlen[j] = d0[j] = d1[j] = 0.0f;
            if (a.want_len) {
                float st_unused, ct;
                agx_np_sincosf(dn[j].lat, st_unused, ct);  // numpy's float32 cos(lat) of the target
                const float v = edge_length_raw(make_float2(sn[j].lat, sn[j].lon), sn[j].cl, make_float2(dn[j].lat, dn[j].lon), ct);
                if (STATS && counted) st_len.add((double)v, v);
                vlen[j] = a.len_invert_now ? __fsub_rn(1.0f, v) : v;
            }
            if (a.want_dir) {
                if (a.dir_rotated) {
                    double e0, e1;
                    edge_direction_rotated(make_float4(sn[j].x, sn[j].y, sn[j].z, 0.f), dn[j].qx, dn[j].qy, dn[j].qw, e0, e1);
                    d0[j] = (float)e0;
                    d1[j] = (float)e1;
                    if (STATS && counted) {
                        st_dir.add(e0, d0[j]);
                        st_dir.add(e1, d1[j]);
                    }
                } else {
                    // directional_edge_features(..., relative_to_rotated_target=False): loc2 - loc1 in float32
                    d0[j] = __fsub_rn(dn[j].lat, sn[j].lat);
                    d1[j] = __fsub_rn(dn[j].lon, sn[j].lon);
                    if (STATS && counted) {
                        st_dir.add((double)d0[j], d0[j]);
                        st_dir.add((double)d1[j], d1[j]);
                    }
                }
            }
        }
        if (J == 2 && live[0] && live[J - 1] && eid[J - 1] == eid[0] + 1 && (eid[0] & 1) == 0) {
            if (a.want_len) *reinterpret_cast<float2*>(a.out_len + eid[0]) = make_float2(vlen[0], vlen[J - 1]);
            if (a.want_dir) *reinterpret_cast<float4*>(a.out_dir + 2 * eid[0]) = make_float4(d0[0], d1[0], d0[J - 1], d1[J - 1]);
        } else {
#pragma unroll
            for (int j = 0; j < J; ++j)
                if (live[j]) {
                    if (a.want_len) a.out_len[eid[j]] = vlen[j];
                    if (a.want_dir) reinterpret_cast<float2*>(a.out_dir)[eid[j]] = make_float2(d0[j], d1[j]);
                }
        }
    }
    if (STATS) {
        __shared__ Stat4 sm[2][ATTR_THREADS / 32];
        st_len = warp_reduce(st_len);
        st_dir = warp_reduce(st_dir);
        int warp = threadIdx.x >> 5;
        if (lane == 0) {
            sm[0][warp] = st_len;
            sm[1][warp] = st_dir;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < ATTR_THREADS / 32; ++w) {
                st_len.merge(sm[0][w]);
                st_dir.merge(sm[1][w]);
            }
            double* p = a.ws + (int64_t)ATTR_STAT_FIELDS * (2 + blockIdx.x);
            st_len.store(p);
            st_dir.store(p + 4);
        }
    }
}

// The same evaluation for a REGULAR edge list - k edges per target, the edges of the i-th target being the columns
// [i k, (i + 1) k) (a KNN result) - organised by TARGET: one lane per target reads the target's coordinates (or record)
// ONCE, evaluates its cos(lat) / rotation quaternion once and walks its k sources.  A third of the target-side
// arithmetic and loads of the edge-centric kernel for k = 3, and the target row is read once per target (its first
// column) instead of once per edge.
template <bool STATS, bool SRC_COORD, bool DST_COORD>
__global__ void __launch_bounds__(ATTR_THREADS, 3) k_edge_attrs_regular(AttrArgs a) {
    Stat4 st_len, st_dir;
    st_len.init();
    st_dir.init();
    const int k = a.regular_k;
    const int64_t n_targets = a.n_edges / k;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_targets; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e0 = i * k;
        const int t = __ldg(a.edst + e0);
        const bool flagged = a.flag_mode != 0 && a.dst_flags[t] != 0;
        if (a.flag_mode == AGX_ATTR_FLAGS_ONLY && !flagged) continue;
        const bool counted = a.flag_mode != AGX_ATTR_FLAGS_SKIP || !flagged;
        const DstNode dn = attr_load_dst<DST_COORD>(a, t, a.want_dir && a.dir_rotated);
        float ct = 0.0f;
        if (a.want_len) {
            float st_unused;
            agx_np_sincosf(dn.lat, st_unused, ct);  // numpy's float32 cos(lat) of the target
        }
        for (int j = 0; j < k; ++j) {
            const int64_t e = e0 + j;
            const SrcNode sn = attr_load_src<SRC_COORD>(a, __ldg(a.esrc + e));
            if (a.want_len) {
                const float v = edge_length_raw(make_float2(sn.lat, sn.lon), sn.cl, make_float2(dn.lat, dn.lon), ct);
                if (STATS && counted) st_len.add((double)v, v);
                a.out_len[e] = a.len_invert_now ? __fsub_rn(1.0f, v) : v;
            }
            if (a.want_dir) {
                float f0, f1;
                if (a.dir_rotated) {
                    double d0, d1;
                    edge_direction_rotated(make_float4(sn.x, sn.y, sn.z, 0.f), dn.qx, dn.qy, dn.qw, d0, d1);
                    f0 = (float)d0;
                    f1 = (float)d1;
                    if (STATS && counted) {
                        st_dir.add(d0, f0);
                        st_dir.add(d1, f1);
                    }
                } else {
                    f0 = __fsub_rn(dn.lat, sn.lat);
                    f1 = __fsub_rn(dn.lon, sn.lon);
                    if (STATS && counted) {
                        st_dir.add((double)f0, f0);
                        st_dir.add((double)f1, f1);
                    }
                }
                reinterpret_cast<float2*>(a.out_dir)[e] = make_float2(f0, f1);
            }
        }
    }
    if (STATS) {
        __shared__ Stat4 sm[2][ATTR_THREADS / 32];
        st_len = warp_reduce(st_len);
        st_dir = warp_reduce(st_dir);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) {
            sm[0][warp] = st_len;
            sm[1][warp] = st_dir;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < ATTR_THREADS / 32; ++w) {
                st_len.merge(sm[0][w]);
                st_dir.merge(sm[1][w]);
            }
            double* p = a.ws + (int64_t)ATTR_STAT_FIELDS * (2 + blockIdx.x);
            st_len.store(p);
            st_dir.store(p + 4);
        }
    }
}

template <bool F64>
__device__ __forceinline__ void scale_array(float* __restrict__ a, int64_t n, float shift32, float div32, double shift,
                                            double mul, int invert) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    int64_t head = ((16 - ((uintptr_t)a & 15)) & 15) >> 2;  // floats before the first 16-byte boundary
    if (head > n) head = n;
    int64_t n_vec = (n - head) >> 2;
    float4* v4 = reinterpret_cast<float4*>(a + head);
    for (int64_t i = tid; i < n_vec; i += stride) {
        float4 v = v4[i];
        v.x = scale_one<F64>(v.x, shift32, div32, shift, mul, invert);
        v.y = scale_one<F64>(v.y, shift32, div32, shift, mul, invert);
        v.z = scale_one<F64>(v.z, shift32, div32, shift, mul, invert);
        v.w = scale_one<F64>(v.w, shift32, div32, shift, mul, invert);
        v4[i] = v;
    }
    int64_t tail0 = head + (n_vec << 2);
    for (int64_t i = tid; i < head + (n - tail0); i += stride) {
        int64_t j = i < head ? i : tail0 + (i - head);
        a[j] = scale_one<F64>(a[j], shift32, div32, shift, mul, invert);
    }
}

__global__ void __launch_bounds__(256) k_attr_scale(float* __restrict__ out_len, int64_t n_len, int len_scale,
                                                     int len_invert, float* __restrict__ out_dir, int64_t n_dir,
                                                     int dir_scale, int dir_f64, const double* __restrict__ ws) {
    if (out_len != nullptr && (len_scale || len_invert))
        scale_array<false>(out_len, n_len, len_scale ? (float)ws[0] : 0.0f, len_scale ? (float)ws[1] : 1.0f, 0.0, 1.0,
                           len_invert);
    if (out_dir != nullptr && dir_scale) {
        if (dir_f64)
            scale_array<true>(out_dir, n_dir, 0.0f, 1.0f, ws[2], ws[3], 0);
        else
            scale_array<false>(out_dir, n_dir, (float)ws[4], (float)ws[5], 0.0, 1.0, 0);
    }
}

// Fold the per-block partials into stats[8] = {len sum, sumsq, min, max, dir sum, sumsq, min, max}.
// One 256-thread block: thread t folds partials t, t+256, ... in order, then a fixed shuffle/shared tree -
// the association order depends only on n_blocks, so the result is reproducible run to run.
__global__ void __launch_bounds__(256) k_attr_fold(const double* __restrict__ ws, int n_blocks, double* __restrict__ stats) {
    Stat4D L, D;
    L.init();
    D.init();
    for (int b = threadIdx.x; b < n_blocks; b += 256) {
        const double* p = ws + (int64_t)ATTR_STAT_FIELDS * (2 + b);
        Stat4D l = {p[0], p[1], p[2], p[3]}, d = {p[4], p[5], p[6], p[7]};
        L.merge(l);
        D.merge(d);
    }
    __shared__ Stat4D sm[2][8];
    L = warp_reduce(L);
    D = warp_reduce(D);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        sm[0][warp] = L;
        sm[1][warp] = D;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) {
            L.merge(sm[0][w]);
            D.merge(sm[1][w]);
        }
        stats[0] = L.sum; stats[1] = L.sumsq; stats[2] = L.mn; stats[3] = L.mx;
        stats[4] = D.sum; stats[5] = D.sumsq; stats[6] = D.mn; stats[7] = D.mx;
    }
}

// Global statistics -> normalisation parameters (normalise.py:33-52).
// ws[0..1] = length (shift, div); ws[2..5] = direction (shift, 1/div, shift, div).
__global__ void k_attr_params(double* __restrict__ ws, const double* __restrict__ stats_sets, int n_sets, int64_t n_edges,
                              int len_norm, int dir_norm) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    // fold the per-shard statistics in order (one set on a single GPU): the same association on every rank
    double stats[8] = {0.0, 0.0, 1e300, -1e300, 0.0, 0.0, 1e300, -1e300};
    for (int r = 0; r < n_sets; ++r)
        for (int b = 0; b < 8; b += 4) {
            const double* p = stats_sets + 8 * r + b;
            stats[b] += p[0];
            stats[b + 1] += p[1];
            stats[b + 2] = fmin(stats[b + 2], p[2]);
            stats[b + 3] = fmax(stats[b + 3], p[3]);
        }
    for (int which = 0; which < 2; ++which) {
        int norm = which ? dir_norm : len_norm;
        double shift = 0.0, div = 1.0;
        if (norm > 0) {
            const double* S = stats + 4 * which;  // sum, sumsq, min, max
            double count = (double)n_edges * (which ? 2.0 : 1.0);
            if (norm == AGX_NORM_L1) div = S[0];
            else if (norm == AGX_NORM_L2) div = sqrt(S[1]);
            else if (norm == AGX_NORM_UNIT_MAX) div = S[3];
            else if (norm == AGX_NORM_UNIT_RANGE) { shift = S[2]; div = S[3] - S[2]; }
            else if (norm == AGX_NORM_UNIT_STD) {
                double mean = S[0] / count;
                double var = S[1] / count - mean * mean;
                double sd = var > 0.0 ? sqrt(var) : 0.0;
                div = sd == 0.0 ? 1.0 : sd;  // normalise.py:46-50: skipped when std == 0
            }
            // a NaN value (an antipodal pair's length) makes numpy's sum, amax, amin and std NaN, so the reference
            // returns NaN everywhere; the sum carries the NaN here, the minimum / maximum (fminf / fmaxf) do not
            if (isnan(S[0])) div = __longlong_as_double(0x7ff8000000000000ll);
        }
        if (which == 0) {
            ws[0] = shift;
            ws[1] = div;
        } else {
            ws[2] = shift;
            ws[3] = 1.0 / div;
            ws[4] = shift;
            ws[5] = div;
        }
    }
}

// the node inputs of one call: per side either a record table or the (lat, lon) coordinates
struct AttrNodes {
    const float* src_rec;
    const float* src_ll;
    const double* dst_rec;
    const float* dst_ll;
};

static int attrs_check(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, const AttrNodes& nd,
                       const double* workspace) {
    AGX_REQUIRE(n_edges >= 0, AGX_ERR_ARG, "agx_edge_attrs: n_edges < 0");
    if (n_edges == 0) return AGX_OK;
    AGX_REQUIRE(edge_src && edge_dst && workspace, AGX_ERR_ARG, "agx_edge_attrs: NULL buffer");
    AGX_REQUIRE((nd.src_rec != nullptr) != (nd.src_ll != nullptr), AGX_ERR_ARG,
                "agx_edge_attrs: give the source nodes as records OR as coordinates");
    AGX_REQUIRE((nd.dst_rec != nullptr) != (nd.dst_ll != nullptr), AGX_ERR_ARG,
                "agx_edge_attrs: give the target nodes as records OR as coordinates");
    AGX_REQUIRE(((uintptr_t)nd.src_rec & 15) == 0 && ((uintptr_t)nd.dst_rec & 15) == 0 && ((uintptr_t)nd.src_ll & 7) == 0 &&
                    ((uintptr_t)nd.dst_ll & 7) == 0,
                AGX_ERR_ARG, "agx_edge_attrs: node records must be 16-byte, coordinates 8-byte aligned");
    return AGX_OK;
}

// the per-edge kernels store a direction as one float2 (J = 1 lanes, k_edge_attrs_regular): a 4-byte aligned out_dir
// (a view that starts at an odd float) would fault there, so every entry point refuses it before any device work
static int attrs_check_dir(const float* out_dir) {
    AGX_REQUIRE(((uintptr_t)out_dir & 7) == 0, AGX_ERR_ARG, "agx_edge_attrs: out_dir must be 8-byte aligned");
    return AGX_OK;
}

static inline int attrs_grid(int64_t n_edges, int j) {
    int grid = agx_grid((n_edges + j - 1) / j, ATTR_THREADS, 3);
    return grid > ATTR_MAX_BLOCKS ? ATTR_MAX_BLOCKS : grid;
}

template <bool STATS, int J>
static void attrs_launch_modes(int grid, cudaStream_t stream, const AttrArgs& a) {
    const bool sc = a.s_rec == nullptr, dc = a.t_rec == nullptr;
    if (sc && dc)
        k_edge_attrs<STATS, J, true, true><<<grid, ATTR_THREADS, 0, stream>>>(a);
    else if (sc)
        k_edge_attrs<STATS, J, true, false><<<grid, ATTR_THREADS, 0, stream>>>(a);
    else if (dc)
        k_edge_attrs<STATS, J, false, true><<<grid, ATTR_THREADS, 0, stream>>>(a);
    else
        k_edge_attrs<STATS, J, false, false><<<grid, ATTR_THREADS, 0, stream>>>(a);
}

template <bool STATS>
static void attrs_launch_regular(int grid, cudaStream_t stream, const AttrArgs& a) {
    const bool sc = a.s_rec == nullptr, dc = a.t_rec == nullptr;
    if (sc && dc)
        k_edge_attrs_regular<STATS, true, true><<<grid, ATTR_THREADS, 0, stream>>>(a);
    else if (sc)
        k_edge_attrs_regular<STATS, true, false><<<grid, ATTR_THREADS, 0, stream>>>(a);
    else if (dc)
        k_edge_attrs_regular<STATS, false, true><<<grid, ATTR_THREADS, 0, stream>>>(a);
    else
        k_edge_attrs_regular<STATS, false, false><<<grid, ATTR_THREADS, 0, stream>>>(a);
}

template <int J>
static void attrs_launch(bool stats, int grid, cudaStream_t stream, const AttrArgs& a) {
    if (stats)
        attrs_launch_modes<true, J>(grid, stream, a);
    else
        attrs_launch_modes<false, J>(grid, stream, a);
}

// pass A: raw values of the local edges -> out_* (float32), and stats[8] when stats is given
static int attrs_raw(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, const AttrNodes& nd, int want_len,
                     int len_invert_now, float* out_len, int want_dir, int dir_rotated, float* out_dir, double* stats,
                     double* workspace, cudaStream_t stream, const uint8_t* dst_flags, int flag_mode,
                     const int32_t* only_list, const int64_t* only_count, int regular_k) {
    int grid = 0;
    if (n_edges > 0 && (want_len || want_dir)) {
        AttrArgs a;
        a.esrc = edge_src;
        a.edst = edge_dst;
        a.n_edges = n_edges;
        a.s_rec = (const float4*)nd.src_rec;
        a.s_ll = (const float2*)nd.src_ll;
        a.t_rec = (const double2*)nd.dst_rec;
        a.t_ll = (const float2*)nd.dst_ll;
        a.want_len = want_len;
        a.len_invert_now = len_invert_now;
        a.want_dir = want_dir;
        a.dir_rotated = dir_rotated;
        a.out_len = out_len;
        a.out_dir = out_dir;
        a.ws = workspace;
        a.dst_flags = dst_flags;
        a.flag_mode = flag_mode;
        a.only_list = only_list;
        a.only_count = only_count;
        a.regular_k = regular_k;
        // two adjacent edges per lane need 8-byte aligned index rows and 8 / 16-byte aligned outputs (a (2, E) list with
        // odd E, or a block that starts at an odd column, is not): scalar lanes then
        const bool aligned = (((uintptr_t)edge_src | (uintptr_t)edge_dst | (uintptr_t)out_len) & 7) == 0 &&
                             ((uintptr_t)out_dir & 15) == 0;
        const int j = (only_list == nullptr && aligned) ? 2 : 1;
        if (only_list == nullptr && regular_k > 0) {
            // a regular-k list (KNN result) walked by target
            grid = attrs_grid(n_edges / regular_k, 1);
            if (stats != nullptr)
                attrs_launch_regular<true>(grid, stream, a);
            else
                attrs_launch_regular<false>(grid, stream, a);
        } else {
            grid = only_list ? 32 : attrs_grid(n_edges, j);
            if (j == 2)
                attrs_launch<2>(stats != nullptr, grid, stream, a);
            else
                attrs_launch<1>(stats != nullptr, grid, stream, a);
        }
        agx_note_launch(1);
    }
    if (stats) {
        k_attr_fold<<<1, 256, 0, stream>>>(workspace, grid, stats);  // grid == 0: the empty statistics
        agx_note_launch(1);
    }
    AGX_LAUNCH_OK();
    return AGX_OK;
}

// pass B: statistics -> parameters, in-place scaling of the raw values
static int attrs_scale(int64_t n_edges, int len_norm, int len_invert, float* out_len, int dir_norm, int dir_rotated,
                       float* out_dir, const double* stats, int n_stat_sets, int64_t n_edges_global, double* workspace,
                       cudaStream_t stream) {
    int want_len = len_norm >= 0, want_dir = dir_norm >= 0;
    bool len_scale = want_len && len_norm > 0, dir_scale = want_dir && dir_norm > 0;
    if (n_edges == 0 || !(len_scale || dir_scale || (want_len && len_invert))) return AGX_OK;
    k_attr_params<<<1, 32, 0, stream>>>(workspace, stats, n_stat_sets, n_edges_global, want_len ? len_norm : 0,
                                        want_dir ? dir_norm : 0);
    int64_t work = (n_edges * (want_dir ? 2 : 1) + 3) / 4;
    k_attr_scale<<<agx_grid(work, 256, 8), 256, 0, stream>>>(want_len ? out_len : nullptr, n_edges, len_scale, len_invert,
                                                           want_dir ? out_dir : nullptr, 2 * n_edges, dir_scale,
                                                           dir_rotated, workspace);
    AGX_LAUNCH_OK();
    agx_note_launch(2);
    return AGX_OK;
}

extern "C" int agx_edge_attrs_stats(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges,
                                    const float* src_rec, const float* src_latlon, const double* dst_rec,
                                    const float* dst_latlon, int want_len, int want_dir, int dir_rotated, float* out_len,
                                    float* out_dir, double* stats, double* workspace, const uint8_t* dst_flags,
                                    int flag_mode, const int32_t* list, const int64_t* count, int regular_k,
                                    void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(regular_k >= 0 && (regular_k == 0 || n_edges % regular_k == 0), AGX_ERR_ARG,
                "agx_edge_attrs_stats: n_edges is not a multiple of regular_k");
    AGX_REQUIRE(stats != nullptr, AGX_ERR_ARG, "agx_edge_attrs_stats: stats is NULL");
    AGX_REQUIRE(workspace != nullptr, AGX_ERR_ARG, "agx_edge_attrs_stats: workspace is NULL");
    AGX_REQUIRE(flag_mode == 0 || flag_mode == AGX_ATTR_FLAGS_SKIP || flag_mode == AGX_ATTR_FLAGS_ONLY, AGX_ERR_ARG,
                "agx_edge_attrs_stats: flag_mode must be 0, 1 (skip) or 2 (only)");
    AGX_REQUIRE((list != nullptr) == (count != nullptr), AGX_ERR_ARG, "agx_edge_attrs_stats: give list and count together");
    AGX_REQUIRE(!list || (flag_mode == AGX_ATTR_FLAGS_ONLY && !dst_flags && regular_k > 0), AGX_ERR_ARG,
                "agx_edge_attrs_stats: a target list replaces dst_flags in flag_mode 2 (only) with regular_k > 0");
    AGX_REQUIRE(list || flag_mode == 0 || dst_flags, AGX_ERR_ARG,
                "agx_edge_attrs_stats: flag_mode 1 (skip) needs dst_flags, 2 (only) dst_flags or a target list");
    const AttrNodes nd = {src_rec, src_latlon, dst_rec, dst_latlon};
    int rc = attrs_check(edge_src, edge_dst, n_edges, nd, workspace);
    if (rc || (rc = attrs_check_dir(out_dir))) return rc;
    AGX_REQUIRE(n_edges == 0 || ((!want_len || out_len) && (!want_dir || out_dir)), AGX_ERR_ARG,
                "agx_edge_attrs_stats: give every requested output buffer");
    // the list IS the set of "only" targets: the kernel then reads no flags
    return attrs_raw(edge_src, edge_dst, n_edges, nd, want_len, 0, out_len, want_dir, dir_rotated, out_dir, stats,
                     workspace, stream, dst_flags, list ? 0 : flag_mode, list, count, regular_k);
}

extern "C" int agx_edge_attrs_apply(int64_t n_edges, int len_norm, int len_invert, float* out_len, int dir_norm,
                                    int dir_rotated, float* out_dir, const double* stats, int n_stat_sets,
                                    int64_t n_edges_global, double* workspace, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    int want_len = len_norm >= 0, want_dir = dir_norm >= 0;
    AGX_REQUIRE(len_norm <= AGX_NORM_UNIT_STD && dir_norm <= AGX_NORM_UNIT_STD, AGX_ERR_ARG, "agx_edge_attrs: unknown norm code");
    AGX_REQUIRE(n_edges >= 0, AGX_ERR_ARG, "agx_edge_attrs_apply: n_edges < 0");
    if (n_edges == 0 || (!want_len && !want_dir)) return AGX_OK;
    if (int rc = attrs_check_dir(out_dir)) return rc;
    AGX_REQUIRE(workspace != nullptr, AGX_ERR_ARG, "agx_edge_attrs_apply: workspace is NULL");
    AGX_REQUIRE(!want_len || out_len, AGX_ERR_ARG, "agx_edge_attrs: out_len is NULL");
    AGX_REQUIRE(!want_dir || out_dir, AGX_ERR_ARG, "agx_edge_attrs: out_dir is NULL");
    bool need_stats = (want_len && len_norm > 0) || (want_dir && dir_norm > 0);
    AGX_REQUIRE(!need_stats || (stats && n_stat_sets >= 1), AGX_ERR_ARG,
                "agx_edge_attrs_apply: this normalisation needs the statistics of every shard");
    AGX_REQUIRE(n_edges_global >= n_edges, AGX_ERR_ARG, "agx_edge_attrs_apply: n_edges_global < n_edges");
    return attrs_scale(n_edges, len_norm, len_invert, out_len, dir_norm, dir_rotated, out_dir, stats, n_stat_sets,
                       n_edges_global, workspace, stream);
}

extern "C" int agx_edge_attrs(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, const float* src_rec,
                              const float* src_latlon, const double* dst_rec, const float* dst_latlon, int len_norm,
                              int len_invert, float* out_len, int dir_norm, int dir_rotated, float* out_dir,
                              double* workspace, int regular_k, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(regular_k >= 0 && (regular_k == 0 || n_edges % regular_k == 0), AGX_ERR_ARG,
                "agx_edge_attrs: n_edges is not a multiple of regular_k");
    int want_len = len_norm >= 0, want_dir = dir_norm >= 0;
    AGX_REQUIRE(len_norm <= AGX_NORM_UNIT_STD && dir_norm <= AGX_NORM_UNIT_STD, AGX_ERR_ARG, "agx_edge_attrs: unknown norm code");
    const AttrNodes nd = {src_rec, src_latlon, dst_rec, dst_latlon};
    int rc = attrs_check(edge_src, edge_dst, n_edges, nd, workspace);
    if (rc || (rc = attrs_check_dir(out_dir))) return rc;
    if (n_edges == 0 || (!want_len && !want_dir)) return AGX_OK;
    AGX_REQUIRE(!want_len || out_len, AGX_ERR_ARG, "agx_edge_attrs: out_len is NULL");
    AGX_REQUIRE(!want_dir || out_dir, AGX_ERR_ARG, "agx_edge_attrs: out_dir is NULL");
    bool need_stats = (want_len && len_norm > 0) || (want_dir && dir_norm > 0);
    double* stats = need_stats ? workspace + 6 : nullptr;  // ws[6..13]: between the parameters and the block partials
    // no normalisation: the raw pass writes the final values (an inversion needs no statistics)
    rc = attrs_raw(edge_src, edge_dst, n_edges, nd, want_len, need_stats ? 0 : len_invert, out_len, want_dir, dir_rotated,
                   out_dir, stats, workspace, stream, nullptr, 0, nullptr, nullptr, regular_k);
    if (rc || !need_stats) return rc;
    return attrs_scale(n_edges, len_norm, len_invert, out_len, dir_norm, dir_rotated, out_dir, stats, 1, n_edges,
                       workspace, stream);
}

// ------------------------------------------------------------------------------------------------
// Azimuth: the initial bearing at the target towards the source, clockwise from north, in [-pi, pi]
// ------------------------------------------------------------------------------------------------
// atan2(sin(dlon) cos(lat_s), cos(lat_t) sin(lat_s) - sin(lat_t) cos(lat_s) cos(dlon)), dlon = lon_s - lon_t, in float64
// from the float32 coordinates, each operation rounded as numpy rounds it (no contraction), stored as float32.  The
// statistics are those of EdgeLength (the float64 of the stored value) in the length slot of the K5 workspace, so the
// global norm is k_attr_fold -> k_attr_params -> k_attr_scale with its NaN rule.  An endpoint outside its node set is
// never read: it raises *bad (an int in workspace word 14, between the statistics and the block partials).
__global__ void __launch_bounds__(ATTR_THREADS) k_edge_azimuth(const int32_t* __restrict__ esrc, const int32_t* __restrict__ edst,
                                                               int64_t n, const float2* __restrict__ s_ll, int64_t n_src,
                                                               const float2* __restrict__ t_ll, int64_t n_dst,
                                                               float* __restrict__ out, double* __restrict__ ws, int stats) {
    Stat4 st;
    st.init();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t s = __ldg(esrc + i), t = __ldg(edst + i);
        if (s < 0 || s >= n_src || t < 0 || t >= n_dst) {
            *reinterpret_cast<int*>(ws + 14) = 1;
            continue;
        }
        const float2 ps = __ldg(s_ll + s), pt = __ldg(t_ll + t);
        double sls, cls, slt, clt, sdl, cdl;
        sincos((double)ps.x, &sls, &cls);
        sincos((double)pt.x, &slt, &clt);
        sincos(__dsub_rn((double)ps.y, (double)pt.y), &sdl, &cdl);
        const double y = __dmul_rn(sdl, cls);
        const double x = __dsub_rn(__dmul_rn(clt, sls), __dmul_rn(__dmul_rn(slt, cls), cdl));
        const float v = (float)atan2(y, x);
        out[i] = v;
        if (stats) st.add((double)v, v);
    }
    if (stats) {
        __shared__ Stat4 sm[ATTR_THREADS / 32];
        st = warp_reduce(st);
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) sm[warp] = st;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < ATTR_THREADS / 32; ++w) st.merge(sm[w]);
            double* p = ws + (int64_t)ATTR_STAT_FIELDS * (2 + blockIdx.x);
            st.store(p);
            Stat4 none;
            none.init();
            none.store(p + 4);  // the direction slot of the fold stays empty
        }
    }
}

extern "C" int agx_edge_azimuth(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, const float* src_latlon,
                                int64_t n_src_nodes, const float* dst_latlon, int64_t n_dst_nodes, int norm, float* out,
                                double* workspace, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AGX_REQUIRE(n_edges >= 0 && n_src_nodes >= 0 && n_dst_nodes >= 0, AGX_ERR_ARG, "agx_edge_azimuth: negative size");
    AGX_REQUIRE(norm >= 0 && norm <= AGX_NORM_UNIT_STD, AGX_ERR_ARG, "agx_edge_azimuth: unknown norm code");
    if (n_edges == 0) return AGX_OK;
    AGX_REQUIRE(edge_src && edge_dst && out && workspace, AGX_ERR_ARG, "agx_edge_azimuth: NULL buffer");
    AGX_REQUIRE((n_src_nodes == 0 || src_latlon) && (n_dst_nodes == 0 || dst_latlon), AGX_ERR_ARG,
                "agx_edge_azimuth: NULL coordinates");
    AGX_REQUIRE((((uintptr_t)src_latlon | (uintptr_t)dst_latlon) & 7) == 0, AGX_ERR_ARG,
                "agx_edge_azimuth: coordinates must be 8-byte aligned");
    AGX_CUDA_OK(cudaMemsetAsync(workspace + 14, 0, sizeof(double), stream));
    const int grid = attrs_grid(n_edges, 1);
    k_edge_azimuth<<<grid, ATTR_THREADS, 0, stream>>>(edge_src, edge_dst, n_edges, (const float2*)src_latlon, n_src_nodes,
                                                      (const float2*)dst_latlon, n_dst_nodes, out, workspace, norm > 0);
    agx_note_launch(1);
    if (norm > 0) {
        k_attr_fold<<<1, 256, 0, stream>>>(workspace, grid, workspace + 6);
        k_attr_params<<<1, 32, 0, stream>>>(workspace, workspace + 6, 1, n_edges, norm, 0);
        k_attr_scale<<<agx_grid((n_edges + 3) / 4, 256, 8), 256, 0, stream>>>(out, n_edges, 1, 0, nullptr, 0, 0, 0, workspace);
        agx_note_launch(3);
    }
    AGX_LAUNCH_OK();
    long long bad = 0;
    int rc = agx_readback(&bad, workspace + 14, 1, stream);
    if (rc) return rc;
    AGX_REQUIRE((int)bad == 0, AGX_ERR_ARG, "agx_edge_azimuth: an edge endpoint is outside [0, num_nodes) of its node set");
    return AGX_OK;
}
