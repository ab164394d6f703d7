/* agx_b200 - C ABI of the B200-native edge-construction path of anemoi-graphs.
 *
 * One shared library (libagx_b200.so, CUDA sm_100a) exports exactly these symbols; the Python
 * host layer (anemoi_graphs_b200/_cabi.py) binds them with ctypes.  Each entry point names the
 * reference interface it replaces (paths relative to /root/reference/src/anemoi/graphs/).
 *
 * Conventions
 *  - every pointer marked DEV is a CUDA device pointer owned by the caller; HOST pointers are
 *    plain host memory.  No torch / C++ types cross the boundary.
 *  - node coordinates are float32 (lat, lon) pairs in RADIANS, interleaved (n x 2), exactly the
 *    layout of `graph[name].x` (nodes/builders/base.py:54,84-101).
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All work is
 *    enqueued on it; functions that return a value through a HOST pointer synchronise the stream.
 *  - return value: 0 on success, a negative AGX_ERR_* code otherwise; agx_last_error() gives a
 *    thread-local message.  Nothing throws; there is no global state besides opaque handles.
 *  - variable-size outputs use count -> (caller allocates) -> fill.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    AGX_ERR_CUDA.
 */
#ifndef AGX_B200_H
#define AGX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGX_ABI_VERSION 4

#define AGX_OK 0
#define AGX_ERR_CUDA -1      /* CUDA runtime / launch failure (includes "no device") */
#define AGX_ERR_ARG -2       /* invalid argument */
#define AGX_ERR_UNSUPPORTED -3 /* valid in the reference, not built yet (message says what) */
#define AGX_ERR_OVERFLOW -4  /* an internal fixed-capacity buffer was too small */

/* normalisation codes: normalise.py:20-55 */
#define AGX_NORM_NONE 0
#define AGX_NORM_L1 1
#define AGX_NORM_L2 2
#define AGX_NORM_UNIT_MAX 3
#define AGX_NORM_UNIT_RANGE 4
#define AGX_NORM_UNIT_STD 5

typedef struct agx_index agx_index_t;

const char* agx_last_error(void);
int agx_abi_version(void);
/* number of kernels this library has launched in the calling process (bench.py "gpu_launches") */
int64_t agx_launch_count(void);

/* ---- neighbour index -------------------------------------------------------------------------
 * Replaces `NearestNeighbors(metric="haversine").fit(coords)` (edges/builder.py:259-260,364-365;
 * utils.py:37-39; generate/masks.py:74): bins the reference points into 6*C*C equi-angular
 * cube-sphere cells (C = cells_per_face, 0 = choose from n and `hint_k` / `hint_radius`).
 * `latlon` must stay valid until agx_index_free.                                               */
int agx_index_build(const float* latlon /*DEV n*2*/, int64_t n, int cells_per_face, int hint_k,
                    double hint_radius, void* stream, agx_index_t** out);
int agx_index_free(agx_index_t* index, void* stream);
int agx_index_info(const agx_index_t* index, int64_t* n, int* cells_per_face);
/* The float32 unit vectors the neighbour search filters with (float64 trig of the float32 (lat, lon), rounded once;
 * every component within 2^-25 + 3e-11 of exact - the bound the FP32 filter margin of agx_knn / agx_radius_* is
 * derived from).  Exposed so that tests can pin that bound; not needed to build a graph.                      */
int agx_search_vectors(const float* latlon /*DEV n*2*/, int64_t n, float* xyz /*DEV n*3*/, void* stream);

/* ---- KNN --------------------------------------------------------------------------------------
 * Replaces `kneighbors_graph(target, n_neighbors=k)` / `kneighbors(...)` (edges/builder.py:261-265,
 * utils.py:62, generate/masks.py:97).  For query q (0 <= q < nq) writes the SET of its k nearest
 * reference points to out_src[q*k .. q*k+k); if out_dst != NULL also out_dst[q*k+j] = dst_base + q
 * (so (out_src, out_dst) are the two rows of edge_index, edges/builder.py:86-87).  Decisions are
 * float64 haversine `rdist` on the float32 inputs (sklearn _dist_metrics.pyx.tp:2639-2648); ties
 * within 2^-40 relative go to the lower index.  out_rdist (optional, nq*k) receives the float64 rdist
 * of every neighbour; with it each row is ascending (rdist, index) under that tie rule.  Without it
 * only the set is defined: the order inside a row is the filter's (FP32 chord, truncated by up to
 * 2^-14 relative) and may differ between runs that process the queries in a different order.
 * stats (optional, DEV int64[4]) += {queries refined in float64, queries with a tie at the k-th
 * boundary, queries needing a wider search, (query, candidate) pairs evaluated by the staged scans on the FP32 pipe}.
 * max_radius (radians; 0 = unlimited) bounds the search, for callers that only ask "is anything within r?"
 * (KNNAreaMaskBuilder.get_mask compares the distance with a margin, generate/masks.py:94-99 - without the bound a
 * query far from a clustered reference set walks the whole sphere): a query whose k-th neighbour lies within
 * max_radius is answered exactly.  For any other query the row holds EVERY reference point within max_radius
 * (with its exact rdist); the remaining slots hold distinct points farther than max_radius, or -1 with
 * rdist = +inf (with out_rdist: after the points, ascending as above).                                      */
int agx_knn(const agx_index_t* index, const float* q_latlon /*DEV nq*2*/, int64_t nq, int k, double max_radius,
            int32_t* out_src /*DEV*/, int32_t* out_dst /*DEV or NULL*/, int64_t dst_base,
            double* out_rdist /*DEV or NULL*/, int64_t* stats /*DEV or NULL*/, void* stream);

/* agx_knn with one more output: tie_flags[q] (DEV nq bytes, zeroed by the caller) is set to 1 for every query whose
 * k-th and (k+1)-th candidates tie within 2^-40 relative - the only queries whose edge set depends on how the
 * reference points are NUMBERED (lower index wins).  A caller that searches before the final numbering is known
 * (device.Provisional: the node order is still being sorted on the host) re-runs exactly these queries afterwards. */
int agx_knn_flagged(const agx_index_t* index, const float* q_latlon /*DEV nq*2*/, int64_t nq, int k, double max_radius,
                    int32_t* out_src /*DEV*/, int32_t* out_dst /*DEV or NULL*/, int64_t dst_base,
                    double* out_rdist /*DEV or NULL*/, int64_t* stats /*DEV or NULL*/, uint8_t* tie_flags /*DEV nq or NULL*/,
                    void* stream);

/* The second half: searches ONLY the queries whose tie_flags byte is set (against an index built over the finally
 * numbered reference points) and overwrites their k slots of out_src; every other query is left untouched.  No
 * compaction and no read-back: a tile of 32 queries without a flagged one costs 32 bytes of traffic, read as two
 * 16-byte words - so tie_flags must be 16-byte aligned (AGX_ERR_ARG otherwise; a cudaMalloc'ed base is, and so is
 * flags + 16 m).                                                                                                */
int agx_knn_redecide(const agx_index_t* index, const float* q_latlon /*DEV nq*2*/, int64_t nq, int k, double max_radius,
                     int32_t* out_src /*DEV nq*k*/, const uint8_t* tie_flags /*DEV nq, 16-byte aligned*/, void* stream);

/* The same re-decision WITHOUT a second index: `index` is still the one built over the provisionally numbered points
 * (the one agx_knn_flagged searched).  Ties go to the lower FINAL label rank[provisional label]; the k slots are
 * written as provisional labels again (order[final label]), so that one relabel pass afterwards treats every slot
 * of the row alike.  rank / order: DEV int64[n_reference], inverse permutations (agx_order_resolve).              */
/* ... and driven by an explicit list of query ids (ascending, *count entries, device memory) instead of the flag
 * array: one thread per listed query, no staging.  rank / order NULL: the index labels are final.               */
int agx_knn_redecide_list(const agx_index_t* index, const float* q_latlon /*DEV nq*2*/, int64_t nq, int k,
                          double max_radius, int32_t* out_src /*DEV nq*k*/, const int32_t* list /*DEV*/,
                          const int64_t* count /*DEV*/, const int64_t* rank /*DEV or NULL*/,
                          const int64_t* order /*DEV or NULL*/, void* stream);
/* Ascending list of the positions of the non-zero bytes of flags[0..n) and its length (both device memory; list has
 * room for n entries); no read-back.                                                                            */
int agx_compact_flags(const uint8_t* flags /*DEV n, 4-byte aligned*/, int64_t n, int32_t* list /*DEV n*/,
                      int64_t* count /*DEV 1*/, void* stream);
int agx_knn_redecide_ranked(const agx_index_t* index, const float* q_latlon /*DEV nq*2*/, int64_t nq, int k,
                            double max_radius, int32_t* out_src /*DEV nq*k*/,
                            const uint8_t* tie_flags /*DEV nq, 16-byte aligned*/, const int64_t* rank /*DEV*/,
                            const int64_t* order /*DEV*/, void* stream);

/* Query order of the tile kernels.  agx_knn / agx_radius_* decide per call whether to walk the queries as given or in
 * a spatially binned order; for >= 262 144 queries the decision samples tile plans and synchronises the stream.
 * A caller that searches ONE query set in several chunks (device.ChunkedGather) reads the first call's decision
 * (agx_last_query_order: 0 as given, 1 binned) and pins it for the rest (agx_set_query_order_mode; -1 = decide per
 * call again), so that the host can enqueue chunk c+1 while chunk c runs.  Both are per host thread.            */
void agx_set_query_order_mode(int mode);
int agx_last_query_order(void);

/* ---- cut-off (radius) search -------------------------------------------------------------------
 * Replaces `radius_neighbors_graph(target, radius)` (edges/builder.py:366): every reference point
 * with rdist <= sin^2(radius/2) (inclusive).  count -> scan -> fill; output grouped by query, in
 * cell-scan order (deterministic).  `offsets` has nq+1 entries; total = offsets[nq].
 * stats (optional, DEV int64[4]) += {pairs decided in float64, pairs within 2^-40 relative of the
 * threshold, 0, 0}.                                                                             */
int agx_radius_count(const agx_index_t* index, const float* q_latlon /*DEV*/, int64_t nq, double radius,
                     int32_t* counts /*DEV nq*/, void* stream);
int agx_exclusive_scan(const int32_t* counts /*DEV n*/, int64_t n, int64_t* offsets /*DEV n+1*/,
                       int64_t* total /*HOST or NULL; sync if given*/, void* stream);
int agx_radius_fill(const agx_index_t* index, const float* q_latlon /*DEV*/, int64_t nq, double radius,
                    const int64_t* offsets /*DEV nq+1*/, int32_t* out_src /*DEV*/, int32_t* out_dst /*DEV*/,
                    int64_t dst_base, int64_t* stats /*DEV or NULL*/, void* stream);

/* ---- grid reference distance --------------------------------------------------------------------
 * Replaces `dists[dists > 0].max()` (utils.py:62-63) on the float64 rdist of a k=2 self query
 * (agx_knn with out_rdist): largest strictly positive value and its flat position.            */
int agx_max_positive(const double* values /*DEV n*/, int64_t n, double* out_value /*HOST*/,
                     int64_t* out_index /*HOST*/, void* stream);
/* Host half of the same (NO device work, all pointers HOST): the nodes the GPU search nominates (those whose
 * nearest-neighbour distance is within rounding of the largest) are re-evaluated with the C library's sin / cos -
 * the calls sklearn's compiled HaversineDistance64 makes (_dist_metrics.pyx.tp:2639-2648) - so that the cut-off
 * radius carries the reference's bits: out_rdist = max over candidates c of min over its n_nb neighbours of
 * rdist(q[c], nb[c][j]) (exact compares; a zero minimum - duplicate points - is skipped like `dists > 0`).   */
int agx_host_reference_rdist(const float* q_latlon /*HOST n_cand*2*/, const float* nb_latlon /*HOST n_cand*n_nb*2*/,
                             int64_t n_cand, int n_nb, double* out_rdist /*HOST*/);

/* ---- node pruning -------------------------------------------------------------------------------------
 * RemoveUnconnectedNodes (processors/post_process.py:45-60 update_edge_indices, :133-149 compute_mask):
 * agx_mark_nodes sets flags[v] = 1 for every endpoint v in an edge row (flags pre-zeroed / pre-seeded by the caller,
 * AGX_ERR_ARG if an endpoint is outside [0, n_nodes)); after agx_exclusive_scan(flags) -> new_index,
 * agx_relabel_nodes rewrites a row in place as new_index[v] - the reference's python dict + Tensor.apply_.       */
int agx_mark_nodes(const int32_t* row /*DEV n*/, int64_t n, int64_t n_nodes, int32_t* flags /*DEV n_nodes*/, void* stream);
int agx_relabel_nodes(int32_t* row /*DEV n, in place*/, int64_t n, const int64_t* new_index /*DEV n_nodes+1*/, void* stream);
/* agx_relabel_nodes over up to 8 rows in ONE launch (rows / lens: HOST arrays of n_rows device pointers / lengths):
 * every index row that was built in a provisional node numbering, rewritten when the order resolves.            */
int agx_relabel_rows(int32_t* const* rows /*HOST n_rows x DEV*/, const int64_t* lens /*HOST n_rows*/, int n_rows,
                     const int64_t* new_index /*DEV*/, void* stream);

/* ---- edge post-processors -----------------------------------------------------------------------------
 * RestrictEdgeLength / SortEdgeIndexBySourceNodes / SortEdgeIndexByTargetNodes (processors/post_process.py of newer
 * releases; replaces pulling edge_index and every attribute to the host, masking / argsorting them there and writing
 * them back).  Each ends in ONE int32 index list applied to every per-edge array of an edge set.
 * agx_restrict_flags: keep[i] = 0 iff edge i is subject to the restriction (src_mask[src] and dst_mask[dst], each mask
 * optional: uint8 per node, non-zero = subject) and its rdist (agx_rdist64 of target, source) > sin^2(max_radius / 2) - the
 * test CutOffEdges applies (agx_radius_*), so the two agree bit for bit; 1 otherwise.  max_radius in radians, >= 0.
 * AGX_ERR_ARG (after the pass, one read-back) if an endpoint is outside [0, n_src_nodes) / [0, n_dst_nodes); keep is
 * then undefined.  The list of kept positions is agx_compact_flags(keep) (keep from cudaMalloc: 4-byte aligned).     */
int agx_restrict_flags(const int32_t* edge_src /*DEV E*/, const int32_t* edge_dst /*DEV E*/, int64_t n_edges,
                       const float* src_latlon /*DEV ns*2*/, int64_t n_src_nodes, const float* dst_latlon /*DEV nt*2*/,
                       int64_t n_dst_nodes, const uint8_t* src_mask /*DEV ns or NULL*/,
                       const uint8_t* dst_mask /*DEV nt or NULL*/, double max_radius, uint8_t* keep /*DEV E*/,
                       void* stream);
/* agx_sort_edges: perm = the stable permutation that orders the columns lexicographically by (key_row, other_row),
 * ascending or (descending != 0) descending; columns equal in both rows keep their input order.  The rows are packed
 * into 64-bit keys as in agx_concat_edges (same kernel, same trimming to the bits the node counts can set) and
 * sorted with CUB's radix SortPairs / SortPairsDescending, positions as values.  Scratch: 20 bytes per edge + CUB's.
 * AGX_ERR_ARG if E >= 2^31 or an endpoint is outside [0, n_key_nodes) / [0, n_other_nodes) (checked by the packing
 * pass, one read-back at the end; perm is then undefined).                                                         */
int agx_sort_edges(const int32_t* key_row /*DEV E*/, const int32_t* other_row /*DEV E*/, int64_t n_edges,
                   int64_t n_key_nodes, int64_t n_other_nodes, int descending, int32_t* perm /*DEV E*/, void* stream);
/* agx_gather_edge_columns: for each of n_arrays <= 8 arrays (src / dst / row_bytes: HOST arrays of DEV pointers and
 * sizes) row j of dst = row index[j] of src, j < n_index, in ONE launch; a caller with more arrays calls again.  An
 * array is any row-major (rows, row_bytes) buffer - the two rows of an edge_index count as two arrays of E rows.  Rows
 * of any byte size up to 2^20 are moved as the widest word (16, 8, 4, 2 or 1 bytes) that divides the row size and both
 * pointers' alignment.  index entries must lie inside every src; dst must not overlap src.  No read-back.            */
int agx_gather_edge_columns(int n_arrays, const void* const* src /*HOST n_arrays x DEV*/,
                            void* const* dst /*HOST n_arrays x DEV*/, const int64_t* row_bytes /*HOST n_arrays*/,
                            const int32_t* index /*DEV n_index*/, int64_t n_index, void* stream);

/* ---- masked node sets -------------------------------------------------------------------------------------
 * NodeMaskingMixin.undo_masking (edges/builder.py:176-193: compact indices of the row-selected coordinates mapped back
 * to node indices through a python dict + np.vectorize) fused into the searches' writes: while maps are set (thread-
 * local, read when a search is launched) agx_knn* / agx_radius_fill store src_map[reference index] / dst_map[query
 * index] instead of the index / dst_base + query.  Maps: DEV int64, ascending (np.where(mask)[0]); NULL = identity.
 * Decisions (ties by lower index) are unaffected: an ascending map preserves the order.  Reset with (NULL, NULL).  */
void agx_set_output_maps(const int64_t* src_map /*DEV or NULL*/, const int64_t* dst_map /*DEV or NULL*/);

/* ---- merged edge lists --------------------------------------------------------------------------------
 * utils.concat_edges (utils.py:66-81: torch.unique(torch.cat([e1, e2], dim=1), dim=1)): the columns of two (2, E) int32
 * edge lists sorted lexicographically by (source, target), duplicates removed - what a second edge builder on the same
 * node pair does to the edge set (edges/builder.py:105-110).  Both lists are packed into 64-bit keys by one kernel,
 * radix-sorted over the key bits the node counts can set, and the distinct keys unpacked into `out`: the caller's
 * RESULT allocation of 2 * (na + nb) int32, which doubles as the sort's alternate buffer - so the scratch besides the
 * result is one key buffer (8 bytes per input edge).  On return (one read-back) the first 2 * n_unique int32 of `out`
 * are the (2, n_unique) result, row-major.                                                                       */
int agx_concat_edges(const int32_t* a_src /*DEV na*/, const int32_t* a_dst, int64_t na, const int32_t* b_src /*DEV nb*/,
                     const int32_t* b_dst, int64_t nb, int64_t n_src_nodes, int64_t n_dst_nodes,
                     int32_t* out /*DEV 2*(na+nb), 8-byte aligned*/, int64_t* n_unique /*HOST*/, void* stream);

/* ---- node ordering, device half ---------------------------------------------------------------------------
 * get_coordinates_ordering (generate/utils.py:15-33): the two (unstable, order-defining) argsorts stay numpy's on the
 * host; given their results this evaluates `order = arange(n)[index_latitude][index_longitude[::-1]]`, its inverse
 * `rank` (rank[order[i]] = i: the map agx_relabel_nodes applies to provisionally numbered index rows) and
 * `x_out = x_in[order]` (nodes/builders/from_refined_icosahedron.py:66) in one kernel.                        */
int agx_order_resolve(const int64_t* index_latitude /*DEV n*/, const int64_t* index_longitude /*DEV n*/, int64_t n,
                      const float* x_in /*DEV n*2*/, float* x_out /*DEV n*2*/, int64_t* order /*DEV n*/,
                      int64_t* rank /*DEV n*/, void* stream);

/* ---- stream gates -------------------------------------------------------------------------------------------
 * What lets the host queue the work that FOLLOWS the node order (tie re-decision, relabel, scaling, device -> host
 * copies) while numpy is still sorting (generate/utils.py:15-33 is host code in the reference and stays host code
 * here): everything queued on `stream` behind agx_gate_wait starts when *gate == 1.  `gate` is one 32-bit word of
 * page-locked HOST memory (cudaHostAlloc / cudaHostRegister), 0 when the wait is queued.  It is opened by
 * agx_gate_open queued on another stream (behind the upload of the order and agx_order_resolve) or, when the sorting
 * thread failed, by a plain CPU store of 1 so that the device never waits for a result that will not come.
 * Implemented with cuStreamWaitValue32 / cuStreamWriteValue32: no SM is occupied while waiting.
 * agx_gate_supported: 1 if both operations work on the current device (one functional self-test per device,
 * remembered); callers keep their un-gated path otherwise.                                                      */
int agx_gate_supported(void);
int agx_gate_wait(const uint32_t* gate /*HOST page-locked*/, void* stream);
int agx_gate_open(uint32_t* gate /*HOST page-locked*/, void* stream);

/* ---- edge attributes ------------------------------------------------------------------------------
 * agx_node_tables: everything the attribute kernel needs from ONE node, as one 32-byte record per role:
 *   src_rec  float[8]  = (x, y, z, cos lat, lat, lon, 0, 0) - float32 unit vector and cos(lat) with numpy's
 *            float32 sin/cos bits (generate/transforms.py:106-110, utils.py:84-103);
 *   dst_rec  double[4] = (qx, qy, qw, bits(lat, lon)) - the float64 quaternion (z = 0) of the rotation taking the
 *            node to the north pole (edges/directional.py:19-37, epsilon-nudge of generate/transforms.py:133-140
 *            included); the 4th double carries the node's float32 (lat, lon) bit patterns (lat in the low word).
 * Either pointer may be NULL (a node set used only as source / only as target).
 * agx_edge_attrs: replaces EdgeLength.compute / EdgeDirection.compute (edges/attributes.py:42-157):
 * raw values (float32 store) + global statistics in one pass over the edges, then - if a norm was asked for -
 * an in-place scaling pass.  len_norm / dir_norm = AGX_NORM_* or -1 to skip the attribute;
 * dir_rotated = luse_rotated_features.  A NaN value (an antipodal pair's length) makes every normalised value of its
 * attribute NaN, as numpy's sum / amax / amin / std do in the reference.
 * out_dir, in this call and in _stats and _apply, must be 8-byte aligned (one float2 store per edge; AGX_ERR_ARG
 * otherwise, before any device work) - a view of an (E, 2) float32 array at any row is.                           */
int agx_node_tables(const float* latlon /*DEV n*2*/, int64_t n, float* src_rec /*DEV n*8 or NULL*/,
                    double* dst_rec /*DEV n*4 or NULL, 32-byte aligned*/, void* stream);
/* Node inputs of the attribute calls, per side EITHER a record table from agx_node_tables (src_rec / dst_rec; small node
 * sets whose tables stay in L2) OR the node set's float32 (lat, lon) coordinates (src_latlon / dst_latlon; large node
 * sets: the kernel evaluates xyz / the rotation quaternion per edge from 8 bytes instead of gathering a 32-byte record
 * that had to be written first) - exactly one of the two pointers of a side is non-NULL.  Both forms give bit-identical
 * attributes.                                                                                                       */
int agx_edge_attrs(const int32_t* edge_src /*DEV E*/, const int32_t* edge_dst /*DEV E*/, int64_t n_edges,
                   const float* src_rec /*DEV or NULL*/, const float* src_latlon /*DEV ns*2 or NULL*/,
                   const double* dst_rec /*DEV or NULL*/, const float* dst_latlon /*DEV nt*2 or NULL*/,
                   int len_norm /*AGX_NORM_* or -1 = skip*/, int len_invert, float* out_len /*DEV E*/,
                   int dir_norm /*AGX_NORM_* or -1 = skip*/, int dir_rotated, float* out_dir /*DEV E*2, 8-byte aligned*/,
                   double* workspace /*DEV, >= agx_edge_attrs_workspace() doubles*/,
                   int regular_k /*k > 0: the edges of the i-th target are columns [i k, (i+1) k) - a KNN result; 0: any list*/,
                   void* stream);
int64_t agx_edge_attrs_workspace(void);
/* The two halves of agx_edge_attrs, for callers that normalise over more than one call: one rank's SHARD of a
 * multi-GPU build, or KNN edges whose sources of a few targets are re-decided later.
 * _stats evaluates the raw values of the edges ONCE, writes them (float32, not yet normalised) to out_len / out_dir -
 * every requested output is required - and reduces them to
 * stats[8] = {len sum, sum of squares, min, max, dir sum, sum of squares, min, max} (float64; an empty set of edges
 * gives {0, 0, +1e300, -1e300}).  Which edges are evaluated and counted, by a per-TARGET flag byte
 * (dst_flags: DEV uint8[n_target_nodes]):
 *   flag_mode 0: every edge (dst_flags is not read);
 *   flag_mode 1 ("skip"): every edge is evaluated and written, edges INTO a flagged target stay out of the statistics;
 *   flag_mode 2 ("only"): only the edges into flagged targets are evaluated, written and counted.  Instead of dst_flags
 *     (then NULL) the flagged targets may be given as a LIST of a regular-k edge list (list = ascending target ids,
 *     *count = its length, both in device memory - agx_compact_flags; the edges of target t are [t k, (t+1) k)): the
 *     few re-decided queries then cost one small launch instead of a pass over every target index.
 * regular_k > 0 without a list: the edges of the i-th target are columns [i k, (i+1) k), walked by target.
 * For KNN edges built while the source numbering was provisional (agx_knn_flagged): mode 1 right after the search,
 * mode 2 after agx_knn_redecide_ranked, each into its own statistics set - the decoder's trigonometry then runs in the
 * shadow of the host sort and only the scaling pass follows it.
 * _apply is the scaling pass: it normalises the n_edges raw values at out_len / out_dir in place with the
 * n_stat_sets statistics sets at stats (8 doubles each; every rank's sets, in rank order - they are folded in that
 * order, so every rank derives bit-identical constants) and the global edge count.  normalise.py:20-55.          */
int agx_edge_attrs_stats(const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, const float* src_rec,
                         const float* src_latlon, const double* dst_rec, const float* dst_latlon, int want_len,
                         int want_dir, int dir_rotated, float* out_len /*DEV E if want_len*/,
                         float* out_dir /*DEV E*2 if want_dir*/, double* stats /*DEV 8*/, double* workspace,
                         const uint8_t* dst_flags /*DEV or NULL*/, int flag_mode /*0, 1 = skip, 2 = only*/,
                         const int32_t* list /*DEV or NULL*/, const int64_t* count /*DEV or NULL*/, int regular_k,
                         void* stream);
int agx_edge_attrs_apply(int64_t n_edges, int len_norm, int len_invert, float* out_len /*DEV E*/, int dir_norm,
                         int dir_rotated, float* out_dir /*DEV E*2, 8-byte aligned*/,
                         const double* stats /*DEV n_stat_sets*8 or NULL if no norm*/, int n_stat_sets,
                         int64_t n_edges_global, double* workspace, void* stream);
/* agx_edge_azimuth (Azimuth): out[e] = float32 of the initial bearing at the target towards the source, in radians,
 * clockwise from north, in [-pi, pi]: atan2(sin(dlon) cos(lat_s), cos(lat_t) sin(lat_s) - sin(lat_t) cos(lat_s) cos(dlon)),
 * dlon = lon_s - lon_t, in float64 from the float32 coordinates (8-byte aligned).  norm = AGX_NORM_*, over the whole
 * edge set with EdgeLength's arithmetic and NaN rule (the K5 fold / parameter / scaling kernels).  AGX_ERR_ARG (after
 * the pass, one read-back) if an endpoint is outside [0, n_src_nodes) / [0, n_dst_nodes): such an endpoint is never
 * read and out is then undefined.                                                                                 */
int agx_edge_azimuth(const int32_t* edge_src /*DEV E*/, const int32_t* edge_dst /*DEV E*/, int64_t n_edges,
                     const float* src_latlon /*DEV ns*2*/, int64_t n_src_nodes, const float* dst_latlon /*DEV nt*2*/,
                     int64_t n_dst_nodes, int norm, float* out /*DEV E*/,
                     double* workspace /*DEV, >= agx_edge_attrs_workspace() doubles*/, void* stream);
/* agx_gaussian_weights (GaussianDistanceWeights): w = exp(-d^2 / (2 sigma^2)) in float64 from lengths[e] (the float32
 * EdgeLength values, unit sphere), normalised with norm = AGX_NORM_* within each group of edges that share a target
 * (edge_dst), rounded to float32 once: out[e] = float32((w - shift[t]) / div[t]).  The statistics of a group are reduced
 * over its edges in the order of perm - which must be agx_sort_edges(key = edge_dst, other = edge_src, ascending) of
 * the same rows, so the endpoints are checked and the result does not depend on the column order - in one fixed tree.
 * unit-std: two passes; a group whose weights are bit-equal is left unnormalised.  A NaN weight makes its group NaN.
 * norm = AGX_NORM_NONE: out = float32(w), and perm / scratch / edge_dst may be NULL.  edge_src and n_src_nodes are not
 * read: the weights depend on the lengths and the target row only.  sigma > 0.  No read-back.
 * scratch: DEV, 16-byte aligned, >= agx_gaussian_weights_scratch_bytes(n_edges, n_dst_nodes) bytes
 * = 32 n_dst + 64 + 48 (E / 1024 + 1) + 32 (2 (E / 1024) + 2) (a (shift, div) table and the group bounds per target, the
 * groups of more than 1024 edges and their partial statistics).                                                    */
int agx_gaussian_weights(const int32_t* edge_src /*DEV E*/, const int32_t* edge_dst /*DEV E*/, int64_t n_edges,
                         int64_t n_src_nodes, int64_t n_dst_nodes, const float* lengths /*DEV E*/, double sigma, int norm,
                         const int32_t* perm /*DEV E or NULL for norm None*/, float* out /*DEV E*/,
                         void* scratch /*DEV or NULL for norm None*/, void* stream);
int64_t agx_gaussian_weights_scratch_bytes(int64_t n_edges, int64_t n_dst_nodes);

/* ---- icosphere + multi-scale edges -------------------------------------------------------------------
 * agx_icosphere: replaces trimesh.creation.icosphere (generate/tri_icosahedron.py:121,173):
 * float64 vertices (10*4^r+2, 3) and int32 faces (20*4^r, 3) of every level 0..max_level, in
 * trimesh's numbering (level-r vertices are a prefix of level-(r+1)); also float32 (lat, lon) of
 * the finest level per generate/transforms.py:34-52.  Buffers sized for the finest level;
 * `faces_all` holds the levels back to back (level r at offset 20*(4^r-1)/3 faces).
 * agx_multiscale_tri: replaces tri_icosahedron.add_edges_to_nx_graph + nx.to_scipy_sparse_array
 * (generate/tri_icosahedron.py:138-224, edges/builder.py:412-455) for global TriNodes: union over the
 * requested levels of vertex pairs within x_hops mesh hops, relabelled by `rank_of_vertex`
 * (position in node_ordering), emitted sorted by (dst, src).  count -> fill via `offsets`.      */
int agx_icosphere(int max_level, double* vertices /*DEV nv*3*/, int32_t* faces_all /*DEV*/,
                  float* latlon /*DEV nv*2 or NULL*/, void* stream);
int agx_multiscale_tri_count(int max_level, const int32_t* faces_all /*DEV*/, const int32_t* levels /*HOST*/,
                             int n_levels, int x_hops, const int32_t* node_ordering /*DEV nv*/,
                             const int32_t* rank_of_vertex /*DEV nv*/, int32_t* counts /*DEV nv*/,
                             int32_t* scratch /*DEV nv*agx_multiscale_scratch_per_node()*/, void* stream);
int64_t agx_multiscale_scratch_per_node(int n_levels, int x_hops);
/* Limited-area / stretched variant (generate/tri_icosahedron.py:177-187,214-215; edges/builder.py:422-432):
 * the graph has n_nodes nodes that are a SUBSET (or a mix of two levels) of icosphere vertices.
 * vertex_map[v] (v < nv(max_level)) = graph position of vertex v, or -1 if the vertex is masked out - the
 * same array serves every level because lower levels are prefixes; node_vertex[l*n_nodes + t] = the vertex
 * of requested level l that graph node t is, or -1.  Mesh edges with a masked endpoint are not walked.  */
int agx_multiscale_tri_count_mapped(int max_level, const int32_t* faces_all /*DEV*/, const int32_t* levels /*HOST*/,
                                    int n_levels, int x_hops, int64_t n_nodes, const int32_t* vertex_map /*DEV*/,
                                    const int32_t* node_vertex /*DEV n_levels*n_nodes*/, int32_t* counts /*DEV n_nodes*/,
                                    int32_t* scratch /*DEV n_nodes*agx_multiscale_scratch_per_node()*/, void* stream);
int agx_multiscale_tri_fill(int64_t n_nodes, const int32_t* counts, const int64_t* offsets /*DEV nv+1*/,
                            const int32_t* scratch, int64_t scratch_per_node, int32_t* out_src,
                            int32_t* out_dst, void* stream);

/* ---- hexagonal (H3) hidden mesh ------------------------------------------------------------------------
 * agx_hex_cells: replaces `h3.uncompact(h3.get_res0_indexes(), res)` + `np.deg2rad(h3.h3_to_geo(idx))`
 * (generate/hex_icosahedron.py:47,99): the float64 (lat, lon) radians of all agx_hex_num_cells(res) =
 * 2 + 120*7^res cell centres of an H3 resolution, in (icosahedron face, lattice i, lattice j) order - H3's own
 * order is a Python set's, the reference re-orders by get_coordinates_ordering anyway - and the pentagon flags.
 * The H3 library itself is not available to this build: the geometry is restated from its published
 * definition (faceijk.c _hex2dToGeo, coordijk.c _downAp7/_downAp7r, geoCoord.c _geoAzDistanceRads) and
 * checked against the two cell centres H3's documentation prints (oracle/h3_restated.py).
 * agx_hex_adjacency: the cells sharing an edge with each cell, nb[6*u + s] (-1 padded), deg[u] = 6 (5 for the 12
 * pentagons), from row 0 of an `agx_knn(k = 7)` self query of the centres: on an aperture-7 grid the 6 nearest
 * centres ARE the edge neighbours (second ring sqrt(3) x farther, gnomonic distortion <= 1.26).  One BFS step
 * over this table = one ring of `h3.k_ring` (generate/hex_icosahedron.py:147).
 * agx_multiscale_adj_count: the multi-scale expansion of agx_multiscale_tri_count over caller-supplied
 * adjacency tables (HOST arrays of n_levels DEV pointers): nb / deg as above; cell_node[l][c] = graph position
 * of the node that level-l cell c stands for (`h3_to_center_child`, hex_icosahedron.py:149-150) or -1;
 * node_cell[l][t] = the inverse or -1.  walk_all = 1 walks the full disk and drops invalid cells afterwards
 * (`k_ring(idx, k) & nodes`), 0 never crosses an invalid cell (the tri rule).  Fill with
 * agx_multiscale_tri_fill; scratch as agx_multiscale_scratch_per_node.                                   */
int64_t agx_hex_num_cells(int res);
int agx_hex_cells(int res, double* latlon /*DEV n*2*/, uint8_t* pentagon /*DEV n or NULL*/, void* stream);
int agx_hex_adjacency(const int32_t* knn7 /*DEV n*7*/, const uint8_t* pentagon /*DEV n*/, int64_t n,
                      int32_t* nb /*DEV n*6*/, int32_t* deg /*DEV n*/, void* stream);
int agx_multiscale_adj_count(int n_levels, const int32_t* const* nb /*HOST[n_levels] of DEV*/,
                             const int32_t* const* deg, const int32_t* const* cell_node,
                             const int32_t* const* node_cell, int x_hops, int walk_all, int64_t n_nodes,
                             int32_t* counts /*DEV n_nodes*/, int32_t* scratch /*DEV*/, void* stream);

/* ---- HEALPix nodes (SURVEY section 2; not on the section-8 path, kept next to the other mesh generators) ---------
 * Replaces `hp.pix2ang(2**resolution, range(npix), nest=True, lonlat=True)` + reshape_coords
 * (nodes/builders/from_healpix.py:61-66): float32 (lat, lon) radians of the 12 * 4^resolution pixel centres in NESTED
 * order.  healpy is not available to this build: HEALPix's published pix2loc is restated and checked against the
 * independent RING-scheme formulas (oracle/healpix_restated.py).                                             */
int agx_healpix_nodes(int resolution /*log2 nside*/, float* latlon /*DEV npix*2*/, void* stream);

/* ---- octahedral reduced Gaussian grid O<n> (ReducedGaussianGridNodes of newer releases) ---------------------------
 * Upstream reads the grid from a downloaded file; O<n> is defined by its construction, which grids.octahedral_grid +
 * latlon_deg_to_x restate on the host (the oracle).
 * agx_gaussian_latitudes: the 2n Gaussian latitudes (roots of the Legendre polynomial P_2n) in float64 degrees, north to
 * south, within 1e-13 degrees of the exact roots; row 2n-1-k is the exact negation of row k.
 * agx_octahedral_nodes: float32 (lat, lon) radians of the 4n(n+9) points from those latitudes, north to south and west to
 * east from 0 degrees; row i (1-based from the nearer pole) holds 4i + 16 points at lon = j * (360 / (4i + 16)) degrees.
 * Bit for bit the oracle's float32 values wherever the latitudes are within float32 rounding (DESIGN section 4).
 * Both: AGX_ERR_ARG for n < 1, for 4n(n+9) > INT32_MAX and for a NULL pointer.                                    */
int agx_gaussian_latitudes(int n, double* lat_deg /*DEV 2n*/, void* stream);
int agx_octahedral_nodes(int n, const double* lat_deg /*DEV 2n*/, float* latlon /*DEV 4n(n+9)*2*/, void* stream);

/* ---- node attribute: spherical Voronoi cell areas (SURVEY section 8f, row N3) -------------------------------
 * Replaces `SphericalVoronoi(points, radius, centre).calculate_areas()` in SphericalAreaWeights.get_raw_values
 * (nodes/attributes.py:199-221), points = latlon_rad_to_cartesian(x) in float32 (generate/transforms.py:106-110).
 * The region of generator p is { x : x.(q - p) <= 0 for all q } with the float32 generators as given (scipy's hull
 * facets); knn = row 0 of an agx_knn self query of the m listed generators (`subset`, NULL = all n, in order), k
 * entries each (self included), ascending; exhaustive = 1 states that the lists hold EVERY generator (k = n), so a cell
 * is complete when they are used up.  areas[i] (float64, indexed by generator) is written for every generator
 * whose cell closed; status[t] (indexed by list position) = 0 done, 1 / 2 = the k neighbours did not close the cell
 * (retry that generator with a larger k), 3 = duplicate generators, 4 = more than 32 cell edges.              */
int agx_voronoi_areas(const float* latlon /*DEV n*2*/, int64_t n, const int32_t* knn /*DEV m*k*/, int k, int exhaustive,
                      const int32_t* subset /*DEV m or NULL*/, int64_t m, double radius, double* areas /*DEV n*/,
                      int32_t* status /*DEV m*/, void* stream);
/* The same for at most 64 generators, whose cells can be wider than a hemisphere (the reference works from 4 generators):
 * exhaustive on the sphere - every pair of bisector planes, both meeting directions, kept iff inside every other
 * half-space; vertices ordered by azimuth about the generator; the same solid-angle sum.  status as above.        */
int agx_voronoi_areas_small(const float* latlon /*DEV n*2*/, int64_t n, const int32_t* subset /*DEV m or NULL*/, int64_t m,
                            double radius, double* areas /*DEV n*/, int32_t* status /*DEV m*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AGX_B200_H */
