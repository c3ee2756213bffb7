/*
 * s3b200 -- C-ABI of the B200-native hot path of Sparse Spatial Sampling (S^3).
 *
 * The reference (JanisGeise/sparseSpatialSampling) has no FFI: its boundary is the Python class
 * surface.  This header is the boundary a maintainer binds with ctypes (see INTEGRATION.md); every
 * entry point names the reference code it replaces (paths relative to the reference repository).
 *
 * Conventions
 *   - every function returns 0 on success, a negative S3_ERR_* code otherwise; the message of the
 *     last failure on the calling thread is returned by s3_last_error(); nothing throws;
 *   - all `d_*` pointers are DEVICE pointers to caller-owned, contiguous buffers; the library only
 *     owns the opaque handles it hands out (s3_knn_t, s3_geom_t);
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, no hidden device sync
 *     unless stated;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef S3B200_H
#define S3B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S3_F32 0
#define S3_F64 1

typedef struct s3_knn s3_knn_t;
typedef struct s3_geom s3_geom_t;
typedef struct s3_topo s3_topo_t;

/* ---- library ---------------------------------------------------------------------------------- */
const char* s3_last_error(void);
int s3_version(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
int64_t s3_launch_count(void);

/* ---- k-nearest-neighbour index over the original point cloud ---------------------------------
 * replaces sklearn KNeighborsRegressor / NearestNeighbors as used in
 *   sparseSpatialSampling/s_cube.py:161-163 (fit), :224, :328, :372 (predict)
 *   sparseSpatialSampling/export.py:120, :423-441 (fit, kneighbors, inverse-distance weights)      */

/* d_coords: fp64 [n, dim] row-major (dim = 2|3); d_values: fp64 [n] regression targets or NULL.
 * Synchronises `stream` once before returning. */
int s3_knn_build(const double* d_coords, int64_t n, int dim, const double* d_values, void* stream,
                 s3_knn_t** out);
int s3_knn_free(s3_knn_t* h);
/* kneighbors(): d_idx int64 [nq, k], d_dist fp64 [nq, k], ascending distance (ties: smaller index) */
int s3_knn_query(const s3_knn_t* h, const double* d_query, int64_t nq, int k, int64_t* d_idx,
                 double* d_dist, void* stream);
/* KNeighborsRegressor(weights="distance").predict(): d_pred fp64 [nq] */
int s3_knn_predict(const s3_knn_t* h, const double* d_query, int64_t nq, int k, double* d_pred,
                   void* stream);
/* ExportData._build_knn_cache (export.py:403-444): idx int32 [nq,k], normalised inverse-distance
 * weights as fp32 [nq,k] and (optional, may be NULL) fp64 [nq,k] */
int s3_knn_tables(const s3_knn_t* h, const double* d_query, int64_t nq, int k, int32_t* d_idx,
                  float* d_w32, double* d_w64, void* stream);

/* Morton (Z-curve) ordering of a point set, used to process the sampled cells in a cache-friendly order:
 * d_perm int32 [n] = indices of the points sorted along the curve                                  */
int s3_morton_order(const double* d_coords, int64_t n, int dim, int32_t* d_perm, void* stream);

/* ---- refinement engine (device side of SamplingTree, sparseSpatialSampling/s_cube.py) -------------
 * Cell state: structure of arrays indexed by the reference's cell index (creation order):
 *   d_center fp64 [cap, dim], d_level int32 [cap], d_gain fp64 [cap], d_metric fp64 [cap],
 *   d_flags uint8 [cap] (bit 0 = leaf, bit 1 = invalid / removed by a geometry).                     */

/* children of `d_parents[i]` get indices first_child + i*2^dim + c, c in CH order
 * (s_cube.py:29,188-194); centre = fl(parent + dir * 0.25*width/2^level) (s_cube.py:399-445,865-902);
 * parents lose, children get the leaf flag (_update_leaf_cells, s_cube.py:243-251)                 */
int s3_cells_refine(double* d_center, int32_t* d_level, uint8_t* d_flags, const int64_t* d_parents,
                    int64_t n_parents, int64_t first_child, int dim, double width, void* stream);

/* SamplingTree._update_gain (s_cube.py:207-241) + numba _update_gain (s_cube.py:1840-1859):
 * KNN/IDW metric at the cell centre and at the 2^dim would-be child centres, sum|m0-mj|, gain.
 * Cells: d_cells[i] (int64 [n]) if non-NULL, else first + i. sdm_order: association of the 8-term
 * sum in 3-D (0 sequential, 1 = torch's 4-lane order); 2-D is always sequential.                    */
int s3_cells_gain(const s3_knn_t* knn, const double* d_center, const int32_t* d_level,
                  const int64_t* d_cells, int64_t first, int64_t n, int k, double width, double gain0,
                  int sdm_order, double* d_metric, double* d_gain, void* stream);

/* _remove_invalid_cells / _check_cell_validity / GeometryObject.check_cell / _apply_mask
 * (s_cube.py:669-732,1816-1837; geometry/geometry_base.py:40-76; the shape files under geometry/).
 * Geometry tables: d_geom_hdr int32 [n_geoms,4] = {type, keep_inside, param offset, n_extra},
 * d_geom_par fp64 flat parameters (layout per type: the classes in sparsespatialsampling_b200/geometry).
 * only_geom >= 0 restricts the test to one geometry; refine_mode = the reference's refine_geometry;
 * apply != 0 additionally marks invalid cells (flags = invalid, gain = 0; s_cube.py:721-731).
 * d_invalid uint8 [n]: 1 where check_cell() returned True for some geometry.
 * Closed triangulated surfaces (GeometrySTL3D, geometry_STL_3d.py:81-124): bit g of `stl_geoms` says that geometry g
 * is of that type and stored in the tiled layout (triangles in Morton order + one bounding box per 128 triangles, see
 * csrc/stl.cuh); those are evaluated by a separate kernel -- one thread per node, triangle tiles streamed through
 * shared memory, tiles and triangles rejected by bounding box -- before the mask kernel combines the flags.
 * `stl_meta` is a HOST array int32 [n_geoms, 2] = {parameter offset, n_triangles} (the header's numbers);
 * stl_geoms = 0 keeps every geometry on the per-thread path.                                          */
int s3_cells_mask(const double* d_center, const int32_t* d_level, const int64_t* d_cells, int64_t first,
                  int64_t n, int dim, double width, const int32_t* d_geom_hdr, const double* d_geom_par,
                  int n_geoms, int only_geom, int refine_mode, int apply, uint8_t* d_invalid,
                  uint8_t* d_flags, double* d_gain, int stl_geoms, const int32_t* stl_meta, void* stream);

/* GeometryObject.check_cell on explicit node sets: d_nodes fp64 [n, n_nodes, dim] -> d_invalid uint8 [n]
 * (geometry/geometry_base.py:150-163 and the per-shape check_cell methods)                           */
int s3_nodes_mask(const double* d_nodes, int64_t n, int n_nodes, int dim, const int32_t* d_geom_hdr,
                  const double* d_geom_par, int n_geoms, int only_geom, int refine_mode,
                  uint8_t* d_invalid, int stl_geoms, const int32_t* stl_meta, void* stream);
/* per-point inside mask of geometry `geom` (the reference's _mask_* / check_triangle / check_tetrahedron) */
int s3_points_inside(const double* d_points, int64_t n, int dim, const int32_t* d_geom_hdr,
                     const double* d_geom_par, int geom, uint8_t* d_inside, int stl_geoms, const int32_t* stl_meta,
                     void* stream);

/* heapq.nlargest(k, leaf, key=(gain, -idx)) (s_cube.py:601-602): radix select + stable radix sort.
 * d_out int64 [k], ordered by (gain descending, index ascending). Requires k <= number of leaves.   */
int s3_select_topk(const double* d_gain, const uint8_t* d_flags, int64_t n_cells, int64_t k,
                   int64_t* d_out, void* stream);
/* implementation switch (tests / benchmarking): 1 = one cooperative launch for k <= 8192 (default), 0 = multi-kernel */
int s3_select_set_fused(int on);

/* ---- cell topology (HOST side, plain integer bookkeeping; all pointers are host pointers) -----------
 * The reference's neighbour pointers and shared node ids are history dependent (see csrc/topology.cu); this
 * handle replays them: Cell.nb / Cell.node_idx / Cell.children of s_cube.py:30-85.
 *   s3_topo_create        _create_first_cell (s_cube.py:338-397): root cell, its 2^d nodes. async != 0: updates
 *                         (refine / refresh / mark_invalid) are queued and applied in order by a native worker thread
 *                         next to the device work; reads wait for the queue, s3_topo_sync reports a queued failure
 *   s3_topo_refine        per parent, in the given order: _assign_neighbors + _assign_indices
 *                         (s_cube.py:904-1186, 1188-1536) as called from _refine_cells / _refine_uniform
 *   s3_topo_refresh       cell.parent.children = _assign_neighbors(cell.parent, children=...) (s_cube.py:611,
 *                         489-490, 826); of_parents != 0: the list holds the parents (s_cube.py:547-549)
 *   s3_topo_mark_invalid  neighbour reset of _remove_invalid_cells (s_cube.py:721-731)
 *   s3_topo_check_nb      _check_nb (s_cube.py:447-464): out int64 [26], returns the count (-1 on bad arguments)
 *   s3_topo_cell          raw pointers of one cell: nb int32 [8|26], node ids int32 [2^d], {parent, children, level}
 *                         (children: first child index, -1 = leaf, -2 = removed)
 *   s3_topo_final         _resort_nodes_and_indices_of_grid + renumber_node_indices_parallel (s_cube.py:734-772,
 *                         1695-1736): faces int32 [n_leaf, 2^d] in cell-list order, vertices fp64 [n_vertices, dim];
 *                         call with faces == NULL first to get the sizes; centers_by_index (optional) fp64
 *                         [n_cells, dim] = the host replay of all cell centres                                  */
int s3_topo_create(int dim, const double* root_center, double width, int async, s3_topo_t** out);
int s3_topo_free(s3_topo_t* h);
int s3_topo_sync(s3_topo_t* h);
int64_t s3_topo_n_cells(s3_topo_t* h);
int64_t s3_topo_n_nodes(s3_topo_t* h);
int s3_topo_refine(s3_topo_t* h, const int64_t* parents, int64_t n);
int s3_topo_refresh(s3_topo_t* h, const int64_t* cells, int64_t n, int of_parents);
int s3_topo_mark_invalid(s3_topo_t* h, const int64_t* cells, int64_t n);
int64_t s3_topo_check_nb(s3_topo_t* h, int64_t cell, int64_t* out);
int s3_topo_cell(s3_topo_t* h, int64_t cell, int32_t* nb_out, int32_t* node_out, int32_t* state_out);
int s3_topo_final(s3_topo_t* h, int64_t* n_leaf_out, int64_t* n_vertices_out, int32_t* faces,
                  double* vertices, double* centers_by_index);

/* sum of metric^2 over the leaves (_compute_captured_metric, s_cube.py:317-336) and of a plain
 * vector (the target norm, s_cube.py:205); d_out fp64 [1]; deterministic reduction tree             */
int s3_leaf_sumsq(const double* d_metric, const uint8_t* d_flags, int64_t n_cells, double* d_out,
                  void* stream);
int s3_sumsq(const double* d_x, int64_t n, double* d_out, void* stream);

/* ---- export-stage interpolation ---------------------------------------------------------------
 * replaces interpolate_data (sparseSpatialSampling/export.py:446-468):
 *   out[c, d, t] = sum_j w[c, j] * data[idx[c, j], d, t]
 * data is the reference's [n_src, n_comp, n_cols] snapshot batch (t contiguous) with explicit strides in
 * ELEMENTS: row_stride between source points, comp_stride between the components of a point; the result
 * [n_cells, n_comp, n_cols] likewise (out_row_stride, out_comp_stride). Dense tensors: comp_stride = n_cols,
 * row_stride = n_comp * n_cols. The kernel is built for row pitches that are multiples of 128 bytes (every warp
 * request then covers whole cache lines; DESIGN.md 3); any stride is accepted: 32-byte aligned strides and base
 * pointers take 256-bit loads (fp32 -> fp32), 16-byte aligned ones the 128-bit path, everything else a scalar one.
 * fp32 rows of up to 768 columns (the time windows of a sharded export) whose SOURCE is 32-byte aligned run in
 * a kernel of their own; it may load, never store, the (< 32) bytes between the last column of a row and the next
 * 32-byte boundary -- inside the row pitch by the alignment rule above.
 * dtypes: (data F32, out F32): w is fp32, fp32 FMA accumulation;
 *         (data F32|F64, out F64): w is fp64, products and sequential adds in fp64 (reference order).
 * d_out_row: optional int32 [n_cells] -- row of `out` that receives cell c (cells may be passed in
 * any processing order, e.g. Morton order); NULL = identity. 1 <= k <= 64.                           */
int s3_interp_gather_strided(const void* d_data, int data_dtype, int64_t n_src, int n_comp, int64_t n_cols,
                             int64_t row_stride, int64_t comp_stride, const int32_t* d_idx, const void* d_w,
                             int64_t n_cells, int k, const int32_t* d_out_row, void* d_out, int out_dtype,
                             int64_t out_row_stride, int64_t out_comp_stride, void* stream);
/* dense special case: data [n_src, row_len], out [n_cells, row_len] */
int s3_interp_gather(const void* d_data, int data_dtype, int64_t n_src, int64_t row_len,
                     const int32_t* d_idx, const void* d_w, int64_t n_cells, int k,
                     const int32_t* d_out_row, void* d_out, int out_dtype, void* stream);

/* ---- reconstruction error of a sampled grid --------------------------------------------------------
 * the exported field `sampled` [n_sampled, n_comp, n_cols] is interpolated back onto the original points with the
 * tables of the other direction (idx int32 / w fp32 [n_points, k]: the original points queried among the cell
 * centres, in processing order; d_out_row int32 [n_points]: the original row of each, NULL = identity) and compared
 * with `original` [n_points, n_comp, n_cols]:
 *   r = sum_j w[p, j] * sampled[idx[p, j], d, t]   (fp32 FMA chain in neighbour order: the bits of the fp32 gather)
 *   e = (double) r - (double) original[out_row[p], d, t]
 * results, fp64 [n_comp, n_cols] each: d_sq_err = sum_p e^2, d_sq_ref = sum_p original^2, d_max_abs = max_p |e|;
 * d_point_sq_err fp64 [n_points, n_comp] (optional, NULL = skipped): sum_t e^2 is ADDED into row out_row[p], so that
 * successive time windows accumulate. Strides in elements and alignment rules as in s3_interp_gather_strided, both
 * fields fp32 (anything else: S3_ERR_UNSUPPORTED). Every sum is reduced in a fixed order that depends on n_points only:
 * the results are bit-identical from run to run, and each column's results do not depend on the other columns of the
 * call (a time window gives the matching columns of the whole batch). 1 <= k <= 64.                      */
int s3_recon_error(const void* d_sampled, int sampled_dtype, int64_t n_sampled, int n_comp, int64_t n_cols,
                   int64_t s_row_stride, int64_t s_comp_stride, const void* d_original, int original_dtype,
                   int64_t n_points, int64_t o_row_stride, int64_t o_comp_stride, const int32_t* d_idx,
                   const float* d_w, const int32_t* d_out_row, int k, double* d_sq_err, double* d_sq_ref,
                   double* d_max_abs, double* d_point_sq_err, void* stream);

/* ---- streaming ingest -----------------------------------------------------------------------------
 * the reference feeds snapshot batches from host memory (export.py:128-167, utils.py:155-226). A window of the
 * time axis of a host field [rows, T] is a pitched 2-D region: one asynchronous copy per window and direction
 * (`kind` 0 = host to device, 1 = device to host; pinned host memory), `width`/pitches in bytes.            */
int s3_copy2d_async(void* dst, int64_t dst_pitch, const void* src, int64_t src_pitch, int64_t width,
                    int64_t height, int kind, void* stream);
/* the window [0, width) (fp32 elements) of the rows d_rows[0..n_rows) of a pitched fp32 matrix `src` into the dense
 * buffer d_dst [n_rows, dst_pitch]. `src` may be PINNED HOST memory (the kernel reads it over PCIe): only the source
 * rows the sampled grid references cross the bus. Pitches in elements; n_ctas = 0: two CTAs per SM.              */
int s3_gather_rows(const float* src, int64_t src_pitch, const int32_t* d_rows, int64_t n_rows, int64_t width,
                   float* d_dst, int64_t dst_pitch, int n_ctas, void* stream);

/* ---- volume-weighted snapshot SVD ---------------------------------------------------------------
 * device side of compute_svd (sparseSpatialSampling/utils.py:302-346), method of snapshots:
 *   B = sqrt(vol) * (A - mean_t(A));  G = B^T B;  G = V diag(s^2) V^T (host, T x T);  U = (A - mean) V / s.
 * A: fp32 [m, t] row-major (vector fields stacked as m = n_cells * D rows, utils.py:337-338), one weight per
 * `vol_div` consecutive rows (vol_div = D).                                                          */

/* temporal mean of every row (utils.py:322): d_mean fp32 [m] */
int s3_svd_row_means(const float* d_a, int64_t m, int64_t t, float* d_mean, void* stream);
/* Gram matrix of the centred, sqrt(volume)-scaled rows (utils.py:322-329 followed by the contraction the
 * reference leaves to LAPACK): d_gram fp64 [t, t] (symmetric, both triangles written).
 * method 1: tcgen05 tensor cores with a 3xTF32 split (fp32-equivalent products), short fp32 accumulation
 *           segments in TMEM, summed in registers and in fp64 across flushes;  method 2: same, single TF32 products;
 * method 0: fp32 CUDA-core tiles (cross-check).                                                      */
int s3_svd_gram(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, int64_t m, int64_t t,
                int method, double* d_gram, void* stream);
/* modes (utils.py:330 / :344 after the un-scaling): d_u fp32 [m, r] = (A - mean) * d_vs, d_vs fp32 [t, r] =
 * V[:, :r] / s[:r]                                                                                    */
int s3_svd_project(const float* d_a, const float* d_mean, const float* d_vs, int64_t m, int64_t t, int r,
                   float* d_u, void* stream);
/* The same projection on the tensor cores: rows centred, weighted by sqrt(vol) and split into TF32 planes as in
 * s3_svd_gram, contracted with d_vs over t by tcgen05 MMAs (method 1 = 3xTF32, 2 = TF32), un-weighted in the epilogue. */
int s3_svd_project_tc(const float* d_a, const float* d_mean, const float* d_vol, int vol_div, const float* d_vs,
                      int64_t m, int64_t t, int r, int method, float* d_u, void* stream);

/* ---- residual of a low-rank model (DMD / truncated POD reconstruction error) ------------------------
 * e[m, t] = (a[m, t] - mean[m]) - sum_j left[m, j] * right_t[t, j]
 * a fp32 [m, t] dense row-major (vector fields stacked as in s3_svd_gram, one vol per vol_div rows);
 * d_mean fp32 [m] or NULL (= 0); d_vol fp32 [m / vol_div] or NULL (= 1); left fp32 [m, q]; right_t fp32 [t, q];
 * 1 <= q <= 512 (larger q: S3_ERR_UNSUPPORTED). The product runs on tcgen05 (3xTF32), e is formed in fp64 and `a` is
 * read once. Outputs, component c = m % vol_div:
 *   d_sq_err  fp64 [vol_div, t] = sum_m vol * e^2
 *   d_sq_ref  fp64 [vol_div, t] = sum_m vol * (a - mean)^2
 *   d_max_abs fp64 [vol_div, t] = max_m |e|
 *   d_row_sq_err fp64 [m] or NULL: sum_t e^2 ADDED into row m
 * Every sum is reduced in a fixed order that depends on m and t only: bit-identical from run to run.        */
int s3_lowrank_error(const float* d_a, int64_t m, int64_t t, const float* d_mean, const float* d_vol, int vol_div,
                     const float* d_left, const float* d_right_t, int q, double* d_sq_err, double* d_sq_ref,
                     double* d_max_abs, double* d_row_sq_err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* S3B200_H */
