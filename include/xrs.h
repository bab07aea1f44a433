/*
 * xrs.h -- C ABI of libxrs.so, the B200 (sm_100a) spatial-resampling kernels.
 *
 * This is the drop-in boundary below the Python entry points
 * (resample_in_space / rectify_dataset / reproject_dataset /
 * affine_transform_dataset).  The reference (xcube-dev/xcube-resampling
 * v0.1.0) has no FFI of its own: its "native" layer is a set of numba-jitted
 * functions and calls into scipy / numpy / PROJ.  Each entry point below
 * replaces one of those and cites it (paths relative to the reference root).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *  - the caller owns every buffer; functions never allocate device memory;
 *  - work is enqueued on the caller's stream (a cudaStream_t passed as void*;
 *    NULL = legacy default stream) and the call returns without synchronising
 *    unless stated otherwise;
 *  - return value 0 = ok, non-zero = error, message via xrs_last_error()
 *    (thread-local);
 *  - images are row-major, spatial dimensions last, pitches in ELEMENTS;
 *  - one call touches exactly one device (the current one).
 */
#ifndef XRS_H_
#define XRS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XRS_VERSION 100 /* 0.1.0 */

/* element types of data variables */
enum xrs_dtype {
    XRS_F32 = 0, XRS_F64 = 1, XRS_U8 = 2, XRS_I8 = 3, XRS_U16 = 4,
    XRS_I16 = 5, XRS_I32 = 6, XRS_U32 = 7, XRS_I64 = 8
};

/* interpolation methods (constants.py:66-70) */
enum xrs_interp { XRS_NEAREST = 0, XRS_BILINEAR = 1, XRS_TRIANGULAR = 2 };

/* aggregation methods (constants.py:34-65) */
enum xrs_agg {
    XRS_AGG_CENTER = 0, XRS_AGG_COUNT = 1, XRS_AGG_FIRST = 2, XRS_AGG_LAST = 3, XRS_AGG_MAX = 4,
    XRS_AGG_MEAN = 5, XRS_AGG_MEDIAN = 6, XRS_AGG_MODE = 7, XRS_AGG_MIN = 8, XRS_AGG_PROD = 9,
    XRS_AGG_STD = 10, XRS_AGG_SUM = 11, XRS_AGG_VAR = 12
};

/* map projections understood by the device code (SURVEY.md 7.5) */
enum xrs_proj_kind {
    XRS_PROJ_GEOGRAPHIC = 0, /* lon/lat degrees (EPSG:4326 always_xy, OGC:CRS84) */
    XRS_PROJ_TMERC = 1,      /* transverse Mercator / UTM, Krueger n-series to n^6 */
    XRS_PROJ_WEBMERC = 2,    /* EPSG:3857 spherical Mercator */
    XRS_PROJ_LAEA = 3        /* Lambert azimuthal equal-area, ellipsoidal (EPSG:3035) */
};

/* A projected or geographic CRS reduced to what the formulas need. */
typedef struct xrs_proj {
    int32_t kind;   /* enum xrs_proj_kind */
    int32_t _pad;
    double a;       /* semi-major axis [m] */
    double inv_f;   /* inverse flattening (0 = sphere) */
    double lon0;    /* central meridian [deg] */
    double lat0;    /* latitude of origin [deg] */
    double k0;      /* scale factor */
    double fe;      /* false easting [m] */
    double fn;      /* false northing [m] */
} xrs_proj;

int xrs_version(void);
int xrs_device_count(void);
const char *xrs_last_error(void);
/* number of kernels this library has launched in the calling process (all threads) */
uint64_t xrs_launch_count(void);

/* Per-kernel timing for bench.py and profiling runs (off by default, no cost when off).  While on,
 * every kernel launch is bracketed by CUDA events on the stream it is launched on.
 * xrs_profile_collect waits for the recorded events, sums them per kernel name and clears the
 * records: names come back newline-separated in `names`, total milliseconds and launch counts in
 * the parallel arrays; returns the number of entries written (<= max_entries). */
int xrs_profile_enable(int32_t on);
int32_t xrs_profile_collect(char *names, int64_t names_len, double *total_ms, int64_t *launches, int32_t max_entries);

/* ------------------------------------------------------------------------
 * Rectification (rectify.py)
 * --------------------------------------------------------------------- */

/* K0 -- per-target-tile source windows.
 * Replaces GridMapping.ij_bboxes_from_xy_bboxes -> compute_ij_bboxes
 * (gridmapping/base.py:565-629, gridmapping/bboxes.py:28-106) for the
 * separable tile boxes of a regular target grid (gridmapping/base.py:521-533):
 * tile (ty,tx) has the x-interval [x_lo[tx], x_hi[tx]] and the y-interval
 * [y_lo[ty], y_hi[ty]], both ALREADY grown by xy_border by the caller (so the
 * comparisons use the same doubles as bboxes.py:60-69).  Single O(S) pass.
 * out_boxes: (nty*ntx, 4) int64 rows (i_min, j_min, i_max, j_max), -1 row if no
 * source point falls into the tile; grown by ij_border and clipped to
 * [0,w]x[0,h] (bboxes.py:90-106).
 * workspace: xrs_tile_src_bboxes_workspace_bytes(ntx, nty) bytes. */
int64_t xrs_tile_src_bboxes_workspace_bytes(int32_t ntx, int32_t nty);
int xrs_tile_src_bboxes(const double *x, const double *y, int64_t src_h, int64_t src_w, int64_t src_pitch,
                        const double *x_lo, const double *x_hi, int32_t ntx, const double *y_lo,
                        const double *y_hi, int32_t nty, int32_t ij_border, int64_t *out_boxes, void *workspace,
                        void *stream);

/* K0 over a ROW SLAB of the swath (multi-GPU: every GPU scans 1/N of the source rows), merged
 * afterwards.  `minform_table` is (ntx*nty, 4) int32 in "min-form" -- (i_min, j_min, -i_max1, -j_max1)
 * in whole-image indices, INT32_MAX = nothing seen (xrs_minform_init) -- so partial tables of
 * different slabs combine with an element-wise MIN: one all-reduce(MIN) between processes, one
 * numpy.minimum between threads.  x / y point at row `j_offset` of the (src_h, src_w) images.
 * xrs_tile_src_bboxes_finalize turns the merged table into the int64 boxes of xrs_tile_src_bboxes
 * (grown by ij_border, clipped to the whole image, bboxes.py:90-106).  The only exchange step of
 * the rectification path. */
int xrs_minform_init(int32_t *table, int64_t n, void *stream);
int xrs_tile_src_bboxes_partial(const double *x, const double *y, int64_t slab_h, int64_t src_w, int64_t src_pitch,
                                int64_t j_offset, const double *x_lo, const double *x_hi, int32_t ntx,
                                const double *y_lo, const double *y_hi, int32_t nty, int32_t *minform_table,
                                void *workspace, void *stream);
int xrs_tile_src_bboxes_finalize(const int32_t *minform_table, int32_t n_tiles, int32_t ij_border, int64_t src_w,
                                 int64_t src_h, int64_t *out_boxes, void *stream);

/* Source footprint of target ROW BANDS (multi-GPU partition, SURVEY 8e; the reference's per-tile
 * source slicing is rectify.py:397-399).  For band b = target rows [band_edges[b], band_edges[b+1])
 * and every group g of xrs_quad_row_group() source quad rows, minform_fp[(b*n_groups + g)*2 ..] holds
 * (c_min, -c_max) over the quads of the scanned slab whose pixel box (grown by 2 px + 1 % of its
 * extent) overlaps the band; INT32_MAX = none.  Every quad that can claim a pixel of the band is
 * inside, so K1 restricted to the footprint (src_col_ranges) gives the same claims as K1 on the
 * whole swath.  n_groups = ceil((src_h - 1) / group); the slab is rows [j_offset, j_offset + slab_h)
 * of the image (include the first row of the next slab so that no quad row is lost) and j_offset
 * must be a multiple of the group size.  band_edges (device, n_bands + 1 values) must ascend; equal
 * neighbours make an empty band, which gets no footprint.  Tables of different slabs merge with MIN. */
int32_t xrs_quad_row_group(void);
int xrs_band_quad_footprints(const double *x, const double *y, int64_t slab_h, int64_t src_w, int64_t src_pitch,
                             int64_t j_offset, int64_t src_h, int64_t dst_h, int64_t dst_w, double x_min, double y_min,
                             double y_max, double x_res, double y_res, int32_t is_j_axis_up,
                             const int32_t *band_edges, int32_t n_bands, int32_t *minform_fp, void *stream);

/* Strided copies between host and device on the copy engines: `slices` windows of `rows` rows of
 * `width_bytes`, row pitches and slice strides in bytes on either side (cudaMemcpy2DAsync per slice,
 * direction inferred from the pointers; host memory should be page-locked).  Ragged footprint
 * uploads and row-band downloads into one shared host array go through this. */
int xrs_copy2d_slices(void *dst, int64_t dst_pitch_bytes, int64_t dst_slice_bytes, const void *src,
                      int64_t src_pitch_bytes, int64_t src_slice_bytes, int64_t width_bytes, int64_t rows,
                      int64_t slices, void *stream);

/* Statistics of 2-D coordinate images that stay on the device (CRS-transformed or pre-downscaled
 * swath coordinates inside rectify_dataset): what GridMapping.from_coords needs from the WHOLE
 * images.  out4 (device, 4 x uint64): [0] 1 if any x > 180 (coords.py:102-103), [1] / [2] bit
 * patterns of the smallest / largest positive cell area of coords.py:226-252 (geographic grids:
 * the reference's metre conversion), ~0 / 0 if there is none, [3] reserved.
 * xrs_lon_360: x < 0 -> x + 360 in place (helpers.py to_lon_360). */
int xrs_coords_stats(const double *x, const double *y, int64_t h, int64_t w, int64_t pitch, int32_t is_geographic,
                     uint64_t *out4, void *stream);
int xrs_lon_360(double *x, int64_t h, int64_t w, int64_t pitch, void *stream);

/* K1 -- source-index (ij) image of a regular target grid.
 * Replaces _compute_target_source_ij / _compute_target_source_ij_block /
 * _compute_target_source_ij_sequential / _line (rectify.py:312-576) including
 * _fdet/_fu/_fv/_fclamp (rectify.py:737-768).  Result is identical to the
 * sequential first-writer-wins scatter: per target pixel the accepting source
 * quad with the smallest row-major index inside the reference tile's source
 * window wins (DESIGN.md "K1 equivalence").
 *   x, y          source coordinate images (src_h, src_w), pitch src_pitch
 *   tile_boxes    (nty*ntx, 4) int64 from xrs_tile_src_bboxes (row-major tiles)
 *   ij            (2, dst_h, dst_w) float64, plane 0 = i (x index), 1 = j
 *   tile_w/h      the reference tile size of the target grid mapping
 *   x_min,y_min,y_max,x_res,y_res,is_j_axis_up  target grid (rectify.py:402-416)
 *   uv_delta      barycentric tolerance (constants.py:80, 1e-3)
 *   row_begin/end only target rows [row_begin, row_end) are computed (multi-GPU row
 *                 bands); ij then is (2, row_end-row_begin, dst_w).  Results do not
 *                 depend on the band split.
 *   src_col_ranges  NULL, or the band's row of the table of xrs_band_quad_footprints: per group
 *                 of xrs_quad_row_group() source quad rows (c_min, -c_max) of the quads whose
 *                 coordinates the caller made resident.  Only those quads are read -- x and y
 *                 may then be buffers in which just the footprint has been uploaded.
 * workspace: xrs_rectify_ij_workspace_bytes(src_h, src_w, row_end - row_begin, dst_w) bytes,
 *            16-byte aligned. */
int64_t xrs_rectify_ij_workspace_bytes(int64_t src_h, int64_t src_w, int64_t dst_rows, int64_t dst_w);
int xrs_rectify_ij(const double *x, const double *y, int64_t src_h, int64_t src_w, int64_t src_pitch,
                   const int64_t *tile_boxes, double *ij, int64_t dst_h, int64_t dst_w, int32_t tile_h,
                   int32_t tile_w, double x_min, double y_min, double y_max, double x_res, double y_res,
                   int32_t is_j_axis_up, double uv_delta, int64_t row_begin, int64_t row_end,
                   const int32_t *src_col_ranges, void *workspace, void *stream);

/* K2 -- gather of all bands through the ij image.
 * Replaces _compute_var_image / _compute_var_image_block /
 * _compute_var_image_sequential / _for_dest_line (rectify.py:579-734).
 *   src_planes_host  HOST array of n_bands device pointers, each pointing at element
 *                    (win_j0, win_i0) of a (src_h, src_w) plane of `dtype`, row pitch
 *                    src_pitch: only the (win_h, win_w) window the ij values reach has
 *                    to be resident (row-band footprints); src_h/src_w stay the full
 *                    image size because neighbour taps clamp at the true image edge.
 *                    A pitch that is a multiple of 16 bytes (and 16-byte aligned planes)
 *                    enables the TMA-staged kernel; anything else runs the direct one.
 *   dst_planes_host  HOST array of n_bands device pointers, each a
 *                    (dst_h, dst_w) plane of `dtype`, contiguous rows
 *   ij               (2, dst_h, dst_w) float64 from xrs_rectify_ij
 *   fill             value written where ij is NaN, converted to dtype like np.full(..., float(fill), dtype)
 *                    on x86 (xrs_casts.h): NaN gives INT32_MIN / INT64_MIN for int32 / int64 and 0 for the
 *                    other integer types, -1 gives 0xFFFFFFFF for uint32.  A double cannot hold every
 *                    int64: fills beyond 2^53 arrive rounded to the nearest double (INT64_MAX as 2^63,
 *                    which converts to INT64_MIN).
 * Arithmetic is float64 without FMA contraction, one cast to dtype at the end with x86's results (an int64
 * sample that rounds to 2^63 stores INT64_MIN).  Nearest samples take the reference's float64 round trip
 * of the source window (rectify.py:628-630): int64 values beyond 2^53 are rounded, INT64_MAX reads back as
 * INT64_MIN; every other dtype is copied unchanged. */
int xrs_gather_ij(const void *const *src_planes_host, void *const *dst_planes_host, int32_t n_bands,
                  int32_t dtype, int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0,
                  int64_t win_w, int64_t win_h, const double *ij, int64_t dst_h, int64_t dst_w, int32_t method,
                  double fill, void *stream);

/* K2, two methods in one pass -- nearest AND bilinear (or triangular) samples of the same bands.
 * Replaces two _compute_var_image passes over the same ij image: the reference calls
 * _rectify_data_array once per output variable (rectify.py:159-174, 263-309), so a dataset that
 * wants the same source bands with both methods walks ij and the source twice.  The nearest sample
 * is always one of the four taps of the bilinear / triangular one (rectify.py:689-698), so one
 * launch reads ij and the source once and writes both results.
 *   dst_interp_planes_host   HOST array of n_bands device pointers: planes for `method`
 *                            (XRS_BILINEAR or XRS_TRIANGULAR)
 *   dst_nearest_planes_host  the same for the nearest-neighbour result
 *   fill_interp, fill_nearest  fill value of either result
 * Everything else as in xrs_gather_ij; results are bit-identical to two xrs_gather_ij calls (which
 * is what runs when the source layout rules out the TMA-staged kernel). */
int xrs_gather_ij2(const void *const *src_planes_host, void *const *dst_interp_planes_host,
                   void *const *dst_nearest_planes_host, int32_t n_bands, int32_t dtype, int64_t src_h,
                   int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w, int64_t win_h,
                   const double *ij, int64_t dst_h, int64_t dst_w, int32_t method, double fill_interp,
                   double fill_nearest, void *stream);

/* K1 + K2 fused -- xrs_rectify_ij followed by xrs_gather_ij without materialising the ij image:
 * the claim stage of K1 runs as usual, then the gather kernel resolves each pixel's fractional
 * source index in registers (same arithmetic, same results) and gathers all bands.  Saves the
 * 16 bytes per target pixel that K1 would write and K2 read back; meant for calls that gather ONE
 * variable (rectify_dataset uses xrs_rectify_ij + xrs_gather_ij when several variables share the
 * ij image).  Arguments as for the two functions; `data_pitch` is the row pitch of the data planes,
 * dst planes are (row_end - row_begin, dst_w); workspace as for xrs_rectify_ij. */
int xrs_rectify_gather(const double *x, const double *y, int64_t src_h, int64_t src_w, int64_t src_pitch,
                       const int64_t *tile_boxes, int64_t dst_h, int64_t dst_w, int32_t tile_h, int32_t tile_w,
                       double x_min, double y_min, double y_max, double x_res, double y_res, int32_t is_j_axis_up,
                       double uv_delta, int64_t row_begin, int64_t row_end, const int32_t *src_col_ranges,
                       void *workspace, const void *const *src_planes_host, void *const *dst_planes_host, int32_t n_bands, int32_t dtype,
                       int64_t data_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w, int64_t win_h, int32_t method,
                       double fill, void *stream);

/* ------------------------------------------------------------------------
 * Reprojection (reproject.py) and CRS point transforms
 * --------------------------------------------------------------------- */

/* K3a -- CRS transform of n points, always_xy axis order.
 * Replaces pyproj.Transformer.from_crs(from_crs, to_crs, always_xy=True).transform(x, y) at
 * reproject.py:483 (_transform_gridpoints), rectify.py:196-204 (_transform_coords) and, with the
 * densified tile edges built by the host, transform_bounds (reproject.py:347,398).  Points that a
 * projection cannot represent come back as NaN (PROJ reports inf).  x_out / y_out may alias the
 * inputs. */
int xrs_transform_points(const xrs_proj *from_crs, const xrs_proj *to_crs, const double *x_in, const double *y_in,
                         double *x_out, double *y_out, int64_t n, void *stream);

/* K3 -- target-pixel CRS transform fused with the gather of all bands.
 * Replaces _transform_gridpoints (reproject.py:472-496) + _reproject_block (reproject.py:268-335);
 * the padded, re-tiled source copy of _reorganize_data_array_slice (reproject.py:499-530) is never
 * materialised -- taps outside the source read `fill`, as da.pad(constant_values=fill) provides.
 *   src_planes_host  HOST array of n_bands device pointers, each at element (win_j0, win_i0) of a
 *                    (src_h, src_w) plane of `dtype`, row pitch src_pitch: only the resident
 *                    (win_h, win_w) window has to be valid memory (row-band footprints)
 *   dst_planes_host  HOST array of n_bands device pointers to (row_end-row_begin, dst_w) planes of
 *                    `out_dtype`: `dtype` for nearest and triangular; for bilinear float64 (what
 *                    numpy's promotion yields in the reference) or `dtype` (value cast once)
 *   src_crs/dst_crs  source and target CRS; points go dst_crs -> src_crs (reproject.py:124-126)
 *   dst_x, dst_y     pixel-centre coordinates of the target grid, (dst_w,) and (dst_h,) float64
 *                    (GridMapping.x_coords / y_coords, regular.py:44-63)
 *   tile_h/w         reference tile size of the target grid mapping; tile t = ty * ntx + tx
 *   tile_x0/y0       per tile: coordinate of window element 0 -- the FLOAT32 value the reference
 *                    stores (reproject.py:427-450) widened to float64
 *   tile_i0/j0       per tile: source index of window element 0 (before padding, may be negative)
 *   tile_win_w/h     common window size of all tiles (reproject.py:407-423); window indices follow
 *                    numpy (negative counts from the end); indices still outside give `fill`
 *                    where the reference raises IndexError
 *   src_x_res/y_res  source resolution (positive); fractional index = (X - x0) / x_res,
 *                    (Y - y0) / -y_res (reproject.py:278-279)
 *   row_begin/end    target rows computed by this call
 * A target pixel whose transform is not finite gets `fill` (the reference indexes garbage). */
int xrs_reproject(const void *const *src_planes_host, void *const *dst_planes_host, int32_t n_bands, int32_t dtype,
                  int32_t out_dtype, int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0,
                  int64_t win_w, int64_t win_h, const xrs_proj *src_crs, const xrs_proj *dst_crs, const double *dst_x,
                  const double *dst_y, int64_t dst_h, int64_t dst_w, int32_t tile_h, int32_t tile_w,
                  const double *tile_x0, const double *tile_y0, const int32_t *tile_i0, const int32_t *tile_j0,
                  int32_t tile_win_w, int32_t tile_win_h, double src_x_res, double src_y_res, int32_t method,
                  double fill, int64_t row_begin, int64_t row_end, void *stream);

/* ------------------------------------------------------------------------
 * Affine resampling and block aggregation (affine.py, coarsen.py)
 * --------------------------------------------------------------------- */

/* K4+K5 -- affine resampling (scale + offset per axis, order 0 or 1) with optional fused block
 * aggregation.  Replaces _resample_array / _downscale / _upscale (affine.py:243-362), i.e.
 * dask_image.ndinterp.affine_transform -> scipy.ndimage.affine_transform(matrix=diag(1.., j_scale,
 * i_scale), offset=(0.., j_off, i_off), order, mode="constant", cval) followed by
 * dask.array.coarsen(agg, {y: f_j, x: f_i}) with the reducers of coarsen.py:50-155 and
 * constants.py:51-65.
 *   src        (n_slices, src_h, src_w) of `dtype`, row pitch src_pitch, slice stride src_slice_stride
 *   dst        (n_slices, dst_h, dst_w) contiguous; element type is `dtype`, except int64 for
 *              agg = mode / count and for sum / prod of integer data (what numpy returns)
 *   j/i_scale, j/i_off  source index = intermediate index * scale + off; the intermediate image is
 *              (dst_h * f_j, dst_w * f_i) (affine.py:287-297 has already divided the scale by f)
 *   order      0 nearest, 1 linear; anything else fails like affine.py:329-335
 *   agg, f_j, f_i  reducer (enum xrs_agg) over f_j x f_i intermediate samples; f_j = f_i = 1: none
 *   slice_blend  1 reproduces scipy's zero-weight read of the neighbouring slice for 3-D float
 *              arrays with order 1 (non-finite values there make the sample NaN; one slice reads itself)
 * Every sample takes scipy's float64 round trip, order 0 included: int64 values beyond 2^53 come back
 * rounded as scipy rounds them (2^52 + 1 -> 2^52 + 2, 2^62 + 1 -> 2^62), -0.0 as +0.0; NaN / out-of-range
 * results and cval in integer outputs convert as scipy's do on x86 (NaN -> INT32_MIN / INT64_MIN for 32- and
 * 64-bit signed types, 0 for the others; 2^63 -> INT64_MIN, above -> INT64_MAX).  */
int xrs_affine(const void *src, void *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
               int64_t src_pitch, int64_t src_slice_stride, int64_t dst_h, int64_t dst_w, double j_scale, double j_off,
               double i_scale, double i_off, int32_t order, double cval, int32_t agg, int32_t f_j, int32_t f_i,
               int32_t slice_blend, void *stream);

/* NaN recovery for order-1 resampling of floating-point data (affine.py:344-360, recover_nans=True):
 * the zero-filled image and the validity mask pass through the same filter and are divided, so a
 * sample next to a NaN keeps the weighted mean of its valid neighbours instead of becoming NaN.
 * The reference takes this branch only if the array holds a NaN at all (xrs_has_nan).  dst is
 * float64 (numpy divides the filtered image by the float64 filtered mask); aggregation as for
 * xrs_affine, carried out on those float64 samples. */
int xrs_has_nan(const void *src, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w, int64_t src_pitch,
                int64_t src_slice_stride, int32_t *flag, void *stream);
int xrs_affine_recover(const void *src, double *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
                       int64_t src_pitch, int64_t src_slice_stride, int64_t dst_h, int64_t dst_w, double j_scale,
                       double j_off, double i_scale, double i_off, double cval, int32_t agg, int32_t f_j, int32_t f_i,
                       int32_t slice_blend, void *stream);

/* K5 alone -- dask.array.coarsen(agg, array, {y: f_j, x: f_i}) with the same reducers
 * (coarsen.py:50-155); f_j, f_i must divide src_h, src_w.  dst as for xrs_affine.  Unlike xrs_affine the
 * values are aggregated as stored (dask never converts them): int64 beyond 2^53 stays exact, -0.0 stays -0.0. */
int xrs_coarsen(const void *src, void *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
                int64_t src_pitch, int64_t src_slice_stride, int32_t agg, int32_t f_j, int32_t f_i, void *stream);

/* ------------------------------------------------------------------------
 * Compressed Zarr v2 / v3 chunks decoded on the device (io.py, the I/O edge)
 * --------------------------------------------------------------------- */

/* codec of one chunk file: missing (the array's fill value), a Blosc-1 frame with an LZ4 / LZ4HC, a Zstd or a Zlib
 * inner codec (numcodecs Blosc, byte shuffle or none, or a frame stored whole; each stream of a Zstd frame is one
 * zstd frame, each stream of a Zlib frame one zlib stream), numcodecs' lz4 (int32 decoded size, then one LZ4 block),
 * numcodecs' zstd (one zstd frame, RFC 8878, without a dictionary; skippable frames may follow it), numcodecs' zlib
 * (one zlib stream, RFC 1950, without a preset dictionary; bytes after its Adler-32 are ignored) or numcodecs' gzip
 * (gzip members, RFC 1952, with NUL bytes between and after them allowed).  Zarr v3's zstd, gzip and blosc codecs
 * write the same streams.
 * XRS_CHUNK_CRC32C is a flag OR-ed into a codec other than XRS_CHUNK_MISSING (Zarr v3's crc32c codec after the
 * compressor): the last 4 bytes of the file are the little-endian CRC-32C (Castagnoli, reflected polynomial
 * 0x82F63B78) of the bytes in front of them, and the codec applies to the length - 4 bytes of that payload.  The
 * call checks the trailer on the device (k_crc32c, before any decoder) and reports XRS_DECODE_CRC32C on a mismatch.
 * `header` holds the payload's first 16 bytes, as for an unflagged file.  A table without the flag is decoded
 * exactly as before. */
enum xrs_chunk_codec {
    XRS_CHUNK_MISSING = 0, XRS_CHUNK_BLOSC = 1, XRS_CHUNK_LZ4 = 2, XRS_CHUNK_ZSTD = 3, XRS_CHUNK_ZLIB = 4,
    XRS_CHUNK_GZIP = 5,
    XRS_CHUNK_CRC32C = 0x100
};

/* One chunk file of a xrs_zarr_decode call (80 bytes); for a sharded Zarr v3 array, one inner chunk: offset / length
 * cover exactly that chunk's bytes. */
typedef struct xrs_zarr_chunk {
    int64_t offset;       /* first byte of the file in `data` */
    int64_t length;       /* bytes of the file (0 when missing) */
    int64_t band, row, col; /* array index of the chunk's element (0, 0, 0); band 0 for 2-D arrays */
    int32_t codec;        /* enum xrs_chunk_codec, optionally | XRS_CHUNK_CRC32C */
    int32_t n_streams;    /* filled by the call */
    int64_t stream_base;  /* filled by the call */
    int64_t scratch;      /* filled by the call: where the decoded chunk goes in the workspace, -1 when missing */
    uint8_t header[16];   /* the first 16 bytes of the file (Blosc header; lz4: the size prefix; zstd: the magic) */
} xrs_zarr_chunk;

/* CF mask-and-scale of the decoded values (io.DecodedSource): the stored value is converted to out_dtype,
 * values equal to one of `fills` become NaN, then * scale (if has_scale), then + offset (if has_offset), each
 * rounded once in out_dtype -- numpy's steps in numpy's order. */
#define XRS_ZARR_CF_MAX_FILLS 16
typedef struct xrs_zarr_cf {
    int32_t out_dtype;    /* XRS_F32 or XRS_F64 */
    int32_t n_fills;      /* <= XRS_ZARR_CF_MAX_FILLS */
    int32_t has_scale, has_offset;
    double scale, offset;
    uint64_t fills[XRS_ZARR_CF_MAX_FILLS]; /* stored-dtype values, native byte order, in the low bytes */
} xrs_zarr_cf;

/* reasons in bits 24-31 of the error word; bits 0-23 hold 1 + the index of the bad chunk in the table */
enum xrs_decode_error {
    XRS_DECODE_BAD_LAYOUT = 1,          /* a block offset or stream size points outside the file */
    XRS_DECODE_OFFSET_ZERO = 2,         /* an LZ4 match offset of 0 */
    XRS_DECODE_OFFSET_BEFORE_START = 3, /* a match reaching before the stream's first decoded byte (Deflate: before
                                           the stream's or the gzip member's first byte) */
    XRS_DECODE_LITERALS_OVERRUN = 4,    /* literals past the decoded size or past the input (Deflate: a literal or
                                           stored block past the decoded size) */
    XRS_DECODE_MATCH_OVERRUN = 5,       /* a match past the decoded size */
    XRS_DECODE_INPUT_OVERRUN = 6,       /* length extension, offset or next token past the input; zstd: a frame
                                           header, block or checksum past the input; Deflate: bits, a stored block,
                                           a gzip header field or a trailer past the input */
    XRS_DECODE_SHORT = 7,               /* the stream ends short of its decoded size */
    /* zstd frames (the reasons above apply to them too; an offset of 0 is a repeat offset of 0), and where noted
     * zlib streams and gzip members */
    XRS_DECODE_BAD_FRAME_HEADER = 8,    /* unknown magic, reserved bit set, a dictionary ID other than 0, a window
                                           beyond 2^31 bytes, or a content size other than the stream's; zlib: a
                                           method other than 8, CINFO > 7, a bad FCHECK or FDICT set; gzip: a
                                           member without the magic or with a method other than 8 */
    XRS_DECODE_BAD_BLOCK = 9,           /* reserved block type, or a compressed block above min(128 KiB, window) */
    XRS_DECODE_BAD_LITERALS = 10,       /* a literals section past its block or above min(128 KiB, window),
                                           treeless literals without a previous tree, or a Huffman stream that does
                                           not decode to exactly its literals */
    XRS_DECODE_BAD_HUFFMAN = 11,        /* a Huffman tree description that is truncated or does not form a tree */
    XRS_DECODE_BAD_FSE = 12,            /* an FSE table description above the table's accuracy log or whose
                                           probabilities do not sum */
    XRS_DECODE_BAD_SEQUENCES = 13,      /* a sequences header past its block, reserved mode bits, a repeated table
                                           without a previous one, an RLE code out of range, or a bitstream not
                                           consumed exactly */
    XRS_DECODE_TRAILING_BYTES = 14,     /* bytes after the frame that are not skippable frames; gzip: bytes after a
                                           member that are neither NUL nor the next member */
    XRS_DECODE_CHECKSUM = 15,           /* the content checksum (XXH64, low 32 bits) does not match; zlib: the
                                           Adler-32; gzip: a member's CRC-32 or ISIZE (its size mod 2^32) */
    /* Deflate streams only (RFC 1951) */
    XRS_DECODE_BAD_DEFLATE_BLOCK = 16,  /* block type 3, or a stored block whose NLEN is not the complement of LEN */
    XRS_DECODE_BAD_DEFLATE_CODES = 17,  /* a dynamic block's code description: more than 286 litlen or 30 distance
                                           codes, an over-subscribed or incomplete set (a litlen or distance set may
                                           be one code of length 1; a distance set may be empty), a repeat code 16
                                           without a previous length or a repeat past the last length, or no
                                           end-of-block code */
    XRS_DECODE_BAD_DEFLATE_SYMBOL = 18, /* litlen symbol 286 / 287, distance symbol 30 / 31, or a code that an
                                           incomplete set leaves unassigned (an empty distance set included) */
    /* files flagged XRS_CHUNK_CRC32C */
    XRS_DECODE_CRC32C = 19              /* the CRC-32C trailer does not match the payload in front of it */
};

/* Decode whole chunk files and place their elements into a pitched (bands, rows, width) slot.
 *   data, data_bytes   the chunk files, concatenated as read from the store
 *   chunks_host        HOST table of n_chunks < 2^24 files (page-locked memory keeps the call asynchronous); the
 *                      call checks each header and fills stream_base / n_streams / scratch, then copies the table to the
 *                      workspace on `stream`: it must stay unchanged until the stream has passed the call
 *   chunk_bands/h/w    chunk shape (chunk_bands 1 for 2-D arrays); dtype: the stored type, big_endian 1 for
 *                      ">" dtypes (values are byte-swapped to native order)
 *   fill_bits          the stored value of a missing chunk, native byte order in the low bytes
 *   cf_host            NULL (values as stored, dst of `dtype`) or CF decoding (dst of cf_host->out_dtype)
 *   img_h, img_w       array height and width: ragged edge chunks are clipped to them
 *   dst                element (band b0, row win_j0, column 0) of the slot; pitch and band stride in elements;
 *                      only rows [win_j0, win_j1) and bands [b0, b0 + nb) are written
 *   workspace          xrs_zarr_decode_workspace_bytes(...) bytes, 256-byte aligned: the table, 32 bytes a stream and
 *                      one decoded chunk per file present; with Zstd streams also one literal buffer per Zstd
 *                      stream of min(S, 128 KiB) bytes, S the largest decoded size of one Zstd stream in the call
 *                      (a numcodecs zstd chunk; for Blosc-Zstd, blocksize / streams of a full block or the last,
 *                      partial block), so a Blosc-Zstd call takes at most about twice the scratch of an LZ4 one;
 *                      Deflate streams (zlib, gzip, Blosc-Zlib) add nothing but their 32-byte descriptors
 *   error_word         device uint32, 0 before the first call; a malformed stream stores its reason and
 *                      chunk there (the first one recorded wins) and the call's results are undefined.  A file
 *                      the call can reject from its header alone fails the call itself, naming the chunk. */
int64_t xrs_zarr_decode_workspace_bytes(xrs_zarr_chunk *chunks_host, int64_t n_chunks, int64_t chunk_bands,
                                        int64_t chunk_h, int64_t chunk_w, int32_t dtype);
int xrs_zarr_decode(const void *data, int64_t data_bytes, xrs_zarr_chunk *chunks_host, int64_t n_chunks,
                    int64_t chunk_bands, int64_t chunk_h, int64_t chunk_w, int32_t dtype, int32_t big_endian,
                    uint64_t fill_bits, const xrs_zarr_cf *cf_host, int64_t img_h, int64_t img_w, void *dst,
                    int64_t dst_pitch, int64_t dst_band_stride, int64_t win_j0, int64_t win_j1, int64_t b0, int64_t nb,
                    void *workspace, int64_t workspace_bytes, uint32_t *error_word, void *stream);

#ifdef __cplusplus
}
#include "xrs_casts.h" /* the conversions behind `fill` and the integer stores above, as C++ templates */
#endif
#endif /* XRS_H_ */
