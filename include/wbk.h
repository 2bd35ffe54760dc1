/* libwbk -- C-ABI of the B200-native WaveBreaking detection path.
 *
 * The reference (skaderli/WaveBreaking v0.3.8) is pure Python and defines no FFI of
 * its own; its boundary is the Python API re-exported in wavebreaking/__init__.py:19-34.
 * This header is the C boundary that the Python host layer (wavebreaking_b200/) binds
 * with ctypes; every entry point names the reference code whose arithmetic it replaces.
 *
 * Conventions
 *  - plain C types only; pointers named d_* are device pointers (in the emulator build
 *    used by the CPU-only tests they are host pointers), h_* are host pointers;
 *  - every function returns WBK_OK (0) or a negative error code; the message of the
 *    last error of the calling thread is returned by wbk_last_error();
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *  - variable-length results live in capacity-bounded device arenas owned by a context;
 *    an overflow yields WBK_ERR_CAPACITY and wbk_caps_needed() tells the sizes that
 *    would have sufficed, so the caller can re-create the context and retry;
 *  - lattice points are packed as x | (y << 16) in a uint32 (x = column on the
 *    periodically extended grid, y = row).
 */
#ifndef WBK_H
#define WBK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WBK_OK 0
#define WBK_ERR_INVALID (-1)
#define WBK_ERR_CUDA (-2)
#define WBK_ERR_CAPACITY (-3)
#define WBK_ERR_NODEVICE (-4)

#define WBK_F32 0
#define WBK_F64 1
#define WBK_I16 2 /* packed NetCDF shorts (input of wbk_smooth / wbk_smooth_contours / wbk_orient / wbk_mflux, and the
                     intensity of wbk_events_raster) */

/* rounding of the smoothing passes (scipy keeps the input dtype, the division by
 * np.sum(weights) promotes float32 to float64 under NumPy >= 2; SURVEY.md A.7) */
#define WBK_ROUND_NONE 0      /* float64 data: all passes in float64 */
#define WBK_ROUND_FIRST 1     /* float32 data, NumPy >= 2: pass 1 rounds its sum to float32, then float64 */
#define WBK_ROUND_ALL 2       /* float32 data, NumPy 1.x: every pass rounds to float32 */

/* per-job status bits (job = one (time step, contour level)) */
#define WBK_ST_SEG_OVERFLOW 1       /* more marching-squares segments than seg_cap */
#define WBK_ST_CONTOUR_OVERFLOW 2   /* more contours than contour_cap */
#define WBK_ST_LATTICE_VERTEX 4     /* informational: a contour vertex fell exactly on a grid vertex (value == level);
                                       the job was linked by the sequential, skimage-exact linker */
#define WBK_ST_PAIR_OVERFLOW 8      /* more streamer candidate pairs than pair_cap */
#define WBK_ST_EVENT_OVERFLOW 16    /* more events than event_cap */
#define WBK_ST_SEL_OVERFLOW 32      /* more full-width contours than sel_cap */
#define WBK_ST_WIDTH_OVERFLOW 64    /* extended grid wider than the shared-memory column tables */
#define WBK_ST_PACK_OVERFLOW 128    /* (job 0 only) packed contour set larger than the caller's buffers */
#define WBK_ST_FETCH_OVERFLOW 256   /* (job 0 only) more events / ring vertices than the caller's fetch buffers */
#define WBK_ST_SPLIT_CHAINS 512     /* (job 0 only) an event leaves and re-enters one side of the last meridian more than
                                       24 times: the device clipper cannot split it, its cells are missing from the
                                       flag grids (an error, not a capacity) */

const char* wbk_last_error(void);
int wbk_version(void);
/* number of CUDA devices visible; WBK_ERR_NODEVICE if none (the library has no CPU path) */
int wbk_device_count(void);

/* ---------------------------------------------------------------------------------------------
 * wavebreaking/processing/spatial.py:60-128  calculate_smoothed_field
 *   `passes` x [scipy.ndimage.convolve(weights=[[0,1,0],[1,2,1],[0,1,0]], mode="wrap") / np.sum(weights) = 6]
 *   then rows {0,1,nlat-2,nlat-1} := NaN (spatial.py:100-107).  All passes are fused in one
 *   launch per WBK_SMOOTH_MAX_FUSED passes.  d_in [ntime,nlat,nlon] (in_dtype), d_out same shape
 *   (out_dtype: F64 for ROUND_NONE / ROUND_FIRST, F32 for ROUND_ALL; passes == 0 needs
 *   out_dtype == in_dtype).  d_tmp (same size as d_out) is needed only if
 *   passes > WBK_SMOOTH_MAX_FUSED, else may be NULL.
 *
 * opts (may be NULL) describes how d_in is stored; the result is always in the ascending orientation:
 *   flip_lat / flip_lon   the latitude / longitude coordinate of d_in is descending
 *                         (utils/data_utils.py:196-213 correct_dimension_orientation; ERA5 files are lat-descending):
 *                         the kernel reads row nlat-1-y / column nlon-1-x, no re-sorted copy is made;
 *   scale, offset, fill   in_dtype == WBK_I16 only: CF packing of NetCDF files, decoded the way xarray does,
 *                         float64(v) * scale_factor + add_offset (two roundings), v == fill -> NaN when has_fill
 *                         (round_mode must be WBK_ROUND_NONE and out_dtype WBK_F64).
 */
#define WBK_SMOOTH_MAX_FUSED 8
typedef struct wbk_smooth_opts {
  int flip_lat, flip_lon;
  double scale, offset;
  int has_fill, fill;
} wbk_smooth_opts;
int wbk_smooth(const void* d_in, int in_dtype, void* d_out, int out_dtype, void* d_tmp, int ntime, int nlat,
               int nlon, int passes, int round_mode, const wbk_smooth_opts* opts, void* stream);

/* tuning knob (process-wide): 64-column halves a warp of the smoothing kernel marches side by side; 0 / 1 = one
 * (default, the faster one on B200: 16 instead of 8 warps per SM), 2 = two (<= 5 passes).  Results do not depend on it. */
void wbk_tune_smooth_halves(int halves);

/* orientation fix (and int16 decode) alone: d_out[t, y, x] = decode(d_in[t, flip_lat ? nlat-1-y : y,
 * flip_lon ? nlon-1-x : x]); output dtype = in_dtype, float64 for WBK_I16 */
int wbk_orient(const void* d_in, int in_dtype, void* d_out, int ntime, int nlat, int nlon, const wbk_smooth_opts* opts,
               void* stream);

/* spatial.py:103 with user-supplied weights / mode: ONE pass of
 * scipy.ndimage.convolve(in, weights, mode, cval=0) (output dtype = dtype, accumulation in
 * double in scipy's tap order), followed by the division by `divisor` (np.sum(weights)) when
 * divide != 0.  mode: 0 wrap ("wrap"/"grid-wrap"), 1 reflect, 2 mirror, 3 nearest, 4 constant.
 * h_weights is the kh x kw kernel as given to scipy (row-major, host memory).
 */
int wbk_convolve2d(const void* d_in, int in_dtype, void* d_out, int out_dtype, int ntime, int nlat, int nlon,
                   const double* h_weights, int kh, int kw, int mode, int divide, double divisor, void* stream);

/* set rows {0..border-1} and {nlat-border..nlat-1} to NaN (spatial.py:106-107) */
int wbk_nan_border(void* d_field, int dtype, int ntime, int nlat, int nlon, int border, void* stream);

/* spatial.py:27-57 calculate_momentum_flux: (u - nanmean_lon(u)) * (v - nanmean_lon(v)).  The zonal means follow
 * numpy.nanmean bit for bit: pairwise summation in the data dtype when longitude is the contiguous axis of the
 * user's array (sequential = 0), plain left-to-right summation when it is not (sequential = 1), float64 quotient
 * rounded to the data dtype.  The flux is computed and written in the stored order of u and v.
 * dtype WBK_I16: u and v are packed NetCDF shorts, packing points at two wbk_smooth_opts (u, then v: scale, offset,
 * fill as for wbk_smooth; flip_lat / flip_lon must be 0), every value is decoded as it is loaded and everything
 * (NaN counts, sums, products) runs on the decoded float64 values; d_out is float64.  packing is NULL for WBK_F32 /
 * WBK_F64 (d_out of the data dtype). */
int wbk_mflux(const void* d_u, const void* d_v, void* d_out, int dtype, int ntime, int nlat, int nlon, int sequential,
              const wbk_smooth_opts* packing, void* stream);

/* utils/data_utils.py:196-213 correct_dimension_orientation: out[t, y, x] = in[t, flip_lat ? nlat-1-y : y,
 * flip_lon ? nlon-1-x : x] */
int wbk_flip(const void* d_in, void* d_out, int dtype, int ntime, int nlat, int nlon, int flip_lat, int flip_lon,
             void* stream);

/* synthetic Rossby-wave PV (SURVEY.md 8d; host mirror: wavebreaking_b200/synthetic.py).
 * h_blobs: [2][n_blob][3] doubles (lat0, lon0, radius); hours: first hour and step. */
int wbk_synth_pv(void* d_out, int dtype, int ntime, int nlat, int nlon, double hour0, double hour_step,
                 const double* h_blobs, int n_blob, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Detection context: owns the capacity-bounded device arenas of one batch of jobs
 * (job = time step x contour level, job = t * nlevels + l: time-outer, level-inner, the row
 * order of utils/index_utils.py:217-258).
 */
typedef struct wbk_caps {
  int max_jobs;    /* time steps x levels per batch */
  int seg_cap;     /* marching-squares segments per job */
  int contour_cap; /* contours per job (before the length / duplicate filters) */
  int sel_cap;     /* full-width contours (exp_lon == max) per job */
  int pair_cap;    /* streamer candidate pairs per full-width contour */
  int event_cap;   /* events per job and index */
} wbk_caps;

typedef struct wbk_ctx wbk_ctx;

/* bytes of device workspace wbk_create() needs for these capacities */
size_t wbk_workspace_bytes(const wbk_caps* caps, int nlat, int nlon, int add);
/* d_workspace: caller-owned device buffer of >= wbk_workspace_bytes() bytes (256-byte aligned) */
int wbk_create(wbk_ctx** out, const wbk_caps* caps, int nlat, int nlon, int add, void* d_workspace,
               size_t workspace_bytes);
int wbk_destroy(wbk_ctx* ctx);

/* wavebreaking/indices/contour_index.py:86-194 calculate_contours (original_coordinates=False)
 * for every (time step, level) of a batch: marching squares on the periodically extended grid
 * (columns [0, nlon+add), extension = re-read of columns [0, add)), skimage's contour assembly
 * order, np.round + keep-first dedupe, the >= 4 points filter, the periodic duplicate filter
 * (:119-147) and the per-contour closed / exp_lon / mean_lat ingredients.  Results stay in the
 * context until the next call.  d_field: [ntime, nlat, nlon], latitude and longitude ascending.
 */
int wbk_contours(wbk_ctx* ctx, const void* d_field, int dtype, int ntime, const double* h_levels, int nlevels,
                 void* stream);
/* calculate_smoothed_field + calculate_contours without re-reading the smoothed field (float32 under NumPy >= 2
 * promotion, float64 or packed int16 input; float64 smoothed output; 1..WBK_SMOOTH_MAX_FUSED passes): the smoothing
 * kernel leaves, next to the smoothed field, two bits per cell and level ("value > level", "is NaN"; ballots of the
 * values it holds in registers) and the marching-squares stage classifies the squares on those bit planes, fetching
 * the four corner values only for the squares a contour crosses.  Results are identical to wbk_smooth followed by
 * wbk_contours.  opts: as for wbk_smooth. */
int wbk_smooth_contours(wbk_ctx* ctx, const void* d_in, int in_dtype, double* d_smoothed, int ntime, int passes,
                        const double* h_levels, int nlevels, const wbk_smooth_opts* opts, void* stream);
/* per-job results of the last wbk_contours (synchronises the stream): number of contours, number
 * of contour points, status bits (WBK_ST_*), and the batch-wide maximum number of distinct
 * columns of a contour (exp_lon.max() / dlon).  Arrays have ntime*nlevels entries. */
int wbk_contours_counts(wbk_ctx* ctx, int* h_ncontours, int* h_npoints, int* h_status, int* h_max_nx, void* stream);
/* pack the batch's contours into caller-owned device arrays (sizes from wbk_contours_counts):
 *   d_job_off [njobs+1]  first contour of every job
 *   d_pt_off  [C+1]      first point of every contour
 *   d_meta    [C*4]      closed, nx (distinct columns), sum of rows y, job
 *   d_pts     [P]        packed points x | y << 16 in contour order
 * h_job_off_in / h_pt_job_off_in: exclusive prefix sums of the per-job counts (host, njobs+1). */
int wbk_contours_pack(wbk_ctx* ctx, const int* h_ncontours, const int* h_npoints, int* d_job_off, int* d_pt_off,
                      int* d_meta, uint32_t* d_pts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Index stage on a packed contour set (wbk_contours_pack layout; may also be uploaded by the
 * caller, e.g. contours passed by the user).
 */
typedef struct wbk_index_params {
  int do_streamers;    /* indices/streamer_index.py:100-275 */
  int do_overturnings; /* indices/overturning_index.py:99-215 */
  int do_cutoffs;      /* indices/cutoff_index.py:83-98 */
  int gmax_nx;         /* exp_lon.max() / dlon over ALL contours of the call (streamer_index.py:106) */
  double dlon, dlat;
  double geo_dis, cont_dis;        /* streamers: km */
  double range_group, ot_min_exp;  /* overturnings: degrees */
  double co_min_exp;               /* cutoffs: degrees */
} wbk_index_params;

/* event kinds */
#define WBK_EV_STREAMER 0
#define WBK_EV_OVERTURNING 1
#define WBK_EV_CUTOFF 2
/* ints per event record: contour (index into the packed set), i1, i2 (streamer base points; cutoff:
 * 0, npts-1), x0, y0, x1, y1 (overturning box min_lon, min_lat, max_lon, max_lat; else bounding box),
 * orientation (overturning: 0 cyclonic, 1 anticyclonic), split (1 if a vertex has x >= nlon and one has
 * x <= nlon-1: needs the meridian split of utils/index_utils.py:148-173), near (streamers; bit 0: the decision
 * that kept this pair had a distance within 1e-9 relative of geo_dis / cont_dis; bit 1: the pair won its group
 * (streamer_index.py:240-247, longest member) against a member whose length is within 1e-12 relative -- a tie that
 * the last bits of the libm decide, the reference may have kept the other member) */
#define WBK_EV_INTS 10
/* doubles per event record: sum(area), sum(area*data), sum(area*intensity), sum(area*x), sum(area*y),
 * number of member cells  (utils/index_utils.py:66-102) */
#define WBK_EV_F64 6

/* d_coords: device doubles  [lat_deg(nlat) | lat_rad(nlat) | cos(lat_rad)(nlat) | cell_area(nlat) | lon_rad(nlon)]
 * (host-built with the libm calls of the reference so that the trig inputs are identical).
 * d_work: device scratch of 2*npoints doubles (along-contour distances and their prefix sums). */
int wbk_index_run(wbk_ctx* ctx, int njobs, int nlevels, const int* d_job_off, const int* d_pt_off, const int* d_meta,
                  const uint32_t* d_pts, int ncontours, int npoints, const double* d_coords, double* d_work,
                  const wbk_index_params* params, void* stream);

/* utils/index_utils.py:35-126 calculate_properties sums and processing/events.py:66-106 to_xarray flags for
 * the events of the last wbk_index_run.  d_data: [ntime, nlat, nlon], latitude and longitude ascending.
 * d_intensity: NULL (its sums are 0) or [ntime, nlat, nlon] of intensity_dtype (WBK_F32 / WBK_F64 / WBK_I16,
 * independent of dtype), stored as intensity_opts describes it (NULL: ascending and not packed; flip_lat / flip_lon:
 * descending latitudes / longitudes; scale, offset, fill: the CF packing of a WBK_I16 intensity, decoded as wbk_smooth
 * does): member cell (t, y, x) of the ascending grid is read from the stored array and widened to double (decoded
 * for WBK_I16), so the sums equal those of a converted (decoded), re-oriented copy bit for bit.  Only member cells
 * are read.
 * d_flags: NULL or int8 [3][ntime][nlat][nlon] (kind-major), zeroed here and set to 1 where an event of that
 * kind is present; events that straddle the last meridian (split = 1 in their record) are clipped on the
 * device (utils/index_utils.py:148-173) and their pieces rasterised too.
 * The flags use the buffer of events.py:75-79, r = (dlon + dlat) / 4 degrees, measured in degrees: on a grid with
 * dlon != dlat a lattice point is flagged when it is inside, on the boundary or closer than r (in degrees) to an
 * edge.  Flag grids need params->dlon / params->dlat to be an exact ratio p / q of integers <= 64 with
 * max(dlon, dlat) / min(dlon, dlat) < 3 (spacings within 1e-9 of each other count as equal); other spacings give
 * WBK_ERR_INVALID with a message.  The property sums use the radius (dlon + dlat) / 4 in index units on any grid
 * (index_utils.py:47-50). */
int wbk_events_raster(wbk_ctx* ctx, const int* d_job_off, const int* d_pt_off, const uint32_t* d_pts,
                      const double* d_coords, const void* d_data, int dtype, const void* d_intensity,
                      int intensity_dtype, const wbk_smooth_opts* intensity_opts, int ntime, int8_t* d_flags,
                      const wbk_index_params* params, void* stream);

/* Near-threshold decisions of the streamer pair scan of the last wbk_index_run (streamer_index.py:130-139): every
 * pair (i < j, |x_i - x_j| <= 120) for which `geo < geo_dis` or `cont > cont_dis` was decided within 1e-9 (relative)
 * of its threshold while the other test passed or was in its band too -- the pairs that were KEPT and the pairs that
 * were REJECTED.  (CUDA's sin / asin differ from glibc's by <= 2 ulp, so these are the only pairs whose membership
 * may differ from the reference.)  Inside the band `cont` is summed in the reference's order (on[i+1] + ... + on[j]).
 * Record = 4 ints: job, contour (index into the packed set), i, j | kept << 28 | geo_in_band << 29 | cont_in_band << 30.
 * Copies min(cap, WBK_NEAR_CAP) records to d_recs and the number of decisions seen to *d_count (device memory,
 * asynchronous). */
#define WBK_NEAR_CAP 4096
int wbk_near_list(wbk_ctx* ctx, int* d_recs, int cap, int* d_count, void* stream);

/* per-kind, per-job event counts of the last wbk_index_run (synchronises): h_counts [3][njobs] */
int wbk_events_counts(wbk_ctx* ctx, int* h_counts, int* h_status, void* stream);
/* events of one kind, job-major in reference row order: h_ints [n][WBK_EV_INTS], h_f64 [n][WBK_EV_F64], h_job [n] */
int wbk_events_fetch(wbk_ctx* ctx, int kind, int n, int* h_ints, double* h_f64, int* h_job, void* stream);

/* generic lattice-polygon rasteriser (to_xarray for arbitrary event tables, and the split pieces):
 * rings in index coordinates of the REAL grid (no folding), ring r = vertices
 * [d_ring_off[r], d_ring_off[r+1]) of d_xy (int32 x,y pairs), written at time index d_ring_t[r].
 * Cells inside (non-zero winding), on the boundary or closer than sqrt(r2) cells to an edge are selected
 * (processing/events.py:75-79).  d_out_i8 != NULL: int8 [ntime][nlat][nlon], selected cells := 1.
 * d_out_f64 != NULL: double [ntime][nlat][nlon], selected cells := d_ring_val[r] where r is the LAST ring
 * (highest index) selecting the cell (events.py:96-102); needs d_owner, int32 [ntime][nlat][nlon] scratch.
 * Outputs are NOT zeroed here. */
int wbk_rasterize_rings(const int* d_xy, const int* d_ring_off, const int* d_ring_t, const double* d_ring_val,
                        int nrings, int nlat, int nlon, int ntime, double r2, int8_t* d_out_i8, double* d_out_f64,
                        int* d_owner, void* stream);

/* processing/events.py:66-106 to_xarray on a regular grid with spacings dlon, dlat (degrees): like
 * wbk_rasterize_rings (same rings, outputs and last-writer rule), with the buffer r = (dlon + dlat) / 4 degrees
 * (events.py:75-79) measured in degrees, so that on a grid with dlon != dlat the buffer is an ellipse in index units.
 * dlon / dlat must be an exact ratio p / q of integers <= 64 with max(dlon, dlat) / min(dlon, dlat) < 3 (spacings
 * within 1e-9 of each other count as equal: r = 1/2 cell); other spacings give WBK_ERR_INVALID with a message. */
int wbk_rasterize_rings_grid(const int* d_xy, const int* d_ring_off, const int* d_ring_t, const double* d_ring_val,
                             int nrings, int nlat, int nlon, int ntime, double dlon, double dlat, int8_t* d_out_i8,
                             double* d_out_f64, int* d_owner, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Sync-free batch plumbing (what wavebreaking_b200/pipeline.py uses): nothing below waits for the device.
 *
 * wbk_contours_pack_auto: like wbk_contours_pack, but the prefix sums run on the device and the caller's
 * buffers are capacity bounded (d_pt_off [cap_contours+1], d_meta [cap_contours*4], d_pts [cap_points]).
 * wbk_index_run may then be called with gmax_nx < 0 (= use the batch maximum found by wbk_contours) and
 * ncontours / npoints = the capacities.
 *
 * wbk_batch_fetch: after wbk_events_raster, gathers ALL events (kind-major, then job, then reference order)
 * into d_out_int [cap_events][WBK_EV_INTS], d_out_f64 [cap_events][WBK_EV_F64], d_out_job [cap_events], the
 * ring vertices of every streamer / cutoff event into d_ring_pts (event e = [d_ring_off[e], d_ring_off[e+1])),
 * and writes the summary record d_summary[16] = contours, points, streamers, overturnings, cutoffs,
 * OR of all status bits, max_nx, split pieces, marching-squares segments, streamer candidate pairs (after the pair
 * scan), near-threshold decisions, active pair-scan tiles, 4 reserved.  The caller copies these buffers to the host
 * and synchronises once. */
int wbk_contours_pack_auto(wbk_ctx* ctx, int* d_job_off, int* d_pt_off, int* d_meta, uint32_t* d_pts, int cap_contours,
                           int cap_points, void* stream);
int wbk_batch_fetch(wbk_ctx* ctx, const int* d_pt_off, const uint32_t* d_pts, int* d_out_int, double* d_out_f64,
                    int* d_out_job, int* d_ring_off, uint32_t* d_ring_pts, int cap_events, int cap_ring, int* d_summary,
                    void* stream);

/* Pieces of the events that straddle the last meridian (utils/index_utils.py:148-173 transform_polygons), as the
 * device clipper of the last wbk_events_raster / wbk_split_clip left them: ring r = vertices
 * [d_ring_off[r], d_ring_off[r+1]) of d_xy (int32 x, y: folded index coordinates of the real grid), d_ring_ev[r] = row of
 * the event in the wbk_batch_fetch tables.  d_count[3] = pieces, vertices, clipper overflow flag (pieces > cap_rings
 * or vertices > cap_vertices: the caller's buffers were too small).  Asynchronous. */
/* Run the device clipper on the straddling events of the last wbk_events_raster when that call had no flag grids
 * (d_flags == NULL; with flag grids the clipper has already run and this is a no-op).  Asynchronous. */
int wbk_split_clip(wbk_ctx* ctx, const int* d_pt_off, const uint32_t* d_pts, void* stream);
int wbk_split_fetch(wbk_ctx* ctx, int* d_ring_ev, int* d_ring_off, int* d_xy, int cap_rings, int cap_vertices,
                    int* d_count, void* stream);

/* Bit-packed copy of flag grids for the device -> host link: cell c of d_flags (int8, != 0 means set) becomes bit
 * (c & 7) of byte c >> 3 of d_packed (numpy.unpackbits(..., bitorder="little") restores the grid).  d_packed holds
 * 4 * ceil(ncells / 32) bytes; d_flags 16-byte aligned, d_packed 4-byte aligned. */
int wbk_pack_flags(const int8_t* d_flags, uint8_t* d_packed, long long ncells, void* stream);

/* Occurrence counts behind a flag-frequency climatology.
 * d_flags : int8 [nkinds][ntime][ncells], the layout wbk_events_raster writes (nkinds = 3, kind stride ntime * ncells,
 *           where ntime is the batch length, not the capacity of the buffer).
 * d_group : int32 [ntime] (device): the group of each time step in [0, ngroups), or -1 = step not counted.  Any value
 *           outside [0, ngroups) is ignored like -1.
 * d_counts: uint32 [ngroups][nkinds][ncells]; counts[g][k][c] += #{t : group[t] == g && flags[k][t][c] != 0}.
 * Several streams may add into the same d_counts at once (atomic adds).  Nothing is zeroed.  16-byte loads are used
 * when ncells % 16 == 0 and d_flags is 16-byte aligned, byte loads otherwise.  ntime == 0 or ncells == 0 is a no-op.
 * Asynchronous. */
int wbk_flag_counts(const int8_t* d_flags, int nkinds, int ntime, long long ncells, const int* d_group, int ngroups,
                    uint32_t* d_counts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Per-kernel device timing (CUDA events on the launching stream around every kernel launch of the
 * library).  wbk_prof_enable(1) starts collecting, wbk_prof_read synchronises the device and returns, for
 * kernel id k < WBK_PROF_NKERNELS, the number of launches and the summed duration in milliseconds since
 * the last wbk_prof_reset().  Names: wbk_prof_name(k). */
#define WBK_PROF_NKERNELS 32
int wbk_prof_enable(int on);
int wbk_prof_reset(void);
int wbk_prof_read(int* h_launches, double* h_ms);
const char* wbk_prof_name(int k);
/* total number of kernel launches issued by the library in this process (always counted) */
long long wbk_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * wavebreaking/processing/events.py:113-241 track_events.  Events are sorted by date on the host; everything
 * that scales with the number of event pairs runs here.
 *
 * wbk_track_candidates (events.py:160-181): d_lo / d_hi [n] give, per event i, the index window [lo, hi) of the
 * events j with 0 < date_j - date_i <= time_range.  Appends every (i, j) of the windows whose integer bounding
 * boxes d_bbox [n][4] = x0, y0, x1, y1 intersect (d_bbox NULL: all of them) to d_pairs [cap][2], in no particular
 * order; *d_count receives the number found (> cap: the caller retries with a larger buffer). */
int wbk_track_candidates(const int* d_lo, const int* d_hi, const int* d_bbox, int n, int* d_pairs, int cap,
                         int* d_count, void* stream);

/* events.py:205-214 with overlap = 0 (`inter.area / union.area > 0`), decided exactly for lattice polygons
 * (integer vertices in [0, 4096)).  d_edges [V][4]: for every vertex its edge x0, y0, x1, y1 to the next vertex of
 * its ring; d_vsign [V]: orientation of the vertex's ring (+1 counter-clockwise, -1 clockwise, 0 degenerate);
 * ring r = vertices [d_ring_off[r], d_ring_off[r+1]), polygon p = rings [d_poly_off[p], d_poly_off[p+1]) (non-zero
 * winding over all rings).  d_result[k]: bit 0 = the polygons of pair k share a region of positive area, bit 1 =
 * their boundaries touch without crossing (decided piece by piece). */
int wbk_track_overlap_exact(const int* d_edges, const int* d_vsign, const int* d_ring_off, const int* d_poly_off,
                            const int* d_pairs, int npairs, int* d_result, void* stream);

/* events.py:205-214 for overlap > 0: float64 areas of event pairs.
 * Polygons are given as rings of double (x, y) vertices: polygon p = rings [d_poly_off[p], d_poly_off[p+1]),
 * ring r = vertices [d_ring_off[r], d_ring_off[r+1]) of d_xy (open rings).  For pair k = (d_pairs[2k],
 * d_pairs[2k+1]) writes d_out[3k..3k+2] = area(A), area(B), area(A n B).
 * Every ring is the region it encloses under non-zero winding, whatever its orientation: area(P) is the sum of
 * |area(ring)| over the rings of P, and a ring of zero area adds nothing.  The parts of one polygon must not overlap
 * each other (such a MultiPolygon is invalid; GEOS does not define its area either).  The arithmetic runs on
 * coordinates relative to the first vertex of A, so lattice pairs give the same areas bit for bit under any integer
 * translation.  d_vsign of wbk_track_overlap_exact follows the same orientation rule. */
int wbk_track_overlap(const double* d_xy, const int* d_ring_off, const int* d_poly_off, const int* d_pairs, int npairs,
                      double* d_out, void* stream);

/* events.py:187-201 by_distance: sklearn's haversine (unit sphere, radians) of the rows d_rad [n][2] of every
 * pair, in sklearn's operand order; d_out [npairs].  CUDA's libm differs from glibc's by <= 2 ulp: the caller
 * re-decides pairs within 1e-9 of its threshold on the host. */
int wbk_track_distance(const double* d_rad, const int* d_pairs, int npairs, double* d_out, void* stream);

/* Tracking polygons of one kind of a batch, read from the device buffers of wbk_batch_fetch / wbk_split_fetch and
 * appended to a caller-owned window in the layout wbk_track_candidates and wbk_track_overlap_exact read
 * (utils/index_utils.py:129-184 transform_polygons, vertex for vertex as pipeline.events_soup builds them).
 * Input: the rows [first, first + n) of d_ev_int [rows][WBK_EV_INTS] (the kind-major gather), their rings
 * d_ring_off [rows + 1] / d_ring_pts (packed x | y << 16), and the npieces device-clipper pieces d_sp_ev / d_sp_off /
 * d_sp_xy.  A row with split == 1 becomes its pieces (in piece order), an overturning (is_box) the box
 * (x1, y0), (x1, y1), (x0, y1), (x0, y0), any other row its ring; x is folded with x % nlon.
 * Output, starting at vertex v0, ring r0 and polygon p0 of the window: d_edges [V][4] (x0, y0, x1, y1 of the edge
 * to the next vertex of the ring), d_vsign [V] (sign of the ring's doubled area), d_win_ring_off (ring r0 + k =
 * vertices [ring_off[r0 + k], ring_off[r0 + k + 1]), absolute), d_win_poly_off (absolute, like the ring offsets) and
 * d_bbox [P][4] (x0, y0, x1, y1; (1, 1, 0, 0) for a polygon without vertices).  nrings / nverts: what this batch adds
 * (the caller knows them from the host copies of the ring and piece offsets).  cap_v / cap_r / cap_p: the sizes of
 * d_edges (and d_vsign), d_win_ring_off and d_win_poly_off in elements; WBK_ERR_INVALID when the batch does not fit
 * or the window would pass 2^31 - 1 vertices, rings or polygons (the offsets are int32).  Asynchronous. */
int wbk_track_append(const int* d_ev_int, const int* d_ring_off, const uint32_t* d_ring_pts, const int* d_sp_ev,
                     const int* d_sp_off, const int* d_sp_xy, int npieces, int first, int n, int is_box, int nlon,
                     long long nrings, long long nverts, int* d_edges, int* d_vsign, int* d_win_ring_off,
                     int* d_win_poly_off, int* d_bbox, long long v0, long long r0, long long p0, long long cap_v,
                     long long cap_r, long long cap_p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WBK_H */
