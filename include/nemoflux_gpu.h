/*
 * nemoflux_gpu.h -- C ABI of libnemoflux_gpu.so: the B200 (sm_100a) transect-flux hot path of
 * pletzer/nemoflux behind the interface nemoflux binds today.
 *
 * What it replaces.  nemoflux reaches its native code through python-mint's ctypes bindings of
 * libmint's C API (mnt_grid_*, mnt_polylineintegral_*; call sites /root/reference/nemoflux/
 * horizgrid.py:23-24, field.py:45-48, field.py:102, fluxplot.py:56) and does the C-grid edge-flux
 * assembly itself in numpy (field.py:145-234).  Each entry point below cites the call it stands for.
 *
 * Conventions (the same as libmint's): every function returns int, 0 = success, non-zero = error
 * code (NFX_E_*), details through nfx_last_error(); objects are opaque and passed as T** like mint's
 * handles; no exception crosses the boundary; the caller owns every array.  Arrays marked "host"
 * are ordinary host memory, arrays marked "device" are CUDA device pointers that the library only
 * borrows (e.g. torch tensor.data_ptr()); `stream` is a cudaStream_t passed as void* (NULL = the
 * legacy default stream).  A handle is bound to the CUDA device that was current when it was
 * created; calls on one handle must be serialised by the caller.
 */
#ifndef NEMOFLUX_GPU_H
#define NEMOFLUX_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFX_OK 0
#define NFX_E_INVALID 1   /* bad argument / call order            */
#define NFX_E_CUDA 2      /* a CUDA runtime call failed           */
#define NFX_E_NOGPU 3     /* no usable CUDA device                */
#define NFX_E_ALLOC 4     /* out of host or device memory         */
#define NFX_E_INTERNAL 5

/* mint.CELL_BY_CELL_DATA (field.py:102): data is (ncells, 4), one private datum per cell edge */
#define NFX_CELL_BY_CELL_DATA 0

/* storage type of uo/vo */
#define NFX_F64 0   /* datagen.py:9 writes float64 */
#define NFX_F32 1   /* real NEMO output            */
/* OR into dtype for nfx_flux_series_host only: the host buffers hold BIG-ENDIAN values, i.e. the bytes of a
 * NetCDF classic file as stored on disk (what scipy.io.netcdf_file memory-maps).  The raw bytes are uploaded and the
 * byte order is swapped on the device, instead of a conversion pass over the data on the host CPU. */
#define NFX_BIG_ENDIAN 0x100

/* summation order of the transect integral */
#define NFX_ORDER_LIST 0  /* emission order: sub-segment by sub-segment, edges 0..3          */
#define NFX_ORDER_MAP 1   /* mint's std::map<(cellId,edgeIndex),weight> order (default)     */

/* ---- tuning options (nfx_set_option / nfx_get_option) ----------------------------------------------------------
 * Process-wide, not thread safe: set them before the calls they affect.  Every value changes speed only, never a
 * result bit (the parity tests sweep them).  The defaults are the measured optimum on B200 (profiles/). */
#define NFX_OPT_K2_VARIANT 1       /* edge-flux kernel of the two-launch path: */
#define NFX_K2_AUTO 0              /*   direct loads, 256-bit for float64 storage, 128-bit for float32 */
#define NFX_K2_LDG 1               /*   direct vectorised global loads, widest legal (256-bit on sm_100a) */
#define NFX_K2_TMA 2               /*   1-D bulk copies (cp.async.bulk + mbarrier) into shared-memory stages */
#define NFX_K2_LDG128 3            /*   direct loads capped at 128 bits */
#define NFX_OPT_K2_UNROLL 2        /* levels in flight per thread (0 = default 5); TMA: tile configuration id */
#define NFX_OPT_K2_BLOCK 3         /* threads per CTA (0 = default 256) */
#define NFX_OPT_FAST_SERIES 4      /* nfx_flux_series with eflux == NULL: 1 (default) fused L2-resident pass where it
                                      is the faster one, 2 always fused, 0 never (two launches) */
#define NFX_OPT_RING_SLOT_MB 5     /* size of one edge-flux ring slot of the fused pass in MB; 0 (default) = automatic:
                                      a time step of up to 8 MB is one panel, larger grids are cut into panels of
                                      about 4 MB (float64 storage) or 8 MB (float32) */
#define NFX_OPT_K2_ALU_MASK 6      /* float32 storage, two-launch K2: which of every 5 levels take the bit-shuffle
                                      conversion instead of F2F (-1 = default, all; 0 = none) */
#define NFX_OPT_FUSED_F32_SHAPE 7  /* fused pass, float32 storage: 10 * vector width + unroll (85, 45, 83, 43; 0 = 45) */
#define NFX_OPT_LAST_SERIES_PATH 8 /* READ ONLY: 1 = the last nfx_flux_series* call took the fused pass, 0 = two
                                      launches, -1 = none yet */
#define NFX_OPT_FUSED_ORDER 9      /* fused pass: bit 0 = visit the (time step, panel) batches panel-major, bit 1 = K3
                                      gathers unrolled x8 (default 3) */
#define NFX_OPT_FUSED_F64_CTAS 10  /* fused pass, float64 storage, 256-bit loads: register budget for 2 or 4 CTAs per
                                      SM (0 = default 3) */
#define NFX_OPT_FUSED_K3_LAG 15    /* fused pass: the K3 items of batch b - lag are queued behind the K2 tiles of batch b
                                      (0 = automatic: one-panel grids the batches the resident CTAs span + 1, else 1) */

#define NFX_OPT_RING_MAX_MB 16      /* fused pass: upper bound of the whole edge-flux ring in MB (0 = default 24) */
#define NFX_OPT_SPARSE_COLUMNS 17   /* fused pass: 0 = K2 reads every column of u, v; 2 = only the groups of columns
                                       whose edge fluxes the transects read (nfx_pli_get_column_groups); 1 (default) =
                                       sparse while those groups are less than 80 % of the grid's.  Same series bits. */
#define NFX_OPT_LAST_SERIES_SPARSE 18  /* READ ONLY: 1 = the last nfx_flux_series* call took the sparse fused pass,
                                          0 = the dense fused pass or two launches, -1 = none yet */

typedef struct nfx_grid nfx_grid;
typedef struct nfx_pli nfx_pli;
typedef struct nfx_vinterp nfx_vinterp;

const char* nfx_last_error(void);
int nfx_version(void);
int nfx_set_option(int option, int value);
int nfx_get_option(int option, int* value);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int nfx_launch_count(int64_t* n);
/* Debug aid (compute-sanitizer is not available on every pool): with NFX_DEBUG_GUARDS=1 in the environment every
 * device buffer the library owns carries 4 KB guard bands; this call synchronises the device, checks them all and
 * returns NFX_E_INTERNAL (details in nfx_last_error) when a kernel wrote before the start or past the end of one.
 * *nbuffers = buffers checked (0 when the guards are off), *ndamaged = buffers with a damaged band. */
int nfx_debug_check_guards(int64_t* nbuffers, int64_t* ndamaged);
/* self-test of the above: overwrites the byte right before (where = 0) or right behind (1) the most recently allocated
 * guarded buffer; refuses to do anything unless NFX_DEBUG_GUARDS is set */
int nfx_debug_poke_guard(int where);

/* ---- mint.Grid: Grid(), setPoints(points), getNumberOfCells()  (horizgrid.py:23-24,30) ---------- */
int nfx_grid_new(nfx_grid** self);
int nfx_grid_del(nfx_grid** self);
/* points: host (ncells,4,3) float64, vertices 0=SW 1=SE 2=NE 3=NW, (lon deg, lat deg, unused);
 * copied to the device (mint borrows the pointer instead, horizgrid.py:24) */
int nfx_grid_set_points(nfx_grid** self, int64_t ncells, const double* points);
int nfx_grid_get_num_cells(nfx_grid** self, int64_t* ncells);
/* the structured shape behind the cell ids (cell = j*nx + i, horizgrid.py:17-22); needed by the
 * compact [eU|eV] flux layout (field.py:209-223), not by the mint-style calls */
int nfx_grid_set_cgrid_shape(nfx_grid** self, int ny, int nx);
/* arc (ncells,4) device: unit-sphere length of edge e -> e+1 (Field.computeArcLengths, field.py:170-181) with the
 * well-conditioned haversine of the lon/lat differences.  NOT bit-compatible with the reference's arccos(a.b) (geo.py:24-27),
 * which the parity path keeps on the host; differences are the reference's own rounding noise (~1e-16/arc). */
int nfx_grid_arc_lengths(nfx_grid** self, double* arc, void* stream);

/* ---- mint.PolylineIntegral  (field.py:45-48, field.py:102, fluxplot.py:56) ----------------------- */
int nfx_pli_new(nfx_pli** self);
int nfx_pli_del(nfx_pli** self);
int nfx_pli_set_grid(nfx_pli** self, nfx_grid* grid);
/* buildLocator(numCellsPerBucket=128, periodX=360., enableFolding=False), field.py:47.  Builds the
 * device-side bounding-box hierarchy ONCE per grid, shared by all transects (the reference rebuilds
 * a locator per transect).  numCellsPerBucket is accepted and ignored, enableFolding must be 0. */
int nfx_pli_build_locator(nfx_pli** self, int num_cells_per_bucket, double period_x, int enable_folding);
/* computeWeights(xyz (npoints,3) float64 host, counterclock=False), field.py:48: one transect */
int nfx_pli_compute_weights(nfx_pli** self, int npoints, const double* xyz, int counterclock);
/* the batched form: ntransects polylines; offsets (ntransects+1) indexes points in xyz (total,3) */
int nfx_pli_compute_weights_batch(nfx_pli** self, int ntransects, const int* offsets, const double* xyz,
                                  int counterclock);
int nfx_pli_get_num_transects(nfx_pli** self, int* ntransects);
/* sub-segments in emission order (transect, segment, ta, cell, image); every output is host memory
 * and may be NULL; transect_offsets has ntransects+1 entries; xia/xib are (n,2), w is (n,4) */
int nfx_pli_get_num_subsegments(nfx_pli** self, int64_t* n);
int nfx_pli_get_subsegments(nfx_pli** self, int64_t* transect_offsets, int64_t* cell, int32_t* seg, int32_t* img,
                            double* ta, double* tb, double* coeff, double* xia, double* xib, double* w);
/* mint's map view: per transect the unique keys cell*4+edge (ascending) and accumulated weights */
int nfx_pli_get_map_size(nfx_pli** self, int64_t* n);
int nfx_pli_get_map(nfx_pli** self, int64_t* transect_offsets, int64_t* keys, double* w);
/* getIntegral(data (ncells,4) float64 host, CELL_BY_CELL_DATA) -> result (field.py:102); for a batch
 * `results` receives ntransects values */
int nfx_pli_get_integral(nfx_pli** self, const double* data, int placement, double* result);
int nfx_pli_get_integrals(nfx_pli** self, const double* data, int placement, int order, double* results);
/* same with data already on the device: data device (nt, ncells, 4), results device (nt, ntransects) */
int nfx_pli_get_integrals_device(nfx_pli** self, const double* data, int nt, int order, double* results,
                                 void* stream);

/* ---- mint.VectorInterp  (field.py:90-95,119-120; the arrow glyphs of the viewer, SURVEY 8f rank 3) ------------ */
int nfx_vinterp_new(nfx_vinterp** self);
int nfx_vinterp_del(nfx_vinterp** self);
int nfx_vinterp_set_grid(nfx_vinterp** self, nfx_grid* grid);
/* buildLocator(numCellsPerBucket=128, periodX=360.), field.py:92: shares the grid's bounding-box hierarchy */
int nfx_vinterp_build_locator(nfx_vinterp** self, int num_cells_per_bucket, double period_x, int enable_folding);
/* findPoints(points (npoints,3) host, tol2=1e-12), field.py:93: containing cell (lowest id) and parametric
 * coordinates of every point; num_not_found may be NULL */
int nfx_vinterp_find_points(nfx_vinterp** self, int64_t npoints, const double* xyz, double tol2, int64_t* num_not_found);
int nfx_vinterp_get_cells(nfx_vinterp** self, int64_t* cell, double* xi);
/* getFaceVectors(data (ncells,4) host, placement=0) -> vectors (npoints,3) host, field.py:94-95 */
int nfx_vinterp_get_face_vectors(nfx_vinterp** self, const double* data, int placement, double* vectors);
/* the same with data (ncells,4) and vectors (npoints,3) on the device */
int nfx_vinterp_get_face_vectors_device(nfx_vinterp** self, const double* data, double* vectors, void* stream);

/* ---- Field.readField + Field.computeIntegratedFlux  (field.py:145-163, 183-234)  = kernel K2 ----- */
/* u, v: device (nt, nz, ncell) of dtype; thickness device (nz) = deptht_bounds[:,1]-[:,0]
 * (field.py:51); arc1/arc2 device (ncell) = arcLengths[:,1], arcLengths[:,2] (field.py:195-196);
 * NaN (and values equal to `fill` when fill is not NaN) count as 0 (field.py:157); sverdrup
 * multiplies by 6371000/1e6 (field.py:225-228).
 * eflux: device (nt, 2*ncell): [t, 0:ncell] = signed eU, [t, ncell:2*ncell] = signed eV. */
int nfx_edgeflux_assemble(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                          const double* arc2, int nt, int nz, int64_t ncell, int sverdrup, double fill,
                          double* eflux, void* stream);
/* the same with a padded level plane: u, v are (nt, nz, ld) with ld >= ncell cells per plane in memory (the
 * device layout is the caller's: ld % 4 == 0 gives 32-byte aligned rows and 256-bit loads for every grid size,
 * ORCA025/ORCA12 planes are only 16-byte aligned when stored densely) */
int nfx_edgeflux_assemble_ld(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                             const double* arc2, int nt, int nz, int64_t ncell, int64_t ld, int sverdrup, double fill,
                             double* eflux, void* stream);
/* SURVEY 8f rank 4 -- per-column, per-level vertical scale factors (NEMO e3u/e3v: partial cells, z*) instead of
 * the 1-D layer thickness of field.py:51: U = sum_k e3u[t,k,c]*u[t,k,c].  e3u, e3v: device, dtype and plane
 * layout of u, v, (e3_nt, nz, ld) with e3_nt = 1 (time-invariant, e.g. e3u_0 of mesh_mask) or nt.
 * Algorithmic bytes double (4 streamed arrays). */
int nfx_edgeflux_assemble_e3(const void* u, const void* v, const void* e3u, const void* e3v, int dtype, int e3_nt,
                             const double* arc1, const double* arc2, int nt, int nz, int64_t ncell, int64_t ld,
                             int sverdrup, double fill, double* eflux, void* stream);
int nfx_flux_series_e3(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                       int e3_nt, const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup,
                       double fill, int order, double* eflux, double* series, void* stream);
/* the (ncell,4) mint layout of field.py:209-223 from the compact one: south edges of row 0 are 0,
 * west edges x-periodic.  eflux device (nt, 2*ncell) -> iv device (nt, ncell, 4) */
int nfx_edgeflux_to_cell_by_cell(const double* eflux, int nt, int ny, int nx, double* iv, void* stream);
/* max |eU|, max |eV| over all nt steps (field.py:230-234); result host (1) */
int nfx_edgeflux_absmax(const double* eflux, int nt, int64_t ncell, double* result, void* stream);

/* ---- the fluxplot.py:51-59 loop = kernel K3, and K2+K3 in one call ------------------------------- */
/* series device (nt, ntransects): sum_n w_n * eflux[t, index(cell_n, edge_n)]; needs
 * nfx_grid_set_cgrid_shape before nfx_pli_compute_weights* */
int nfx_pli_integrate(nfx_pli** self, const double* eflux, int nt, int order, double* series, void* stream);
/* nfx_flux_series: eflux may be NULL -- then the edge fluxes are not materialised in HBM at all: K2 writes
 * them into a small ring that stays in L2 and K3 consumes them from there (the fast path).  With eflux != NULL
 * the (nt, 2*ncell) array is produced as by nfx_edgeflux_assemble. */
int nfx_flux_series(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                    const double* arc1, const double* arc2, int nt, int nz, int sverdrup, double fill, int order,
                    double* eflux, double* series, void* stream);
int nfx_flux_series_ld(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                       const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup, double fill,
                       int order, double* eflux, double* series, void* stream);
/* Flux series per layer of model levels (extension, no counterpart in the reference).  layer_levels: HOST (nlayers+1)
 * int, strictly ascending, 0 <= layer_levels[0], layer_levels[nlayers] <= nz; layer i = levels
 * [layer_levels[i], layer_levels[i+1]).  Exactly one of thickness / (e3u, e3v) as in nfx_flux_series / _e3.
 * series device (nt, nlayers, ntransects); eflux NULL (fused pass where the policy allows) or device
 * (nt, nlayers, 2*ncell).  Layer i is nfx_flux_series* with the thickness (or e3) zeroed outside the layer, bit for bit
 * on finite data; an infinity on a level outside the layer does not reach it.  u, v (and e3u, e3v) are read once
 * whatever the layering.  An invalid layering (nlayers < 1, not strictly ascending, outside [0, nz],
 * nt * nlayers * npanels over INT_MAX) returns NFX_E_INVALID before anything is launched. */
int nfx_flux_series_layers(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                           int e3_nt, const double* thickness, const double* arc1, const double* arc2, int nt, int nz,
                           int64_t ld, int nlayers, const int* layer_levels, int sverdrup, double fill, int order,
                           double* eflux, double* series, void* stream);
/* Transport section (extension, no counterpart in the reference): the flux of every sub-segment (cell crossing, the
 * emission order of nfx_pli_get_subsegments) per layer of model levels.  Arguments as nfx_flux_series_layers without
 * order and eflux; section device (nt, nlayers, nsub):
 *   section[t, i, s] = ((w[s,0]*E[idx[4s]] + w[s,1]*E[idx[4s+1]]) + w[s,2]*E[idx[4s+2]]) + w[s,3]*E[idx[4s+3]]
 * with idx the list-order compact flux index (E, W, N, S edges; -1 = 0), E the layer-i edge flux exactly as
 * nfx_flux_series_layers writes it into eflux, separate multiplies and adds (no FMA): summing a transect's sub-segments
 * gives its layered series to rounding.  One launch per 65535 time steps, asynchronous on `stream`, no spin waits (it
 * neither sets nor reports the handle's fused-pass error flag).  An invalid layering, a NULL pointer or transects
 * computed without nfx_grid_set_cgrid_shape return NFX_E_INVALID before anything is launched; nt == 0 or no
 * sub-segment launches nothing. */
int nfx_flux_section(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                     int e3_nt, const double* thickness, const double* arc1, const double* arc2, int nt, int nz,
                     int64_t ld, int nlayers, const int* layer_levels, int sverdrup, double fill, double* section,
                     void* stream);
/* Time-mean transport section (extension): the section of nfx_flux_section summed over windows of time steps.
 * Arguments as nfx_flux_section, plus window_bounds (host, nwindows + 1 step indices relative to the steps passed,
 * 0 <= b0 < b1 < ... < bK <= nt): window w covers the steps [b_w, b_{w+1}); steps outside [b0, bK) are not read.
 * sums device (nwindows, nlayers, nsub):
 *   sums[w, i, s] = (((+0 + sec[b_w, i, s]) + sec[b_w + 1, i, s]) + ...) + sec[b_{w+1} - 1, i, s]
 * with sec exactly the value nfx_flux_section computes, every add a separate round-to-nearest double add in ascending
 * step order (so a one-step window of -0 holds +0).  continue_first != 0: window 0 starts from the partial sums already
 * in sums[0] instead of +0, so a window split over several calls (in step order) sums to the bits of one call.  The
 * mean is sums / (b_{w+1} - b_w), left to the caller.  Launches split so that gridDim.y <= 65535; asynchronous on
 * `stream`.  An invalid layering or window list (nt == 0 has none), nwindows * nlayers * nsub overflowing, or any
 * refusal of nfx_flux_section returns NFX_E_INVALID before anything is launched; no sub-segment launches nothing. */
int nfx_flux_section_window_sums(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                                 int dtype, int e3_nt, const double* thickness, const double* arc1, const double* arc2,
                                 int nt, int nz, int64_t ld, int nlayers, const int* layer_levels, int sverdrup,
                                 double fill, int nwindows, const int* window_bounds, int continue_first, double* sums,
                                 void* stream);
/* Class transport (extension): the flux across every transect binned by a T-grid field c (temperature, salinity,
 * density...).  Arguments as nfx_flux_section with one layer per level, plus the class field cfield (device, c_nt x nz
 * planes of ld values, the dtype of u, v; c_nt = 1: time-invariant, or nt), its missing-value marker cfill (NaN = none;
 * compared in the storage type, as fill) and class_bounds (host, nclasses + 1 strictly ascending doubles, +-inf
 * allowed, no NaN; 1 <= nclasses <= 96).  classes device (nt, nclasses, M):
 *   classes[t, j, m] = sum over the crossings s of transect m and the levels k with b_j <= c[t|0, k, cell(s)] < b_{j+1}
 *                      of f[t, k, s], the value nfx_flux_section computes for the one-level layer k
 * A level whose class value is NaN, the marker, below b0 or at or above bK counts nowhere.  Sum order: per crossing
 * and class the levels in ascending order from +0; the crossings of a transect in tiles of 32 in emission order, each
 * folded by a fixed shuffle tree (lane l + lane l + o, o = 16, 8, 4, 2, 1); the tiles in ascending order from +0.  The
 * bits depend only on the inputs.  Asynchronous on `stream`, except that the bounds (and, on the first call after
 * computeWeights, the crossing tiles) are copied from pageable host memory, which waits for the work already queued on
 * `stream`.  The bounds, tiles and partial sums are scratch of the handle: calls on one handle must not run
 * concurrently on different streams.  Invalid bounds, too many classes, a NULL pointer, or
 * transects computed without nfx_grid_set_cgrid_shape return NFX_E_INVALID before anything is launched; nt == 0 or no
 * crossing launches nothing and leaves `classes` as it is. */
int nfx_flux_classes(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                     int e3_nt, const double* thickness, const double* arc1, const double* arc2, int nt, int nz,
                     int64_t ld, const void* cfield, int c_nt, double cfill, int nclasses, const double* class_bounds,
                     int sverdrup, double fill, double* classes, void* stream);
/* Tracer transport (extension): heat, salt, freshwater... carried across every transect, per layer of model levels.
 * Arguments as nfx_flux_section, plus the tracer (device, tr_nt x nz planes of ld values at the T points, the dtype of
 * u, v; tr_nt = 1: time-invariant, or nt), its missing-value marker tfill (NaN = none; compared in the storage type, as
 * fill; NaN is always missing) and a reference value ref.  Every edge is one C-grid face between two T cells: E eU[c]
 * (c, east(c)), W eU[west(c)] (west(c), c), N eV[c] (c, north(c); none in the top row), S eV[south(c)] (south(c), c);
 * east / west wrap x-periodically.  At level k the face value is
 *   q = 0.5 * (tau_a + tau_b) - ref (both sides present), tau_a - ref (one side present), 0 (neither)
 * and per crossing, layer and edge A_e = sum over the layer's levels in ascending order from +0 of (d_k * u_e,k) * q_e,k
 * (d_k: thickness or e3u/e3v; u with NaN and `fill` as 0).  The crossing's value is nfx_flux_section's operations on
 * the 4 sums A_e (arcs, sverdrup, the sign of eV, the weights in edge order); every operation is rounded on its own, in
 * double.  With tau == 1 and ref == 0 it is nfx_flux_section's value bit for bit.
 *   section device (nt, nlayers, nsub) or NULL: that value;
 *   series  device (nt, nlayers, M) or NULL: the crossings of every transect in tiles of 32 in emission order, each
 *           folded by a fixed shuffle tree (lane l + lane l + o, o = 16, 8, 4, 2, 1), the tiles in ascending order
 *           from +0 (the sum order of nfx_flux_classes).
 * One of series, section may be NULL, not both.  The bits depend only on the inputs.  Asynchronous on `stream`, except
 * that the layering (when it differs from the previous call's) and, on the first call after computeWeights, the
 * crossing tiles are copied from pageable host memory, which waits for the work already queued on `stream`.  The tiles
 * and partial sums are scratch of the handle: calls on one handle must not run concurrently on different streams.  A
 * NULL pointer, tr_nt not in {1, nt}, a bad layering, or transects computed without nfx_grid_set_cgrid_shape return
 * NFX_E_INVALID before anything is launched; nt == 0 or no crossing launches nothing and leaves the outputs as they
 * are.  Units: tracer units x flux units (heat in W: rho0 * cp x the result with metre metrics; freshwater:
 * -1 / S_ref x the result with ref = S_ref). */
int nfx_flux_tracer(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                    int e3_nt, const double* thickness, const double* arc1, const double* arc2, int nt, int nz,
                    int64_t ld, const void* tracer, int tr_nt, double tfill, double ref, int nlayers,
                    const int* layer_levels, int sverdrup, double fill, double* series, double* section,
                    void* stream);
/* The device-path series calls (nfx_flux_series*, nfx_flux_series_range*) are asynchronous on `stream`.  Their fused
 * pass spins on per-batch counters with a bound; a pass that ever overflowed it aborts and leaves NaN in `series`.
 * nfx_pli_series_status synchronises `stream` and reports that: returns 0 with *status = 0 when every pass launched
 * on the handle so far completed, NFX_E_INTERNAL with *status = 1 otherwise (the flag is cleared by the report).
 * The flag is sticky: the next nfx_flux_series* call on the handle fails with NFX_E_INTERNAL as well, so an aborted
 * pass is never handed back silently.  (mint's getIntegral is synchronous and returns ier != 0 on failure,
 * field.py:102; this is the asynchronous equivalent.) */
int nfx_pli_series_status(nfx_pli** self, void* stream, int* status);
/* Read-only HBM ceiling of the current device with the access pattern of the edge-flux kernels (level planes of two
 * arrays, 256-bit evict-first loads, K2's arithmetic, no stores): best of `reps` launches over the caller's device
 * buffer (32-byte aligned, >= 9.3 GB, contents arbitrary) in GB/s.  Measurement aid for bench.py's roofline. */
int nfx_probe_read_bandwidth(const void* buf, int64_t nbytes, int reps, double* gbs, void* stream);
/* The same walk over a list of column groups only (the access pattern of the sparse fused pass): groups device
 * (ngroups) int32, ascending indices of 256-bit vectors (4 doubles) of the probe's 362 x 332 plane, each < 30046.
 * *gbs counts the bytes of the listed groups only. */
int nfx_probe_read_bandwidth_groups(const void* buf, int64_t nbytes, const int32_t* groups, int64_t ngroups, int reps,
                                    double* gbs, void* stream);
/* Column groups of the sparse fused pass for uo/vo of `dtype` (its panel size), summation `order` and `vec` columns
 * per group (1, 2, 4 or 8): per panel q, groups[panel_offsets[q] .. panel_offsets[q+1]) are the ascending panel-local
 * group indices g (columns [g*vec, g*vec+vec) of the panel) in which the transects read eU or eV.  Host outputs, each
 * may be NULL: panel_offsets (npanels + 1), groups (*ngroups). */
int nfx_pli_get_column_groups(nfx_pli** self, int dtype, int order, int vec, int64_t* panel_offsets, int32_t* groups,
                              int64_t* ngroups);
/* Finer-than-time-step sharding over GPUs.  The fused pass works on batches b = t*npanels + q (time step t of
 * the nt resident ones, panel q of npanels panels of panel_cells consecutive cells); this call runs only the
 * batches [batch_begin, batch_end) and returns PARTIAL sums in series (nt, ntransects): complete for the time
 * steps whose panels all lie in the range, contributions of the missing panels are 0.  The owner of the other
 * panels adds its part (nemoflux_b200/dist.py).  Always the fused pass. */
int nfx_pli_get_num_panels(nfx_pli** self, int* npanels, int64_t* panel_cells);   /* float64 storage */
int nfx_pli_get_num_panels_dtype(nfx_pli** self, int dtype, int* npanels, int64_t* panel_cells);
int nfx_flux_series_range(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                          const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup, double fill,
                          int order, int64_t batch_begin, int64_t batch_end, double* series, void* stream);
/* the same sub-range of batches with per-column scale factors (arguments as nfx_flux_series_e3) */
int nfx_flux_series_range_e3(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                             int e3_nt, const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup,
                             double fill, int order, int64_t batch_begin, int64_t batch_end, double* series,
                             void* stream);
/* Chunked NetCDF-4 / HDF5 variables decoded on the device, behind the host-to-device copy of the COMPRESSED bytes
 * (what subsetNEMO.py:78 `zlib=True` and NEMO's XIOS output produce; the reference inflates them on one host thread
 * inside netCDF4/HDF5, field.py:22-35,149).  comp: device buffer holding the chunks as stored in the file, chunk c at
 * byte offset in_off[c] (a multiple of 16), in_size[c] bytes; in_off / in_size / chunk_start are HOST arrays.
 * filters: NFX_H5_DEFLATE (zlib stream per chunk, RFC 1950/1951: stored, fixed and dynamic blocks; Adler-32 verified),
 * NFX_H5_SHUFFLE (byte planes -> elements), NFX_H5_FLETCHER32 (the 4-byte trailer is dropped, not verified).
 * chunk_dims / dst_dims: extents (rank <= 4) of a chunk and of the destination array, a dense C-order array of
 * elem_size-byte elements at dst; chunk_start[c*rank + d] = index in dst of the chunk's first element along d (may be
 * negative / beyond the end: elements outside dst -- the padding of edge chunks, time steps outside the slab -- are
 * dropped).  swap_bytes != 0 reverses the bytes of every element (big-endian data).  status (host, nchunks, may be
 * NULL): 0 or the reason a chunk was rejected; any rejected chunk makes the call return NFX_E_INVALID.  Synchronises
 * `stream` before returning. */
#define NFX_H5_DEFLATE 1
#define NFX_H5_SHUFFLE 2
#define NFX_H5_FLETCHER32 4
int nfx_h5_decode_chunks(const void* comp, int64_t comp_bytes, int64_t nchunks, const int64_t* in_off, const int64_t* in_size,
                         int filters, int elem_size, int rank, const int64_t* chunk_dims, const int64_t* dst_dims,
                         const int64_t* chunk_start, int swap_bytes, void* dst, int32_t* status, void* stream);
/* Threading / stream rules (as for a libmint handle: single-threaded, not re-entrant): a handle owns scratch (ring,
 * partial sums, counters, staging buffers) that every call on it re-uses, so calls on ONE handle must be issued from
 * one thread and one stream at a time; different handles are independent.  The host-buffer entry points below run on
 * two private non-blocking streams of the handle and synchronise them before returning: borrowed DEVICE arrays they
 * are given (e3_on_device) must be complete when the call is made. */
/* everything from HOST buffers (the call a non-CUDA host makes): u, v host (nt,nz,ny,nx), thickness
 * host (nz), arc1/arc2 host (ncell); series host (nt, ntransects).  Streams time chunks through
 * double-buffered device staging (host buffers may be pinned or pageable). chunk_steps <= 0 = auto */
int nfx_flux_series_host(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                         const double* arc1, const double* arc2, int nt, int nz, int sverdrup, double fill,
                         int order, int chunk_steps, double* series);
/* the same with per-column scale factors instead of thickness (SURVEY 8f rank 4; what a NEMO mesh_mask or a
 * variable-volume run provides): e3u, e3v of the dtype (and byte order) of u, v.  e3_on_device != 0: borrowed
 * DEVICE arrays (e3_nt, nz, ncell) the caller uploaded once (the time-invariant e3u_0/e3v_0 of a mesh_mask);
 * else HOST arrays: e3_nt == 1 is uploaded once per call, e3_nt == nt is streamed in the chunks next to u, v. */
int nfx_flux_series_host_e3(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                            int e3_nt, int e3_on_device, const double* arc1, const double* arc2, int nt, int nz,
                            int sverdrup, double fill, int order, int chunk_steps, double* series);
/* nfx_flux_series_layers from HOST buffers: arguments as nfx_flux_series_host / _host_e3 (exactly one of thickness and
 * (e3u, e3v)), layer_levels as nfx_flux_series_layers; series host (nt, nlayers, ntransects). */
int nfx_flux_series_layers_host(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                                int dtype_flags, int e3_nt, int e3_on_device, const double* thickness,
                                const double* arc1, const double* arc2, int nt, int nz, int nlayers,
                                const int* layer_levels, int sverdrup, double fill, int order, int chunk_steps,
                                double* series);
/* nfx_flux_section from HOST buffers: arguments as nfx_flux_series_layers_host without order (native or
 * NFX_BIG_ENDIAN data, chunk_steps, e3 on the device or on the host, time-invariant or per step);
 * section host (nt, nlayers, nsub). */
int nfx_flux_section_host(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                          int dtype_flags, int e3_nt, int e3_on_device, const double* thickness, const double* arc1,
                          const double* arc2, int nt, int nz, int nlayers, const int* layer_levels, int sverdrup,
                          double fill, int chunk_steps, double* section);
/* nfx_flux_section_window_sums from HOST buffers: arguments as nfx_flux_section_host plus nwindows, window_bounds,
 * continue_first; sums host (nwindows, nlayers, nsub), read (window 0, continue_first) and written.  Only the steps
 * [b0, bK) are uploaded.  The device stages the window sums a chunk touches (two slots of at most
 * min(nwindows, chunk_steps + 1) windows, not nt steps) and copies back the windows every chunk completes.  The bits do
 * not depend on chunk_steps or the byte order. */
int nfx_flux_section_window_sums_host(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                                      int dtype_flags, int e3_nt, int e3_on_device, const double* thickness,
                                      const double* arc1, const double* arc2, int nt, int nz, int nlayers,
                                      const int* layer_levels, int sverdrup, double fill, int nwindows,
                                      const int* window_bounds, int continue_first, int chunk_steps, double* sums);
/* nfx_flux_classes from HOST buffers: arguments as nfx_flux_section_host plus cfield (host, c_nt x nz x ncell in the
 * dtype and byte order of u, v: streamed with them when c_nt == nt, uploaded once when c_nt == 1), cfill, nclasses,
 * class_bounds; classes host (nt, nclasses, M).  The bits do not depend on chunk_steps or the byte order and are
 * those of nfx_flux_classes. */
int nfx_flux_classes_host(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                          int dtype_flags, int e3_nt, int e3_on_device, const double* thickness, const double* arc1,
                          const double* arc2, int nt, int nz, const void* cfield, int c_nt, double cfill, int nclasses,
                          const double* class_bounds, int sverdrup, double fill, int chunk_steps, double* classes);
/* nfx_flux_tracer from HOST buffers: arguments as nfx_flux_section_host plus tracer (host, tr_nt x nz x ncell in the
 * dtype and byte order of u, v: streamed with them when tr_nt == nt, uploaded once when tr_nt == 1), tfill, ref;
 * series host (nt, nlayers, M) and / or section host (nt, nlayers, nsub), one of them may be NULL.  The bits do not
 * depend on chunk_steps or the byte order and are those of nfx_flux_tracer. */
int nfx_flux_tracer_host(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                         int dtype_flags, int e3_nt, int e3_on_device, const double* thickness, const double* arc1,
                         const double* arc2, int nt, int nz, const void* tracer, int tr_nt, double tfill, double ref,
                         int nlayers, const int* layer_levels, int sverdrup, double fill, int chunk_steps,
                         double* series, double* section);

#ifdef __cplusplus
}
#endif
#endif
