// Shared declarations of libnemoflux_gpu.so (sm_100a).  See include/nemoflux_gpu.h for the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/nemoflux_gpu.h"

namespace nfx {

struct Error : public std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

void set_last_error(const std::string& m);
void count_launch(int n = 1);

#define NFX_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            throw nfx::Error(NFX_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));     \
    } while (0)

#define NFX_REQUIRE(cond, msg)                                      \
    do {                                                            \
        if (!(cond)) throw nfx::Error(NFX_E_INVALID, (msg));        \
    } while (0)

// Debug guard bands (NFX_DEBUG_GUARDS=1 in the environment): every DevBuf is allocated with kGuardBytes of 0xA5 on
// both sides and registered; nfx_debug_check_guards() synchronises the device and reports every guard byte that was
// overwritten.  The pool's boxes refuse compute-sanitizer (profiles/r2_sanitizer_closed.log); this catches what its
// memcheck would catch for writes past either end of a library-owned buffer.
constexpr size_t kGuardBytes = 4096;
bool guards_enabled();
void guard_register(void* raw, size_t payload_bytes);
void guard_unregister(void* raw);

// owning device buffer
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    void* raw = nullptr;   // what cudaMalloc returned (differs from p only with guard bands)
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() {
        if (raw) {
            if (raw != (void*)p) guard_unregister(raw);
            cudaFree(raw);
        }
        p = nullptr;
        raw = nullptr;
        n = 0;
    }
    void alloc(size_t count) {
        release();
        if (count == 0) count = 1;
        const size_t bytes = count * sizeof(T);
        const bool guard = guards_enabled();
        const size_t payload = guard ? (bytes + 255) & ~(size_t)255 : bytes;
        cudaError_t e = cudaMalloc(&raw, payload + (guard ? 2 * kGuardBytes : 0));
        if (e != cudaSuccess) {
            raw = nullptr;
            throw Error(NFX_E_ALLOC, std::string("cudaMalloc: ") + cudaGetErrorString(e));
        }
        if (guard) {
            p = reinterpret_cast<T*>(static_cast<unsigned char*>(raw) + kGuardBytes);
            guard_register(raw, bytes);
        } else {
            p = static_cast<T*>(raw);
        }
        n = count;
    }
    void ensure(size_t count) {
        if (count > n) alloc(count);
    }
};

// Bump allocator over one persistent device buffer: the temporaries of computeWeights (tens of bytes per
// sub-segment, 0.8 GB on an ORCA12 grid with 1024 transects) cost more in cudaMalloc/cudaFree than their kernels.
// Everything taken from an Arena is used on ONE stream, so rewinding (`used = mark`) is safe in stream order.
template <typename T>
struct View {
    T* p = nullptr;
};
struct Arena {
    unsigned char* base = nullptr;
    size_t cap = 0, used = 0;
    template <typename T>
    View<T> take(size_t count) {
        const size_t bytes = (std::max<size_t>(count, 1) * sizeof(T) + 255) & ~(size_t)255;
        if (used + bytes > cap) throw Error(NFX_E_INTERNAL, "scratch arena overflow");
        View<T> v;
        v.p = reinterpret_cast<T*>(base + used);
        used += bytes;
        return v;
    }
};

// ---- K1 data ------------------------------------------------------------------------------------
constexpr int kFan = 32;  // bounding-box hierarchy fan-out = warp width

struct GridDev {
    int device = 0;
    int64_t ncell = 0;
    int ny = 0, nx = 0;          // optional structured shape (0 = unknown)
    DevBuf<double2> verts;       // (ncell*4) lon,lat
    // locator (built by nfx_pli_build_locator, cached on the grid so every pli shares it)
    bool locator_built = false;
    int64_t nl1 = 0, nl2 = 0, nl3 = 0;
    DevBuf<double4> box1, box2, box3;  // xmin, xmax, ymin, ymax; level k groups 32 boxes of level k-1
    double mean_cell = 0.0;      // sqrt(bounding-box area / ncell): scale for the sub-segment count estimate of K1
};

// CSR of (flux index, weight) per transect
struct Csr {
    int64_t nnz = 0;
    DevBuf<int64_t> rowptr;  // (M+1)
    DevBuf<int32_t> idx;
    const double* w = nullptr;  // borrowed: PliDev::w (list order) or PliDev::map_w (map order)
};

// Work plan of the fused K2+K3 pass: the compact CSR of every transect regrouped by panel of cells and cut into
// sub-rows of at most kSubRow entries (bounded work per warp).  Sub-rows are ordered by (panel, transect, chunk);
// idx is the panel-local index into a (2, panel_cols) slab [eU | eV]; entries that always read 0 are dropped.
struct PanelPlan {
    bool built = false;
    int64_t panel_cells = 0;
    int npanels = 0;
    int64_t nnz = 0;
    int64_t nsr = 0;              // number of sub-rows
    int max_sr_per_panel = 0;
    DevBuf<int64_t> rowptr;       // (npanels*M + 1) entry offsets of the (panel, transect) rows
    DevBuf<int32_t> idx;
    DevBuf<double> w;
    DevBuf<int64_t> sr_ptr;       // (nsr + 1) entry offsets of the sub-rows
    DevBuf<int64_t> panel_sr;     // (npanels + 1) first sub-row of every panel
    DevBuf<int64_t> tr_ptr;       // (M + 1) per transect: range in tr_sr
    DevBuf<int64_t> tr_sr;        // (nsr) sub-row ids of every transect, ascending
    std::vector<int64_t> h_panel_sr;   // host copy of panel_sr
    // Column groups: per panel, ascending, the panel-local indices g of the groups of grp_vec columns [g*vec, g*vec+vec)
    // in which idx reads u or v.  The K2 tiles of the sparse fused pass load only these (built for the vector width
    // of the pass, see build_column_groups; grp_vec = 0: not built for this plan yet).
    int grp_vec = 0;
    int64_t ngroups = 0;          // groups in the list, all panels
    int64_t ngroups_all = 0;      // groups of grp_vec columns the panels hold (the dense pass loads all of them)
    int max_grp_per_panel = 0;
    DevBuf<int32_t> grp;
    DevBuf<int64_t> grp_ptr;      // (npanels + 1) offsets into grp
};
constexpr int64_t kSubRow = 4096;

struct PliDev {
    GridDev* grid = nullptr;   // borrowed; never dereferenced by nfx_pli_del (the grid may already be gone)
    int device = 0;
    double period_x = 360.0;
    bool locator_requested = false;
    int ntransects = 0;
    int64_t nsub = 0;
    // sub-segments, emission order
    DevBuf<int64_t> sub_offsets;  // (M+1) per transect
    DevBuf<int32_t> cell, seg, img;
    DevBuf<double> ta, tb, coeff, xia, xib, w;  // xia/xib (n,2), w (n,4)
    // mint map view
    int64_t nmap = 0;
    DevBuf<int64_t> map_offsets;  // (M+1)
    DevBuf<int64_t> map_keys;     // cell*4+edge
    DevBuf<double> map_w;
    // CSRs: [order][layout]; layout 0 = (ncell,4) cell-by-cell data, 1 = compact [eU|eV]
    Csr csr[2][2];
    bool has_compact = false;
    PanelPlan plan[2];            // per summation order
    DevBuf<double> ring, partial;  // L2-resident eflux ring and per-panel partial sums of the fused pass
    DevBuf<int> fused_sync;        // work counter, error flag, per-batch completion counters
    DevBuf<int> fused_sticky_buf;  // device: 1 once any fused pass on this handle aborted
    int* h_fused_err = nullptr;    // pinned: error flag of the fused passes launched so far, copied back behind every
                                   // launch (sticky until reported by the next call on the handle / nfx_pli_series_status)
    DevBuf<unsigned char> scratch; // computeWeights temporaries (Arena), kept between calls when small
    int64_t nsub_hint = 0;         // sub-segments of the previous computeWeights: sizes the record list of the next
    size_t scratch_hint = 0;       // bytes the arena ended with
    DevBuf<int64_t> scan_tmp;
    DevBuf<int> batch_map;         // fused pass: order in which the (time step, panel) batches are visited
    std::vector<int> h_batch_map;
    int64_t batch_map_key[4] = {-1, -1, -1, -1};   // (batch_begin, batch_end, npanels, order) of the cached map
    std::vector<int64_t> h_sub_offsets, h_map_offsets;
    DevBuf<int> levels;            // layered series: device copy of the layer boundaries of the last layered call
    std::vector<int> h_levels;     // ... and its host copy (the upload is skipped when they are unchanged)
    DevBuf<int> windows;           // time-mean section: device copy of the window bounds of the last call
    // scratch reused by the host-buffer entry points
    DevBuf<double> scratch_data, scratch_res;
    // persistent staging of nfx_flux_series_host (two slots)
    DevBuf<unsigned char> stage_u[2], stage_v[2], stage_e3u[2], stage_e3v[2];
    DevBuf<double> stage_eflux[2], stage_series, stage_thick, stage_arc1, stage_arc2;
    DevBuf<double> stage_windows[2];   // time-mean section: the window sums a chunk touches (two slots)
    DevBuf<unsigned char> stage_cf[2];  // class transport: the class field of a chunk (two slots), or of every step
    // class transport: warp tiles of the crossings (class_ntiles + 1 starts, per transect the range of its tiles), built
    // on first use after computeWeights (class_ntiles < 0: not built); the bounds of the last call; partial sums
    int64_t class_ntiles = -1;
    std::vector<int64_t> h_class_tiles, h_class_tr_tiles;
    DevBuf<int64_t> class_tiles, class_tr_tiles;
    DevBuf<double> class_bounds, class_partial;
    cudaStream_t copy_stream = nullptr, compute_stream = nullptr;
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
};

// mint.VectorInterp (nfx_k4_vinterp.cu)
struct VInterpDev {
    GridDev* grid = nullptr;
    int device = 0;
    double period_x = 360.0;
    int64_t npts = 0;
    DevBuf<int32_t> cell;   // containing cell of every point, -1 = not found
    DevBuf<double> xi;      // (npts, 2) parametric coordinates
    DevBuf<double> scratch_data, scratch_vec;
};
void vinterp_find_points(VInterpDev& vi, int64_t npts, const double* xyz_host, double tol2, cudaStream_t s);
void vinterp_face_vectors(VInterpDev& vi, const double* data_dev, double* vec_dev, cudaStream_t s);

// K1 (nfx_k1_intersect.cu)
void grid_upload_points(GridDev& g, int64_t ncells, const double* points_host);
void grid_build_locator(GridDev& g, cudaStream_t s);
void grid_arc_lengths(GridDev& g, double* arc_dev, cudaStream_t s);
void pli_compute_weights(PliDev& p, int ntransects, const int* offsets, const double* xyz, int counterclock,
                         cudaStream_t s);

// K2 (nfx_k2_edgeflux.cu)
struct K2Options {
    int variant = NFX_K2_AUTO;
    int unroll = 0;   // 0 = default
    int block = 0;    // 0 = default
    int alu_mask = -1;  // float32 storage: levels (of each batch of 5) converted on the ALU; -1 = built-in choice
};
void edgeflux_assemble(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                       const double* arc2, int nt, int nz, int64_t ncell, int sverdrup, double fill, double* eflux,
                       const K2Options& opt, cudaStream_t s);
void edgeflux_assemble_panel(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                             const double* arc2, int nt, int nz, int64_t ncols, int64_t ld, int sverdrup, double fill,
                             double* eflux, int keep_l2, const K2Options& opt, cudaStream_t s,
                             const void* e3u = nullptr, const void* e3v = nullptr, int64_t e3_tstride = 0,
                             int nlayers = 1, const int* levels = nullptr);
void edgeflux_to_cell_by_cell(const double* eflux, int nt, int ny, int nx, double* iv, cudaStream_t s);
void edgeflux_absmax(const double* eflux, int nt, int64_t ncell, double* result_host, cudaStream_t s);
void bswap_inplace(void* p, size_t n, int esize, cudaStream_t s);   // big-endian file bytes -> native, on the device

// K3 (nfx_k3_reduce.cu)
void csr_integrate(const Csr& c, int ntransects, const double* data, int64_t stride_t, int nt, double* series,
                   cudaStream_t s);
void rows_integrate(const int64_t* rowptr, const int32_t* idx, const double* w, int nrows, int64_t nnz,
                    const double* data, int64_t stride_t, int nt, double* out, int64_t out_stride_t, cudaStream_t s);
void reduce_subrows(const double* partial, int nt, int64_t nsr, const int64_t* tr_ptr, const int64_t* tr_sr,
                    int ntransects, double* series, cudaStream_t s);
void build_panel_plan(PliDev& p, int order, int64_t panel_cells, cudaStream_t s);
void build_column_groups(PanelPlan& pl, int64_t ncell, int ntransects, int vec, cudaStream_t s);

// K2+K3 fused persistent pass (nfx_k23_fused.cu)
void flux_series_fused(PliDev& p, PanelPlan& pl, const void* u, const void* v, int dtype, const double* thickness,
                       const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup, double fill,
                       int64_t batch_begin, int64_t batch_end, double* out, cudaStream_t s, const void* e3u = nullptr,
                       const void* e3v = nullptr, int64_t e3_tstride = 0, int nlayers = 1, const int* levels = nullptr);
int fused_tile_columns(int dtype, const void* u, const void* v, int64_t ncell, int64_t ld, int64_t panel,
                       uintptr_t more_bits = 0);
int fused_error_flag(PliDev& p, cudaStream_t s);
void fused_check_sticky_error(PliDev& p);   // throws if a fused pass launched earlier on this handle aborted
void h5_decode_chunks(const void* comp_dev, int64_t comp_bytes, int64_t nchunks, const int64_t* in_off,
                      const int64_t* in_size, int filters, int elem_size, int rank, const int64_t* chunk_dims,
                      const int64_t* dst_dims, const int64_t* chunk_start, int swap_bytes, void* dst_dev,
                      int32_t* status_host, cudaStream_t s);   // nfx_inflate.cu
double probe_read_bandwidth(const void* buf, int64_t nbytes, int reps, double* sink, cudaStream_t s);   // nfx_probe.cu
extern int g_fused_f32_shape;
extern int g_fused_order;
extern int g_fused_k3_lag;
extern int g_fused_ring_max_mb;
extern int g_fused_f64_ctas;
extern int g_sparse_columns;
extern int g_last_series_sparse;
double probe_read_bandwidth_groups(const void* buf, int64_t nbytes, const int32_t* groups, int64_t ngroups, int reps,
                                   double* sink, cudaStream_t s);   // nfx_probe.cu
int k3_group_for(int64_t nnz, int64_t nrows);

// transport section (nfx_section.cu): section (nt, nlayers, nsub) from the list-order compact CSR (idx, w: 4 entries per
// sub-segment); exactly one of thickness and (e3u, e3v); levels: device (nlayers + 1), nullptr = one layer [0, nz)
void flux_section(const void* u, const void* v, int dtype, const double* thickness, const void* e3u, const void* e3v,
                  int64_t e3_tstride, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                  int64_t nsub, int64_t ncell, int64_t ld, int nt, int nz, int nlayers, const int* levels, int sverdrup,
                  double fill, double* section, cudaStream_t s);
// ... summed over windows of time steps (nfx_section.cu): sums ((nwin, nlayers, nsub) from window w0 on) += the section
// of the steps [bounds[w], bounds[w+1]) clipped to [t_first, t_end), in ascending step order; u, v (and per-step e3) hold
// the steps from t_first on; bounds: device (all windows + 1); continue_first: window w0 continues the partial sums in
// `sums`, else every window starts from +0
void flux_section_windows(const void* u, const void* v, int dtype, const double* thickness, const void* e3u,
                          const void* e3v, int64_t e3_tstride, const double* arc1, const double* arc2,
                          const int32_t* idx, const double* w, int64_t nsub, int64_t ncell, int64_t ld, int nz,
                          int nlayers, const int* levels, int sverdrup, double fill, const int* bounds, int w0, int nwin,
                          int t_first, int t_end, int continue_first, double* sums, cudaStream_t s);
// class transport (nfx_section.cu): classes (nt, K, M), the per-level section flux of every crossing binned by the class
// field at its cell (cfield (1 or nt, nz, ld) of the dtype of u, v; c_tstride 0 or nz * ld) into the classes
// [bounds[j], bounds[j+1]) (device, K + 1 ascending doubles).  tile_start (ntiles + 1): the warp tiles of at most 32
// crossings of one transect, tr_tiles (M + 1) the tiles of every transect; partial: scratch of
// partial_steps * ntiles * K doubles, the steps are run in batches of at most partial_steps.
constexpr int kClassMax = 96;   // the per-thread class sums of a 256-thread CTA: 2 KB of shared memory per class
void flux_classes(const void* u, const void* v, int dtype, const double* thickness, const void* e3u, const void* e3v,
                  int64_t e3_tstride, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                  const int32_t* cell, const void* cfield, int64_t c_tstride, double cfill, const double* bounds, int K,
                  const int64_t* tile_start, int64_t ntiles, const int64_t* tr_tiles, int ntransects, int64_t ncell,
                  int64_t ld, int nt, int nz, int sverdrup, double fill, double* partial, int partial_steps,
                  double* classes, cudaStream_t s);
// tracer transport (nfx_section.cu): per layer (levels: device, nlayers + 1) the section flux of every crossing with
// each edge's level terms weighted by the tracer at its C-grid face (tracer (1 or nt, nz, ld) of the dtype of u, v;
// tr_tstride 0 or nz * ld; the grid nx cells wide).  section (nt, nlayers, nsub) and / or series (nt, nlayers, M), the
// crossings folded over the warp tiles of flux_classes; partial: scratch of partial_steps * ntiles * nlayers doubles
// (with series), the steps are run in batches of at most partial_steps.
void flux_tracer(const void* u, const void* v, int dtype, const double* thickness, const void* e3u, const void* e3v,
                 int64_t e3_tstride, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                 const int32_t* cell, const void* tracer, int64_t tr_tstride, double tfill, double ref,
                 const int64_t* tile_start, int64_t ntiles, const int64_t* tr_tiles, int ntransects, int64_t nsub,
                 int64_t ncell, int nx, int64_t ld, int nt, int nz, int nlayers, const int* levels, int sverdrup,
                 double fill, double* partial, int partial_steps, double* series, double* section, cudaStream_t s);

}  // namespace nfx
