// extern "C" entry points of libnemoflux_gpu.so -- see include/nemoflux_gpu.h.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "nfx_common.cuh"

namespace nfx {

static thread_local std::string g_last_error;
static std::atomic<int64_t> g_launches{0};
static K2Options g_k2opt;
static int g_fast_series = 1;             // NFX_OPT_FAST_SERIES
static int g_last_series_fused = -1;      // NFX_OPT_LAST_SERIES_PATH (read only): path of the last nfx_flux_series* call
static int64_t g_slot_bytes = 0;          // NFX_OPT_RING_SLOT_MB, 0 = automatic (slot_bytes_for)

// ---- debug guard bands (see nfx_common.cuh) ---------------------------------------------------------------------
struct GuardRec {
    void* raw;
    size_t payload;
};
static std::mutex g_guard_mu;
static std::vector<GuardRec> g_guards;

bool guards_enabled() {
    static const bool on = [] {
        const char* e = std::getenv("NFX_DEBUG_GUARDS");
        return e && std::atoi(e) != 0;
    }();
    return on;
}

void guard_register(void* raw, size_t payload_bytes) {
    unsigned char* b = static_cast<unsigned char*>(raw);
    cudaMemset(b, 0xA5, kGuardBytes);
    // the tail guard starts right behind the payload (not behind its 256-byte rounding): an overrun by one element shows
    const size_t rounded = (payload_bytes + 255) & ~(size_t)255;
    cudaMemset(b + kGuardBytes + payload_bytes, 0xA5, rounded - payload_bytes + kGuardBytes);
    std::lock_guard<std::mutex> lk(g_guard_mu);
    g_guards.push_back({raw, payload_bytes});
}

static int64_t g_guard_checked = 0;        // buffers checked so far (alive at a check, or at their release)
static int64_t g_guard_damaged_freed = 0;  // damaged buffers found at release time, not yet reported
static std::string g_guard_freed_report;

// one buffer: true when a guard byte was overwritten (the caller synchronised the device)
static bool guard_damaged(const GuardRec& g, std::string* report) {
    const size_t rounded = (g.payload + 255) & ~(size_t)255;
    const size_t tail = rounded - g.payload + kGuardBytes;
    std::vector<unsigned char> h(kGuardBytes + tail);
    unsigned char* b = static_cast<unsigned char*>(g.raw);
    if (cudaMemcpy(h.data(), b, kGuardBytes, cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(h.data() + kGuardBytes, b + kGuardBytes + g.payload, tail, cudaMemcpyDeviceToHost) != cudaSuccess) {
        cudaGetLastError();
        return false;   // context gone (interpreter shutdown): nothing to check
    }
    int64_t first = -1, count = 0;
    for (size_t i = 0; i < h.size(); ++i)
        if (h[i] != 0xA5) {
            if (first < 0) first = (int64_t)i;
            ++count;
        }
    if (count && report && report->size() < 2000) {
        const bool head = first < (int64_t)kGuardBytes;
        *report += "buffer of " + std::to_string(g.payload) + " bytes: " + std::to_string(count) +
                   " guard bytes overwritten, first " +
                   (head ? std::to_string((int64_t)kGuardBytes - first) + " bytes BEFORE the start"
                         : std::to_string(first - (int64_t)kGuardBytes) + " bytes PAST the end") + "; ";
    }
    return count != 0;
}

// a buffer that is freed is checked first: a test that drops its handles before the check must not hide an overrun
void guard_unregister(void* raw) {
    std::lock_guard<std::mutex> lk(g_guard_mu);
    for (size_t i = 0; i < g_guards.size(); ++i)
        if (g_guards[i].raw == raw) {
            if (cudaDeviceSynchronize() == cudaSuccess) {
                ++g_guard_checked;
                if (guard_damaged(g_guards[i], &g_guard_freed_report)) ++g_guard_damaged_freed;
            } else {
                cudaGetLastError();
            }
            g_guards[i] = g_guards.back();
            g_guards.pop_back();
            return;
        }
}

// number of library-owned buffers with a damaged guard band (after a device synchronise), buffers freed since the last
// check included; details in *report.  *nbuffers = buffers checked since the last call.
static int64_t guard_check_all(std::string* report, int64_t* nbuffers) {
    std::lock_guard<std::mutex> lk(g_guard_mu);
    NFX_CUDA(cudaDeviceSynchronize());
    int64_t bad = g_guard_damaged_freed;
    if (report) *report += g_guard_freed_report;
    for (const GuardRec& g : g_guards) bad += guard_damaged(g, report) ? 1 : 0;
    if (nbuffers) *nbuffers = g_guard_checked + (int64_t)g_guards.size();
    g_guard_checked = 0;
    g_guard_damaged_freed = 0;
    g_guard_freed_report.clear();
    return bad;
}

void set_last_error(const std::string& m) { g_last_error = m; }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

static void require_gpu(int* dev) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        throw Error(NFX_E_NOGPU, std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e)
                                                                                           : "device count is 0"));
    }
    NFX_CUDA(cudaGetDevice(dev));
}

template <typename F>
static int guarded(F&& f) {
    try {
        cudaGetLastError();  // a stale non-sticky error of an earlier call must not be blamed on this one
        f();
        return NFX_OK;
    } catch (const Error& e) {
        set_last_error(e.what());
        return e.code;
    } catch (const std::bad_alloc&) {
        set_last_error("out of host memory");
        return NFX_E_ALLOC;
    } catch (const std::exception& e) {
        set_last_error(e.what());
        return NFX_E_INTERNAL;
    } catch (...) {
        set_last_error("unknown error");
        return NFX_E_INTERNAL;
    }
}

static void free_host_path(PliDev& p) {
    for (int i = 0; i < 2; ++i) {
        if (p.ev_ready[i]) cudaEventDestroy(p.ev_ready[i]);
        if (p.ev_done[i]) cudaEventDestroy(p.ev_done[i]);
        p.ev_ready[i] = p.ev_done[i] = nullptr;
    }
    if (p.copy_stream) cudaStreamDestroy(p.copy_stream);
    if (p.compute_stream) cudaStreamDestroy(p.compute_stream);
    p.copy_stream = p.compute_stream = nullptr;
    if (p.h_fused_err) cudaFreeHost(p.h_fused_err);
    p.h_fused_err = nullptr;
}

// K2+K3 with the edge fluxes kept in L2 (nfx_k23_fused.cu): one persistent launch; large grids are cut into
// panels of cells whose (2, panel) slab of edge fluxes fits a ring slot, their partial sums are added at the end.
// ring slot = one batch of edge fluxes.  A time step that fits 8 MB is ONE panel (ORCA1 class).  Larger grids are cut
// into panels of about 4 MB for float64 storage and 8 MB for float32 (same-box A/B over 2 / 4 / 8 / 16 MB,
// profiles/r2_fused_experiments.md: float64 +1.8 % (ORCA025) and +2.5 % (ORCA12) with 4 MB against 8 MB, float32
// -1.4 % and -5 %); NFX_OPT_RING_SLOT_MB overrides both.
static int64_t single_panel_bytes() { return g_slot_bytes > 0 ? g_slot_bytes : (int64_t)8 << 20; }
static int64_t slot_bytes_for(int dtype) {
    if (g_slot_bytes > 0) return g_slot_bytes;
    return dtype == NFX_F64 ? (int64_t)4 << 20 : (int64_t)8 << 20;
}
static int64_t fused_panel_cells(int64_t ncell, int dtype) {
    if (ncell * 16 <= single_panel_bytes()) return ncell;
    const int64_t sb = slot_bytes_for(dtype);
    const int64_t np0 = (ncell * 16 + sb - 1) / sb;
    return ((ncell + np0 - 1) / np0 + 1023) / 1024 * 1024;
}

static void flux_series_fast(PliDev& p, const void* u, const void* v, int dtype, const double* thickness,
                             const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup,
                             double fill, int order, double* series, cudaStream_t stream, int64_t batch_begin = 0,
                             int64_t batch_end = -1, const void* e3u = nullptr, const void* e3v = nullptr,
                             int64_t e3_tstride = 0) {
    NFX_REQUIRE(order == NFX_ORDER_LIST || order == NFX_ORDER_MAP, "order must be NFX_ORDER_LIST or NFX_ORDER_MAP");
    NFX_REQUIRE(p.csr[order][0].rowptr.p != nullptr, "computeWeights was not called");
    NFX_REQUIRE(p.has_compact, "nfx_grid_set_cgrid_shape must be called before computeWeights for the flux path");
    const int64_t ncell = p.grid->ncell;
    const int M = p.ntransects;
    if (nt <= 0 || M <= 0) return;
    fused_check_sticky_error(p);   // an earlier pass on this handle that aborted is reported here, not swallowed
    const int64_t panel = fused_panel_cells(ncell, dtype);
    PanelPlan& pl = p.plan[order];
    if (!pl.built || pl.panel_cells != panel) build_panel_plan(p, order, panel, stream);
    p.partial.ensure((size_t)nt * std::max<int64_t>(pl.nsr, 1));
    if (batch_end < 0) batch_end = (int64_t)nt * pl.npanels;
    flux_series_fused(p, pl, u, v, dtype, thickness, arc1, arc2, nt, nz, ld, sverdrup, fill, batch_begin, batch_end,
                      p.partial.p, stream, e3u, e3v, e3_tstride);
    reduce_subrows(p.partial.p, nt, pl.nsr, pl.tr_ptr.p, pl.tr_sr.p, M, series, stream);
}

// NFX_OPT_FAST_SERIES: 1 (default) = the fused pass when the edge fluxes of one time step fit a ring slot (one
// panel: ORCA1-class grids, 3-10 % faster than two launches) and, on larger grids that need several panels, when the
// level rows allow the widest loads (256-bit for float64, >= 128-bit for float32: -8..-11 % time in the same-box
// A/B); the two-launch path otherwise.  2 = always fused, 0 = never.
static bool use_fused(const PliDev& p, int dtype, const void* u, const void* v, int64_t ld) {
    if (g_fast_series == 2) return true;
    if (g_fast_series == 0 || !p.grid) return false;
    const int64_t ncell = p.grid->ncell;
    const int vec = fused_tile_columns(dtype, u, v, ncell, ld, fused_panel_cells(ncell, dtype));
    // float32 storage: fused with 128-bit loads or wider (-8..-11 % time against two launches, same-box A/B)
    if (dtype != NFX_F64) return vec >= 4;
    if (ncell * 16 <= single_panel_bytes()) return true;
    // several panels: only with 256-bit loads (32-byte aligned rows), where the same-box A/B shows -8 % time
    return vec == 4;
}

// the same decision with per-column scale factors (four streams; the fused kernels use 128-bit loads there):
// float64 when one panel holds a time step of edge fluxes, float32 as above
static bool use_fused_e3(const PliDev& p, int dtype, const void* u, const void* v, const void* e3u, const void* e3v,
                         int64_t e3_tstride, int64_t ld) {
    if (g_fast_series == 2) return true;
    if (g_fast_series == 0 || !p.grid) return false;
    const int64_t ncell = p.grid->ncell;
    if (dtype == NFX_F64) return ncell * 16 <= single_panel_bytes();
    const uintptr_t more = (uintptr_t)e3u | (uintptr_t)e3v | (uintptr_t)(e3_tstride * 4);
    return fused_tile_columns(dtype, u, v, ncell, ld, fused_panel_cells(ncell, dtype), more) >= 4;
}

static const Csr& pick_csr(PliDev& p, int order, int layout) {
    NFX_REQUIRE(order == NFX_ORDER_LIST || order == NFX_ORDER_MAP, "order must be NFX_ORDER_LIST or NFX_ORDER_MAP");
    NFX_REQUIRE(p.csr[order][0].rowptr.p != nullptr, "computeWeights was not called");
    if (layout == 1)
        NFX_REQUIRE(p.has_compact, "nfx_grid_set_cgrid_shape must be called before computeWeights for the flux path");
    return p.csr[order][layout];
}

}  // namespace nfx

using namespace nfx;

struct nfx_grid {
    GridDev d;
};
struct nfx_pli {
    PliDev d;
};
struct nfx_vinterp {
    VInterpDev d;
};

template <typename T>
static void d2h(T* dst, const T* src, size_t n) {
    if (dst && n) NFX_CUDA(cudaMemcpy(dst, src, sizeof(T) * n, cudaMemcpyDeviceToHost));
}

extern "C" {

const char* nfx_last_error(void) { return g_last_error.c_str(); }
int nfx_version(void) { return 100; }

int nfx_set_option(int option, int value) {
    return guarded([&] {
        switch (option) {
            case NFX_OPT_K2_VARIANT:
                NFX_REQUIRE(value >= NFX_K2_AUTO && value <= NFX_K2_LDG128, "bad K2 variant");
                g_k2opt.variant = value;
                break;
            case NFX_OPT_K2_UNROLL: g_k2opt.unroll = value; break;
            case NFX_OPT_K2_BLOCK: g_k2opt.block = value; break;
            case NFX_OPT_K2_ALU_MASK: g_k2opt.alu_mask = value; break;
            case NFX_OPT_FUSED_F32_SHAPE: g_fused_f32_shape = value; break;
            case NFX_OPT_FUSED_ORDER: g_fused_order = value; break;
            case NFX_OPT_FUSED_F64_CTAS: g_fused_f64_ctas = value; break;
            case NFX_OPT_FUSED_K3_LAG:
                NFX_REQUIRE(value >= 0 && value <= 60, "NFX_OPT_FUSED_K3_LAG must be 0..60");
                g_fused_k3_lag = value;
                break;
            case NFX_OPT_RING_MAX_MB:
                NFX_REQUIRE(value >= 0 && value <= 120, "NFX_OPT_RING_MAX_MB must be 0..120");
                g_fused_ring_max_mb = value;
                break;
            case NFX_OPT_LAST_SERIES_PATH: throw Error(NFX_E_INVALID, "NFX_OPT_LAST_SERIES_PATH is read only");
            case NFX_OPT_FAST_SERIES:
                NFX_REQUIRE(value >= 0 && value <= 2, "NFX_OPT_FAST_SERIES must be 0, 1 or 2");
                g_fast_series = value;
                break;
            case NFX_OPT_SPARSE_COLUMNS:
                NFX_REQUIRE(value >= 0 && value <= 2, "NFX_OPT_SPARSE_COLUMNS must be 0, 1 or 2");
                g_sparse_columns = value;
                break;
            case NFX_OPT_LAST_SERIES_SPARSE: throw Error(NFX_E_INVALID, "NFX_OPT_LAST_SERIES_SPARSE is read only");
            case NFX_OPT_RING_SLOT_MB:
                NFX_REQUIRE(value >= 0 && value <= 64, "ring slot must be 1..64 MB (0 = automatic)");
                g_slot_bytes = (int64_t)value << 20;
                break;
            default: throw Error(NFX_E_INVALID, "unknown option");
        }
    });
}

int nfx_get_option(int option, int* value) {
    return guarded([&] {
        NFX_REQUIRE(value, "NULL value");
        switch (option) {
            case NFX_OPT_K2_VARIANT: *value = g_k2opt.variant; break;
            case NFX_OPT_K2_UNROLL: *value = g_k2opt.unroll; break;
            case NFX_OPT_K2_BLOCK: *value = g_k2opt.block; break;
            case NFX_OPT_K2_ALU_MASK: *value = g_k2opt.alu_mask; break;
            case NFX_OPT_FUSED_F32_SHAPE: *value = g_fused_f32_shape; break;
            case NFX_OPT_FUSED_ORDER: *value = g_fused_order; break;
            case NFX_OPT_FUSED_F64_CTAS: *value = g_fused_f64_ctas; break;
            case NFX_OPT_FUSED_K3_LAG: *value = g_fused_k3_lag; break;
            case NFX_OPT_RING_MAX_MB: *value = g_fused_ring_max_mb; break;
            case NFX_OPT_LAST_SERIES_PATH: *value = g_last_series_fused; break;
            case NFX_OPT_FAST_SERIES: *value = g_fast_series; break;
            case NFX_OPT_RING_SLOT_MB: *value = (int)(g_slot_bytes >> 20); break;
            case NFX_OPT_SPARSE_COLUMNS: *value = g_sparse_columns; break;
            case NFX_OPT_LAST_SERIES_SPARSE: *value = g_last_series_sparse; break;
            default: throw Error(NFX_E_INVALID, "unknown option");
        }
    });
}

int nfx_debug_check_guards(int64_t* nbuffers, int64_t* ndamaged) {
    return guarded([&] {
        NFX_REQUIRE(ndamaged, "NULL pointer");
        if (nbuffers) *nbuffers = 0;
        *ndamaged = 0;
        if (!guards_enabled()) return;
        int dev;
        require_gpu(&dev);
        std::string report;
        *ndamaged = guard_check_all(&report, nbuffers);
        if (*ndamaged) throw Error(NFX_E_INTERNAL, "guard bands damaged: " + report);
    });
}

int nfx_debug_poke_guard(int where) {
    return guarded([&] {
        NFX_REQUIRE(guards_enabled(), "NFX_DEBUG_GUARDS is not set");
        std::lock_guard<std::mutex> lk(g_guard_mu);
        NFX_REQUIRE(!g_guards.empty(), "no guarded buffer yet");
        const GuardRec& g = g_guards.back();
        unsigned char* b = static_cast<unsigned char*>(g.raw);
        NFX_CUDA(cudaMemset(where == 0 ? b + kGuardBytes - 1 : b + kGuardBytes + g.payload, 0, 1));
    });
}

int nfx_launch_count(int64_t* n) {
    if (!n) return NFX_E_INVALID;
    *n = g_launches.load();
    return NFX_OK;
}

// ---- grid -------------------------------------------------------------------------------------------
int nfx_grid_new(nfx_grid** self) {
    return guarded([&] {
        NFX_REQUIRE(self, "NULL handle");
        int dev;
        require_gpu(&dev);
        *self = new nfx_grid();
        (*self)->d.device = dev;
    });
}

int nfx_grid_del(nfx_grid** self) {
    return guarded([&] {
        NFX_REQUIRE(self, "NULL handle");
        if (*self) {
            DeviceGuard g((*self)->d.device);
            delete *self;
        }
        *self = nullptr;
    });
}

int nfx_grid_set_points(nfx_grid** self, int64_t ncells, const double* points) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        DeviceGuard g((*self)->d.device);
        grid_upload_points((*self)->d, ncells, points);
    });
}

int nfx_grid_get_num_cells(nfx_grid** self, int64_t* ncells) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && ncells, "NULL handle");
        *ncells = (*self)->d.ncell;
    });
}

int nfx_grid_set_cgrid_shape(nfx_grid** self, int ny, int nx) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        NFX_REQUIRE(ny > 0 && nx > 0, "ny and nx must be positive");
        NFX_REQUIRE((*self)->d.ncell == 0 || (int64_t)ny * nx == (*self)->d.ncell, "ny*nx differs from the cell count");
        (*self)->d.ny = ny;
        (*self)->d.nx = nx;
    });
}

int nfx_grid_arc_lengths(nfx_grid** self, double* arc, void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        DeviceGuard g((*self)->d.device);
        grid_arc_lengths((*self)->d, arc, (cudaStream_t)stream);
    });
}

// ---- polyline integral -------------------------------------------------------------------------------
int nfx_pli_new(nfx_pli** self) {
    return guarded([&] {
        NFX_REQUIRE(self, "NULL handle");
        int dev;
        require_gpu(&dev);
        *self = new nfx_pli();
        (*self)->d.device = dev;
    });
}

int nfx_pli_del(nfx_pli** self) {
    return guarded([&] {
        NFX_REQUIRE(self, "NULL handle");
        if (*self) {
            DeviceGuard g((*self)->d.device);
            free_host_path((*self)->d);
            delete *self;
        }
        *self = nullptr;
    });
}

int nfx_pli_set_grid(nfx_pli** self, nfx_grid* grid) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && grid, "NULL handle");
        (*self)->d.grid = &grid->d;
        (*self)->d.device = grid->d.device;
    });
}

int nfx_pli_build_locator(nfx_pli** self, int num_cells_per_bucket, double period_x, int enable_folding) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "buildLocator: setGrid was not called");
        NFX_REQUIRE(num_cells_per_bucket > 0, "buildLocator: numCellsPerBucket must be positive");
        NFX_REQUIRE(enable_folding == 0, "buildLocator: enableFolding is not supported (nemoflux passes False)");
        NFX_REQUIRE(period_x >= 0.0, "buildLocator: periodX must be >= 0");
        DeviceGuard g(p.grid->device);
        grid_build_locator(*p.grid, nullptr);
        NFX_CUDA(cudaStreamSynchronize(nullptr));
        p.period_x = period_x;
        p.locator_requested = true;
    });
}

int nfx_pli_compute_weights_batch(nfx_pli** self, int ntransects, const int* offsets, const double* xyz,
                                  int counterclock) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "computeWeights: setGrid was not called");
        DeviceGuard g(p.grid->device);
        pli_compute_weights(p, ntransects, offsets, xyz, counterclock, nullptr);
    });
}

int nfx_pli_compute_weights(nfx_pli** self, int npoints, const double* xyz, int counterclock) {
    if (npoints < 0) {
        set_last_error("computeWeights: negative number of points");
        return NFX_E_INVALID;
    }
    const int offsets[2] = {0, npoints};
    return nfx_pli_compute_weights_batch(self, 1, offsets, xyz, counterclock);
}

int nfx_pli_get_num_transects(nfx_pli** self, int* ntransects) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && ntransects, "NULL handle");
        *ntransects = (*self)->d.ntransects;
    });
}

int nfx_pli_get_num_subsegments(nfx_pli** self, int64_t* n) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && n, "NULL handle");
        *n = (*self)->d.nsub;
    });
}

int nfx_pli_get_subsegments(nfx_pli** self, int64_t* transect_offsets, int64_t* cell, int32_t* seg, int32_t* img,
                            double* ta, double* tb, double* coeff, double* xia, double* xib, double* w) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        const size_t n = (size_t)p.nsub;
        if (transect_offsets)
            for (int m = 0; m <= p.ntransects; ++m) transect_offsets[m] = p.h_sub_offsets[m];
        if (cell && n) {
            std::vector<int32_t> tmp(n);
            d2h(tmp.data(), p.cell.p, n);
            for (size_t i = 0; i < n; ++i) cell[i] = tmp[i];
        }
        d2h(seg, p.seg.p, n);
        d2h(img, p.img.p, n);
        d2h(ta, p.ta.p, n);
        d2h(tb, p.tb.p, n);
        d2h(coeff, p.coeff.p, n);
        d2h(xia, p.xia.p, 2 * n);
        d2h(xib, p.xib.p, 2 * n);
        d2h(w, p.w.p, 4 * n);
    });
}

int nfx_pli_get_map_size(nfx_pli** self, int64_t* n) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && n, "NULL handle");
        *n = (*self)->d.nmap;
    });
}

int nfx_pli_get_map(nfx_pli** self, int64_t* transect_offsets, int64_t* keys, double* w) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        if (transect_offsets)
            for (int m = 0; m <= p.ntransects; ++m) transect_offsets[m] = p.h_map_offsets[m];
        d2h(keys, p.map_keys.p, (size_t)p.nmap);
        d2h(w, p.map_w.p, (size_t)p.nmap);
    });
}

int nfx_pli_get_integrals_device(nfx_pli** self, const double* data, int nt, int order, double* results,
                                 void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        const Csr& c = pick_csr(p, order, 0);
        csr_integrate(c, p.ntransects, data, p.grid->ncell * 4, nt, results, (cudaStream_t)stream);
    });
}

int nfx_pli_get_integrals(nfx_pli** self, const double* data, int placement, int order, double* results) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && data && results, "NULL pointer");
        NFX_REQUIRE(placement == NFX_CELL_BY_CELL_DATA, "only CELL_BY_CELL_DATA placement is supported");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        const Csr& c = pick_csr(p, order, 0);
        const size_t n = (size_t)p.grid->ncell * 4;
        p.scratch_data.ensure(n);
        p.scratch_res.ensure((size_t)std::max(p.ntransects, 1));
        NFX_CUDA(cudaMemcpy(p.scratch_data.p, data, sizeof(double) * n, cudaMemcpyHostToDevice));
        csr_integrate(c, p.ntransects, p.scratch_data.p, (int64_t)n, 1, p.scratch_res.p, nullptr);
        NFX_CUDA(cudaMemcpy(results, p.scratch_res.p, sizeof(double) * p.ntransects, cudaMemcpyDeviceToHost));
    });
}

int nfx_pli_get_integral(nfx_pli** self, const double* data, int placement, double* result) {
    if (self && *self && (*self)->d.ntransects != 1) {
        set_last_error("getIntegral: the handle holds a batch; use nfx_pli_get_integrals");
        return NFX_E_INVALID;
    }
    return nfx_pli_get_integrals(self, data, placement, NFX_ORDER_MAP, result);
}

// ---- mint.VectorInterp (field.py:90-95,119-120) ----------------------------------------------------------
int nfx_vinterp_new(nfx_vinterp** self) {
    return guarded([&] {
        NFX_REQUIRE(self, "NULL handle");
        int dev;
        require_gpu(&dev);
        *self = new nfx_vinterp();
        (*self)->d.device = dev;
    });
}

int nfx_vinterp_del(nfx_vinterp** self) {
    return guarded([&] {
        NFX_REQUIRE(self, "NULL handle");
        if (*self) {
            DeviceGuard g((*self)->d.device);
            delete *self;
        }
        *self = nullptr;
    });
}

int nfx_vinterp_set_grid(nfx_vinterp** self, nfx_grid* grid) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && grid, "NULL handle");
        (*self)->d.grid = &grid->d;
        (*self)->d.device = grid->d.device;
    });
}

int nfx_vinterp_build_locator(nfx_vinterp** self, int num_cells_per_bucket, double period_x, int enable_folding) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        VInterpDev& vi = (*self)->d;
        NFX_REQUIRE(vi.grid, "buildLocator: setGrid was not called");
        NFX_REQUIRE(num_cells_per_bucket > 0 && period_x >= 0.0 && enable_folding == 0, "buildLocator: bad arguments");
        DeviceGuard g(vi.grid->device);
        grid_build_locator(*vi.grid, nullptr);
        NFX_CUDA(cudaStreamSynchronize(nullptr));
        vi.period_x = period_x;
    });
}

int nfx_vinterp_find_points(nfx_vinterp** self, int64_t npoints, const double* xyz, double tol2, int64_t* num_not_found) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        VInterpDev& vi = (*self)->d;
        NFX_REQUIRE(vi.grid, "findPoints: setGrid was not called");
        DeviceGuard g(vi.grid->device);
        vinterp_find_points(vi, npoints, xyz, tol2, nullptr);
        if (num_not_found) {
            std::vector<int32_t> h((size_t)std::max<int64_t>(npoints, 1));
            if (npoints) NFX_CUDA(cudaMemcpy(h.data(), vi.cell.p, sizeof(int32_t) * npoints, cudaMemcpyDeviceToHost));
            int64_t bad = 0;
            for (int64_t i = 0; i < npoints; ++i) bad += h[i] < 0;
            *num_not_found = bad;
        }
    });
}

int nfx_vinterp_get_cells(nfx_vinterp** self, int64_t* cell, double* xi) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        VInterpDev& vi = (*self)->d;
        NFX_REQUIRE(vi.grid, "setGrid was not called");
        DeviceGuard g(vi.grid->device);
        if (vi.npts == 0) return;
        if (cell) {
            std::vector<int32_t> h((size_t)vi.npts);
            NFX_CUDA(cudaMemcpy(h.data(), vi.cell.p, sizeof(int32_t) * vi.npts, cudaMemcpyDeviceToHost));
            for (int64_t i = 0; i < vi.npts; ++i) cell[i] = h[i];
        }
        if (xi) NFX_CUDA(cudaMemcpy(xi, vi.xi.p, sizeof(double) * 2 * vi.npts, cudaMemcpyDeviceToHost));
    });
}

int nfx_vinterp_get_face_vectors(nfx_vinterp** self, const double* data, int placement, double* vectors) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && data && vectors, "NULL pointer");
        NFX_REQUIRE(placement == NFX_CELL_BY_CELL_DATA, "only CELL_BY_CELL_DATA placement is supported");
        VInterpDev& vi = (*self)->d;
        NFX_REQUIRE(vi.grid, "getFaceVectors: setGrid was not called");
        DeviceGuard g(vi.grid->device);
        if (vi.npts == 0) return;
        const size_t n = (size_t)vi.grid->ncell * 4;
        vi.scratch_data.ensure(n);
        vi.scratch_vec.ensure((size_t)vi.npts * 3);
        NFX_CUDA(cudaMemcpy(vi.scratch_data.p, data, sizeof(double) * n, cudaMemcpyHostToDevice));
        vinterp_face_vectors(vi, vi.scratch_data.p, vi.scratch_vec.p, nullptr);
        NFX_CUDA(cudaMemcpy(vectors, vi.scratch_vec.p, sizeof(double) * 3 * vi.npts, cudaMemcpyDeviceToHost));
    });
}

int nfx_vinterp_get_face_vectors_device(nfx_vinterp** self, const double* data, double* vectors, void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && data && vectors, "NULL pointer");
        VInterpDev& vi = (*self)->d;
        NFX_REQUIRE(vi.grid, "getFaceVectors: setGrid was not called");
        DeviceGuard g(vi.grid->device);
        vinterp_face_vectors(vi, data, vectors, (cudaStream_t)stream);
    });
}

// ---- K2 / K3 on device buffers -------------------------------------------------------------------------
int nfx_edgeflux_assemble(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                          const double* arc2, int nt, int nz, int64_t ncell, int sverdrup, double fill,
                          double* eflux, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        edgeflux_assemble(u, v, dtype, thickness, arc1, arc2, nt, nz, ncell, sverdrup, fill, eflux, g_k2opt,
                          (cudaStream_t)stream);
    });
}

int nfx_edgeflux_assemble_ld(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                             const double* arc2, int nt, int nz, int64_t ncell, int64_t ld, int sverdrup, double fill,
                             double* eflux, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        NFX_REQUIRE(ld >= ncell, "ld must be >= ncell");
        edgeflux_assemble_panel(u, v, dtype, thickness, arc1, arc2, nt, nz, ncell, ld, sverdrup, fill, eflux, 0, g_k2opt,
                                (cudaStream_t)stream);
    });
}

int nfx_edgeflux_assemble_e3(const void* u, const void* v, const void* e3u, const void* e3v, int dtype, int e3_nt,
                             const double* arc1, const double* arc2, int nt, int nz, int64_t ncell, int64_t ld,
                             int sverdrup, double fill, double* eflux, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        NFX_REQUIRE(e3u && e3v, "e3u / e3v is NULL");
        NFX_REQUIRE(ld >= ncell, "ld must be >= ncell");
        NFX_REQUIRE(e3_nt == 1 || e3_nt == nt, "e3u/e3v must hold 1 (time-invariant) or nt time steps");
        edgeflux_assemble_panel(u, v, dtype, nullptr, arc1, arc2, nt, nz, ncell, ld, sverdrup, fill, eflux, 0, g_k2opt,
                                (cudaStream_t)stream, e3u, e3v, e3_nt == 1 ? 0 : (int64_t)nz * ld);
    });
}

int nfx_flux_series_e3(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                       int e3_nt, const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup,
                       double fill, int order, double* eflux, double* series, void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        NFX_REQUIRE(u && v && e3u && e3v && arc1 && arc2 && series, "NULL pointer");
        const int64_t ncell = p.grid->ncell;
        NFX_REQUIRE(ld >= ncell, "ld must be >= the number of cells");
        NFX_REQUIRE(e3_nt == 1 || e3_nt == nt, "e3u/e3v must hold 1 (time-invariant) or nt time steps");
        const int64_t e3_tstride = e3_nt == 1 ? 0 : (int64_t)nz * ld;
        g_last_series_fused = 0;
        g_last_series_sparse = 0;
        if (eflux == nullptr && use_fused_e3(p, dtype, u, v, e3u, e3v, e3_tstride, ld)) {
            g_last_series_fused = 1;
            flux_series_fast(p, u, v, dtype, nullptr, arc1, arc2, nt, nz, ld, sverdrup, fill, order, series,
                             (cudaStream_t)stream, 0, -1, e3u, e3v, e3_tstride);
            return;
        }
        const Csr& c = pick_csr(p, order, 1);
        if (eflux == nullptr) {
            p.stage_eflux[0].ensure((size_t)nt * 2 * ncell);
            eflux = p.stage_eflux[0].p;
        }
        edgeflux_assemble_panel(u, v, dtype, nullptr, arc1, arc2, nt, nz, ncell, ld, sverdrup, fill, eflux, 0, g_k2opt,
                                (cudaStream_t)stream, e3u, e3v, e3_tstride);
        csr_integrate(c, p.ntransects, eflux, ncell * 2, nt, series, (cudaStream_t)stream);
    });
}

int nfx_edgeflux_to_cell_by_cell(const double* eflux, int nt, int ny, int nx, double* iv, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        edgeflux_to_cell_by_cell(eflux, nt, ny, nx, iv, (cudaStream_t)stream);
    });
}

int nfx_edgeflux_absmax(const double* eflux, int nt, int64_t ncell, double* result, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        edgeflux_absmax(eflux, nt, ncell, result, (cudaStream_t)stream);
    });
}

int nfx_pli_integrate(nfx_pli** self, const double* eflux, int nt, int order, double* series, void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        const Csr& c = pick_csr(p, order, 1);
        csr_integrate(c, p.ntransects, eflux, p.grid->ncell * 2, nt, series, (cudaStream_t)stream);
    });
}

int nfx_flux_series_ld(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                       const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup, double fill,
                       int order, double* eflux, double* series, void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        NFX_REQUIRE(u && v && thickness && arc1 && arc2 && series, "NULL pointer");
        const int64_t ncell = p.grid->ncell;
        NFX_REQUIRE(ld >= ncell, "ld must be >= the number of cells");
        g_last_series_fused = 0;
        g_last_series_sparse = 0;
        if (eflux == nullptr && use_fused(p, dtype, u, v, ld)) {
            g_last_series_fused = 1;
            flux_series_fast(p, u, v, dtype, thickness, arc1, arc2, nt, nz, ld, sverdrup, fill, order, series,
                             (cudaStream_t)stream);
            return;
        }
        const Csr& c = pick_csr(p, order, 1);
        if (eflux == nullptr) {   // two-launch path with an internal eflux array
            p.stage_eflux[0].ensure((size_t)nt * 2 * ncell);
            eflux = p.stage_eflux[0].p;
        }
        edgeflux_assemble_panel(u, v, dtype, thickness, arc1, arc2, nt, nz, ncell, ld, sverdrup, fill, eflux, 0, g_k2opt,
                                (cudaStream_t)stream);
        csr_integrate(c, p.ntransects, eflux, ncell * 2, nt, series, (cudaStream_t)stream);
    });
}

int nfx_pli_series_status(nfx_pli** self, void* stream, int* status) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        if (status) *status = 0;
        if (!p.grid) return;
        DeviceGuard g(p.grid->device);
        NFX_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
        if (p.h_fused_err && *(volatile int*)p.h_fused_err != 0) {
            if (status) *status = 1;
            fused_check_sticky_error(p);   // resets the flag and throws
        }
    });
}

int nfx_h5_decode_chunks(const void* comp, int64_t comp_bytes, int64_t nchunks, const int64_t* in_off, const int64_t* in_size,
                         int filters, int elem_size, int rank, const int64_t* chunk_dims, const int64_t* dst_dims,
                         const int64_t* chunk_start, int swap_bytes, void* dst, int32_t* status, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        h5_decode_chunks(comp, comp_bytes, nchunks, in_off, in_size, filters, elem_size, rank, chunk_dims, dst_dims,
                         chunk_start, swap_bytes, dst, status, (cudaStream_t)stream);
    });
}

int nfx_probe_read_bandwidth(const void* buf, int64_t nbytes, int reps, double* gbs, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        NFX_REQUIRE(buf && gbs, "NULL pointer");
        DevBuf<double> sink;
        sink.alloc(1);
        *gbs = probe_read_bandwidth(buf, nbytes, reps, sink.p, (cudaStream_t)stream);
    });
}

int nfx_probe_read_bandwidth_groups(const void* buf, int64_t nbytes, const int32_t* groups, int64_t ngroups, int reps,
                                    double* gbs, void* stream) {
    return guarded([&] {
        int dev;
        require_gpu(&dev);
        NFX_REQUIRE(buf && groups && gbs, "NULL pointer");
        DevBuf<double> sink;
        sink.alloc(1);
        *gbs = probe_read_bandwidth_groups(buf, nbytes, groups, ngroups, reps, sink.p, (cudaStream_t)stream);
    });
}

int nfx_pli_get_column_groups(nfx_pli** self, int dtype, int order, int vec, int64_t* panel_offsets, int32_t* groups,
                              int64_t* ngroups) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        NFX_REQUIRE(dtype == NFX_F64 || dtype == NFX_F32, "dtype must be NFX_F64 or NFX_F32");
        NFX_REQUIRE(vec == 1 || vec == 2 || vec == 4 || vec == 8, "vec must be 1, 2, 4 or 8");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid && p.grid->ncell > 0, "setGrid / setPoints was not called");
        NFX_REQUIRE(order == NFX_ORDER_LIST || order == NFX_ORDER_MAP, "order must be NFX_ORDER_LIST or NFX_ORDER_MAP");
        NFX_REQUIRE(p.csr[order][0].rowptr.p != nullptr, "computeWeights was not called");
        DeviceGuard g(p.grid->device);
        const int64_t panel = fused_panel_cells(p.grid->ncell, dtype);
        PanelPlan& pl = p.plan[order];
        if (!pl.built || pl.panel_cells != panel) build_panel_plan(p, order, panel, nullptr);
        if (pl.grp_vec != vec) build_column_groups(pl, p.grid->ncell, p.ntransects, vec, nullptr);
        NFX_CUDA(cudaStreamSynchronize(nullptr));
        if (ngroups) *ngroups = pl.ngroups;
        d2h(panel_offsets, pl.grp_ptr.p, (size_t)pl.npanels + 1);
        d2h(groups, pl.grp.p, (size_t)pl.ngroups);
    });
}

int nfx_pli_get_num_panels_dtype(nfx_pli** self, int dtype, int* npanels, int64_t* panel_cells) {
    return guarded([&] {
        NFX_REQUIRE(self && *self && npanels, "NULL pointer");
        NFX_REQUIRE(dtype == NFX_F64 || dtype == NFX_F32, "dtype must be NFX_F64 or NFX_F32");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid && p.grid->ncell > 0, "setGrid / setPoints was not called");
        const int64_t pc = fused_panel_cells(p.grid->ncell, dtype);
        *npanels = (int)((p.grid->ncell + pc - 1) / pc);
        if (panel_cells) *panel_cells = pc;
    });
}

int nfx_pli_get_num_panels(nfx_pli** self, int* npanels, int64_t* panel_cells) {
    return nfx_pli_get_num_panels_dtype(self, NFX_F64, npanels, panel_cells);
}

int nfx_flux_series_range(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                          const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup, double fill,
                          int order, int64_t batch_begin, int64_t batch_end, double* series, void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        NFX_REQUIRE(u && v && thickness && arc1 && arc2 && series, "NULL pointer");
        NFX_REQUIRE(ld >= p.grid->ncell, "ld must be >= the number of cells");
        g_last_series_fused = 1;
        flux_series_fast(p, u, v, dtype, thickness, arc1, arc2, nt, nz, ld, sverdrup, fill, order, series,
                         (cudaStream_t)stream, batch_begin, batch_end);
    });
}

int nfx_flux_series_range_e3(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v, int dtype,
                             int e3_nt, const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup,
                             double fill, int order, int64_t batch_begin, int64_t batch_end, double* series,
                             void* stream) {
    return guarded([&] {
        NFX_REQUIRE(self && *self, "NULL handle");
        PliDev& p = (*self)->d;
        NFX_REQUIRE(p.grid, "setGrid was not called");
        DeviceGuard g(p.grid->device);
        NFX_REQUIRE(u && v && e3u && e3v && arc1 && arc2 && series, "NULL pointer");
        NFX_REQUIRE(ld >= p.grid->ncell, "ld must be >= the number of cells");
        NFX_REQUIRE(e3_nt == 1 || e3_nt == nt, "e3u/e3v must hold 1 (time-invariant) or nt time steps");
        g_last_series_fused = 1;
        flux_series_fast(p, u, v, dtype, nullptr, arc1, arc2, nt, nz, ld, sverdrup, fill, order, series,
                         (cudaStream_t)stream, batch_begin, batch_end, e3u, e3v, e3_nt == 1 ? 0 : (int64_t)nz * ld);
    });
}

int nfx_flux_series(nfx_pli** self, const void* u, const void* v, int dtype, const double* thickness,
                    const double* arc1, const double* arc2, int nt, int nz, int sverdrup, double fill, int order,
                    double* eflux, double* series, void* stream) {
    if (!(self && *self && (*self)->d.grid)) {
        set_last_error("NULL handle or setGrid was not called");
        return NFX_E_INVALID;
    }
    return nfx_flux_series_ld(self, u, v, dtype, thickness, arc1, arc2, nt, nz, (*self)->d.grid->ncell, sverdrup, fill,
                              order, eflux, series, stream);
}

// ---- everything from host buffers: double-buffered H2D staging, K2+K3 per chunk --------------------------
// e3u/e3v (optional): per-column scale factors instead of `thickness`.  e3_on_device: borrowed device arrays
// (e3_nt, nz, ncell) of the dtype of u, v; else host arrays -- e3_nt == 1 is uploaded once per call, e3_nt == nt
// travels in the chunks next to u and v (same byte order as u, v).
static void flux_series_host_impl(nfx_pli** self, const void* u, const void* v, int dtype_flags, const double* thickness,
                                  const void* e3u, const void* e3v, int e3_nt, int e3_on_device, const double* arc1,
                                  const double* arc2, int nt, int nz, int sverdrup, double fill, int order,
                                  int chunk_steps, double* series) {
    NFX_REQUIRE(self && *self, "NULL handle");
    const bool e3 = e3u != nullptr || e3v != nullptr;
    NFX_REQUIRE(u && v && arc1 && arc2 && series, "NULL pointer");
    NFX_REQUIRE(e3 ? (e3u && e3v) : thickness != nullptr, "needs the layer thickness or both of e3u, e3v");
    NFX_REQUIRE(nt >= 0 && nz > 0, "bad sizes");
    NFX_REQUIRE(!e3 || e3_nt == 1 || e3_nt == nt, "e3u/e3v must hold 1 (time-invariant) or nt time steps");
    const bool big_endian = (dtype_flags & NFX_BIG_ENDIAN) != 0;
    const int dtype = dtype_flags & ~NFX_BIG_ENDIAN;
    NFX_REQUIRE(dtype == NFX_F64 || dtype == NFX_F32, "dtype must be NFX_F64 or NFX_F32 (optionally | NFX_BIG_ENDIAN)");
    PliDev& p = (*self)->d;
    NFX_REQUIRE(p.grid, "setGrid was not called");
    DeviceGuard g(p.grid->device);
    const Csr& c = pick_csr(p, order, 1);
    const int64_t ncell = p.grid->ncell;
    const int M = p.ntransects;
    if (nt == 0 || M == 0) return;
    const size_t esize = dtype == NFX_F64 ? 8 : 4;
    const size_t step_bytes = esize * (size_t)nz * (size_t)ncell;
    const bool e3_streamed = e3 && !e3_on_device && e3_nt == nt && nt > 1;
    if (chunk_steps <= 0) {
        const size_t target = (size_t)256 << 20;  // per variable and slot
        chunk_steps = (int)std::max<size_t>(1, target / step_bytes);
    }
    chunk_steps = std::min(chunk_steps, nt);
    if (!p.copy_stream) {
        NFX_CUDA(cudaStreamCreateWithFlags(&p.copy_stream, cudaStreamNonBlocking));
        NFX_CUDA(cudaStreamCreateWithFlags(&p.compute_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            NFX_CUDA(cudaEventCreateWithFlags(&p.ev_ready[i], cudaEventDisableTiming));
            NFX_CUDA(cudaEventCreateWithFlags(&p.ev_done[i], cudaEventDisableTiming));
        }
    }
    for (int i = 0; i < 2; ++i) {
        p.stage_u[i].ensure(step_bytes * chunk_steps);
        p.stage_v[i].ensure(step_bytes * chunk_steps);
        if (e3_streamed) {
            p.stage_e3u[i].ensure(step_bytes * chunk_steps);
            p.stage_e3v[i].ensure(step_bytes * chunk_steps);
        }
    }
    p.stage_series.ensure((size_t)nt * M);
    p.stage_arc1.ensure(ncell);
    p.stage_arc2.ensure(ncell);
    cudaStream_t cs = p.copy_stream, ks = p.compute_stream;
    if (!e3) {
        p.stage_thick.ensure(nz);
        NFX_CUDA(cudaMemcpyAsync(p.stage_thick.p, thickness, sizeof(double) * nz, cudaMemcpyHostToDevice, ks));
    }
    NFX_CUDA(cudaMemcpyAsync(p.stage_arc1.p, arc1, sizeof(double) * ncell, cudaMemcpyHostToDevice, ks));
    NFX_CUDA(cudaMemcpyAsync(p.stage_arc2.p, arc2, sizeof(double) * ncell, cudaMemcpyHostToDevice, ks));
    const void* d_e3u = e3u;   // device addresses of the scale factors of the first time step of a chunk
    const void* d_e3v = e3v;
    if (e3 && !e3_on_device && !e3_streamed) {   // host, time-invariant (or a single step): once per call
        p.stage_e3u[0].ensure(step_bytes);
        p.stage_e3v[0].ensure(step_bytes);
        NFX_CUDA(cudaMemcpyAsync(p.stage_e3u[0].p, e3u, step_bytes, cudaMemcpyHostToDevice, ks));
        NFX_CUDA(cudaMemcpyAsync(p.stage_e3v[0].p, e3v, step_bytes, cudaMemcpyHostToDevice, ks));
        if (big_endian) {
            bswap_inplace(p.stage_e3u[0].p, step_bytes / esize, (int)esize, ks);
            bswap_inplace(p.stage_e3v[0].p, step_bytes / esize, (int)esize, ks);
        }
        d_e3u = p.stage_e3u[0].p;
        d_e3v = p.stage_e3v[0].p;
    }
    const bool fused = e3 ? use_fused_e3(p, dtype, nullptr, nullptr, nullptr, nullptr, 0, ncell)
                          : use_fused(p, dtype, nullptr, nullptr, ncell);
    if (!fused)
        for (int i = 0; i < 2; ++i) p.stage_eflux[i].ensure((size_t)chunk_steps * 2 * ncell);
    int slot = 0;
    bool used[2] = {false, false};
    for (int t0 = 0; t0 < nt; t0 += chunk_steps, slot ^= 1) {
        const int n = std::min(chunk_steps, nt - t0);
        if (used[slot]) NFX_CUDA(cudaStreamWaitEvent(cs, p.ev_done[slot], 0));
        const size_t off = (size_t)t0 * step_bytes;
        const void* src[4] = {(const unsigned char*)u + off, (const unsigned char*)v + off,
                              e3_streamed ? (const unsigned char*)e3u + off : nullptr,
                              e3_streamed ? (const unsigned char*)e3v + off : nullptr};
        unsigned char* dst[4] = {p.stage_u[slot].p, p.stage_v[slot].p, e3_streamed ? p.stage_e3u[slot].p : nullptr,
                                 e3_streamed ? p.stage_e3v[slot].p : nullptr};
        for (int q = 0; q < 4; ++q) {
            if (!src[q]) continue;
            NFX_CUDA(cudaMemcpyAsync(dst[q], src[q], step_bytes * n, cudaMemcpyHostToDevice, cs));
            if (big_endian)   // file bytes as stored: swap on the device, behind the copy on the copy stream
                bswap_inplace(dst[q], step_bytes * n / esize, (int)esize, cs);
        }
        NFX_CUDA(cudaEventRecord(p.ev_ready[slot], cs));
        NFX_CUDA(cudaStreamWaitEvent(ks, p.ev_ready[slot], 0));
        const void* ce3u = nullptr;
        const void* ce3v = nullptr;
        int64_t e3_tstride = 0;
        if (e3_streamed) {
            ce3u = dst[2];
            ce3v = dst[3];
            e3_tstride = (int64_t)nz * ncell;
        } else if (e3) {
            const bool per_step = e3_on_device && e3_nt == nt && nt > 1;
            e3_tstride = per_step ? (int64_t)nz * ncell : 0;
            ce3u = (const unsigned char*)d_e3u + (per_step ? off : 0);
            ce3v = (const unsigned char*)d_e3v + (per_step ? off : 0);
        }
        double* out = p.stage_series.p + (size_t)t0 * M;
        if (fused) {
            flux_series_fast(p, dst[0], dst[1], dtype, e3 ? nullptr : p.stage_thick.p, p.stage_arc1.p, p.stage_arc2.p, n,
                             nz, ncell, sverdrup, fill, order, out, ks, 0, -1, ce3u, ce3v, e3_tstride);
        } else {
            edgeflux_assemble_panel(dst[0], dst[1], dtype, e3 ? nullptr : p.stage_thick.p, p.stage_arc1.p,
                                    p.stage_arc2.p, n, nz, ncell, ncell, sverdrup, fill, p.stage_eflux[slot].p, 0, g_k2opt,
                                    ks, ce3u, ce3v, e3_tstride);
            csr_integrate(c, M, p.stage_eflux[slot].p, ncell * 2, n, out, ks);
        }
        NFX_CUDA(cudaEventRecord(p.ev_done[slot], ks));
        used[slot] = true;
    }
    NFX_CUDA(cudaMemcpyAsync(series, p.stage_series.p, sizeof(double) * (size_t)nt * M, cudaMemcpyDeviceToHost, ks));
    NFX_CUDA(cudaStreamSynchronize(ks));
    NFX_CUDA(cudaStreamSynchronize(cs));
    g_last_series_fused = fused ? 1 : 0;
    if (!fused) g_last_series_sparse = 0;
    if (fused && fused_error_flag(p, ks) != 0)
        throw Error(NFX_E_INTERNAL, "fused K2+K3 pass aborted (a bounded wait overflowed)");
}

int nfx_flux_series_host(nfx_pli** self, const void* u, const void* v, int dtype_flags, const double* thickness,
                         const double* arc1, const double* arc2, int nt, int nz, int sverdrup, double fill, int order,
                         int chunk_steps, double* series) {
    return guarded([&] {
        NFX_REQUIRE(thickness, "NULL pointer");
        flux_series_host_impl(self, u, v, dtype_flags, thickness, nullptr, nullptr, 0, 0, arc1, arc2, nt, nz, sverdrup,
                              fill, order, chunk_steps, series);
    });
}

int nfx_flux_series_host_e3(nfx_pli** self, const void* u, const void* v, const void* e3u, const void* e3v,
                            int dtype_flags, int e3_nt, int e3_on_device, const double* arc1, const double* arc2, int nt,
                            int nz, int sverdrup, double fill, int order, int chunk_steps, double* series) {
    return guarded([&] {
        NFX_REQUIRE(e3u && e3v, "e3u / e3v is NULL");
        flux_series_host_impl(self, u, v, dtype_flags, nullptr, e3u, e3v, e3_nt, e3_on_device, arc1, arc2, nt, nz,
                              sverdrup, fill, order, chunk_steps, series);
    });
}

}  // extern "C"
