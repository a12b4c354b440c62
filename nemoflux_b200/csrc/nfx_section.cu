// Transport section (sm_100a): the flux of every sub-segment (cell crossing) of every transect, per layer of model
// levels and time step, in the emission order of K1.
//
//   section[t, i, s] = ((w[s,0]*E_i[idx[4s]] + w[s,1]*E_i[idx[4s+1]]) + w[s,2]*E_i[idx[4s+2]]) + w[s,3]*E_i[idx[4s+3]]
//
// idx is the list-order compact CSR of K1 (flux_index: E -> eU[c], W -> eU[west], N -> eV[c], S -> eV[south], -1 for
// the south edge of row 0, whose flux is 0), E_i the layer-i edge flux exactly as the layered K2 writes it: the
// k-ascending sum of dz[k] * u (e3u * u) from +0 over the levels of the layer, times arc1 (times -arc2 for eV), times
// 6.371 with sverdrup; every product and sum a separate __dmul_rn / __dadd_rn.  float32 values go through the plain
// conversion (clean()): the bits are those of K2's clean_scaled() path by construction.
//
// Nothing is reduced across sub-segments, so this is a direct gather pass: one thread per (time step, sub-segment),
// consecutive sub-segments in consecutive lanes.  Per level a thread loads the 4 columns its edges read (and, with
// E3, the 4 scale factors at the same places), UNROLL levels in flight, and keeps 4 running column sums; at every
// layer boundary it finishes the 4 edge fluxes, combines them with the weights and stores one value (coalesced over
// s, streaming).  The loads allocate in L1: a crossing's E column is its zonal neighbour's W column, and the lanes
// of a zonal run share 32-byte sectors.
//
// Bytes: per (time step, level) the 32-byte sectors of u/v (and e3u/e3v) the list index touches, plus 8 bytes per
// (time step, layer, sub-segment) written.
#include "nfx_common.cuh"
#include "nfx_stream_ops.cuh"

namespace nfx {

namespace {

using namespace dev;

constexpr int kSectionBlock = 256;

// levels in flight per thread (4 loads per level, 8 with E3) and CTAs per SM: 80 registers without E3, 124-128 with
// (the E3 instances spill at 80, profiles/r5_section_ptxas.md)
template <typename T, bool E3>
struct SectionShape {
    static constexpr int unroll = E3 ? (sizeof(T) == 8 ? 2 : 3) : 4;
    static constexpr int ctas = E3 ? 2 : 3;
};

template <typename T, bool E3>
__global__ void __launch_bounds__(kSectionBlock, SectionShape<T, E3>::ctas)
k_flux_section(const T* __restrict__ u, const T* __restrict__ v, const T* __restrict__ e3u, const T* __restrict__ e3v,
               int64_t e3_tstride, const double* __restrict__ dz, const double* __restrict__ arc1,
               const double* __restrict__ arc2, const int32_t* __restrict__ idx, const double* __restrict__ w,
               int64_t nsub, int64_t ncell, int64_t ld, int nz, int nlayers, const int* __restrict__ levels, double scale,
               int use_scale, T fill, int has_fill, int64_t t0, double* __restrict__ section) {
    constexpr int UNROLL = SectionShape<T, E3>::unroll;
    extern __shared__ double s_dz[];                        // [nz] dz (without E3), then [nlayers + 1] boundaries
    int* s_lev = reinterpret_cast<int*>(s_dz + (E3 ? 0 : nz));
    if constexpr (!E3)
        for (int k = threadIdx.x; k < nz; k += kSectionBlock) s_dz[k] = dz[k];
    for (int i = threadIdx.x; i <= nlayers; i += kSectionBlock)
        s_lev[i] = levels ? levels[i] : (i == 0 ? 0 : nz);  // levels == nullptr: one layer, the whole column
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * kSectionBlock + threadIdx.x;
    if (s >= nsub) return;
    const int64_t t = t0 + blockIdx.y;
    const T* pc[4];        // column of every edge at level 0 of step t
    const T* pe[4];        // E3: its scale factors
    double arc[4], wt[4], acc[4];
    bool live[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int32_t j = idx[4 * s + e];
        live[e] = j >= 0;
        const bool isv = j >= ncell;
        const int64_t col = !live[e] ? 0 : isv ? j - ncell : j;   // idx < 0: a harmless address, the flux is 0
        pc[e] = (isv ? v : u) + t * nz * ld + col;
        pe[e] = E3 ? (isv ? e3v : e3u) + t * e3_tstride + col : nullptr;
        arc[e] = !live[e] ? 0.0 : isv ? -arc2[col] : arc1[col];   // eV = (-sum) * arc2: the negation is exact
        wt[e] = w[4 * s + e];
        acc[e] = 0.0;
    }
    double* out = section + (t * nlayers) * nsub + s;
    int layer = 0, next = s_lev[1];
    const int kend = s_lev[nlayers];
    int k = s_lev[0];
    // level kk into the 4 column sums; after the last level of a layer: the 4 edge fluxes, their weighted sum in
    // edge order, one streaming store (the layering is the same for every thread: the branch does not diverge)
    auto step = [&](int kk, const T (&x)[4], const T (&ex)[4]) {
        const double d = E3 ? 0.0 : s_dz[kk];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const double de = E3 ? clean<T>(ex[e], fill, has_fill) : d;
            acc[e] = __dadd_rn(acc[e], __dmul_rn(de, clean<T>(x[e], fill, has_fill)));
        }
        if (kk + 1 == next) {
            double r = 0.0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                // the eflux value of K2: (sum * arc) [* 6.371], -sum * arc2 for eV; 0 for the south edge of row 0
                double f = __dmul_rn(acc[e], arc[e]);
                if (use_scale) f = __dmul_rn(f, scale);
                f = live[e] ? f : 0.0;
                r = e == 0 ? __dmul_rn(wt[0], f) : __dadd_rn(r, __dmul_rn(wt[e], f));
                acc[e] = 0.0;
            }
            __stcs(out + (int64_t)layer * nsub, r);
            ++layer;
            next = layer < nlayers ? s_lev[layer + 1] : -1;
        }
    };
    for (; k + UNROLL <= kend; k += UNROLL) {
        T x[UNROLL][4], ex[UNROLL][4];
#pragma unroll
        for (int q = 0; q < UNROLL; ++q)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                x[q][e] = __ldg(pc[e] + (int64_t)(k + q) * ld);
                if constexpr (E3) ex[q][e] = __ldg(pe[e] + (int64_t)(k + q) * ld);
            }
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) step(k + q, x[q], ex[q]);
    }
    for (; k < kend; ++k) {
        T x[4], ex[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            x[e] = __ldg(pc[e] + (int64_t)k * ld);
            if constexpr (E3) ex[e] = __ldg(pe[e] + (int64_t)k * ld);
        }
        step(k, x, ex);
    }
}

// Time-mean section: the sums over windows of time steps of the section above.  One thread per (window, layer,
// sub-segment), consecutive sub-segments in consecutive lanes; y = window * nlayers + layer.  Window w covers the steps
// [bounds[w], bounds[w+1]) clipped to the steps [t_first, t_end) the arrays hold (u, v, e3 start at step t_first).
// The thread walks the window's steps in ascending order; per step it sums the layer's levels into the 4 column sums,
// forms the step's section value with the operations of k_flux_section and adds it to the running window sum:
//   sum = (((+0 | the stored partial sum) + sec[t0]) + sec[t0 + 1]) + ...       (every add a __dadd_rn)
// The first window the launch covers (w0) continues the partial sum stored in `sums` when continue_first is set.  One
// streaming store per (window, layer, sub-segment); the loads per (step, level, edge) are those of k_flux_section.
template <typename T, bool E3>
__global__ void __launch_bounds__(kSectionBlock, SectionShape<T, E3>::ctas)
k_flux_section_windows(const T* __restrict__ u, const T* __restrict__ v, const T* __restrict__ e3u,
                       const T* __restrict__ e3v, int64_t e3_tstride, const double* __restrict__ dz,
                       const double* __restrict__ arc1, const double* __restrict__ arc2,
                       const int32_t* __restrict__ idx, const double* __restrict__ w, int64_t nsub, int64_t ncell,
                       int64_t ld, int nz, int nlayers, const int* __restrict__ levels, double scale, int use_scale,
                       T fill, int has_fill, const int* __restrict__ bounds, int w0, int t_first, int t_end,
                       int continue_first, int64_t y0, double* __restrict__ sums) {
    constexpr int UNROLL = SectionShape<T, E3>::unroll;
    extern __shared__ double s_dz[];                        // [nz] dz (without E3), then [nlayers + 1] boundaries
    int* s_lev = reinterpret_cast<int*>(s_dz + (E3 ? 0 : nz));
    if constexpr (!E3)
        for (int k = threadIdx.x; k < nz; k += kSectionBlock) s_dz[k] = dz[k];
    for (int i = threadIdx.x; i <= nlayers; i += kSectionBlock)
        s_lev[i] = levels ? levels[i] : (i == 0 ? 0 : nz);
    __syncthreads();
    const int64_t s = (int64_t)blockIdx.x * kSectionBlock + threadIdx.x;
    if (s >= nsub) return;
    const int64_t y = y0 + blockIdx.y;                      // (window - w0) * nlayers + layer
    const int win = w0 + (int)(y / nlayers);
    const int layer = (int)(y % nlayers);
    const int tb = max(bounds[win], t_first) - t_first, te = min(bounds[win + 1], t_end) - t_first;
    const int kbeg = s_lev[layer], kend = s_lev[layer + 1];
    const T* pc[4];        // column of every edge at level kbeg of step 0
    const T* pe[4];
    double arc[4], wt[4];
    bool live[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int32_t j = idx[4 * s + e];
        live[e] = j >= 0;
        const bool isv = j >= ncell;
        const int64_t col = !live[e] ? 0 : isv ? j - ncell : j;
        pc[e] = (isv ? v : u) + (int64_t)kbeg * ld + col;
        pe[e] = E3 ? (isv ? e3v : e3u) + (int64_t)kbeg * ld + col : nullptr;
        arc[e] = !live[e] ? 0.0 : isv ? -arc2[col] : arc1[col];
        wt[e] = w[4 * s + e];
    }
    double* out = sums + y * nsub + s;
    double total = continue_first && y < nlayers ? __ldcs(out) : 0.0;
    for (int t = tb; t < te; ++t) {
        const int64_t tu = (int64_t)t * nz * ld, tx = (int64_t)t * e3_tstride;
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        auto level = [&](int kk, const T (&x)[4], const T (&ex)[4]) {
            const double d = E3 ? 0.0 : s_dz[kk];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const double de = E3 ? clean<T>(ex[e], fill, has_fill) : d;
                acc[e] = __dadd_rn(acc[e], __dmul_rn(de, clean<T>(x[e], fill, has_fill)));
            }
        };
        int k = kbeg;
        for (; k + UNROLL <= kend; k += UNROLL) {
            T x[UNROLL][4], ex[UNROLL][4];
#pragma unroll
            for (int q = 0; q < UNROLL; ++q)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    x[q][e] = __ldg(pc[e] + tu + (int64_t)(k - kbeg + q) * ld);
                    if constexpr (E3) ex[q][e] = __ldg(pe[e] + tx + (int64_t)(k - kbeg + q) * ld);
                }
#pragma unroll
            for (int q = 0; q < UNROLL; ++q) level(k + q, x[q], ex[q]);
        }
        for (; k < kend; ++k) {
            T x[4], ex[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                x[e] = __ldg(pc[e] + tu + (int64_t)(k - kbeg) * ld);
                if constexpr (E3) ex[e] = __ldg(pe[e] + tx + (int64_t)(k - kbeg) * ld);
            }
            level(k, x, ex);
        }
        double r = 0.0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            double f = __dmul_rn(acc[e], arc[e]);
            if (use_scale) f = __dmul_rn(f, scale);
            f = live[e] ? f : 0.0;
            r = e == 0 ? __dmul_rn(wt[0], f) : __dadd_rn(r, __dmul_rn(wt[e], f));
        }
        total = __dadd_rn(total, r);
    }
    __stcs(out, total);
}

template <typename T, bool E3>
void launch_section_windows(const void* u, const void* v, const void* e3u, const void* e3v, int64_t e3_tstride,
                            const double* dz, const double* arc1, const double* arc2, const int32_t* idx,
                            const double* w, int64_t nsub, int64_t ncell, int64_t ld, int nz, int nlayers,
                            const int* levels, int sverdrup, double fill, const int* bounds, int w0, int nwin,
                            int t_first, int t_end, int continue_first, double* sums, cudaStream_t s) {
    const double scale = 6371000.0 / 1.e6;
    const int has_fill = !(fill != fill);
    const size_t smem = (E3 ? 0 : sizeof(double) * nz) + sizeof(int) * (nlayers + 1);
    const unsigned gx = (unsigned)((nsub + kSectionBlock - 1) / kSectionBlock);
    const int64_t ny = (int64_t)nwin * nlayers;
    for (int64_t y0 = 0; y0 < ny; y0 += 65535) {
        dim3 grid(gx, (unsigned)std::min<int64_t>(65535, ny - y0));
        k_flux_section_windows<T, E3><<<grid, kSectionBlock, smem, s>>>(
            (const T*)u, (const T*)v, (const T*)e3u, (const T*)e3v, e3_tstride, dz, arc1, arc2, idx, w, nsub, ncell,
            ld, nz, nlayers, levels, scale, sverdrup, (T)fill, has_fill, bounds, w0, t_first, t_end, continue_first,
            y0, sums);
        count_launch();
        NFX_CUDA(cudaGetLastError());
    }
}

template <typename T, bool E3>
void launch_section(const void* u, const void* v, const void* e3u, const void* e3v, int64_t e3_tstride,
                    const double* dz, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                    int64_t nsub, int64_t ncell, int64_t ld, int nt, int nz, int nlayers, const int* levels,
                    int sverdrup, double fill, double* section, cudaStream_t s) {
    const double scale = 6371000.0 / 1.e6;   // field.py:12,226, as K2
    const int has_fill = !(fill != fill);
    const size_t smem = (E3 ? 0 : sizeof(double) * nz) + sizeof(int) * (nlayers + 1);
    const unsigned gx = (unsigned)((nsub + kSectionBlock - 1) / kSectionBlock);
    for (int t0 = 0; t0 < nt; t0 += 65535) {
        dim3 grid(gx, (unsigned)std::min(65535, nt - t0));
        k_flux_section<T, E3><<<grid, kSectionBlock, smem, s>>>(
            (const T*)u, (const T*)v, (const T*)e3u, (const T*)e3v, e3_tstride, dz, arc1, arc2, idx, w, nsub, ncell, ld,
            nz, nlayers, levels, scale, sverdrup, (T)fill, has_fill, t0, section);
        count_launch();
        NFX_CUDA(cudaGetLastError());
    }
}

}  // namespace

void flux_section(const void* u, const void* v, int dtype, const double* thickness, const void* e3u, const void* e3v,
                  int64_t e3_tstride, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                  int64_t nsub, int64_t ncell, int64_t ld, int nt, int nz, int nlayers, const int* levels, int sverdrup,
                  double fill, double* section, cudaStream_t s) {
    NFX_REQUIRE(u && v && arc1 && arc2 && idx && w && section, "section: NULL pointer");
    NFX_REQUIRE((e3u == nullptr) == (e3v == nullptr) && (thickness != nullptr) != (e3u != nullptr),
                "section: needs exactly one of thickness and (e3u, e3v)");
    NFX_REQUIRE(nz > 0 && nz <= 3000 && nt >= 0 && ld >= ncell, "section: bad sizes");
    NFX_REQUIRE(nsub / kSectionBlock < 2147483647ll, "section: too many sub-segments");
    if (nt == 0 || nsub == 0) return;
    const bool e3 = e3u != nullptr;
    if (dtype == NFX_F64) {
        if (e3)
            launch_section<double, true>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, nsub, ncell, ld, nt, nz,
                                         nlayers, levels, sverdrup, fill, section, s);
        else
            launch_section<double, false>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, nsub, ncell, ld, nt,
                                          nz, nlayers, levels, sverdrup, fill, section, s);
    } else {
        NFX_REQUIRE(dtype == NFX_F32, "section: dtype must be NFX_F64 or NFX_F32");
        if (e3)
            launch_section<float, true>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, nsub, ncell, ld, nt, nz,
                                        nlayers, levels, sverdrup, fill, section, s);
        else
            launch_section<float, false>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, nsub, ncell, ld, nt,
                                         nz, nlayers, levels, sverdrup, fill, section, s);
    }
}

void flux_section_windows(const void* u, const void* v, int dtype, const double* thickness, const void* e3u,
                          const void* e3v, int64_t e3_tstride, const double* arc1, const double* arc2,
                          const int32_t* idx, const double* w, int64_t nsub, int64_t ncell, int64_t ld, int nz,
                          int nlayers, const int* levels, int sverdrup, double fill, const int* bounds, int w0, int nwin,
                          int t_first, int t_end, int continue_first, double* sums, cudaStream_t s) {
    NFX_REQUIRE(u && v && arc1 && arc2 && idx && w && bounds && sums, "section windows: NULL pointer");
    NFX_REQUIRE((e3u == nullptr) == (e3v == nullptr) && (thickness != nullptr) != (e3u != nullptr),
                "section windows: needs exactly one of thickness and (e3u, e3v)");
    NFX_REQUIRE(nz > 0 && nz <= 3000 && nwin >= 0 && t_first <= t_end && ld >= ncell, "section windows: bad sizes");
    NFX_REQUIRE(nsub / kSectionBlock < 2147483647ll, "section windows: too many sub-segments");
    if (nwin == 0 || nsub == 0) return;
    const bool e3 = e3u != nullptr;
#define NFX_SECTION_WINDOWS(T, E3)                                                                                    \
    launch_section_windows<T, E3>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, nsub, ncell, ld, nz,     \
                                  nlayers, levels, sverdrup, fill, bounds, w0, nwin, t_first, t_end, continue_first,  \
                                  sums, s)
    if (dtype == NFX_F64) {
        if (e3)
            NFX_SECTION_WINDOWS(double, true);
        else
            NFX_SECTION_WINDOWS(double, false);
    } else {
        NFX_REQUIRE(dtype == NFX_F32, "section windows: dtype must be NFX_F64 or NFX_F32");
        if (e3)
            NFX_SECTION_WINDOWS(float, true);
        else
            NFX_SECTION_WINDOWS(float, false);
    }
#undef NFX_SECTION_WINDOWS
}

}  // namespace nfx
