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

// The operation sequence of one crossing, shared by the section kernels.  section_edges: the column of u or v every
// edge of sub-segment s reads (at offset `off`, its scale factor at `e3_off`), the factor that turns a column sum into
// K2's edge flux, its weight, and whether it is live (idx -1: the south edge of row 0, whose flux is 0).
template <typename T, bool E3>
__device__ __forceinline__ void section_edges(const T* __restrict__ u, const T* __restrict__ v, const T* __restrict__ e3u,
                                              const T* __restrict__ e3v, const double* __restrict__ arc1,
                                              const double* __restrict__ arc2, const int32_t* __restrict__ idx,
                                              const double* __restrict__ w, int64_t s, int64_t ncell, int64_t off,
                                              int64_t e3_off, const T* (&pc)[4], const T* (&pe)[4], double (&arc)[4],
                                              double (&wt)[4], bool (&live)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int32_t j = idx[4 * s + e];
        live[e] = j >= 0;
        const bool isv = j >= ncell;
        const int64_t col = !live[e] ? 0 : isv ? j - ncell : j;   // idx < 0: a harmless address, the flux is 0
        pc[e] = (isv ? v : u) + off + col;
        pe[e] = E3 ? (isv ? e3v : e3u) + e3_off + col : nullptr;
        arc[e] = !live[e] ? 0.0 : isv ? -arc2[col] : arc1[col];   // eV = (-sum) * arc2: the negation is exact
        wt[e] = w[4 * s + e];
    }
}

// the 4 columns (and, with E3, their scale factors) of one level, `off` / `e3_off` past the pointers of section_edges
template <typename T, bool E3>
__device__ __forceinline__ void section_load(const T* const (&pc)[4], const T* const (&pe)[4], int64_t off,
                                             int64_t e3_off, T (&x)[4], T (&ex)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        x[e] = __ldg(pc[e] + off);
        if constexpr (E3) ex[e] = __ldg(pe[e] + e3_off);
    }
}

// one level into the 4 column sums: acc += dz (or e3) * u, NaN and the marker as 0
template <typename T, bool E3>
__device__ __forceinline__ void section_level(double (&acc)[4], double d, const T (&x)[4], const T (&ex)[4], T fill,
                                              int has_fill) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const double de = E3 ? clean<T>(ex[e], fill, has_fill) : d;
        acc[e] = __dadd_rn(acc[e], __dmul_rn(de, clean<T>(x[e], fill, has_fill)));
    }
}

// the section value of 4 column sums: the eflux value of K2 per edge ((sum * arc) [* 6.371], -sum * arc2 for eV; 0 for
// the south edge of row 0), their weighted sum in edge order
__device__ __forceinline__ double section_value(const double (&acc)[4], const double (&arc)[4], const double (&wt)[4],
                                                const bool (&live)[4], double scale, int use_scale) {
    double r = 0.0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        double f = __dmul_rn(acc[e], arc[e]);
        if (use_scale) f = __dmul_rn(f, scale);
        f = live[e] ? f : 0.0;
        r = e == 0 ? __dmul_rn(wt[0], f) : __dadd_rn(r, __dmul_rn(wt[e], f));
    }
    return r;
}

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
    double arc[4], wt[4], acc[4] = {0.0, 0.0, 0.0, 0.0};
    bool live[4];
    section_edges<T, E3>(u, v, e3u, e3v, arc1, arc2, idx, w, s, ncell, t * nz * ld, t * e3_tstride, pc, pe, arc, wt,
                         live);
    double* out = section + (t * nlayers) * nsub + s;
    int layer = 0, next = s_lev[1];
    const int kend = s_lev[nlayers];
    int k = s_lev[0];
    // level kk into the 4 column sums; after the last level of a layer: the section value, one streaming store (the
    // layering is the same for every thread: the branch does not diverge)
    auto step = [&](int kk, const T (&x)[4], const T (&ex)[4]) {
        section_level<T, E3>(acc, E3 ? 0.0 : s_dz[kk], x, ex, fill, has_fill);
        if (kk + 1 == next) {
            const double r = section_value(acc, arc, wt, live, scale, use_scale);
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[e] = 0.0;
            __stcs(out + (int64_t)layer * nsub, r);
            ++layer;
            next = layer < nlayers ? s_lev[layer + 1] : -1;
        }
    };
    for (; k + UNROLL <= kend; k += UNROLL) {
        T x[UNROLL][4], ex[UNROLL][4];
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) section_load<T, E3>(pc, pe, (int64_t)(k + q) * ld, (int64_t)(k + q) * ld, x[q], ex[q]);
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) step(k + q, x[q], ex[q]);
    }
    for (; k < kend; ++k) {
        T x[4], ex[4];
        section_load<T, E3>(pc, pe, (int64_t)k * ld, (int64_t)k * ld, x, ex);
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
    section_edges<T, E3>(u, v, e3u, e3v, arc1, arc2, idx, w, s, ncell, (int64_t)kbeg * ld, (int64_t)kbeg * ld, pc, pe,
                         arc, wt, live);
    double* out = sums + y * nsub + s;
    double total = continue_first && y < nlayers ? __ldcs(out) : 0.0;
    for (int t = tb; t < te; ++t) {
        const int64_t tu = (int64_t)t * nz * ld, tx = (int64_t)t * e3_tstride;
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        int k = kbeg;
        for (; k + UNROLL <= kend; k += UNROLL) {
            T x[UNROLL][4], ex[UNROLL][4];
#pragma unroll
            for (int q = 0; q < UNROLL; ++q)
                section_load<T, E3>(pc, pe, tu + (int64_t)(k - kbeg + q) * ld, tx + (int64_t)(k - kbeg + q) * ld, x[q],
                                    ex[q]);
#pragma unroll
            for (int q = 0; q < UNROLL; ++q)
                section_level<T, E3>(acc, E3 ? 0.0 : s_dz[k + q], x[q], ex[q], fill, has_fill);
        }
        for (; k < kend; ++k) {
            T x[4], ex[4];
            section_load<T, E3>(pc, pe, tu + (int64_t)(k - kbeg) * ld, tx + (int64_t)(k - kbeg) * ld, x, ex);
            section_level<T, E3>(acc, E3 ? 0.0 : s_dz[k], x, ex, fill, has_fill);
        }
        total = __dadd_rn(total, section_value(acc, arc, wt, live, scale, use_scale));
    }
    __stcs(out, total);
}

// Class transport: the flux across every transect binned by a T-grid field c (temperature, salinity, density...).
// One thread per (time step, crossing), the crossings of one transect in warp tiles of at most 32 consecutive
// crossings (tile_start, K1's emission order; a tile never spans two transects), 8 tiles per CTA.  Per level the
// thread gathers its 4 columns as k_flux_section does, forms the crossing's level flux with the section's operations
// (a one-level layer: the bits of fluxSection(layers=range(nz+1))), loads c at its cell and level, finds the class
// j with b_j <= c < b_{j+1} by a search over the bounds in shared memory and adds the flux to its own sum of class j
// in shared memory (s_acc[j][thread]: no two threads share a word).  NaN, the marker cfill and values outside
// [b0, bK) count nowhere.  After the last level each warp folds its 32 per-crossing sums of every class with a fixed
// shuffle tree into one partial value per (step, tile, class); k_reduce_class_tiles adds a transect's tiles in
// ascending order.  No atomics: the bits depend on nothing but the inputs.
// levels in flight of k_flux_classes (5 loads per level, 9 with E3) and CTAs per SM: the section's, one level fewer
// without E3 (4 levels spill at 80 registers, profiles/r7_classes_ptxas.md)
template <typename T, bool E3>
struct ClassShape {
    static constexpr int unroll = E3 ? SectionShape<T, E3>::unroll : 3;
    static constexpr int ctas = SectionShape<T, E3>::ctas;
};

template <typename T, bool E3>
__global__ void __launch_bounds__(kSectionBlock, ClassShape<T, E3>::ctas)
k_flux_classes(const T* __restrict__ u, const T* __restrict__ v, const T* __restrict__ e3u, const T* __restrict__ e3v,
               int64_t e3_tstride, const double* __restrict__ dz, const double* __restrict__ arc1,
               const double* __restrict__ arc2, const int32_t* __restrict__ idx, const double* __restrict__ w,
               const int32_t* __restrict__ cell, const T* __restrict__ cf, int64_t c_tstride, T cfill, int has_cfill,
               const double* __restrict__ bounds, int K, const int64_t* __restrict__ tile_start, int64_t ntiles,
               int64_t ncell, int64_t ld, int nz, double scale, int use_scale, T fill, int has_fill, int64_t t0,
               double* __restrict__ partial) {
    constexpr int UNROLL = ClassShape<T, E3>::unroll;
    extern __shared__ double s_mem[];
    double* s_acc = s_mem;                                  // [K][kSectionBlock] per-thread class sums
    double* s_b = s_acc + (size_t)K * kSectionBlock;        // [K + 1] bounds
    double* s_dz = s_b + K + 1;                             // [nz] dz (without E3)
    for (int i = threadIdx.x; i <= K; i += kSectionBlock) s_b[i] = bounds[i];
    if constexpr (!E3)
        for (int k = threadIdx.x; k < nz; k += kSectionBlock) s_dz[k] = dz[k];
    for (int j = 0; j < K; ++j) s_acc[j * kSectionBlock + threadIdx.x] = 0.0;
    __syncthreads();
    const int64_t tile = (int64_t)blockIdx.x * (kSectionBlock / 32) + threadIdx.x / 32;
    if (tile >= ntiles) return;                             // the whole warp
    const int lane = threadIdx.x & 31;
    const int64_t t = t0 + blockIdx.y;
    const int64_t s = tile_start[tile] + lane;
    double* acc_j = s_acc + threadIdx.x;                    // this thread's sum of class j: acc_j[j * kSectionBlock]
    if (s < tile_start[tile + 1]) {
        const T* pc[4];
        const T* pe[4];
        double arc[4], wt[4];
        bool live[4];
        section_edges<T, E3>(u, v, e3u, e3v, arc1, arc2, idx, w, s, ncell, t * nz * ld, t * e3_tstride, pc, pe, arc,
                             wt, live);
        const T* pcl = cf + t * c_tstride + cell[s];
        int top = 1;                                        // the largest power of two <= K + 1
        while (2 * top <= K + 1) top *= 2;
        auto level = [&](int kk, const T (&x)[4], const T (&ex)[4], T c) {
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
            section_level<T, E3>(acc, E3 ? 0.0 : s_dz[kk], x, ex, fill, has_fill);
            const double f = section_value(acc, arc, wt, live, scale, use_scale);
            const double xc = (double)c;
            if (xc != xc || (has_cfill && c == cfill)) return;
            int pos = 0;                                    // the number of bounds <= xc
            for (int h = top; h > 0; h >>= 1)
                if (pos + h <= K + 1 && s_b[pos + h - 1] <= xc) pos += h;
            if (pos >= 1 && pos <= K) acc_j[(pos - 1) * kSectionBlock] = __dadd_rn(acc_j[(pos - 1) * kSectionBlock], f);
        };
        int k = 0;
        for (; k + UNROLL <= nz; k += UNROLL) {
            T x[UNROLL][4], ex[UNROLL][4], c[UNROLL];
#pragma unroll
            for (int q = 0; q < UNROLL; ++q) {
                section_load<T, E3>(pc, pe, (int64_t)(k + q) * ld, (int64_t)(k + q) * ld, x[q], ex[q]);
                c[q] = __ldg(pcl + (int64_t)(k + q) * ld);
            }
#pragma unroll
            for (int q = 0; q < UNROLL; ++q) level(k + q, x[q], ex[q], c[q]);
        }
        for (; k < nz; ++k) {
            T x[4], ex[4];
            section_load<T, E3>(pc, pe, (int64_t)k * ld, (int64_t)k * ld, x, ex);
            level(k, x, ex, __ldg(pcl + (int64_t)k * ld));
        }
    }
    __syncwarp();
    // lane l adds lane l + o for o = 16, 8, 4, 2, 1 (absent crossings hold +0): one value per (step, tile, class)
    double* out = partial + ((int64_t)blockIdx.y * ntiles + tile) * K;
    for (int j = 0; j < K; ++j) {
        double a = acc_j[j * kSectionBlock];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a = __dadd_rn(a, __shfl_down_sync(0xffffffffu, a, o));
        if (lane == 0) out[j] = a;
    }
}

// classes[t, j, m] = the tiles of transect m added in ascending order from +0 (partial: the steps from t0 on)
__global__ void k_reduce_class_tiles(const double* __restrict__ partial, int nt, int64_t ntiles, int K,
                                     const int64_t* __restrict__ tr_tiles, int ntransects, int64_t t0,
                                     double* __restrict__ classes) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)nt * ntransects * K) return;
    const int j = (int)(i % K);
    const int m = (int)(i / K % ntransects);
    const int64_t t = i / ((int64_t)K * ntransects);
    double a = 0.0;
    for (int64_t g = tr_tiles[m]; g < tr_tiles[m + 1]; ++g) a = __dadd_rn(a, partial[(t * ntiles + g) * K + j]);
    classes[((t0 + t) * K + j) * ntransects + m] = a;
}

// Tracer transport: the flux of every crossing weighted by a tracer tau (temperature, salinity...) taken at the C-grid
// face of each of its edges.  Face of edge e of crossing s in cell c (flux_index order S, E, N, W):
//   S: eV[south(c)], the T cells south(c) and c      E: eU[c], c and east(c)
//   N: eV[c], c and north(c) (none in the top row)   W: eU[west(c)], west(c) and c        (east / west x-periodic)
// At level k the face value q is 0.5 * (tau_a + tau_b) - ref with both sides present, tau_a - ref with one side, 0 with
// none (missing: NaN or the marker tfill, compared in the storage type).  Per layer and edge the thread sums
// A_e += (d_k * u_e,k) * q_e,k over the layer's levels in ascending order from +0 (d_k: dz, or e3u / e3v; u cleaned as
// in section_level) and turns the 4 sums into the crossing's value with section_value.  With tau == 1 and ref == 0,
// q == 1 and every term is the section's: the value is fluxSection's bit for bit.
// One thread per (time step, crossing) in the warp tiles of k_flux_classes; the lanes past the end of a tile run the
// tile's first crossing and count +0, so every lane reaches the shuffles.  Per level the thread gathers its 4 columns
// (section_load) and the tracer at 5 cells: c is shared by all 4 faces.  At a layer boundary it forms the value once,
// stores it to `section` (streaming) and / or folds the tile with the shuffle tree of k_flux_classes into
// partial[(step - t0, tile, layer)], which k_reduce_class_tiles adds up per transect (K = nlayers).
// levels in flight (9 loads per level, 13 with E3) and CTAs per SM: 122-128 registers, no spills; every shape with 3
// CTAs per SM (80 registers) spills, even with one level in flight (profiles/r8_tracer_ptxas.md)
template <typename T, bool E3>
struct TracerShape {
    static constexpr int unroll = E3 ? 1 : 3;
    static constexpr int ctas = 2;
};

// the face value q of a face between the T cells a and b (has_b false: no cell b)
template <typename T>
__device__ __forceinline__ double face_tracer(T a, T b, bool has_b, T tfill, int has_tfill, double ref) {
    const bool pa = !(a != a) && !(has_tfill && a == tfill);
    const bool pb = has_b && !(b != b) && !(has_tfill && b == tfill);
    if (pa && pb) return __dsub_rn(__dmul_rn(0.5, __dadd_rn((double)a, (double)b)), ref);
    if (pa) return __dsub_rn((double)a, ref);
    if (pb) return __dsub_rn((double)b, ref);
    return 0.0;
}

template <typename T, bool E3>
__global__ void __launch_bounds__(kSectionBlock, TracerShape<T, E3>::ctas)
k_flux_tracer(const T* __restrict__ u, const T* __restrict__ v, const T* __restrict__ e3u, const T* __restrict__ e3v,
              int64_t e3_tstride, const double* __restrict__ dz, const double* __restrict__ arc1,
              const double* __restrict__ arc2, const int32_t* __restrict__ idx, const double* __restrict__ w,
              const int32_t* __restrict__ cell, const T* __restrict__ tr, int64_t tr_tstride, T tfill, int has_tfill,
              double ref, const int64_t* __restrict__ tile_start, int64_t ntiles, int64_t nsub, int64_t ncell, int nx,
              int64_t ld, int nz, int nlayers, const int* __restrict__ levels, double scale, int use_scale, T fill,
              int has_fill, int64_t t0, double* __restrict__ section, double* __restrict__ partial) {
    constexpr int UNROLL = TracerShape<T, E3>::unroll;
    extern __shared__ double s_dz[];                        // [nz] dz (without E3), then [nlayers + 1] boundaries
    int* s_lev = reinterpret_cast<int*>(s_dz + (E3 ? 0 : nz));
    if constexpr (!E3)
        for (int k = threadIdx.x; k < nz; k += kSectionBlock) s_dz[k] = dz[k];
    for (int i = threadIdx.x; i <= nlayers; i += kSectionBlock)
        s_lev[i] = levels ? levels[i] : (i == 0 ? 0 : nz);  // levels == nullptr: one layer, the whole column
    __syncthreads();
    const int64_t tile = (int64_t)blockIdx.x * (kSectionBlock / 32) + threadIdx.x / 32;
    if (tile >= ntiles) return;                             // the whole warp
    const int lane = threadIdx.x & 31;
    const int64_t t = t0 + blockIdx.y;
    const int64_t s0 = tile_start[tile] + lane;
    const bool present = s0 < tile_start[tile + 1];
    const int64_t s = present ? s0 : tile_start[tile];
    const T* pc[4];
    const T* pe[4];
    double arc[4], wt[4], acc[4] = {0.0, 0.0, 0.0, 0.0};
    bool live[4];
    section_edges<T, E3>(u, v, e3u, e3v, arc1, arc2, idx, w, s, ncell, t * nz * ld, t * e3_tstride, pc, pe, arc, wt,
                         live);
    // the tracer at c and at its east, west, north and south neighbours (no north cell in the top row, no south cell in
    // row 0: c itself, a harmless address; the S edge of row 0 is not live)
    const int64_t c = cell[s];
    const int i = (int)(c % nx);
    const bool has_n = c + nx < ncell;
    const T* pt = tr + t * tr_tstride + c;
    const int64_t o_e = i + 1 < nx ? 1 : 1 - nx, o_w = i >= 1 ? -1 : nx - 1, o_n = has_n ? nx : 0,
                  o_s = c >= nx ? -(int64_t)nx : 0;
    double* sec = section ? section + (t * nlayers) * nsub + s : nullptr;
    double* part = partial ? partial + ((int64_t)blockIdx.y * ntiles + tile) * nlayers : nullptr;
    int layer = 0, next = s_lev[1];
    const int kend = s_lev[nlayers];
    int k = s_lev[0];
    // level kk into the 4 tracer-weighted column sums; after the last level of a layer: the value, stored and / or
    // folded over the tile (the layering is the same for every thread: the branch does not diverge)
    auto step = [&](int kk, const T (&x)[4], const T (&ex)[4], const T (&ta)[5]) {
        const double q[4] = {face_tracer<T>(ta[4], ta[0], true, tfill, has_tfill, ref),
                             face_tracer<T>(ta[0], ta[1], true, tfill, has_tfill, ref),
                             face_tracer<T>(ta[0], ta[3], has_n, tfill, has_tfill, ref),
                             face_tracer<T>(ta[2], ta[0], true, tfill, has_tfill, ref)};
        const double d = E3 ? 0.0 : s_dz[kk];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const double de = E3 ? clean<T>(ex[e], fill, has_fill) : d;
            acc[e] = __dadd_rn(acc[e], __dmul_rn(__dmul_rn(de, clean<T>(x[e], fill, has_fill)), q[e]));
        }
        if (kk + 1 == next) {
            const double r = section_value(acc, arc, wt, live, scale, use_scale);
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[e] = 0.0;
            if (sec && present) __stcs(sec + (int64_t)layer * nsub, r);
            if (part) {
                double a = present ? r : 0.0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) a = __dadd_rn(a, __shfl_down_sync(0xffffffffu, a, o));
                if (lane == 0) part[layer] = a;
            }
            ++layer;
            next = layer < nlayers ? s_lev[layer + 1] : -1;
        }
    };
    // the 5 tracer values of level kk: c, east, west, north, south
    auto load_tracer = [&](int kk, T (&ta)[5]) {
        const T* p = pt + (int64_t)kk * ld;
        ta[0] = __ldg(p);
        ta[1] = __ldg(p + o_e);
        ta[2] = __ldg(p + o_w);
        ta[3] = __ldg(p + o_n);
        ta[4] = __ldg(p + o_s);
    };
    for (; k + UNROLL <= kend; k += UNROLL) {
        T x[UNROLL][4], ex[UNROLL][4], ta[UNROLL][5];
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) {
            section_load<T, E3>(pc, pe, (int64_t)(k + q) * ld, (int64_t)(k + q) * ld, x[q], ex[q]);
            load_tracer(k + q, ta[q]);
        }
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) step(k + q, x[q], ex[q], ta[q]);
    }
    for (; k < kend; ++k) {
        T x[4], ex[4], ta[5];
        section_load<T, E3>(pc, pe, (int64_t)k * ld, (int64_t)k * ld, x, ex);
        load_tracer(k, ta);
        step(k, x, ex, ta);
    }
}

template <typename T, bool E3>
void launch_tracer(const void* u, const void* v, const void* e3u, const void* e3v, int64_t e3_tstride,
                   const double* dz, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                   const int32_t* cell, const void* tracer, int64_t tr_tstride, double tfill, double ref,
                   const int64_t* tile_start, int64_t ntiles, const int64_t* tr_tiles, int ntransects, int64_t nsub,
                   int64_t ncell, int nx, int64_t ld, int nt, int nz, int nlayers, const int* levels, int sverdrup,
                   double fill, double* partial, int partial_steps, double* series, double* section, cudaStream_t s) {
    const double scale = 6371000.0 / 1.e6;
    const size_t smem = (E3 ? 0 : sizeof(double) * nz) + sizeof(int) * (nlayers + 1);
    const unsigned gx = (unsigned)((ntiles + kSectionBlock / 32 - 1) / (kSectionBlock / 32));
    const int batch = series ? std::min(partial_steps, 65535) : 65535;
    for (int t0 = 0; t0 < nt; t0 += batch) {
        const int n = std::min(batch, nt - t0);
        k_flux_tracer<T, E3><<<dim3(gx, (unsigned)n), kSectionBlock, smem, s>>>(
            (const T*)u, (const T*)v, (const T*)e3u, (const T*)e3v, e3_tstride, dz, arc1, arc2, idx, w, cell,
            (const T*)tracer, tr_tstride, (T)tfill, !(tfill != tfill), ref, tile_start, ntiles, nsub, ncell, nx, ld, nz,
            nlayers, levels, scale, sverdrup, (T)fill, !(fill != fill), t0, section, series ? partial : nullptr);
        count_launch();
        NFX_CUDA(cudaGetLastError());
        if (!series) continue;
        const int64_t nr = (int64_t)n * ntransects * nlayers;
        k_reduce_class_tiles<<<(unsigned)((nr + 255) / 256), 256, 0, s>>>(partial, n, ntiles, nlayers, tr_tiles,
                                                                         ntransects, t0, series);
        count_launch();
        NFX_CUDA(cudaGetLastError());
    }
}

template <typename T, bool E3>
void launch_classes(const void* u, const void* v, const void* e3u, const void* e3v, int64_t e3_tstride,
                    const double* dz, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                    const int32_t* cell, const void* cfield, int64_t c_tstride, double cfill, const double* bounds,
                    int K, const int64_t* tile_start, int64_t ntiles, const int64_t* tr_tiles, int ntransects,
                    int64_t ncell, int64_t ld, int nt, int nz, int sverdrup, double fill, double* partial,
                    int partial_steps, double* classes, cudaStream_t s) {
    const double scale = 6371000.0 / 1.e6;
    const size_t smem = sizeof(double) * ((size_t)K * kSectionBlock + K + 1 + (E3 ? 0 : nz));
    NFX_CUDA(cudaFuncSetAttribute(k_flux_classes<T, E3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned gx = (unsigned)((ntiles + kSectionBlock / 32 - 1) / (kSectionBlock / 32));
    const int batch = std::min(partial_steps, 65535);
    for (int t0 = 0; t0 < nt; t0 += batch) {
        const int n = std::min(batch, nt - t0);
        k_flux_classes<T, E3><<<dim3(gx, (unsigned)n), kSectionBlock, smem, s>>>(
            (const T*)u, (const T*)v, (const T*)e3u, (const T*)e3v, e3_tstride, dz, arc1, arc2, idx, w, cell,
            (const T*)cfield, c_tstride, (T)cfill, !(cfill != cfill), bounds, K, tile_start, ntiles, ncell, ld, nz, scale,
            sverdrup, (T)fill, !(fill != fill), t0, partial);
        count_launch();
        NFX_CUDA(cudaGetLastError());
        const int64_t nr = (int64_t)n * ntransects * K;
        k_reduce_class_tiles<<<(unsigned)((nr + 255) / 256), 256, 0, s>>>(partial, n, ntiles, K, tr_tiles, ntransects,
                                                                         t0, classes);
        count_launch();
        NFX_CUDA(cudaGetLastError());
    }
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

void flux_classes(const void* u, const void* v, int dtype, const double* thickness, const void* e3u, const void* e3v,
                  int64_t e3_tstride, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                  const int32_t* cell, const void* cfield, int64_t c_tstride, double cfill, const double* bounds, int K,
                  const int64_t* tile_start, int64_t ntiles, const int64_t* tr_tiles, int ntransects, int64_t ncell,
                  int64_t ld, int nt, int nz, int sverdrup, double fill, double* partial, int partial_steps,
                  double* classes, cudaStream_t s) {
    NFX_REQUIRE(u && v && arc1 && arc2 && idx && w && cell && cfield && bounds && tile_start && tr_tiles && partial &&
                    classes, "classes: NULL pointer");
    NFX_REQUIRE((e3u == nullptr) == (e3v == nullptr) && (thickness != nullptr) != (e3u != nullptr),
                "classes: needs exactly one of thickness and (e3u, e3v)");
    NFX_REQUIRE(nz > 0 && nz <= 3000 && nt >= 0 && ld >= ncell && partial_steps >= 1, "classes: bad sizes");
    NFX_REQUIRE(K >= 1 && K <= kClassMax, "classes: K must be in [1, " + std::to_string(kClassMax) + "]");
    NFX_REQUIRE(ntiles / (kSectionBlock / 32) < 2147483647ll, "classes: too many sub-segments");
    if (nt == 0 || ntiles == 0) return;
    const bool e3 = e3u != nullptr;
#define NFX_CLASSES(T, E3)                                                                                            \
    launch_classes<T, E3>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, cell, cfield, c_tstride, cfill,  \
                          bounds, K, tile_start, ntiles, tr_tiles, ntransects, ncell, ld, nt, nz, sverdrup, fill,     \
                          partial, partial_steps, classes, s)
    if (dtype == NFX_F64) {
        if (e3)
            NFX_CLASSES(double, true);
        else
            NFX_CLASSES(double, false);
    } else {
        NFX_REQUIRE(dtype == NFX_F32, "classes: dtype must be NFX_F64 or NFX_F32");
        if (e3)
            NFX_CLASSES(float, true);
        else
            NFX_CLASSES(float, false);
    }
#undef NFX_CLASSES
}

void flux_tracer(const void* u, const void* v, int dtype, const double* thickness, const void* e3u, const void* e3v,
                 int64_t e3_tstride, const double* arc1, const double* arc2, const int32_t* idx, const double* w,
                 const int32_t* cell, const void* tracer, int64_t tr_tstride, double tfill, double ref,
                 const int64_t* tile_start, int64_t ntiles, const int64_t* tr_tiles, int ntransects, int64_t nsub,
                 int64_t ncell, int nx, int64_t ld, int nt, int nz, int nlayers, const int* levels, int sverdrup,
                 double fill, double* partial, int partial_steps, double* series, double* section, cudaStream_t s) {
    NFX_REQUIRE(u && v && arc1 && arc2 && idx && w && cell && tracer && tile_start && tr_tiles &&
                    (series || section) && (!series || partial), "tracer: NULL pointer");
    NFX_REQUIRE((e3u == nullptr) == (e3v == nullptr) && (thickness != nullptr) != (e3u != nullptr),
                "tracer: needs exactly one of thickness and (e3u, e3v)");
    NFX_REQUIRE(nz > 0 && nz <= 3000 && nt >= 0 && ld >= ncell && nx > 0 && ncell % nx == 0 && partial_steps >= 1,
                "tracer: bad sizes");
    NFX_REQUIRE(ntiles / (kSectionBlock / 32) < 2147483647ll, "tracer: too many sub-segments");
    if (nt == 0 || ntiles == 0) return;
    const bool e3 = e3u != nullptr;
#define NFX_TRACER(T, E3)                                                                                             \
    launch_tracer<T, E3>(u, v, e3u, e3v, e3_tstride, thickness, arc1, arc2, idx, w, cell, tracer, tr_tstride, tfill,  \
                         ref, tile_start, ntiles, tr_tiles, ntransects, nsub, ncell, nx, ld, nt, nz, nlayers, levels, \
                         sverdrup, fill, partial, partial_steps, series, section, s)
    if (dtype == NFX_F64) {
        if (e3)
            NFX_TRACER(double, true);
        else
            NFX_TRACER(double, false);
    } else {
        NFX_REQUIRE(dtype == NFX_F32, "tracer: dtype must be NFX_F64 or NFX_F32");
        if (e3)
            NFX_TRACER(float, true);
        else
            NFX_TRACER(float, false);
    }
#undef NFX_TRACER
}

}  // namespace nfx
