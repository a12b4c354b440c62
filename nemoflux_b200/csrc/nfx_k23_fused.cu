// K2+K3 fused, persistent: the whole flux time series in ONE launch, edge fluxes never reach HBM.
//
// Why: measured with tools/readbw.cu on a B200 the u/v stream alone runs at 7.47 TB/s, but writing the
// edge fluxes (1.3 % of the traffic) costs 10 % (DRAM read/write turnarounds), 5 % with evict-first stores,
// and 0.4 % when they go, with L2::evict_last, to a small ring that is overwritten while still in L2.  K3
// then gathers from L2 instead of HBM.  Cutting the work into batches launched one after the other loses
// more to launch tails than it wins (profiles/r1_fused_notes.md), hence one persistent kernel.
//
// Work is cut into batches b = (pseudo-step s, panel q of cells) whose (2, panel) slab of edge fluxes fits a
// ring slot; the ring has R slots.  A pseudo-step s = t * nlayers + i is time step t restricted to layer i, the
// levels [levels[i], levels[i+1]) (levels == nullptr: one layer, the whole column -- the plain series).
// Work items are handed out in a fixed global order by an atomic counter:
//     ... | K2 tiles of batch b (ntiles items) | K3 items of batch b-1 (nk3 items) | K2 tiles of b+1 | ...
// K2 item: z-sum over the layer's levels + metric factors for 256*VEC columns (field.py:145-163, 195-196, 225-228),
//          written to ring slot b % R; waits (b >= R) until K3 of batch b-R has finished reading that slot.
// K3 item: 8 sub-rows (<= 4096 CSR entries of one transect inside panel q) x batch b: one warp per sub-row gathers
//          from the slot (L2) and writes its partial sum; waits until all K2 tiles of batch b are done.
// The batches are visited panel-major (batch_map), so a panel's slice of the CSR stays in L2 across time steps.
// Every wait is on items with a SMALLER id, i.e. items already taken by a running CTA -> no deadlock, whatever
// the number of resident CTAs.  Spins are bounded; on overflow an error flag is raised instead of hanging.
//
// The per-column sums are the ones of nfx_k2_edgeflux.cu (bit-identical edge fluxes); the transect sums use the
// same lane-strided + shuffle-tree scheme as nfx_k3_reduce.cu on sub-rows, so the series agrees with the
// two-launch path to rounding (tested to 1e-13 of sum |w f|) and is deterministic run to run.
#include <algorithm>

#include "nfx_common.cuh"
#include "nfx_stream_ops.cuh"

namespace nfx {

int g_fused_f32_shape = 0;   // NFX_OPT_FUSED_F32_SHAPE (tuning knob)
int g_fused_f64_ctas = 0;    // NFX_OPT_FUSED_F64_CTAS (tuning knob): 2 or 4 resident CTAs per SM instead of 3
int g_fused_ring_max_mb = 0;  // NFX_OPT_RING_MAX_MB: upper bound of the whole ring (0 = 24 MB)
int g_fused_k3_lag = 0;      // NFX_OPT_FUSED_K3_LAG: 0 = automatic, else the lag of the K3 items in batches
int g_fused_order = 3;       // NFX_OPT_FUSED_ORDER: bit 0 = visit the batches panel-major, bit 1 = K3 gathers unrolled x8
                             // (same-box A/B, profiles/r1_fused_order_ab.md: -3 % and -1 % time on multi-panel grids)
int g_sparse_columns = 1;    // NFX_OPT_SPARSE_COLUMNS: 0 = dense, 1 = automatic, 2 = always sparse
int g_last_series_sparse = -1;   // NFX_OPT_LAST_SERIES_SPARSE (read only)
// automatic mode takes the sparse pass while its groups are less than this share of the panels' groups
constexpr double kSparseMaxShare = 0.8;

namespace {

using namespace dev;

constexpr int kFusedBlock = 256;
constexpr int kFusedF64Ctas = 3;   // float64 storage: 80 registers; -2.5 % time against 4 CTAs x 64 registers,
                                   // -6 % against 2 CTAs x 114 registers (profiles/r1_fused_ctas_ab.md)
constexpr int kWarps = kFusedBlock / 32;
constexpr unsigned kSpinLimit = 1u << 27;

struct FusedArgs {
    const void* u;
    const void* v;
    const void* e3u;        // E3 kernels: per-column, per-level scale factors (dtype and plane layout of u, v) ...
    const void* e3v;
    int64_t e3_tstride;     // ... elements per time step of e3u/e3v, 0 = time-invariant
    const double* dz;
    const double* arc1;
    const double* arc2;
    double* ring;           // ring_slots slots of slot_elems doubles: [eU(panel) | eV(panel)]
    double* out;            // (nt * nlayers, nsr) partial sums of the sub-rows
    const int64_t* sr_ptr;    // (nsr + 1) entry offsets of the sub-rows
    const int64_t* panel_sr;  // (npanels + 1) first sub-row of every panel
    int64_t nsr;
    const int32_t* idx;
    const double* w;
    int* sync;              // [0] work counter, [1] error flag, [2 .. 2+nb) K2 tiles done, [2+nb .. 2+2nb) K3 items done
    int64_t ncell, ld, panel, slot_elems;   // ld = cells per level plane in memory (>= ncell)
    int nt, nz, ntransects, npanels, nbatches, ntiles, nk3, ring_slots;
    const int* batch_map;   // (nbatches) global batch index s * npanels + q of the b-th batch visited
    const int32_t* grp;     // sparse pass: PanelPlan::grp (column groups of VEC the K2 tiles load), nullptr = dense
    const int64_t* grp_ptr;
    int k3_lag;             // the K3 items of batch b - k3_lag are queued behind the K2 tiles of batch b
    int k3_unroll8;
    double scale, fill;
    int use_scale, has_fill;
    const int* levels;      // (nlayers + 1) ascending level boundaries, nullptr = one layer [0, nz)
    int nlayers;
};

__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// thread 0 spins until *flag >= target, then the CTA continues; returns false on overflow (error raised)
__device__ __forceinline__ bool cta_wait(const int* flag, int target, int* err, int* s_ok) {
    if (threadIdx.x == 0) {
        unsigned spins = 0;
        int ok = 1;
        while (ld_acquire(flag) < target) {
            __nanosleep(64);
            if (++spins > kSpinLimit || ld_acquire(err) != 0) {
                atomicExch(err, 1);
                ok = 0;
                break;
            }
        }
        *s_ok = ok;
    }
    __syncthreads();
    const bool ok = *s_ok != 0;
    __syncthreads();
    return ok;
}

// resident CTAs per SM the register allocation is bounded for (0 = the default of the shape)
template <typename T, int VEC, int UNROLL, bool E3 = false>
constexpr int fused_min_ctas(int wanted) {
    if (wanted > 0) return wanted;
    if (E3) return 3;   // four streams: 80 registers hold the loads of a batch without spilling
    if (sizeof(T) == 4) return (VEC == 8 && UNROLL == 5) ? 3 : 4;
    return kFusedF64Ctas;
}

// E3: e3u[t,k,c] / e3v[t,k,c] replace the 1-D thickness dz[k] (SURVEY 8f rank 4), the arithmetic of
// k2_edgeflux_ldg<..., E3 = true> (nfx_k2_edgeflux.cu) operation for operation -> the same edge fluxes bit for bit
// LAYERED: the batches are (pseudo-step, panel) pairs and the K2 tiles sum the levels of the pseudo-step's layer; a
// template flag, so that the whole-column instances (levels == nullptr) keep their registers
template <typename T, int VEC, int UNROLL, int CTAS = 0, bool E3 = false, bool LAYERED = false>
__global__ void __launch_bounds__(kFusedBlock, fused_min_ctas<T, VEC, UNROLL, E3>(CTAS))
k23_fused(const FusedArgs a) {
    extern __shared__ double s_dz[];
    __shared__ int s_item;
    __shared__ int s_ok;
    // float32 storage: levels go through clean_scaled() (nfx_stream_ops.cuh) with dz * 2^896 in s_dz[nz..2nz)
    constexpr bool kScaled = sizeof(T) == 4;
    int big = 0;
    if constexpr (!E3) {
        for (int k = threadIdx.x; k < a.nz; k += kFusedBlock) {
            const double d = a.dz[k];
            s_dz[k] = d;
            if constexpr (kScaled) {
                s_dz[a.nz + k] = d * kScaleUp;
                big |= !(fabs(d) < kScaleLimit);
            }
        }
    }
    const bool redo_all = __syncthreads_or(big) != 0;
    using P = Pack<T, VEC>;
    using V = typename P::type;
    const T* __restrict__ u = reinterpret_cast<const T*>(a.u);
    const T* __restrict__ v = reinterpret_cast<const T*>(a.v);
    const T* __restrict__ e3u = reinterpret_cast<const T*>(a.e3u);
    const T* __restrict__ e3v = reinterpret_cast<const T*>(a.e3v);
    int* counter = a.sync;
    int* err = a.sync + 1;
    int* k2done = a.sync + 2;
    int* k3done = a.sync + 2 + a.nbatches;
    const int per_batch = a.ntiles + a.nk3;
    const int64_t nitems = (int64_t)(a.nbatches + a.k3_lag) * per_batch;
    const uint64_t pol = l2_evict_last_policy();
    const uint64_t pol_ef = l2_evict_first_policy();
    const T fill = (T)a.fill;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;

    // Tried and dropped (same-box A/B, profiles/r1_fused_notes.md): fetching the next item id while the current
    // item runs (a K3 item parked behind a K2 tile delays the release of its ring slot: +20 % time at ORCA1
    // size, +3 % at ORCA12 size) and items of two column groups (+10 % time on large grids).
    for (;;) {
        if (threadIdx.x == 0) s_item = atomicAdd(counter, 1);
        __syncthreads();
        const int64_t item = s_item;
        __syncthreads();
        if (item >= nitems) break;
        const int bb = (int)(item / per_batch);
        const int r = (int)(item - (int64_t)bb * per_batch);
        if (r < a.ntiles) {
            // ------------------------------- K2 tile of batch bb -------------------------------
            const int b = bb;
            if (b >= a.nbatches) continue;
            if (b >= a.ring_slots && !cta_wait(k3done + (b - a.ring_slots), a.nk3, err, &s_ok)) break;
            const int gb = a.batch_map[b];
            const int64_t ps = gb / a.npanels;
            const int q = gb - (int)ps * a.npanels;
            // layered: the sums of the whole column with dz (e3) zeroed outside the layer
            const int64_t t = LAYERED ? ps / a.nlayers : ps;
            const int kbeg = LAYERED ? a.levels[ps - t * a.nlayers] : 0;
            const int kend = LAYERED ? a.levels[ps - t * a.nlayers + 1] : a.nz;
            const int64_t pc0 = (int64_t)q * a.panel;
            const int64_t pc = min(a.panel, a.ncell - pc0);
            int64_t cl = ((int64_t)r * kFusedBlock + threadIdx.x) * VEC;   // column inside the panel
            if (a.grp) {   // sparse: the r-th 256 groups of the panel's list; a tile past its end loads nothing
                const int64_t gi = a.grp_ptr[q] + (int64_t)r * kFusedBlock + threadIdx.x;
                cl = gi < a.grp_ptr[q + 1] ? (int64_t)a.grp[gi] * VEC : pc;
            }
            if (cl < pc) {
                const int64_t c = pc0 + cl;
                const T* pu = u + t * a.nz * a.ld + c;
                const T* pv = v + t * a.nz * a.ld + c;
                const T* pe = E3 ? e3u + t * a.e3_tstride + c : nullptr;
                const T* pf = E3 ? e3v + t * a.e3_tstride + c : nullptr;
                double su[VEC], sv[VEC];
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    su[e] = 0.0;
                    sv[e] = 0.0;
                }
                float amax = 0.f;
                int k = kbeg;
                for (; k + UNROLL <= kend; k += UNROLL) {
                    V ru[UNROLL], rv[UNROLL], re[E3 ? UNROLL : 1], rf[E3 ? UNROLL : 1];
#pragma unroll
                    for (int qq = 0; qq < UNROLL; ++qq) {
                        ru[qq] = ld_stream(reinterpret_cast<const V*>(pu + (int64_t)(k + qq) * a.ld), pol_ef);
                        rv[qq] = ld_stream(reinterpret_cast<const V*>(pv + (int64_t)(k + qq) * a.ld), pol_ef);
                        if constexpr (E3) {
                            re[qq] = ld_stream(reinterpret_cast<const V*>(pe + (int64_t)(k + qq) * a.ld), pol_ef);
                            rf[qq] = ld_stream(reinterpret_cast<const V*>(pf + (int64_t)(k + qq) * a.ld), pol_ef);
                        }
                    }
#pragma unroll
                    for (int qq = 0; qq < UNROLL; ++qq) {
                        pin(ru[qq]);
                        pin(rv[qq]);
                        if constexpr (E3) {
                            pin(re[qq]);
                            pin(rf[qq]);
                        }
                    }
#pragma unroll
                    for (int qq = 0; qq < UNROLL; ++qq) {
                        T x[VEC], y[VEC], ex[VEC], ey[VEC];
                        P::unpack(ru[qq], x);
                        P::unpack(rv[qq], y);
                        if constexpr (E3) {
                            P::unpack(re[qq], ex);
                            P::unpack(rf[qq], ey);
                        }
                        const double d = E3 ? 0.0 : s_dz[(kScaled ? a.nz : 0) + k + qq];
#pragma unroll
                        for (int e = 0; e < VEC; ++e) {
                            if constexpr (kScaled && E3) {
                                // both factors come from float32: undo the 2^-896 of each bit shuffle exactly
                                const double du = __dmul_rn(clean_scaled(ex[e], fill, a.has_fill, amax), kScaleUp);
                                const double dv = __dmul_rn(clean_scaled(ey[e], fill, a.has_fill, amax), kScaleUp);
                                const double xu = __dmul_rn(clean_scaled(x[e], fill, a.has_fill, amax), kScaleUp);
                                const double xv = __dmul_rn(clean_scaled(y[e], fill, a.has_fill, amax), kScaleUp);
                                su[e] = __dadd_rn(su[e], __dmul_rn(du, xu));
                                sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, xv));
                            } else if constexpr (kScaled) {
                                su[e] = __dadd_rn(su[e], __dmul_rn(d, clean_scaled(x[e], fill, a.has_fill, amax)));
                                sv[e] = __dadd_rn(sv[e], __dmul_rn(d, clean_scaled(y[e], fill, a.has_fill, amax)));
                            } else {
                                const double du = E3 ? clean<T>(ex[e], fill, a.has_fill) : d;
                                const double dv = E3 ? clean<T>(ey[e], fill, a.has_fill) : d;
                                su[e] = __dadd_rn(su[e], __dmul_rn(du, clean<T>(x[e], fill, a.has_fill)));
                                sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean<T>(y[e], fill, a.has_fill)));
                            }
                        }
                    }
                }
                for (; k < kend; ++k) {
                    T x[VEC], y[VEC], ex[VEC], ey[VEC];
                    P::unpack(ld_stream(reinterpret_cast<const V*>(pu + (int64_t)k * a.ld), pol_ef), x);
                    P::unpack(ld_stream(reinterpret_cast<const V*>(pv + (int64_t)k * a.ld), pol_ef), y);
                    if constexpr (E3) {
                        P::unpack(ld_stream(reinterpret_cast<const V*>(pe + (int64_t)k * a.ld), pol_ef), ex);
                        P::unpack(ld_stream(reinterpret_cast<const V*>(pf + (int64_t)k * a.ld), pol_ef), ey);
                    }
                    const double d = E3 ? 0.0 : s_dz[k];
#pragma unroll
                    for (int e = 0; e < VEC; ++e) {
                        const double du = E3 ? clean<T>(ex[e], fill, a.has_fill) : d;
                        const double dv = E3 ? clean<T>(ey[e], fill, a.has_fill) : d;
                        su[e] = __dadd_rn(su[e], __dmul_rn(du, clean<T>(x[e], fill, a.has_fill)));
                        sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean<T>(y[e], fill, a.has_fill)));
                    }
                }
                if constexpr (kScaled) {
                    if (redo_all || !(amax <= 3.402823466e38f)) {   // rare: an infinity in this thread's columns
#pragma unroll
                        for (int e = 0; e < VEC; ++e) {
                            su[e] = 0.0;
                            sv[e] = 0.0;
                        }
#pragma unroll 1
                        for (int kk = kbeg; kk < kend; ++kk) {
                            const double d = E3 ? 0.0 : s_dz[kk];
#pragma unroll
                            for (int e = 0; e < VEC; ++e) {
                                const double du = E3 ? clean<T>(pe[(int64_t)kk * a.ld + e], fill, a.has_fill) : d;
                                const double dv = E3 ? clean<T>(pf[(int64_t)kk * a.ld + e], fill, a.has_fill) : d;
                                su[e] = __dadd_rn(su[e], __dmul_rn(du, clean<T>(pu[(int64_t)kk * a.ld + e], fill, a.has_fill)));
                                sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean<T>(pv[(int64_t)kk * a.ld + e], fill, a.has_fill)));
                            }
                        }
                    }
                }
                double* ou = a.ring + (int64_t)(b % a.ring_slots) * a.slot_elems + cl;
                double* ov = ou + pc;
                const int nvalid = (int)min((int64_t)VEC, pc - cl);   // the last vector may hang over the panel end
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    if (e < nvalid) {
                        double fu = __dmul_rn(su[e], a.arc1[c + e]);
                        double fv = __dmul_rn(-sv[e], a.arc2[c + e]);
                        if (a.use_scale) {
                            fu = __dmul_rn(fu, a.scale);
                            fv = __dmul_rn(fv, a.scale);
                        }
                        su[e] = fu;
                        sv[e] = fv;
                    }
                }
                const bool pair_ok = (VEC % 2 == 0) && ((pc & 1) == 0) && ((a.slot_elems & 1) == 0);
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    if (pair_ok && (e % 2 == 0) && e + 1 < nvalid) {
                        st_stream2(ou + e, su[e], su[e + 1 < VEC ? e + 1 : e], 1, pol);
                        st_stream2(ov + e, sv[e], sv[e + 1 < VEC ? e + 1 : e], 1, pol);
                    } else if (e < nvalid && !(pair_ok && (e % 2 == 1))) {
                        st_stream1(ou + e, su[e], 1, pol);
                        st_stream1(ov + e, sv[e], 1, pol);
                    }
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {   // the barrier orders the CTA's stores before this fence (cumulativity)
                __threadfence();
                atomicAdd(k2done + b, 1);
            }
        } else {
            // ------------------------- K3 item of batch bb - k3_lag -------------------------
            // queued far enough behind the batch's K2 tiles that they are done when a CTA takes the item: with a lag
            // of 1 a CTA that took a K3 item sat idle until the slowest tile of the batch before finished (-4 % with
            // float32 storage, where the K3 items of a time step weigh twice as much against its K2 tiles)
            const int b = bb - a.k3_lag;
            if (b < 0 || b >= a.nbatches) continue;
            if (!cta_wait(k2done + b, a.ntiles, err, &s_ok)) break;
            __threadfence();
            const int gb = a.batch_map[b];
            const int64_t ps = gb / a.npanels;
            const int q = gb - (int)ps * a.npanels;
            {
                // one warp per sub-row (<= kSubRow entries): lane-strided partial sums, fixed shuffle tree
                const int64_t sr = a.panel_sr[q] + (int64_t)(r - a.ntiles) * kWarps + wid;
                if (sr < a.panel_sr[q + 1]) {
                    const int64_t r0 = a.sr_ptr[sr], r1 = a.sr_ptr[sr + 1];
                    const double* d = a.ring + (int64_t)(b % a.ring_slots) * a.slot_elems;
                    double acc = 0.0;
                    if (a.k3_unroll8) {
#pragma unroll 8
                        for (int64_t n = r0 + lane; n < r1; n += 32) acc = fma(a.w[n], __ldcg(d + a.idx[n]), acc);
                    } else {
#pragma unroll 4
                        for (int64_t n = r0 + lane; n < r1; n += 32) acc = fma(a.w[n], __ldcg(d + a.idx[n]), acc);
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                    if (lane == 0) a.out[ps * a.nsr + sr] = acc;
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                atomicAdd(k3done + b, 1);
            }
        }
    }
}


__global__ void k_or_flag(const int* flag, int* sticky) {
    if (*flag != 0) *sticky = 1;
}

// dynamic shared memory of the launch being prepared (2 * nz doubles): the occupancy query uses the real size; the
// answer is cached per device for the common case (nz <= 128, where registers, not shared memory, bound the occupancy)
thread_local size_t t_fused_smem = sizeof(double) * 256;

template <typename T, int VEC, int UNROLL, int CTAS = 0, bool E3 = false, bool LAYERED = false>
int fused_grid() {
    static int grid[64] = {0};   // per device ordinal
    int dev = 0;
    NFX_CUDA(cudaGetDevice(&dev));
    const bool small = t_fused_smem <= sizeof(double) * 256;
    int& g = grid[dev & 63];
    if (g == 0 || !small) {
        int sms = 0, per_sm = 0;
        NFX_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        NFX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k23_fused<T, VEC, UNROLL, CTAS, E3, LAYERED>, kFusedBlock,
                                                               std::max(t_fused_smem, sizeof(double) * 256)));
        const int n = sms * std::max(per_sm, 1);
        if (!small) return n;
        g = n;
    }
    return g;
}

template <typename T, int VEC, int UNROLL, int CTAS = 0, bool E3 = false>
void launch_fused(const FusedArgs& a, cudaStream_t s) {
    if (a.levels)
        k23_fused<T, VEC, UNROLL, CTAS, E3, true>
            <<<fused_grid<T, VEC, UNROLL, CTAS, E3, true>(), kFusedBlock, sizeof(double) * a.nz * 2, s>>>(a);
    else
        k23_fused<T, VEC, UNROLL, CTAS, E3>
            <<<fused_grid<T, VEC, UNROLL, CTAS, E3>(), kFusedBlock, sizeof(double) * a.nz * 2, s>>>(a);
}

// e3u/e3v kernels: four streamed arrays, so half the columns per thread of the thickness kernels keep the same
// number of loads in flight at the same register budget (float64: 2 columns x 5 levels, float32: 4 x 3)
int fused_grid_e3(int dtype, int vec) {
    if (dtype == NFX_F64) return vec == 2 ? fused_grid<double, 2, 5, 0, true>() : fused_grid<double, 1, 5, 0, true>();
    return vec == 4 ? fused_grid<float, 4, 3, 0, true>() : fused_grid<float, 1, 5, 0, true>();
}

int fused_grid_for(int dtype, int vec, int unroll, int ctas) {
    if (dtype == NFX_F64) {
        if (vec == 4) return ctas == 2 ? fused_grid<double, 4, 5, 2>() : ctas == 4 ? fused_grid<double, 4, 5, 4>() : fused_grid<double, 4, 5>();
        return vec == 2 ? fused_grid<double, 2, 5>() : fused_grid<double, 1, 5>();
    }
    if (unroll == 3) return vec == 8 ? fused_grid<float, 8, 3>() : fused_grid<float, 4, 3>();
    if (vec == 4 && ctas == 3) return fused_grid<float, 4, 5, 3>();
    return vec == 8 ? fused_grid<float, 8, 5>() : vec == 4 ? fused_grid<float, 4, 5>() : fused_grid<float, 1, 5>();
}

}  // namespace

// warps per CSR row from the mean row length: short rows -> one warp each (8 rows per CTA), long rows -> the CTA
int k3_group_for(int64_t nnz, int64_t nrows) {
    const int64_t avg = nrows > 0 ? nnz / nrows : 0;
    return avg >= 4096 ? 8 : avg >= 1024 ? 4 : avg >= 256 ? 2 : 1;
}

int fused_tile_columns(int dtype, const void* u, const void* v, int64_t ncell, int64_t ld, int64_t panel,
                       uintptr_t more_bits) {
    // widest vector the alignment of every level row and panel start allows (more_bits: further base addresses)
    const uintptr_t bits = ((uintptr_t)u) | ((uintptr_t)v) | more_bits;
    const bool a16 = (bits & 15) == 0, a32 = (bits & 31) == 0;
    // rows start at multiples of ld, panels at multiples of `panel`; the last panel ends at ncell
    // (a vector may hang over the end of the last panel when the plane is padded: ld >= ncell rounded up)
    auto fits = [&](int64_t vec) {
        return ld % vec == 0 && (panel % vec == 0 || panel == ncell) && (ncell % vec == 0 || ld >= (ncell + vec - 1) / vec * vec);
    };
    if (dtype == NFX_F64) {
        if (a32 && fits(4)) return 4;
        if (a16 && fits(2)) return 2;
        return 1;
    }
    if (a32 && fits(8)) return 8;
    if (a16 && fits(4)) return 4;
    return 1;
}

void flux_series_fused(PliDev& p, PanelPlan& pl, const void* u, const void* v, int dtype, const double* thickness,
                       const double* arc1, const double* arc2, int nt, int nz, int64_t ld, int sverdrup, double fill,
                       int64_t batch_begin, int64_t batch_end, double* out, cudaStream_t s, const void* e3u,
                       const void* e3v, int64_t e3_tstride, int nlayers, const int* levels) {
    const int64_t ncell = p.grid->ncell;
    const int M = p.ntransects;
    const bool e3 = e3u != nullptr;
    NFX_REQUIRE((e3u == nullptr) == (e3v == nullptr), "fused pass: e3u and e3v go together");
    NFX_REQUIRE(thickness || e3, "fused pass: needs the layer thickness or e3u/e3v");
    int vec = fused_tile_columns(dtype, u, v, ncell, ld, pl.panel_cells,
                                 (uintptr_t)e3u | (uintptr_t)e3v | (uintptr_t)(e3_tstride * (dtype == NFX_F64 ? 8 : 4)));
    int unroll = 5;
    if (e3) {
        vec = dtype == NFX_F64 ? std::min(vec, 2) : (vec >= 4 ? 4 : 1);
        unroll = (dtype != NFX_F64 && vec == 4) ? 3 : 5;
    } else if (dtype != NFX_F64 && vec >= 4) {
        // float32 storage: 128-bit loads x 5 levels at 64 registers (4 CTAs per SM) beat 256-bit loads at 80
        // registers (3 CTAs per SM) by 20 % (profiles/r1_f32_alu_sweep.md); the option is a tuning knob
        const int shape = g_fused_f32_shape > 0 ? g_fused_f32_shape : 45;   // 10 * vector width + unroll
        vec = std::min(vec, shape / 10 >= 8 ? 8 : 4);
        unroll = shape % 10 == 3 ? 3 : 5;
    }
    FusedArgs a;
    a.u = u;
    a.v = v;
    a.e3u = e3u;
    a.e3v = e3v;
    a.e3_tstride = e3_tstride;
    a.dz = thickness;
    a.arc1 = arc1;
    a.arc2 = arc2;
    a.ncell = ncell;
    a.ld = ld;
    a.panel = pl.panel_cells;
    a.slot_elems = 2 * std::min(pl.panel_cells, ncell);
    a.nt = nt;
    a.nz = nz;
    a.nlayers = nlayers;
    a.levels = levels;
    NFX_REQUIRE(nlayers >= 1 && (levels != nullptr || nlayers == 1), "fused pass: bad layering");
    const int64_t nps = (int64_t)nt * nlayers;   // pseudo-steps (t, layer)
    a.ntransects = M;
    a.npanels = pl.npanels;
    NFX_REQUIRE(batch_begin >= 0 && batch_begin <= batch_end && batch_end <= nps * pl.npanels,
                "fused pass: bad batch range");
    a.nbatches = (int)(batch_end - batch_begin);
    a.k3_unroll8 = (g_fused_order >> 1) & 1;
    // sparse pass: the K2 tiles walk the plan's column groups, i.e. only the vectors of u, v whose edge fluxes a K3 item
    // reads.  Every edge flux K3 reads is computed as in the dense pass: the series is the same bit for bit.
    bool sparse = false;
    if (g_sparse_columns != 0) {
        if (pl.grp_vec != vec) build_column_groups(pl, ncell, M, vec, s);
        sparse = g_sparse_columns == 2 || (double)pl.ngroups < kSparseMaxShare * (double)pl.ngroups_all;
    }
    g_last_series_sparse = sparse ? 1 : 0;
    a.grp = sparse ? pl.grp.p : nullptr;
    a.grp_ptr = sparse ? pl.grp_ptr.p : nullptr;
    const int64_t item_cols = (int64_t)kFusedBlock * vec;
    a.ntiles = sparse ? std::max(1, (pl.max_grp_per_panel + kFusedBlock - 1) / kFusedBlock)
                      : (int)((std::min(pl.panel_cells, ncell) + item_cols - 1) / item_cols);
    a.nk3 = std::max(1, (pl.max_sr_per_panel + kWarps - 1) / kWarps);
    a.scale = 6371000.0 / 1.e6;
    a.fill = fill;
    a.use_scale = sverdrup;
    a.has_fill = !(fill != fill);
    a.sr_ptr = pl.sr_ptr.p;
    a.panel_sr = pl.panel_sr.p;
    a.nsr = pl.nsr;
    a.idx = pl.idx.p;
    a.w = pl.w.p;
    a.out = out;
    NFX_REQUIRE(nz <= 3000, "edgeflux: at most 3000 levels (dz and dz * 2^896 live in 48 KB of shared memory)");
    NFX_REQUIRE((int64_t)(a.nbatches + 64) * (a.ntiles + a.nk3) < 2000000000ll, "fused pass: too many work items");
    // enough slots that every resident CTA finds a K2 tile while the K3 of older batches drains (x2 margin),
    // but no more than ring_max of evict-last lines in the 126 MB L2
    int ctas = 0;   // 0 = the default register budget of the shape
    if (dtype == NFX_F64 && vec == 4 && (g_fused_f64_ctas == 2 || g_fused_f64_ctas == 4)) ctas = g_fused_f64_ctas;
    if (dtype != NFX_F64 && vec == 4 && unroll == 5 && g_fused_f64_ctas == 3) ctas = 3;
    t_fused_smem = sizeof(double) * (size_t)nz * 2;
    const int resident = e3 ? fused_grid_e3(dtype, vec) : fused_grid_for(dtype, vec, unroll, ctas);
    int slots = (2 * resident + a.ntiles - 1) / a.ntiles + 1;
    // the whole ring stays under 24 MB: beyond that (32 MB: float32 storage on ORCA12, 4 slots of 8 MB) L2 starts writing
    // the evict-last lines back to HBM -- ncu: 228 MB of DRAM writes per 2 time steps -- and the pass loses 2.5 %
    // (profiles/r2_fused_experiments.md)
    const int64_t ring_max = (int64_t)(g_fused_ring_max_mb > 0 ? g_fused_ring_max_mb : 24) << 20;
    const int64_t cap = std::max<int64_t>(3, ring_max / (a.slot_elems * 8));
    slots = (int)std::min<int64_t>(std::max(slots, 3), cap);
    // lag of the K3 items.  One-panel grids (a batch = a whole time step, fewer tiles than resident CTAs): the batches
    // the resident CTAs span + 1, so that a batch's tiles have all FINISHED, not just been handed out, when its K3
    // items come up (same-box A/B, profiles/r2_fused_experiments.md: ORCA1 float32 +2.8..3.8 %, float64 +-0).  Grids
    // of several panels keep 1: a longer lag means more live ring slots, and there it costs 2 %.  The ring must hold
    // the batches in between (slots > lag).
    int lag = g_fused_k3_lag > 0 ? g_fused_k3_lag : pl.npanels == 1 ? (resident + a.ntiles - 1) / a.ntiles + 1 : 1;
    lag = (int)std::max<int64_t>(1, std::min<int64_t>(lag, cap - 2));
    slots = (int)std::min<int64_t>(std::max(slots, lag + 2), cap);
    a.k3_lag = lag;
    a.ring_slots = slots;
    p.ring.ensure((size_t)(a.slot_elems * slots));
    NFX_CUDA(cudaMemsetAsync(out, 0xFF, sizeof(double) * (size_t)nps * std::max<int64_t>(pl.nsr, 1), s));   // NaN: a pass that
    // aborts (bounded spin overflow) must not leave plausible numbers behind.  Sub-rows of batches outside
    // [batch_begin, batch_end) belong to other ranks: they contribute 0 here.
    if (pl.nsr > 0) {
        auto zero_rows = [&](int64_t b0, int64_t b1) {   // batches [b0, b1) -> contiguous runs of sub-rows per pseudo-step
            while (b0 < b1) {
                const int64_t t = b0 / pl.npanels, q0 = b0 - t * pl.npanels;
                const int64_t q1 = std::min<int64_t>(pl.npanels, q0 + (b1 - b0));
                const int64_t r0 = pl.h_panel_sr[q0], r1 = pl.h_panel_sr[q1];
                if (r1 > r0)
                    NFX_CUDA(cudaMemsetAsync(out + t * pl.nsr + r0, 0, sizeof(double) * (size_t)(r1 - r0), s));
                b0 += q1 - q0;
            }
        };
        zero_rows(0, batch_begin);
        zero_rows(batch_end, nps * pl.npanels);
    }
    if (a.nbatches == 0) return;
    {
        // visiting order of the batches.  Time-major: (t, q) as numbered.  Panel-major: all local time steps of
        // panel 0, then of panel 1, ... -- the panel's slice of the CSR (weights, indices) and of the metric
        // arrays is reused from L2 for every time step instead of being re-read from HBM once per step.
        const int order = g_fused_order & 1;
        const int64_t key[4] = {batch_begin, batch_end, pl.npanels, order};
        if (!std::equal(key, key + 4, p.batch_map_key) || p.batch_map.p == nullptr) {
            p.h_batch_map.resize((size_t)a.nbatches);
            for (int b = 0; b < a.nbatches; ++b) p.h_batch_map[(size_t)b] = (int)(batch_begin + b);
            if (order == 1 && pl.npanels > 1) {
                const int np = pl.npanels;
                std::stable_sort(p.h_batch_map.begin(), p.h_batch_map.end(),
                                 [np](int x, int y) { return x % np < y % np; });
            }
            p.batch_map.ensure((size_t)a.nbatches);
            NFX_CUDA(cudaMemcpyAsync(p.batch_map.p, p.h_batch_map.data(), sizeof(int) * (size_t)a.nbatches,
                                     cudaMemcpyHostToDevice, s));
            std::copy(key, key + 4, p.batch_map_key);
        }
        a.batch_map = p.batch_map.p;
    }
    p.fused_sync.ensure((size_t)(2 + 2 * a.nbatches));
    a.ring = p.ring.p;
    a.sync = p.fused_sync.p;
    NFX_CUDA(cudaMemsetAsync(a.sync, 0, sizeof(int) * (2 + 2 * a.nbatches), s));
    if (e3) {
        if (dtype == NFX_F64) {
            if (vec == 2) launch_fused<double, 2, 5, 0, true>(a, s);
            else launch_fused<double, 1, 5, 0, true>(a, s);
        } else {
            if (vec == 4) launch_fused<float, 4, 3, 0, true>(a, s);
            else launch_fused<float, 1, 5, 0, true>(a, s);
        }
    } else if (dtype == NFX_F64) {
        if (vec == 4 && ctas == 2) launch_fused<double, 4, 5, 2>(a, s);
        else if (vec == 4 && ctas == 4) launch_fused<double, 4, 5, 4>(a, s);
        else if (vec == 4) launch_fused<double, 4, 5>(a, s);
        else if (vec == 2) launch_fused<double, 2, 5>(a, s);
        else launch_fused<double, 1, 5>(a, s);
    } else {
        if (unroll == 3 && vec == 8) launch_fused<float, 8, 3>(a, s);
        else if (unroll == 3 && vec == 4) launch_fused<float, 4, 3>(a, s);
        else if (vec == 8) launch_fused<float, 8, 5>(a, s);
        else if (vec == 4 && ctas == 3) launch_fused<float, 4, 5, 3>(a, s);
        else if (vec == 4) launch_fused<float, 4, 5>(a, s);
        else launch_fused<float, 1, 5>(a, s);
    }
    count_launch();
    NFX_CUDA(cudaGetLastError());
    // the error flag travels to a pinned word behind the pass: the next call on the handle (or nfx_pli_series_status)
    // reports an aborted pass instead of handing back NaN with return code 0.  k_or_flag keeps it sticky.
    if (!p.h_fused_err) {
        NFX_CUDA(cudaHostAlloc((void**)&p.h_fused_err, sizeof(int), cudaHostAllocDefault));
        *p.h_fused_err = 0;
        p.fused_sticky_buf.alloc(1);
        NFX_CUDA(cudaMemsetAsync(p.fused_sticky_buf.p, 0, sizeof(int), s));
    }
    k_or_flag<<<1, 1, 0, s>>>(a.sync + 1, p.fused_sticky_buf.p);
    count_launch();
    NFX_CUDA(cudaMemcpyAsync(p.h_fused_err, p.fused_sticky_buf.p, sizeof(int), cudaMemcpyDeviceToHost, s));
}

void fused_check_sticky_error(PliDev& p) {
    if (p.h_fused_err && *(volatile int*)p.h_fused_err != 0) {
        *(volatile int*)p.h_fused_err = 0;
        if (p.fused_sticky_buf.p) cudaMemset(p.fused_sticky_buf.p, 0, sizeof(int));
        throw Error(NFX_E_INTERNAL, "a fused K2+K3 pass launched earlier on this handle aborted (a bounded wait "
                                    "overflowed): its flux series is NaN");
    }
}

// error flag of the last fused pass (1 = a bounded spin overflowed); synchronises the stream
int fused_error_flag(PliDev& p, cudaStream_t s) {
    int h[2] = {0, 0};
    if (!p.fused_sync.p) return 0;
    NFX_CUDA(cudaMemcpyAsync(h, p.fused_sync.p, sizeof h, cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaStreamSynchronize(s));
    return h[1];
}

}  // namespace nfx
