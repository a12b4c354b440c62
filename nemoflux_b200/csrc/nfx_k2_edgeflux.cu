// K2: C-grid edge-flux assembly (sm_100a), HBM-bound streaming kernel.
//
// Replaces Field.readField (NaN -> 0, sum over z of thickness*field, /root/reference/nemoflux/
// field.py:145-163) and Field.computeIntegratedFlux (eU = +U*arc1, eV = -V*arc2, optional Sverdrup
// factor, field.py:183-228) for ALL time steps of a chunk in one launch.
//
//   eflux[t, c]         = (sum_k dz[k]*u[t,k,c]) * arc1[c] (* 6.371)
//   eflux[t, ncell + c] = -(sum_k dz[k]*v[t,k,c]) * arc2[c] (* 6.371)
//
// The (ncell,4) array of field.py:209-223 is NOT materialised on the fast path: K1 remaps
// (cell, edge) to an index into this compact [eU | eV] layout.  nfx_edgeflux_to_cell_by_cell builds
// it on request for the mint-style getIntegral(data) call.
//
// The z-sum runs k = 0..nz-1 per column with separate multiply and add (no FMA), fp64, so the result
// is bit-identical to the sequential CPU restatement (oracle/nfx_oracle.c orc_edgeflux_step).
//
// Algorithmic bytes: 2 * sizeof(T) * nz per cell and time step (u and v read once).  Roofline: HBM.
#include <cuda.h>

#include <algorithm>

#include "nfx_common.cuh"
#include "nfx_stream_ops.cuh"

namespace nfx {

namespace {

using namespace dev;

// One thread owns VEC adjacent columns of one time step; blockIdx.y = time step.
// LAYERED: blockIdx.y + ps0 = t * nlayers + i is a pseudo-step, time step t summed over the levels [levels[i],
// levels[i+1]) of layer i: the sums of the whole column with dz (e3) zeroed outside the layer, bit for bit on finite
// data.  A template flag, so that the whole-column instances keep their registers.
// E3: per-column, per-level scale factors e3u/e3v (NEMO's vertical metric, partial cells / z*) replace the 1-D
// layer thickness dz[k] of field.py:51 -- two more streamed arrays, same layout as u/v (SURVEY 8f rank 4).
// ALU_MASK (float32 storage): bit q set = level q of every batch of UNROLL levels goes through clean_scaled()
// (bit shuffle on the ALU, dz scaled by 2^896) instead of an F2F on the XU pipe; same bits either way
template <typename T, int VEC, int UNROLL, int BLOCK, bool E3, int ALU_MASK, bool LAYERED = false>
__global__ void __launch_bounds__(BLOCK)
k2_edgeflux_ldg(const T* __restrict__ u, const T* __restrict__ v, const double* __restrict__ dz,
                const double* __restrict__ arc1, const double* __restrict__ arc2, double* __restrict__ eflux, int nz,
                int64_t ncell, int64_t ld, double scale, int use_scale, T fill, int has_fill, int keep_l2,
                const T* __restrict__ e3u, const T* __restrict__ e3v, int64_t e3_tstride,
                const int* __restrict__ levels, int nlayers, int64_t ps0) {
    // ncell = columns handled by this launch (a panel of the grid), ld = cells per level plane (row stride of u, v)
    extern __shared__ double s_dz[];   // [nz] dz, then (ALU_MASK != 0) [nz] dz * 2^896
    bool redo = false;                 // ALU_MASK: recompute this thread's columns with clean() (saw an infinity)
    if constexpr (!E3) {
        int big = 0;
        for (int k = threadIdx.x; k < nz; k += BLOCK) {
            const double d = dz[k];
            s_dz[k] = d;
            if constexpr (ALU_MASK != 0) {
                s_dz[nz + k] = d * kScaleUp;
                big |= !(fabs(d) < kScaleLimit);
            }
        }
        if constexpr (ALU_MASK != 0)
            redo = __syncthreads_or(big) != 0;   // absurd thickness: the scaled factors could overflow
        else
            __syncthreads();
    }
    float amax = 0.f;
    using P = Pack<T, VEC>;
    using V = typename P::type;
    int64_t ps = blockIdx.y, t = ps;
    int k0 = 0, k1 = nz;
    if constexpr (LAYERED) {
        ps += ps0;
        t = ps / nlayers;
        k0 = levels[ps - t * nlayers];
        k1 = levels[ps - t * nlayers + 1];
    }
    const int64_t c0 = ((int64_t)blockIdx.x * BLOCK + threadIdx.x) * VEC;
    if (c0 >= ncell) return;
    const T* pu = u + t * nz * ld + c0;
    const T* pv = v + t * nz * ld + c0;
    const T* pe = E3 ? e3u + t * e3_tstride + c0 : nullptr;   // e3_tstride = 0: time-invariant scale factors
    const T* pf = E3 ? e3v + t * e3_tstride + c0 : nullptr;
    const uint64_t pol = keep_l2 ? l2_evict_last_policy() : 0;
    const uint64_t pol_ef = l2_evict_first_policy();
    double su[VEC], sv[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        su[e] = 0.0;
        sv[e] = 0.0;
    }
    int k = k0;
    for (; k + UNROLL <= k1; k += UNROLL) {
        V ru[UNROLL], rv[UNROLL], re[E3 ? UNROLL : 1], rf[E3 ? UNROLL : 1];
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) {
            ru[q] = ld_stream(reinterpret_cast<const V*>(pu + (int64_t)(k + q) * ld), pol_ef);
            rv[q] = ld_stream(reinterpret_cast<const V*>(pv + (int64_t)(k + q) * ld), pol_ef);
            if constexpr (E3) {
                re[q] = ld_stream(reinterpret_cast<const V*>(pe + (int64_t)(k + q) * ld), pol_ef);
                rf[q] = ld_stream(reinterpret_cast<const V*>(pf + (int64_t)(k + q) * ld), pol_ef);
            }
        }
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) {
            pin(ru[q]);
            pin(rv[q]);
            if constexpr (E3) {
                pin(re[q]);
                pin(rf[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < UNROLL; ++q) {
            T a[VEC], b[VEC], ea[VEC], eb[VEC];
            P::unpack(ru[q], a);
            P::unpack(rv[q], b);
            if constexpr (E3) {
                P::unpack(re[q], ea);
                P::unpack(rf[q], eb);
            }
            const bool kScaled = (ALU_MASK >> q) & 1;   // compile-time after unrolling
            const double d = E3 ? 0.0 : s_dz[(kScaled ? nz : 0) + k + q];
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                if (kScaled && E3) {
                    // both factors come from float32: undo the 2^-896 of each bit shuffle with an exact multiply
                    const double du = __dmul_rn(clean_scaled(ea[e], fill, has_fill, amax), kScaleUp);
                    const double dv = __dmul_rn(clean_scaled(eb[e], fill, has_fill, amax), kScaleUp);
                    const double xu = __dmul_rn(clean_scaled(a[e], fill, has_fill, amax), kScaleUp);
                    const double xv = __dmul_rn(clean_scaled(b[e], fill, has_fill, amax), kScaleUp);
                    su[e] = __dadd_rn(su[e], __dmul_rn(du, xu));
                    sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, xv));
                    continue;
                }
                const double du = E3 ? clean<T>(ea[e], fill, has_fill) : d;
                const double dv = E3 ? clean<T>(eb[e], fill, has_fill) : d;
                if (kScaled) {
                    su[e] = __dadd_rn(su[e], __dmul_rn(du, clean_scaled(a[e], fill, has_fill, amax)));
                    sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean_scaled(b[e], fill, has_fill, amax)));
                } else {
                    su[e] = __dadd_rn(su[e], __dmul_rn(du, clean<T>(a[e], fill, has_fill)));
                    sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean<T>(b[e], fill, has_fill)));
                }
            }
        }
    }
    for (; k < k1; ++k) {
        T a[VEC], b[VEC], ea[VEC], eb[VEC];
        P::unpack(ld_stream(reinterpret_cast<const V*>(pu + (int64_t)k * ld), pol_ef), a);
        P::unpack(ld_stream(reinterpret_cast<const V*>(pv + (int64_t)k * ld), pol_ef), b);
        if constexpr (E3) {
            P::unpack(ld_stream(reinterpret_cast<const V*>(pe + (int64_t)k * ld), pol_ef), ea);
            P::unpack(ld_stream(reinterpret_cast<const V*>(pf + (int64_t)k * ld), pol_ef), eb);
        }
        const double d = E3 ? 0.0 : s_dz[k];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
            const double du = E3 ? clean<T>(ea[e], fill, has_fill) : d;
            const double dv = E3 ? clean<T>(eb[e], fill, has_fill) : d;
            su[e] = __dadd_rn(su[e], __dmul_rn(du, clean<T>(a[e], fill, has_fill)));
            sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean<T>(b[e], fill, has_fill)));
        }
    }
    if constexpr (ALU_MASK != 0) {
        redo = redo || !(amax <= 3.402823466e38f);
        if (redo) {                    // rare: an infinity in this thread's columns -- plain conversion, same order
#pragma unroll
            for (int e = 0; e < VEC; ++e) {
                su[e] = 0.0;
                sv[e] = 0.0;
            }
#pragma unroll 1
            for (int kk = k0; kk < k1; ++kk) {
                const double d = E3 ? 0.0 : s_dz[kk];
#pragma unroll
                for (int e = 0; e < VEC; ++e) {
                    const double du = E3 ? clean<T>(pe[(int64_t)kk * ld + e], fill, has_fill) : d;
                    const double dv = E3 ? clean<T>(pf[(int64_t)kk * ld + e], fill, has_fill) : d;
                    su[e] = __dadd_rn(su[e], __dmul_rn(du, clean<T>(pu[(int64_t)kk * ld + e], fill, has_fill)));
                    sv[e] = __dadd_rn(sv[e], __dmul_rn(dv, clean<T>(pv[(int64_t)kk * ld + e], fill, has_fill)));
                }
            }
        }
    }
    double* ou = eflux + ps * 2 * ncell + c0;
    double* ov = ou + ncell;
    // the last vector of a row may hang over the end of the grid (padded planes, ld > ncell): loads are safe,
    // metric factors and stores are only touched for the nvalid real columns
    const int nvalid = (int)min((int64_t)VEC, ncell - c0);
    double fu[VEC], fv[VEC];
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        fu[e] = 0.0;
        fv[e] = 0.0;
        if (e < nvalid) {
            fu[e] = __dmul_rn(su[e], arc1[c0 + e]);
            fv[e] = __dmul_rn(-sv[e], arc2[c0 + e]);
            if (use_scale) {
                fu[e] = __dmul_rn(fu[e], scale);
                fv[e] = __dmul_rn(fv[e], scale);
            }
        }
    }
    // 16-byte stores need even (t*2*ncell + c0) and (ncell): true whenever ncell is even and VEC is even
    const bool pair_ok = (VEC % 2 == 0) && ((ncell & 1) == 0);
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        if (pair_ok && (e % 2 == 0) && e + 1 < nvalid) {
            st_stream2(ou + e, fu[e], fu[e + 1 < VEC ? e + 1 : e], keep_l2, pol);
            st_stream2(ov + e, fv[e], fv[e + 1 < VEC ? e + 1 : e], keep_l2, pol);
        } else if (e < nvalid && !(pair_ok && (e % 2 == 1))) {   // odd e: already written with e-1
            st_stream1(ou + e, fu[e], keep_l2, pol);
            st_stream1(ov + e, fv[e], keep_l2, pol);
        }
    }
}

struct E3Args {
    const void* e3u = nullptr;
    const void* e3v = nullptr;
    int64_t tstride = 0;
};

struct LayerArgs {
    const int* levels = nullptr;   // device (n + 1) level boundaries, nullptr = one layer, the whole column
    int n = 1;
};

template <typename T, int VEC, int UNROLL, int BLOCK>
void launch_ldg(const T* u, const T* v, const double* dz, const double* arc1, const double* arc2, double* eflux, int nt,
                int nz, int64_t ncell, int64_t ld, double scale, int use_scale, T fill, int has_fill, int keep_l2,
                const E3Args& e3, int alu_mask, cudaStream_t s) {
    const int64_t nthreads = (ncell + VEC - 1) / VEC;
    dim3 grid((unsigned)((nthreads + BLOCK - 1) / BLOCK), (unsigned)nt);
    // float32: every level through the bit-shuffle conversion (profiles/r1_f32_alu_sweep.md: 5.09 -> 6.37 TB/s)
    constexpr int kAluMask = (sizeof(T) == 4) ? 0x1f : 0;
    if (e3.e3u)   // float32: every level through the bit shuffle (restored exactly by one multiply per value)
        k2_edgeflux_ldg<T, VEC, UNROLL, BLOCK, true, (sizeof(T) == 4 ? (1 << UNROLL) - 1 : 0)><<<grid, BLOCK, sizeof(double) * nz, s>>>(
            u, v, dz, arc1, arc2, eflux, nz, ncell, ld, scale, use_scale, fill, has_fill, keep_l2, (const T*)e3.e3u,
            (const T*)e3.e3v, e3.tstride, nullptr, 1, 0);
    else if (alu_mask >= 0 && sizeof(T) == 4 && UNROLL == 5) {
        switch (alu_mask) {
#define NFX_ALU_CASE(M)                                                                                             \
    case M:                                                                                                         \
        k2_edgeflux_ldg<T, VEC, UNROLL, BLOCK, false, (sizeof(T) == 4 && UNROLL == 5) ? M : 0>                      \
            <<<grid, BLOCK, sizeof(double) * nz * 2, s>>>(u, v, dz, arc1, arc2, eflux, nz, ncell, ld, scale,      \
                                                          use_scale, fill, has_fill, keep_l2, nullptr, nullptr, 0,  \
                                                          nullptr, 1, 0);                                            \
        break;
            NFX_ALU_CASE(0)
            NFX_ALU_CASE(0x01)
            NFX_ALU_CASE(0x09)
            NFX_ALU_CASE(0x15)
            NFX_ALU_CASE(0x1f)
#undef NFX_ALU_CASE
            default: throw Error(NFX_E_INVALID, "edgeflux: unsupported ALU conversion mask");
        }
    } else
        k2_edgeflux_ldg<T, VEC, UNROLL, BLOCK, false, kAluMask><<<grid, BLOCK, sizeof(double) * nz * 2, s>>>(
            u, v, dz, arc1, arc2, eflux, nz, ncell, ld, scale, use_scale, fill, has_fill, keep_l2, nullptr, nullptr, 0,
            nullptr, 1, 0);
}

// layered sums: nt * nlayers pseudo-steps in launches of at most 65535 (gridDim.y), block of 256, every float32 level
// through the bit shuffle -- the default shape of launch_ldg (the K2 tuning options change speed, never bits)
template <typename T, int VEC, int UNROLL, bool E3>
void launch_ldg_layers(const T* u, const T* v, const double* dz, const double* arc1, const double* arc2, double* eflux,
                       int nt, int nz, int64_t ncell, int64_t ld, double scale, int use_scale, T fill, int has_fill,
                       int keep_l2, const E3Args& e3, const LayerArgs& ly, cudaStream_t s) {
    constexpr int kBlock = 256;
    constexpr int kAluMask = sizeof(T) == 4 ? (E3 ? (1 << UNROLL) - 1 : 0x1f) : 0;
    static_assert(E3 || UNROLL == 5, "whole-column shape: 5 levels per batch");
    const int64_t nthreads = (ncell + VEC - 1) / VEC;
    const int64_t nps = (int64_t)nt * ly.n;
    for (int64_t ps0 = 0; ps0 < nps; ps0 += 65535) {
        dim3 grid((unsigned)((nthreads + kBlock - 1) / kBlock), (unsigned)std::min<int64_t>(65535, nps - ps0));
        k2_edgeflux_ldg<T, VEC, UNROLL, kBlock, E3, kAluMask, true><<<grid, kBlock, sizeof(double) * nz * 2, s>>>(
            u, v, dz, arc1, arc2, eflux, nz, ncell, ld, scale, use_scale, fill, has_fill, keep_l2, (const T*)e3.e3u,
            (const T*)e3.e3v, e3.tstride, ly.levels, ly.n, ps0);
    }
}

template <typename T, int VEC>
void dispatch_ldg(const T* u, const T* v, const double* dz, const double* arc1, const double* arc2, double* eflux, int nt,
                  int nz, int64_t ncell, int64_t ld, double scale, int use_scale, T fill, int has_fill, int keep_l2,
                  const E3Args& e3, const LayerArgs& ly, const K2Options& opt, cudaStream_t s) {
    // four float32 streams (e3u/e3v): 15 levels in flight at 80 registers stream 14 % faster than 5 at 72
    // (6.37 vs 5.58 TB/s, tools/e3_bench.py --k2-unroll); every other shape is within 1 % from 3 to 15
    const int unroll = opt.unroll > 0 ? opt.unroll : (e3.e3u && sizeof(T) == 4 && VEC > 1) ? 15 : 5;
    const int block = opt.block > 0 ? opt.block : 256;
    if (ly.levels) {
        if (!e3.e3u)
            launch_ldg_layers<T, VEC, 5, false>(u, v, dz, arc1, arc2, eflux, nt, nz, ncell, ld, scale, use_scale, fill,
                                                has_fill, keep_l2, e3, ly, s);
        else if (sizeof(T) == 4 && VEC > 1)
            launch_ldg_layers<T, VEC, 15, true>(u, v, dz, arc1, arc2, eflux, nt, nz, ncell, ld, scale, use_scale, fill,
                                                has_fill, keep_l2, e3, ly, s);
        else
            launch_ldg_layers<T, VEC, 5, true>(u, v, dz, arc1, arc2, eflux, nt, nz, ncell, ld, scale, use_scale, fill,
                                               has_fill, keep_l2, e3, ly, s);
        return;
    }
#define NFX_K2_CASE(U, B)                                                                                          \
    if (unroll == U && block == B) {                                                                               \
        launch_ldg<T, VEC, U, B>(u, v, dz, arc1, arc2, eflux, nt, nz, ncell, ld, scale, use_scale, fill, has_fill,  \
                                 keep_l2, e3, opt.alu_mask, s);                                                    \
        return;                                                                                                    \
    }
    NFX_K2_CASE(5, 256)
    NFX_K2_CASE(3, 256)
    NFX_K2_CASE(15, 256)
    NFX_K2_CASE(5, 128)
    NFX_K2_CASE(5, 512)
#undef NFX_K2_CASE
    throw Error(NFX_E_INVALID, "edgeflux: unsupported (unroll, block) option pair");
}


// ---------------------------------------------------------------------------------------------------------
// TMA-staged variant: a persistent CTA per SM; one producer thread streams level tiles from HBM into a ring
// of shared-memory stages with 1-D bulk copies (cp.async.bulk ... mbarrier::complete_tx, SASS UBLKCP) and
// consumer warps run the z-sum out of shared memory.  Bytes in flight per SM = STAGES * KL * 2 * TC * sizeof(T)
// (up to ~200 KB), independent of registers and of the compiler's load scheduling -- the direct-load kernel
// above keeps only ~64 KB in flight per SM and stalls on the long scoreboard.
// Needs 16-byte aligned rows: ncell * sizeof(T) % 16 == 0.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
        "l"(src), "r"(bytes), "r"(bar), "l"(policy)
        : "memory");
}

template <typename T, int N>
struct alignas(sizeof(T) * N) Cols {
    T v[N];
};

// TC columns per tile, KL levels per stage, CT consumer threads (+32 producer), CPT = TC/CT columns per thread
template <typename T, int TC, int KL, int STAGES, int CT>
__global__ void __launch_bounds__(CT + 32, 1)
k2_edgeflux_tma(const T* __restrict__ u, const T* __restrict__ v, const double* __restrict__ dz,
                const double* __restrict__ arc1, const double* __restrict__ arc2, double* __restrict__ eflux, int nt, int nz,
                int64_t ncell, int ntiles, double scale, int use_scale, T fill, int has_fill) {
    constexpr int CPT = TC / CT;
    static_assert(TC % CT == 0 && (CPT * sizeof(T)) % 8 == 0, "bad tile shape");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* s_u = reinterpret_cast<T*>(smem_raw);                                      // [STAGES][KL][TC]
    T* s_v = s_u + (size_t)STAGES * KL * TC;                                      // [STAGES][KL][TC]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_v + (size_t)STAGES * KL * TC);  // full[STAGES], empty[STAGES]
    double* s_dz = reinterpret_cast<double*>(bars + 2 * STAGES);                  // [nz]
    const int tid = threadIdx.x;
    for (int k = tid; k < nz; k += CT + 32) s_dz[k] = dz[k];
    if (tid == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(smem_u32(bars + i), 1);                 // full: the producer's expect_tx arrive
            mbar_init(smem_u32(bars + STAGES + i), CT / 32);  // empty: one arrive per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t nitems = (int64_t)nt * ntiles;
    const int nk = (nz + KL - 1) / KL;
    if (tid >= CT) {
        // ---- producer warp: one elected lane issues the bulk copies ----
        if (tid == CT) {
            uint64_t policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            uint32_t it = 0;
            for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x) {
                const int64_t t = w / ntiles;
                const int64_t c0 = (w - t * ntiles) * TC;
                const int ncols = (int)min((int64_t)TC, ncell - c0);
                const uint32_t row_bytes = (uint32_t)(ncols * sizeof(T));
                const T* gu = u + t * nz * ncell + c0;
                const T* gv = v + t * nz * ncell + c0;
                for (int kb = 0; kb < nk; ++kb, ++it) {
                    const int stage = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    const int k0 = kb * KL;
                    const int kl = min(KL, nz - k0);
                    const uint32_t full = smem_u32(bars + stage), empty = smem_u32(bars + STAGES + stage);
                    mbar_wait(empty, ph ^ 1);
                    mbar_expect_tx(full, 2u * kl * row_bytes);
                    T* du = s_u + ((size_t)stage * KL) * TC;
                    T* dv = s_v + ((size_t)stage * KL) * TC;
                    for (int q = 0; q < kl; ++q) {
                        bulk_g2s(smem_u32(du + (size_t)q * TC), gu + (int64_t)(k0 + q) * ncell, row_bytes, full, policy);
                        bulk_g2s(smem_u32(dv + (size_t)q * TC), gv + (int64_t)(k0 + q) * ncell, row_bytes, full, policy);
                    }
                }
            }
        }
        return;
    }
    // ---- consumers ----
    using CV = Cols<T, CPT>;
    const int lane = tid & 31;
    uint32_t it = 0;
    for (int64_t w = blockIdx.x; w < nitems; w += gridDim.x) {
        const int64_t t = w / ntiles;
        const int64_t c0 = (w - t * ntiles) * TC;
        const int64_t c = c0 + (int64_t)tid * CPT;
        double su[CPT], sv[CPT];
#pragma unroll
        for (int e = 0; e < CPT; ++e) {
            su[e] = 0.0;
            sv[e] = 0.0;
        }
        for (int kb = 0; kb < nk; ++kb, ++it) {
            const int stage = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            const int k0 = kb * KL;
            const int kl = min(KL, nz - k0);
            mbar_wait(smem_u32(bars + stage), ph);
            const T* pu = s_u + ((size_t)stage * KL) * TC + tid * CPT;
            const T* pv = s_v + ((size_t)stage * KL) * TC + tid * CPT;
            if (kl == KL) {
#pragma unroll
                for (int q = 0; q < KL; ++q) {
                    const CV a = *reinterpret_cast<const CV*>(pu + (size_t)q * TC);
                    const CV b = *reinterpret_cast<const CV*>(pv + (size_t)q * TC);
                    const double d = s_dz[k0 + q];
#pragma unroll
                    for (int e = 0; e < CPT; ++e) {
                        su[e] = __dadd_rn(su[e], __dmul_rn(d, clean<T>(a.v[e], fill, has_fill)));
                        sv[e] = __dadd_rn(sv[e], __dmul_rn(d, clean<T>(b.v[e], fill, has_fill)));
                    }
                }
            } else {
                for (int q = 0; q < kl; ++q) {
                    const CV a = *reinterpret_cast<const CV*>(pu + (size_t)q * TC);
                    const CV b = *reinterpret_cast<const CV*>(pv + (size_t)q * TC);
                    const double d = s_dz[k0 + q];
#pragma unroll
                    for (int e = 0; e < CPT; ++e) {
                        su[e] = __dadd_rn(su[e], __dmul_rn(d, clean<T>(a.v[e], fill, has_fill)));
                        sv[e] = __dadd_rn(sv[e], __dmul_rn(d, clean<T>(b.v[e], fill, has_fill)));
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(bars + STAGES + stage));   // this warp is done with the stage
        }
        if (c < ncell) {
            double* ou = eflux + t * 2 * ncell + c;
            double* ov = ou + ncell;
            const int nvalid = (int)min((int64_t)CPT, ncell - c);   // even: ncell and c are even on this path
#pragma unroll
            for (int e = 0; e < CPT; e += 2) {
                if (e < nvalid) {
                    double fu0 = __dmul_rn(su[e], arc1[c + e]), fu1 = __dmul_rn(su[e + 1], arc1[c + e + 1]);
                    double fv0 = __dmul_rn(-sv[e], arc2[c + e]), fv1 = __dmul_rn(-sv[e + 1], arc2[c + e + 1]);
                    if (use_scale) {
                        fu0 = __dmul_rn(fu0, scale);
                        fu1 = __dmul_rn(fu1, scale);
                        fv0 = __dmul_rn(fv0, scale);
                        fv1 = __dmul_rn(fv1, scale);
                    }
                    st_stream2(ou + e, fu0, fu1);
                    st_stream2(ov + e, fv0, fv1);
                }
            }
        }
    }
}

template <typename T, int TC, int KL, int STAGES, int CT>
void launch_tma(const T* u, const T* v, const double* dz, const double* arc1, const double* arc2, double* eflux, int nt,
                int nz, int64_t ncell, double scale, int use_scale, T fill, int has_fill, cudaStream_t s) {
    int dev = 0, num_sms = 0;   // queried per call: a few hundred ns, right for every device of the process
    NFX_CUDA(cudaGetDevice(&dev));
    NFX_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t smem = 2 * sizeof(T) * (size_t)STAGES * KL * TC + sizeof(uint64_t) * 2 * STAGES + sizeof(double) * nz;
    auto kern = k2_edgeflux_tma<T, TC, KL, STAGES, CT>;
    NFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));   // per device
    NFX_REQUIRE(smem <= 227 * 1024, "edgeflux (TMA): too many levels for the shared-memory ring");
    const int ntiles = (int)((ncell + TC - 1) / TC);
    const int64_t nitems = (int64_t)nt * ntiles;
    const int grid = (int)std::min<int64_t>(nitems, num_sms);
    kern<<<grid, CT + 32, smem, s>>>(u, v, dz, arc1, arc2, eflux, nt, nz, ncell, ntiles, scale, use_scale, fill, has_fill);
}

// ---- (ncell,4) layout of field.py:209-223 -------------------------------------------------------------
__global__ void k_to_cell_by_cell(const double* __restrict__ eflux, int ny, int nx, double* __restrict__ iv) {
    const int64_t ncell = (int64_t)ny * nx;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncell) return;
    const int64_t t = blockIdx.y;
    const double* eU = eflux + t * 2 * ncell;
    const double* eV = eU + ncell;
    const int64_t j = c / nx, i = c - j * nx;
    const double south = j >= 1 ? eV[c - nx] : 0.0;          // row 0 never written (field.py:61,219)
    const double west = i >= 1 ? eU[c - 1] : eU[c + nx - 1];  // x-periodic (field.py:223)
    double2* o = reinterpret_cast<double2*>(iv + (t * ncell + c) * 4);
    o[0] = make_double2(south, eU[c]);
    o[1] = make_double2(eV[c], west);
}

__global__ void k_absmax(const double* __restrict__ x, int64_t n, unsigned long long* __restrict__ out) {
    double m = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double a = fabs(x[i]);
        if (a > m) m = a;  // NaN never wins
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// in-place byte-order swap of n elements of 4 or 8 bytes, 16 bytes per thread and iteration
template <int ESIZE>
__global__ void k_bswap(uint4* __restrict__ p, int64_t nvec, unsigned char* __restrict__ tail, int ntail_elems) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
        uint4 x = p[i];
        x.x = __byte_perm(x.x, 0, 0x0123);
        x.y = __byte_perm(x.y, 0, 0x0123);
        x.z = __byte_perm(x.z, 0, 0x0123);
        x.w = __byte_perm(x.w, 0, 0x0123);
        if (ESIZE == 8) x = make_uint4(x.y, x.x, x.w, x.z);
        p[i] = x;
    }
    if (blockIdx.x == 0 && threadIdx.x < ntail_elems) {   // fewer than 16 bytes left over
        unsigned char* q = tail + threadIdx.x * ESIZE;
#pragma unroll
        for (int b = 0; b < ESIZE / 2; ++b) {
            const unsigned char c = q[b];
            q[b] = q[ESIZE - 1 - b];
            q[ESIZE - 1 - b] = c;
        }
    }
}

}  // namespace

void bswap_inplace(void* p, size_t n, int esize, cudaStream_t s) {
    NFX_REQUIRE(esize == 4 || esize == 8, "bswap: element size must be 4 or 8");
    NFX_REQUIRE(((uintptr_t)p & 15) == 0, "bswap: buffer must be 16-byte aligned");
    if (n == 0) return;
    const size_t bytes = n * (size_t)esize;
    const int64_t nvec = (int64_t)(bytes / 16);
    unsigned char* tail = (unsigned char*)p + (size_t)nvec * 16;
    const int ntail = (int)((bytes - (size_t)nvec * 16) / (size_t)esize);
    const int grid = (int)std::min<int64_t>(148 * 8, std::max<int64_t>(1, (nvec + 255) / 256));
    if (esize == 8)
        k_bswap<8><<<grid, 256, 0, s>>>((uint4*)p, nvec, tail, ntail);
    else
        k_bswap<4><<<grid, 256, 0, s>>>((uint4*)p, nvec, tail, ntail);
    count_launch();
    NFX_CUDA(cudaGetLastError());
}

// One launch over `ncols` adjacent columns (a panel of the grid, pointers already offset to its first column)
// and `nt` time steps; ld = cells per level plane.  eflux: (nt, 2*ncols).  Layered (levels: device, nlayers + 1
// ascending level boundaries): eflux (nt, nlayers, 2*ncols), layer i summed over the levels [levels[i], levels[i+1]);
// always the direct-load kernel (the TMA variant sums whole columns only).  Any nt: more than 65535 steps run in
// slices of 65535.
void edgeflux_assemble_panel(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                             const double* arc2, int nt, int nz, int64_t ncols, int64_t ld, int sverdrup, double fill,
                             double* eflux, int keep_l2, const K2Options& opt, cudaStream_t s, const void* e3u,
                             const void* e3v, int64_t e3_tstride, int nlayers, const int* levels) {
    NFX_REQUIRE(u && v && arc1 && arc2 && eflux, "edgeflux: NULL pointer");
    NFX_REQUIRE((e3u == nullptr) == (e3v == nullptr), "edgeflux: e3u and e3v go together");
    NFX_REQUIRE(thickness || e3u, "edgeflux: needs the layer thickness or e3u/e3v");
    E3Args e3;
    e3.e3u = e3u;
    e3.e3v = e3v;
    e3.tstride = e3_tstride;
    LayerArgs ly;
    ly.levels = levels;
    ly.n = nlayers;
    NFX_REQUIRE(nlayers >= 1 && (levels != nullptr || nlayers == 1), "edgeflux: bad layering");
    NFX_REQUIRE(nt >= 0 && nz > 0 && ncols > 0 && ld >= ncols, "edgeflux: bad sizes");
    NFX_REQUIRE(dtype == NFX_F64 || dtype == NFX_F32, "edgeflux: dtype must be NFX_F64 or NFX_F32");
    NFX_REQUIRE(nz <= 3000, "edgeflux: at most 3000 levels (dz and dz * 2^896 live in 48 KB of shared memory)");
    if (nt == 0) return;
    if (nt > 65535) {
        // gridDim.y carries the time steps: slices of at most 65535 steps, each a call of its own on the arrays offset
        // to its first step (every slice picks its load width from its own addresses; the bits do not depend on it)
        const int64_t esize = dtype == NFX_F64 ? 8 : 4;
        for (int t0 = 0; t0 < nt; t0 += 65535) {
            const int64_t off = (int64_t)t0 * nz * ld * esize, e3_off = (int64_t)t0 * e3_tstride * esize;
            edgeflux_assemble_panel((const char*)u + off, (const char*)v + off, dtype, thickness, arc1, arc2,
                                    std::min(65535, nt - t0), nz, ncols, ld, sverdrup, fill,
                                    eflux + (int64_t)t0 * nlayers * 2 * ncols, keep_l2, opt, s,
                                    e3u ? (const char*)e3u + e3_off : nullptr, e3v ? (const char*)e3v + e3_off : nullptr,
                                    e3_tstride, nlayers, levels);
        }
        return;
    }
    const double scale = 6371000.0 / 1.e6;  // field.py:12,226
    const int has_fill = !(fill != fill);
    const uintptr_t addr_bits = ((uintptr_t)u) | ((uintptr_t)v) | ((uintptr_t)eflux) | ((uintptr_t)e3u) | ((uintptr_t)e3v) |
                                (uintptr_t)(e3_tstride * (dtype == NFX_F64 ? 8 : 4));
    const bool aligned16 = (addr_bits & 15) == 0;
    const bool aligned32 = (addr_bits & 31) == 0 && opt.variant != NFX_K2_LDG128;
    const bool want_tma = (opt.variant == NFX_K2_TMA) && ld == ncols && !e3u && !levels;
    if (want_tma && aligned16 && dtype == NFX_F64 && ncols % 2 == 0) {
        const int cfg = opt.unroll;   // tile configuration selector for the sweep (0 = default)
        const double* pu = (const double*)u;
        const double* pv = (const double*)v;
#define NFX_TMA_CASE(ID, TC, KL, ST, CT)                                                                             \
    if (cfg == ID) {                                                                                                 \
        launch_tma<double, TC, KL, ST, CT>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, scale, sverdrup, fill, \
                                           has_fill, s);                                                             \
        count_launch();                                                                                              \
        NFX_CUDA(cudaGetLastError());                                                                                \
        return;                                                                                                      \
    }
        NFX_TMA_CASE(0, 1024, 5, 2, 512)
        NFX_TMA_CASE(1, 512, 5, 4, 256)
        NFX_TMA_CASE(2, 512, 3, 8, 256)
        NFX_TMA_CASE(3, 512, 5, 5, 256)
        NFX_TMA_CASE(4, 1024, 3, 4, 512)
        NFX_TMA_CASE(5, 512, 5, 5, 128)
        NFX_TMA_CASE(6, 256, 5, 10, 128)
        NFX_TMA_CASE(7, 512, 15, 1, 256)
        NFX_TMA_CASE(8, 512, 5, 2, 256)
#undef NFX_TMA_CASE
        throw Error(NFX_E_INVALID, "edgeflux (TMA): unknown tile configuration");
    }
    if (dtype == NFX_F64) {
        const double* pu = (const double*)u;
        const double* pv = (const double*)v;
        if (aligned32 && ld % 4 == 0 && (ncols % 4 == 0 || ld >= (ncols + 3) / 4 * 4))
            dispatch_ldg<double, 4>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, ld, scale, sverdrup, fill,
                                    has_fill, keep_l2, e3, ly, opt, s);
        else if (aligned16 && ld % 2 == 0 && (ncols % 2 == 0 || ld >= (ncols + 1) / 2 * 2))
            dispatch_ldg<double, 2>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, ld, scale, sverdrup, fill,
                                    has_fill, keep_l2, e3, ly, opt, s);
        else
            dispatch_ldg<double, 1>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, ld, scale, sverdrup, fill,
                                    has_fill, keep_l2, e3, ly, opt, s);
    } else {
        const float* pu = (const float*)u;
        const float* pv = (const float*)v;
        // float32: 128-bit loads (72 registers, 3 CTAs per SM) stream 15 % faster than 256-bit loads (2 CTAs per SM)
        // -- profiles/r1_f32_alu_sweep.md; the 256-bit shape stays selectable with NFX_K2_LDG
        const bool wide = opt.variant == NFX_K2_LDG;
        if (wide && aligned32 && ld % 8 == 0 && (ncols % 8 == 0 || ld >= (ncols + 7) / 8 * 8))
            dispatch_ldg<float, 8>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, ld, scale, sverdrup,
                                   (float)fill, has_fill, keep_l2, e3, ly, opt, s);
        else if (aligned16 && ld % 4 == 0 && (ncols % 4 == 0 || ld >= (ncols + 3) / 4 * 4))
            dispatch_ldg<float, 4>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, ld, scale, sverdrup,
                                   (float)fill, has_fill, keep_l2, e3, ly, opt, s);
        else
            dispatch_ldg<float, 1>(pu, pv, thickness, arc1, arc2, eflux, nt, nz, ncols, ld, scale, sverdrup,
                                   (float)fill, has_fill, keep_l2, e3, ly, opt, s);
    }
    count_launch();
    NFX_CUDA(cudaGetLastError());
}

void edgeflux_assemble(const void* u, const void* v, int dtype, const double* thickness, const double* arc1,
                       const double* arc2, int nt, int nz, int64_t ncell, int sverdrup, double fill, double* eflux,
                       const K2Options& opt, cudaStream_t s) {
    edgeflux_assemble_panel(u, v, dtype, thickness, arc1, arc2, nt, nz, ncell, ncell, sverdrup, fill, eflux, 0, opt, s,
                            nullptr, nullptr, 0);
}

void edgeflux_to_cell_by_cell(const double* eflux, int nt, int ny, int nx, double* iv, cudaStream_t s) {
    NFX_REQUIRE(eflux && iv, "to_cell_by_cell: NULL pointer");
    NFX_REQUIRE(nt >= 0 && ny > 0 && nx > 0 && nt <= 65535, "to_cell_by_cell: bad sizes");
    if (nt == 0) return;
    const int64_t ncell = (int64_t)ny * nx;
    dim3 grid((unsigned)((ncell + 255) / 256), (unsigned)nt);
    k_to_cell_by_cell<<<grid, 256, 0, s>>>(eflux, ny, nx, iv);
    count_launch();
    NFX_CUDA(cudaGetLastError());
}

void edgeflux_absmax(const double* eflux, int nt, int64_t ncell, double* result_host, cudaStream_t s) {
    NFX_REQUIRE(eflux && result_host, "absmax: NULL pointer");
    DevBuf<unsigned long long> d;
    d.alloc(1);
    NFX_CUDA(cudaMemsetAsync(d.p, 0, sizeof(unsigned long long), s));
    const int64_t n = (int64_t)nt * 2 * ncell;
    if (n > 0) {
        k_absmax<<<148 * 8, 256, 0, s>>>(eflux, n, d.p);
        count_launch();
        NFX_CUDA(cudaGetLastError());
    }
    unsigned long long bits = 0;
    NFX_CUDA(cudaMemcpyAsync(&bits, d.p, sizeof bits, cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaStreamSynchronize(s));
    double r;
    memcpy(&r, &bits, sizeof r);
    *result_host = r;
}

}  // namespace nfx
