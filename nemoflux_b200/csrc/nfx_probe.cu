// Read-only HBM ceiling of the device the library runs on, measured with K2's own access pattern.
//
// The driver-written peak (MEASURED_PEAKS.json) is a COPY rate (reads + writes share the bus, 6.3-6.5 TB/s on these
// parts); the flux-series pass only reads.  nfx_probe_read_bandwidth walks a caller-owned buffer the way
// k2_edgeflux_ldg / k23_fused walk uo and vo -- one CTA per tile of columns, nz level planes, two arrays, 256-bit
// evict-first loads, 5 levels of both arrays in flight, K2's multiply-add per value -- and stores nothing, so
// bench.py can quote the pass against the ceiling of the box it runs on instead of a constant from another machine.
// nfx_probe_read_bandwidth_groups does the same walk over a list of 256-bit column groups only: the access pattern of
// the sparse fused pass, which is judged against that ceiling rather than the dense one.
#include "nfx_common.cuh"
#include "nfx_stream_ops.cuh"

namespace nfx {
namespace {

using namespace dev;

constexpr int kProbeBlock = 256;
constexpr int kProbeUnroll = 5;

// GROUPS: thread i reads the 256-bit vector groups[i] of every plane instead of vector i (the sparse fused pass)
template <bool GROUPS>
__global__ void __launch_bounds__(kProbeBlock, 3)
k_probe_read(const double4x* __restrict__ a, const double4x* __restrict__ b, int64_t plane4, const int32_t* groups,
             int64_t nwalk, int nz, double* sink) {
    const int64_t i = (int64_t)blockIdx.x * kProbeBlock + threadIdx.x;
    if (i >= nwalk) return;
    const int64_t c = GROUPS ? (int64_t)groups[i] : i;
    const double4x* pa = a + (int64_t)blockIdx.y * nz * plane4 + c;
    const double4x* pb = b + (int64_t)blockIdx.y * nz * plane4 + c;
    double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int k = 0; k + kProbeUnroll <= nz; k += kProbeUnroll) {
        double4x v[kProbeUnroll], w[kProbeUnroll];
#pragma unroll
        for (int q = 0; q < kProbeUnroll; ++q) {
            v[q] = ld_stream(pa + (int64_t)(k + q) * plane4);
            w[q] = ld_stream(pb + (int64_t)(k + q) * plane4);
        }
#pragma unroll
        for (int q = 0; q < kProbeUnroll; ++q) {
            pin(v[q]);
            pin(w[q]);
        }
#pragma unroll
        for (int q = 0; q < kProbeUnroll; ++q) {
            const double d = 1.0 + 0.25 * (k + q);
            const double x[8] = {v[q].x, v[q].y, v[q].z, v[q].w, w[q].x, w[q].y, w[q].z, w[q].w};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const double y = (x[e] != x[e]) ? 0.0 : x[e];
                s[e] = __dadd_rn(s[e], __dmul_rn(d, y));
            }
        }
    }
    double t = 0.0;
#pragma unroll
    for (int e = 0; e < 8; ++e) t += s[e];
    if (t == 1.2345e300) *sink = t;   // never true for real data: keeps the loads alive without a store
}

}  // namespace

// buf: device buffer of nbytes (32-byte aligned, contents arbitrary), treated as two arrays of (nt, 75, plane)
// doubles with the ORCA1 plane of 120 184 cells; walks every vector of a plane, or only groups[0 .. ngroups) when
// groups != nullptr; returns the best of `reps` launches in GB/s of the bytes walked
static double probe_walk(const void* buf, int64_t nbytes, const int32_t* groups, int64_t ngroups, int reps, double* sink,
                         cudaStream_t s) {
    NFX_REQUIRE(buf && (((uintptr_t)buf) & 31) == 0, "probe: the buffer must be 32-byte aligned");
    const int64_t plane4 = 30046;   // 362 x 332 cells / 4
    const int nz = 75;
    const int64_t step_bytes = 32 * plane4 * nz;
    const int64_t nt = (nbytes / 2) / step_bytes;
    NFX_REQUIRE(nt >= 64, "probe: the buffer must hold at least 9.3 GB (64 time steps of two arrays)");
    NFX_REQUIRE(!groups || (ngroups > 0 && ngroups <= plane4), "probe: 1 .. 30046 groups");
    const int64_t nt_use = std::min<int64_t>(nt, 65535);
    const int64_t nwalk = groups ? ngroups : plane4;
    const double4x* a = reinterpret_cast<const double4x*>(buf);
    const double4x* b = a + nt_use * nz * plane4;
    const dim3 grid((unsigned)((nwalk + kProbeBlock - 1) / kProbeBlock), (unsigned)nt_use);
    auto launch = [&] {
        if (groups) k_probe_read<true><<<grid, kProbeBlock, 0, s>>>(a, b, plane4, groups, nwalk, nz, sink);
        else k_probe_read<false><<<grid, kProbeBlock, 0, s>>>(a, b, plane4, nullptr, nwalk, nz, sink);
        count_launch();
    };
    cudaEvent_t e0, e1;
    NFX_CUDA(cudaEventCreate(&e0));
    NFX_CUDA(cudaEventCreate(&e1));
    double best = 0.0;
    try {
        launch();   // warm-up
        for (int r = 0; r < std::max(reps, 1); ++r) {
            NFX_CUDA(cudaEventRecord(e0, s));
            launch();
            NFX_CUDA(cudaEventRecord(e1, s));
            NFX_CUDA(cudaEventSynchronize(e1));
            float ms = 0.f;
            NFX_CUDA(cudaEventElapsedTime(&ms, e0, e1));
            best = std::max(best, 2.0 * (double)nt_use * 32.0 * nz * (double)nwalk / (ms * 1e-3) / 1e9);
        }
        NFX_CUDA(cudaGetLastError());
    } catch (...) {
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        throw;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return best;
}

double probe_read_bandwidth(const void* buf, int64_t nbytes, int reps, double* sink, cudaStream_t s) {
    return probe_walk(buf, nbytes, nullptr, 0, reps, sink, s);
}

double probe_read_bandwidth_groups(const void* buf, int64_t nbytes, const int32_t* groups, int64_t ngroups, int reps,
                                   double* sink, cudaStream_t s) {
    NFX_REQUIRE(groups, "probe: NULL group list");
    return probe_walk(buf, nbytes, groups, ngroups, reps, sink, s);
}

}  // namespace nfx
