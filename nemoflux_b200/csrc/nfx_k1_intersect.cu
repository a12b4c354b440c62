// K1: polyline-segment x curvilinear-cell intersection on the lon-lat grid (sm_100a).
//
// Replaces mint.PolylineIntegral.buildLocator + computeWeights (call site
// /root/reference/nemoflux/field.py:44-49: periodX=360, counterclock=False, enableFolding=False).
//
// Pipeline (all on the device, one-off per set of transects):
//   locator : 3-level bounding-box hierarchy with fan-out 32 (one warp reduces one node)
//   count   : ONE WARP PER (TARGET SEGMENT, x-period image, piece of the segment): lanes test 32 boxes / 32 cells
//             at a time, ballot-compact the accepted cells; the hits are also appended to a record list
//   scan    : exclusive scan of the per-warp counts
//   fill    : scatter of the record list into (cell, image, ta, tb); the same traversal again when the list
//             (sized from an estimate) was too small
//   sort    : per segment by (ta, cell, image): chunks of 4096 keys sorted in shared memory, then merge rank
//   weights : duplicity coefficient, inverse bilinear map (Newton, fixed operation order), 4 edge
//             weights per sub-segment with mint's edge order 0=S 1=E 2=N 3=W and sign convention
//   map     : mint's std::map<(cell,edge),weight> view and the CSR lists consumed by K3
//
// Arithmetic of the geometric predicates uses __dadd_rn/__dmul_rn/__ddiv_rn only (never contracted
// into FMA), in a fixed order, so the emitted (cell, edge, weight) lists are reproducible bit for bit.
#include <math_constants.h>

#include <algorithm>
#include <cmath>

#include "nfx_common.cuh"

namespace nfx {

namespace {

constexpr double kEps = 10.0 * 2.220446049250313e-16;
constexpr double kEps100 = 100.0 * kEps;
constexpr int kNewtonMaxIt = 20;
constexpr double kNewtonTol = 1.0e-15;
constexpr double kMargin = 1.0e-7;  // candidate filter margin (degrees); superset filter only

__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// point-in-quad: z component of (p - v_i) x (p - v_{i+1}) >= -tol on the 4 CCW edges
__device__ __forceinline__ bool contains_point(const double2 (&v)[4], double px, double py) {
    bool inside = true;
#pragma unroll
    for (int i0 = 0; i0 < 4; ++i0) {
        const int i1 = (i0 + 1) & 3;
        const double d0x = dsub(px, v[i0].x), d0y = dsub(py, v[i0].y);
        const double d1x = dsub(px, v[i1].x), d1y = dsub(py, v[i1].y);
        const double cross = dsub(dmul(d0x, d1y), dmul(d0y, d1x));
        if (cross < -kEps) inside = false;
    }
    return inside;
}

// line parameters where segment a->b meets the quad; returns count, min in ta, max in tb.
// Ties keep the first-inserted minimum / last-inserted maximum (what a stable sort would give).
__device__ __forceinline__ int collect_lambdas(const double2 (&v)[4], double ax, double ay, double bx, double by,
                                               double& ta, double& tb) {
    int n = 0;
    double lo = 0.0, hi = 0.0;
    auto push = [&](double l) {
        if (n == 0) {
            lo = l;
            hi = l;
        } else {
            if (l < lo) lo = l;
            if (l >= hi) hi = l;
        }
        ++n;
    };
    if (contains_point(v, ax, ay)) push(0.0);
    if (contains_point(v, bx, by)) push(1.0);
    const double m0 = dsub(bx, ax);
    const double m2 = dsub(by, ay);
#pragma unroll
    for (int i0 = 0; i0 < 4; ++i0) {
        const int i1 = (i0 + 1) & 3;
        const double q0x = v[i0].x, q0y = v[i0].y, q1x = v[i1].x, q1y = v[i1].y;
        const double m1 = dsub(q0x, q1x);
        const double m3 = dsub(q0y, q1y);
        const double r0 = dsub(q0x, ax);
        const double r1 = dsub(q0y, ay);
        const double det = dsub(dmul(m0, m3), dmul(m1, m2));
        const double s0 = dsub(dmul(m3, r0), dmul(m1, r1));
        const double s1 = dsub(dmul(m0, r1), dmul(m2, r0));
        if (fabs(det) > kEps) {
            const double l = ddiv(s0, det);
            const double mu = ddiv(s1, det);
            if (l >= -kEps100 && l <= 1.0 + kEps100 && mu >= -kEps100 && mu <= 1.0 + kEps100) push(l);
        } else if (fabs(s0) < kEps && fabs(s1) < kEps) {
            const double u2 = dadd(dmul(m0, m0), dmul(m2, m2));
            const double t0x = dsub(q1x, ax);
            const double t0y = dsub(q1y, ay);
            const double lA = ddiv(dadd(dmul(r0, m0), dmul(r1, m2)), u2);
            const double lB = ddiv(dadd(dmul(t0x, m0), dmul(t0y, m2)), u2);
            const double lmin = lA < lB ? lA : lB;
            const double lmax = lA < lB ? lB : lA;
            if (!(lmin > 1.0 + kEps || lmax < -kEps)) {
                const double la = lmin > 0.0 ? lmin : 0.0;
                const double lb = lmax < 1.0 ? lmax : 1.0;
                if (fabs(dsub(lb, la)) > kEps) {
                    push(la);
                    push(lb);
                }
            }
        }
    }
    ta = lo;
    tb = hi;
    return n;
}

// inverse bilinear map, Newton from (1/2,1/2)
__device__ __forceinline__ void param_coords(const double2 (&v)[4], double px, double py, double& xi0, double& xi1) {
    const double bx = dsub(v[1].x, v[0].x), by = dsub(v[1].y, v[0].y);
    const double cx = dsub(v[3].x, v[0].x), cy = dsub(v[3].y, v[0].y);
    const double dx = dadd(dsub(v[0].x, v[1].x), dsub(v[2].x, v[3].x));
    const double dy = dadd(dsub(v[0].y, v[1].y), dsub(v[2].y, v[3].y));
    double s = 0.5, t = 0.5;
    for (int it = 0; it < kNewtonMaxIt; ++it) {
        const double st = dmul(s, t);
        const double fx = dsub(dadd(dadd(dadd(v[0].x, dmul(bx, s)), dmul(cx, t)), dmul(dx, st)), px);
        const double fy = dsub(dadd(dadd(dadd(v[0].y, dmul(by, s)), dmul(cy, t)), dmul(dy, st)), py);
        const double j00 = dadd(bx, dmul(dx, t));
        const double j01 = dadd(cx, dmul(dx, s));
        const double j10 = dadd(by, dmul(dy, t));
        const double j11 = dadd(cy, dmul(dy, s));
        const double det = dsub(dmul(j00, j11), dmul(j01, j10));
        const double ds = ddiv(dsub(dmul(fy, j01), dmul(fx, j11)), det);
        const double dt = ddiv(dsub(dmul(fx, j10), dmul(fy, j00)), det);
        s = dadd(s, ds);
        t = dadd(t, dt);
        if (fabs(ds) < kNewtonTol && fabs(dt) < kNewtonTol) break;
    }
    xi0 = s;
    xi1 = t;
}

// conservative "segment certainly misses the box" (margin expanded)
__device__ __forceinline__ bool seg_box_reject(double ax, double ay, double bx, double by, double xmin, double xmax,
                                               double ymin, double ymax) {
    const double sxmin = fmin(ax, bx), sxmax = fmax(ax, bx), symin = fmin(ay, by), symax = fmax(ay, by);
    if (sxmax < xmin - kMargin || sxmin > xmax + kMargin || symax < ymin - kMargin || symin > ymax + kMargin)
        return true;
    const double dx = bx - ax, dy = by - ay;
    const double mt = kMargin * (fabs(dx) + fabs(dy)) + kMargin * kMargin;
    const double c0 = dx * (ymin - ay) - dy * (xmin - ax);
    const double c1 = dx * (ymin - ay) - dy * (xmax - ax);
    const double c2 = dx * (ymax - ay) - dy * (xmax - ax);
    const double c3 = dx * (ymax - ay) - dy * (xmin - ax);
    if (c0 > mt && c1 > mt && c2 > mt && c3 > mt) return true;
    if (c0 < -mt && c1 < -mt && c2 < -mt && c3 < -mt) return true;
    return false;
}

// ---- locator ------------------------------------------------------------------------------------
__global__ void k_pack_points(const double* __restrict__ pts, double2* __restrict__ verts, int64_t nvert) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nvert) verts[i] = make_double2(pts[3 * i], pts[3 * i + 1]);
}

__device__ __forceinline__ double4 warp_box(double4 b) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        b.x = fmin(b.x, __shfl_xor_sync(0xffffffffu, b.x, o));
        b.y = fmax(b.y, __shfl_xor_sync(0xffffffffu, b.y, o));
        b.z = fmin(b.z, __shfl_xor_sync(0xffffffffu, b.z, o));
        b.w = fmax(b.w, __shfl_xor_sync(0xffffffffu, b.w, o));
    }
    return b;
}

__global__ void k_build_box1(const double2* __restrict__ verts, int64_t ncell, double4* __restrict__ box1, int64_t nl1) {
    const int lane = threadIdx.x & 31;
    const int64_t node = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (node >= nl1) return;
    const int64_t c = node * kFan + lane;
    double4 b = make_double4(CUDART_INF, -CUDART_INF, CUDART_INF, -CUDART_INF);
    if (c < ncell) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double2 p = verts[c * 4 + k];
            b.x = fmin(b.x, p.x);
            b.y = fmax(b.y, p.x);
            b.z = fmin(b.z, p.y);
            b.w = fmax(b.w, p.y);
        }
    }
    b = warp_box(b);
    if (lane == 0) box1[node] = b;
}

__global__ void k_build_box2(const double4* __restrict__ box1, int64_t nl1, double4* __restrict__ box2, int64_t nl2) {
    const int lane = threadIdx.x & 31;
    const int64_t node = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (node >= nl2) return;
    const int64_t k = node * kFan + lane;
    double4 b = make_double4(CUDART_INF, -CUDART_INF, CUDART_INF, -CUDART_INF);
    if (k < nl1) b = box1[k];
    b = warp_box(b);
    if (lane == 0) box2[node] = b;
}

// ---- traversal: one warp per (segment, image, piece) ------------------------------------------------
// A long segment (an ORCA12 diagonal crosses ~7 000 cells) would keep one warp busy for 16 ms while the rest of the
// GPU idles, so every (segment, image) is cut into kPieces parameter ranges [k/P, (k+1)/P]: the warp of a piece
// walks the box hierarchy with the piece's own end points (a filter only), runs the exact routine on the FULL
// segment -- same arithmetic, same ta/tb as before -- and keeps a cell iff its ta falls into the piece's range.
// The point p(ta) lies on the cell and on that piece, so the piece always sees the cell as a candidate (margin
// 1e-7 deg against 1e-13 of rounding), and exactly one piece keeps it.  The order inside a segment is restored by
// the sort that follows, as before.
constexpr int kPieces = 8;

struct SegIn {
    double p0x, p0y, p1x, p1y;
};

// ballot of "box first+lane may be crossed by the segment (qa, qb)"
__device__ __forceinline__ unsigned box_hits(const double4* __restrict__ boxes, int64_t nbox, int64_t first, int lane,
                                             double qax, double qay, double qbx, double qby) {
    const int64_t k = first + lane;
    bool hit = false;
    if (k < nbox) {
        const double4 b = boxes[k];
        hit = !seg_box_reject(qax, qay, qbx, qby, b.x, b.y, b.z, b.w);
    }
    return __ballot_sync(0xffffffffu, hit);
}

__device__ __forceinline__ int piece_of(double ta) {
    const int k = (int)floor(ta * (double)kPieces);
    return k < 0 ? 0 : (k >= kPieces ? kPieces - 1 : k);
}

// Speculative record of the count pass: every accepted cell is also appended to a list (warp id, index inside the
// warp's output, cell, ta, tb) in chunks of kRecChunk slots that a warp takes with one atomic.  When the list was
// large enough (host estimate of the number of sub-segments), the fill pass is a plain scatter of the records
// (k_scatter_records) instead of a second traversal; when it overflowed, the fill traversal runs as before.
constexpr int kRecChunk = 32;
struct RecList {
    unsigned long long* nchunks;   // chunks handed out (may exceed cap_chunks: overflow)
    int64_t cap_chunks;
    int32_t* w;                    // -1 = unused slot
    int32_t* idx;
    int32_t* cell;
    double* ta;
    double* tb;
};

template <bool FILL>
__global__ void __launch_bounds__(128)
k1_traverse(const double2* __restrict__ verts, int64_t ncell, const double4* __restrict__ box1, int64_t nl1,
            const double4* __restrict__ box2, int64_t nl2, const double4* __restrict__ box3, int64_t nl3,
            const SegIn* __restrict__ segs, int nseg, int nimg,
            double period_x, int64_t* __restrict__ counts, const int64_t* __restrict__ offsets,
            int32_t* __restrict__ o_cell, int32_t* __restrict__ o_img, double* __restrict__ o_ta,
            double* __restrict__ o_tb, const RecList rec) {
    const int lane = threadIdx.x & 31;
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= (int64_t)nseg * nimg * kPieces) return;
    int64_t chunk_base = -1;       // record list: first slot of the warp's current chunk
    int chunk_used = kRecChunk;
    const int piece = (int)(w % kPieces);
    const int64_t wi = w / kPieces;
    const int seg = (int)(wi / nimg);
    const int img = (int)(wi % nimg) - (nimg == 3 ? 1 : 0);
    const SegIn sg = segs[seg];
    int64_t count = 0;
    if (!(sg.p0x == sg.p1x && sg.p0y == sg.p1y)) {
        const double shift = dmul((double)img, period_x);
        const double ax = dadd(sg.p0x, shift), bx = dadd(sg.p1x, shift);
        const double ay = sg.p0y, by = sg.p1y;
        // end points of this piece: candidate filter only
        const double l0 = (double)piece / kPieces, l1 = (double)(piece + 1) / kPieces;
        const double qax = ax + (bx - ax) * l0, qay = ay + (by - ay) * l0;
        const double qbx = ax + (bx - ax) * l1, qby = ay + (by - ay) * l1;
        const int64_t base = FILL ? offsets[w] : 0;
        // three levels of boxes, 32 children each: the warp tests 32 boxes at a time, descends into every hit
        for (int64_t n3b = 0; n3b < nl3; n3b += 32) {
            for (unsigned m3 = box_hits(box3, nl3, n3b, lane, qax, qay, qbx, qby); m3; m3 &= m3 - 1) {
                const int64_t node3 = n3b + (__ffs(m3) - 1);
                for (unsigned m2 = box_hits(box2, nl2, node3 * kFan, lane, qax, qay, qbx, qby); m2; m2 &= m2 - 1) {
                    const int64_t node2 = node3 * kFan + (__ffs(m2) - 1);
                    for (unsigned m1 = box_hits(box1, nl1, node2 * kFan, lane, qax, qay, qbx, qby); m1; m1 &= m1 - 1) {
                        const int64_t c = (node2 * kFan + (__ffs(m1) - 1)) * kFan + lane;   // one cell per lane
                        bool accept = false;
                        double ta = 0.0, tb = 0.0;
                        if (c < ncell) {
                            double2 v[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) v[k] = verts[c * 4 + k];
                            const double xmin = fmin(fmin(v[0].x, v[1].x), fmin(v[2].x, v[3].x));
                            const double xmax = fmax(fmax(v[0].x, v[1].x), fmax(v[2].x, v[3].x));
                            const double ymin = fmin(fmin(v[0].y, v[1].y), fmin(v[2].y, v[3].y));
                            const double ymax = fmax(fmax(v[0].y, v[1].y), fmax(v[2].y, v[3].y));
                            if (!seg_box_reject(qax, qay, qbx, qby, xmin, xmax, ymin, ymax)) {
                                const int n = collect_lambdas(v, ax, ay, bx, by, ta, tb);
                                accept = (n >= 2) && (fabs(dsub(tb, ta)) > kEps100) && piece_of(ta) == piece;
                            }
                        }
                        const unsigned macc = __ballot_sync(0xffffffffu, accept);
                        if (FILL && accept) {
                            const int64_t pos = base + count + __popc(macc & ((1u << lane) - 1u));
                            o_cell[pos] = (int32_t)c;
                            o_img[pos] = img;
                            o_ta[pos] = ta;
                            o_tb[pos] = tb;
                        }
                        if (!FILL && rec.cap_chunks > 0 && macc) {
                            const int nacc = __popc(macc);
                            if (chunk_used + nacc > kRecChunk) {   // the hits of one ballot stay in one chunk
                                if (chunk_base >= 0 && chunk_base / kRecChunk < rec.cap_chunks)
                                    for (int i = chunk_used + lane; i < kRecChunk; i += 32) rec.w[chunk_base + i] = -1;
                                unsigned long long b = 0;
                                if (lane == 0) b = atomicAdd(rec.nchunks, 1ull);
                                b = __shfl_sync(0xffffffffu, b, 0);
                                chunk_base = (int64_t)b * kRecChunk;
                                chunk_used = 0;
                            }
                            if (accept && chunk_base / kRecChunk < rec.cap_chunks) {
                                const int rk = __popc(macc & ((1u << lane) - 1u));
                                const int64_t r = chunk_base + chunk_used + rk;
                                rec.w[r] = (int32_t)w;
                                rec.idx[r] = (int32_t)(count + rk);
                                rec.cell[r] = (int32_t)c;
                                rec.ta[r] = ta;
                                rec.tb[r] = tb;
                            }
                            chunk_used += nacc;
                        }
                        count += __popc(macc);
                    }
                }
            }
        }
    }
    if (!FILL && rec.cap_chunks > 0 && chunk_base >= 0 && chunk_base / kRecChunk < rec.cap_chunks)
        for (int i = chunk_used + lane; i < kRecChunk; i += 32) rec.w[chunk_base + i] = -1;
    if (!FILL && lane == 0) counts[w] = count;
}

// fill pass from the record list: slot r of warp w goes to offsets[w] + idx -- the layout of k1_traverse<true>
__global__ void k_scatter_records(const RecList rec, int64_t nslots, const int64_t* __restrict__ offsets, int nimg,
                                  int32_t* __restrict__ o_cell, int32_t* __restrict__ o_img, double* __restrict__ o_ta,
                                  double* __restrict__ o_tb) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nslots) return;
    const int32_t w = rec.w[r];
    if (w < 0) return;
    const int64_t pos = offsets[w] + rec.idx[r];
    o_cell[pos] = rec.cell[r];
    o_img[pos] = (int32_t)((w / kPieces) % nimg) - (nimg == 3 ? 1 : 0);
    o_ta[pos] = rec.ta[r];
    o_tb[pos] = rec.tb[r];
}

// ---- exclusive scan (int64), 3 passes ---------------------------------------------------------------
constexpr int kScanBlock = 1024;

__device__ __forceinline__ int64_t block_exclusive_scan(int64_t x, int64_t* total) {
    __shared__ int64_t warp_sums[32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t v = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += y;
    }
    if (lane == 31) warp_sums[wid] = v;
    __syncthreads();
    if (wid == 0) {
        int64_t s = warp_sums[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        warp_sums[lane] = s;
    }
    __syncthreads();
    const int64_t before = wid > 0 ? warp_sums[wid - 1] : 0;
    if (total) *total = warp_sums[31];
    const int64_t res = before + v - x;
    __syncthreads();
    return res;
}

__global__ void k_scan_local(const int64_t* __restrict__ in, int64_t* __restrict__ out, int64_t n,
                             int64_t* __restrict__ block_sums) {
    const int64_t i = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
    const int64_t x = i < n ? in[i] : 0;
    int64_t total;
    const int64_t ex = block_exclusive_scan(x, &total);
    if (i < n) out[i] = ex;
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// single block: exclusive scan of block_sums in place (loops over chunks), writes grand total to out_total
__global__ void k_scan_sums(int64_t* __restrict__ sums, int64_t nb, int64_t* __restrict__ out_total) {
    __shared__ int64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t b = 0; b < nb; b += kScanBlock) {
        const int64_t i = b + threadIdx.x;
        const int64_t x = i < nb ? sums[i] : 0;
        int64_t total;
        const int64_t ex = block_exclusive_scan(x, &total);
        const int64_t c = carry;
        if (i < nb) sums[i] = ex + c;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *out_total = carry;
}

__global__ void k_scan_add(int64_t* __restrict__ out, int64_t n, const int64_t* __restrict__ block_sums) {
    const int64_t i = (int64_t)blockIdx.x * kScanBlock + threadIdx.x;
    if (i < n) out[i] += block_sums[blockIdx.x];
}

// out has n+1 entries: out[n] = total
void exclusive_scan(const int64_t* in, int64_t* out, int64_t n, DevBuf<int64_t>& tmp, cudaStream_t s) {
    const int64_t nb = std::max<int64_t>(1, (n + kScanBlock - 1) / kScanBlock);
    tmp.ensure((size_t)nb);
    k_scan_local<<<(unsigned)nb, kScanBlock, 0, s>>>(in, out, n, tmp.p);
    k_scan_sums<<<1, kScanBlock, 0, s>>>(tmp.p, nb, out + n);
    k_scan_add<<<(unsigned)nb, kScanBlock, 0, s>>>(out, n, tmp.p);
    count_launch(3);
    NFX_CUDA(cudaGetLastError());
}

inline unsigned nblk(int64_t n, int b) { return (unsigned)std::max<int64_t>(1, (n + b - 1) / b); }

// ---- sort inside groups ------------------------------------------------------------------------------
// Each group g owns [goff[g], goff[g+1]).  Keys are (ka (double, optional), kb (int64)); all keys in a group are
// distinct.  Result: perm[goff[g] + rank(i)] = i.  Two launches: (1) every chunk of kSortChunk keys is sorted in
// shared memory (bitonic network) into a scratch copy; (2) every key adds up its lower bound in each sorted chunk
// of its group -- n * ceil(n / kSortChunk) * log2(kSortChunk) steps instead of the n^2 comparisons of a plain
// rank sort (groups reach 28 000 keys on an ORCA12 grid: 43 ms -> 2 ms for 10 M keys).
constexpr int kSortChunk = 4096;
constexpr int kSortBlock = 512;
constexpr int kRankBlock = 256;

template <bool HAS_KA>
__device__ __forceinline__ bool key_less(double a1, int64_t b1, double a2, int64_t b2) {
    if (HAS_KA) return (a1 < a2) || (a1 == a2 && b1 < b2);
    return b1 < b2;
}

template <bool HAS_KA>
__global__ void __launch_bounds__(kSortBlock)
k_chunk_sort(const double* __restrict__ ka, const int64_t* __restrict__ kb, const int64_t* __restrict__ goff,
             double* __restrict__ ska, int64_t* __restrict__ skb) {
    extern __shared__ unsigned char s_raw[];
    int64_t* s_b = reinterpret_cast<int64_t*>(s_raw);
    double* s_a = reinterpret_cast<double*>(s_raw + sizeof(int64_t) * kSortChunk);
    const int64_t g0 = goff[blockIdx.x], n = goff[blockIdx.x + 1] - g0;
    const int64_t c0 = (int64_t)blockIdx.y * kSortChunk;
    if (c0 >= n) return;
    const int m = (int)min((int64_t)kSortChunk, n - c0);
    int P = 32;                        // network size: next power of two >= m
    while (P < m) P <<= 1;
    for (int i = threadIdx.x; i < P; i += kSortBlock) {
        s_b[i] = i < m ? kb[g0 + c0 + i] : INT64_MAX;     // padding sorts to the end
        if (HAS_KA) s_a[i] = i < m ? ka[g0 + c0 + i] : CUDART_INF;
    }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < P; i += kSortBlock) {
                const int l = i ^ j;
                if (l > i) {
                    const double ai = HAS_KA ? s_a[i] : 0.0, al = HAS_KA ? s_a[l] : 0.0;
                    const int64_t bi = s_b[i], bl = s_b[l];
                    const bool up = (i & k) == 0;
                    if (key_less<HAS_KA>(al, bl, ai, bi) == up) {
                        s_b[i] = bl;
                        s_b[l] = bi;
                        if (HAS_KA) {
                            s_a[i] = al;
                            s_a[l] = ai;
                        }
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < m; i += kSortBlock) {
        skb[g0 + c0 + i] = s_b[i];
        if (HAS_KA) ska[g0 + c0 + i] = s_a[i];
    }
}

template <bool HAS_KA>
__global__ void __launch_bounds__(kRankBlock)
k_merge_rank(const double* __restrict__ ka, const int64_t* __restrict__ kb, const double* __restrict__ ska,
             const int64_t* __restrict__ skb, const int64_t* __restrict__ goff, int64_t* __restrict__ perm) {
    const int64_t g0 = goff[blockIdx.x], n = goff[blockIdx.x + 1] - g0;
    const int64_t i = (int64_t)blockIdx.y * kRankBlock + threadIdx.x;
    if (i >= n) return;
    const double my_a = HAS_KA ? ka[g0 + i] : 0.0;
    const int64_t my_b = kb[g0 + i];
    int64_t rank = 0;
    for (int64_t c0 = 0; c0 < n; c0 += kSortChunk) {
        const double* ca = ska + g0 + c0;
        const int64_t* cb = skb + g0 + c0;
        int lo = 0, hi = (int)min((int64_t)kSortChunk, n - c0);   // first position whose key is not less than mine
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (key_less<HAS_KA>(HAS_KA ? ca[mid] : 0.0, cb[mid], my_a, my_b))
                lo = mid + 1;
            else
                hi = mid;
        }
        rank += lo;
    }
    perm[g0 + rank] = g0 + i;
}

// groups of `ngroups` rows, the longest has max_len keys; ska/skb: scratch of the size of the key arrays
template <bool HAS_KA>
void sort_in_groups(const double* ka, const int64_t* kb, const int64_t* goff, int ngroups, int64_t max_len, double* ska,
                    int64_t* skb, int64_t* perm, cudaStream_t s) {
    if (ngroups <= 0 || max_len <= 0) return;
    const size_t smem = (sizeof(int64_t) + (HAS_KA ? sizeof(double) : 0)) * kSortChunk;
    if (smem > 48 * 1024)   // per device and cheap: set on every call
        NFX_CUDA(cudaFuncSetAttribute(k_chunk_sort<HAS_KA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_chunk_sort<HAS_KA><<<dim3((unsigned)ngroups, nblk(max_len, kSortChunk)), kSortBlock, smem, s>>>(ka, kb, goff, ska, skb);
    k_merge_rank<HAS_KA><<<dim3((unsigned)ngroups, nblk(max_len, kRankBlock)), kRankBlock, 0, s>>>(ka, kb, ska, skb, goff,
                                                                                                   perm);
    count_launch(2);
    NFX_CUDA(cudaGetLastError());
}

__global__ void k_make_sort1_key(const int32_t* __restrict__ cell, const int32_t* __restrict__ img, int64_t n,
                                 int64_t* __restrict__ kb) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) kb[i] = (int64_t)cell[i] * 4 + (img[i] + 1);
}

__global__ void k_apply_sort1(const int64_t* __restrict__ perm, int64_t n, const int32_t* __restrict__ cell_in,
                              const int32_t* __restrict__ img_in, const double* __restrict__ ta_in,
                              const double* __restrict__ tb_in, int32_t* __restrict__ cell, int32_t* __restrict__ img,
                              double* __restrict__ ta, double* __restrict__ tb) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t src = perm[i];
    cell[i] = cell_in[src];
    img[i] = img_in[src];
    ta[i] = ta_in[src];
    tb[i] = tb_in[src];
}

// segment id of every sub-segment (local to its transect) from the per-segment offsets
__global__ void k_fill_seg_ids(const int64_t* __restrict__ seg_off, int nseg, const int32_t* __restrict__ seg_local,
                               int32_t* __restrict__ seg_of_sub) {
    const int s = blockIdx.x;
    if (s >= nseg) return;
    const int64_t a = seg_off[s], b = seg_off[s + 1];
    const int32_t id = seg_local ? seg_local[s] : s;
    for (int64_t i = a + threadIdx.x; i < b; i += blockDim.x) seg_of_sub[i] = id;
}

// ---- weights: one thread per sub-segment -------------------------------------------------------------
__global__ void __launch_bounds__(128)
k1_weights(const double2* __restrict__ verts, const SegIn* __restrict__ segs, const int32_t* __restrict__ seg_global,
           const int64_t* __restrict__ seg_off, const int32_t* __restrict__ cell, const int32_t* __restrict__ img,
           const double* __restrict__ ta, const double* __restrict__ tb, int64_t n, double period_x, int counterclock,
           double* __restrict__ coeff, double* __restrict__ xia, double* __restrict__ xib, double* __restrict__ w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int sgid = seg_global[i];
    const int64_t seg_end = seg_off[sgid + 1];
    const double ta0 = ta[i], tb0 = tb[i];
    double cf = 1.0;
    if (i + 1 < seg_end) {
        const double ta1 = ta[i + 1], tb1 = tb[i + 1];
        const double hi = tb0 < tb1 ? tb0 : tb1;
        const double lo = ta0 > ta1 ? ta0 : ta1;
        double ov = dsub(hi, lo);
        if (ov < 0.0) ov = 0.0;
        cf = dsub(1.0, ddiv(ov, dsub(tb0, ta0)));
    }
    const int64_t c = cell[i];
    double2 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = verts[c * 4 + k];
    const SegIn sg = segs[sgid];
    const double shift = dmul((double)img[i], period_x);
    const double ax = dadd(sg.p0x, shift), bx = dadd(sg.p1x, shift);
    const double ddx = dsub(bx, ax), ddy = dsub(sg.p1y, sg.p0y);
    const double pax = dadd(ax, dmul(ta0, ddx)), pay = dadd(sg.p0y, dmul(ta0, ddy));
    const double pbx = dadd(ax, dmul(tb0, ddx)), pby = dadd(sg.p0y, dmul(tb0, ddy));
    double a0, a1, b0, b1;
    param_coords(v, pax, pay, a0, a1);
    param_coords(v, pbx, pby, b0, b1);
    const double dxi0 = dsub(b0, a0), dxi1 = dsub(b1, a1);
    const double xm0 = dmul(0.5, dadd(a0, b0)), xm1 = dmul(0.5, dadd(a1, b1));
    const double sgn = counterclock ? -1.0 : 1.0;
    coeff[i] = cf;
    xia[2 * i] = a0;
    xia[2 * i + 1] = a1;
    xib[2 * i] = b0;
    xib[2 * i + 1] = b1;
    w[4 * i + 0] = dmul(dmul(dxi0, dsub(1.0, xm1)), cf);
    w[4 * i + 1] = dmul(dmul(dxi1, xm0), cf);
    w[4 * i + 2] = dmul(sgn, dmul(dmul(dxi0, xm1), cf));
    w[4 * i + 3] = dmul(sgn, dmul(dmul(dxi1, dsub(1.0, xm0)), cf));
}

// ---- mint map view + CSR lists ------------------------------------------------------------------------
__global__ void k_make_sort2_key(const int32_t* __restrict__ cell, int64_t n, int64_t* __restrict__ kb) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) kb[i] = ((int64_t)cell[i] << 32) | (i & 0xffffffffll);
}

// flags[i] = 1 when sorted position i starts a new (transect, cell) run
__global__ void k_run_flags(const int64_t* __restrict__ perm, const int32_t* __restrict__ cell,
                            const int64_t* __restrict__ toff, int ntransects, int64_t n, int64_t* __restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool start = (i == 0) || (cell[perm[i]] != cell[perm[i - 1]]);
    if (!start) {
        // a transect boundary between i-1 and i?  binary search the transect of i
        int lo = 0, hi = ntransects;  // toff[lo] <= i < toff[hi]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (toff[mid] <= i) lo = mid; else hi = mid;
        }
        start = (toff[lo] == i);
    }
    flags[i] = start ? 1 : 0;
}

__global__ void k_map_fill(const int64_t* __restrict__ perm, const int32_t* __restrict__ cell,
                           const double* __restrict__ w, const int64_t* __restrict__ flags,
                           const int64_t* __restrict__ uidx, int64_t n, int64_t* __restrict__ map_keys,
                           double* __restrict__ map_w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || flags[i] == 0) return;
    const int64_t u = uidx[i];
    const int64_t c = cell[perm[i]];
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    bool first = true;
    int64_t j = i;
    do {  // contributions to one key are added in emission order (std::map operator+=)
        const int64_t src = perm[j];
        if (first) {
            s0 = w[4 * src + 0];
            s1 = w[4 * src + 1];
            s2 = w[4 * src + 2];
            s3 = w[4 * src + 3];
            first = false;
        } else {
            s0 = dadd(s0, w[4 * src + 0]);
            s1 = dadd(s1, w[4 * src + 1]);
            s2 = dadd(s2, w[4 * src + 2]);
            s3 = dadd(s3, w[4 * src + 3]);
        }
        ++j;
    } while (j < n && flags[j] == 0);
    map_keys[4 * u + 0] = c * 4 + 0;
    map_keys[4 * u + 1] = c * 4 + 1;
    map_keys[4 * u + 2] = c * 4 + 2;
    map_keys[4 * u + 3] = c * 4 + 3;
    map_w[4 * u + 0] = s0;
    map_w[4 * u + 1] = s1;
    map_w[4 * u + 2] = s2;
    map_w[4 * u + 3] = s3;
}

// map_offsets[m] = 4 * uidx[toff[m]] (uidx has n+1 entries)
__global__ void k_map_offsets(const int64_t* __restrict__ toff, int ntransects, const int64_t* __restrict__ uidx,
                              int64_t* __restrict__ moff) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m <= ntransects) moff[m] = 4 * uidx[toff[m]];
}

// flux index of (cell, edge) in the compact [eU | eV] layout, field.py:209-223; -1 = always zero
__device__ __forceinline__ int32_t flux_index(int64_t key, int ny, int nx) {
    const int64_t cell = key >> 2;
    const int e = (int)(key & 3);
    const int64_t ncell = (int64_t)ny * nx;
    const int64_t j = cell / nx, i = cell - j * nx;
    switch (e) {
        case 1: return (int32_t)cell;
        case 3: return (int32_t)(i >= 1 ? cell - 1 : cell + nx - 1);
        case 2: return (int32_t)(ncell + cell);
        default: return j >= 1 ? (int32_t)(ncell + cell - nx) : -1;
    }
}

// layout 0: idx = key; layout 1: compact
__global__ void k_csr_from_keys(const int64_t* __restrict__ keys, int64_t n, int ny, int nx, int32_t* __restrict__ idx0,
                                int32_t* __restrict__ idx1) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t k = keys[i];
    idx0[i] = (int32_t)k;
    if (idx1) idx1[i] = flux_index(k, ny, nx);
}

__global__ void k_list_keys(const int32_t* __restrict__ cell, int64_t nsub, int64_t* __restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 4 * nsub) keys[i] = (int64_t)cell[i >> 2] * 4 + (i & 3);
}

__global__ void k_scale_offsets(const int64_t* __restrict__ in, int n, int64_t mult, int64_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] * mult;
}


// ---- panel plan: CSR rows (panel, transect) -------------------------------------------------------------
constexpr int kMaxPanels = 64;

// one warp per transect, 32 consecutive entries per step.  Entries that fall into the same panel keep their order
// (rank inside the step from __match_any_sync, running position per panel in shared memory) -> every
// (panel, transect) row lists its entries in the order of the transect's CSR row: deterministic sums.
constexpr int kPanelRowsWarps = 4;
template <bool FILL>
__global__ void k_panel_rows(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ idx,
                             const double* __restrict__ w, int ntransects, int64_t ncell, int64_t panel_cells,
                             int npanels, int64_t* __restrict__ counts, const int64_t* __restrict__ prow,
                             int32_t* __restrict__ pidx, double* __restrict__ pw) {
    extern __shared__ int64_t s_pos[];   // [warps per block][npanels]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int m = blockIdx.x * kPanelRowsWarps + wid;
    if (m >= ntransects) return;         // whole warps leave together
    int64_t* pos = s_pos + (int64_t)wid * npanels;
    for (int q = lane; q < npanels; q += 32) pos[q] = FILL ? prow[(int64_t)q * ntransects + m] : 0;
    __syncwarp();
    const int64_t end = rowptr[m + 1];
    for (int64_t base = rowptr[m]; base < end; base += 32) {
        const int64_t n = base + lane;
        const int32_t f = n < end ? idx[n] : -1;
        const bool act = f >= 0;         // f < 0: south edge of row 0, always 0 (field.py:61,219)
        const int is_v = act && f >= ncell;
        const int64_t c = is_v ? f - ncell : f;
        const int q = act ? (int)(c / panel_cells) : npanels + lane;   // inactive lanes: a key of their own
        const unsigned same = __match_any_sync(0xffffffffu, q);
        const int rank = __popc(same & ((1u << lane) - 1u));
        const int64_t p0 = act ? pos[q] : 0;
        __syncwarp();
        if (act && rank == 0) pos[q] = p0 + __popc(same);
        __syncwarp();
        if (FILL && act) {
            const int64_t c0 = (int64_t)q * panel_cells;
            const int64_t pc = min(panel_cells, ncell - c0);
            pidx[p0 + rank] = (int32_t)((c - c0) + (is_v ? pc : 0));
            pw[p0 + rank] = w[n];
        }
    }
    if (!FILL)
        for (int q = lane; q < npanels; q += 32) counts[(int64_t)q * ntransects + m] = pos[q];
}

// ---- column groups of the sparse fused pass: panel q holds the groups [q * gpp, q * gpp + gpp) of vec columns ------
__global__ void k_group_flags(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ idx, int ntransects,
                              int64_t ncell, int64_t panel_cells, int vec, int64_t gpp, int64_t* __restrict__ flags) {
    const int q = blockIdx.y;
    const int64_t pc = min(panel_cells, ncell - (int64_t)q * panel_cells);
    const int64_t e1 = rowptr[(int64_t)(q + 1) * ntransects];
    for (int64_t n = rowptr[(int64_t)q * ntransects] + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < e1;
         n += (int64_t)gridDim.x * blockDim.x) {
        const int64_t f = idx[n];   // [eU | eV] of the panel: u column f, or v column f - pc
        flags[q * gpp + (f < pc ? f : f - pc) / vec] = 1;
    }
}

// grp[pos[i]] = panel-local index of every flagged group i, grp_ptr[q] = position of the first group of panel q
__global__ void k_group_compact(const int64_t* __restrict__ flags, const int64_t* __restrict__ pos, int64_t ng,
                                int64_t gpp, int npanels, int32_t* __restrict__ grp, int64_t* __restrict__ grp_ptr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ng && flags[i]) grp[pos[i]] = (int32_t)(i % gpp);
    if (i <= npanels) grp_ptr[i] = pos[min(i * gpp, ng)];
}

}  // namespace

// A one-off per (plan, vector width): runs on the first fused pass after computeWeights, outside any time-step loop.
void build_column_groups(PanelPlan& pl, int64_t ncell, int ntransects, int vec, cudaStream_t s) {
    NFX_REQUIRE(pl.built, "column groups: the panel plan is not built");
    NFX_REQUIRE(pl.npanels == 1 || pl.panel_cells % vec == 0, "column groups: a group would straddle two panels");
    const int64_t gpp = (pl.panel_cells + vec - 1) / vec;
    const int64_t ng = (ncell + vec - 1) / vec;   // = (npanels - 1) * gpp + the groups of the last panel
    DevBuf<int64_t> flags, pos, tmp;
    flags.alloc((size_t)ng);
    pos.alloc((size_t)ng + 1);
    NFX_CUDA(cudaMemsetAsync(flags.p, 0, sizeof(int64_t) * ng, s));
    if (pl.nnz > 0) {
        const int64_t per_panel = std::max<int64_t>(1, pl.nnz / pl.npanels);
        const dim3 grid(nblk(std::min<int64_t>(per_panel, (int64_t)256 * 1024), 256), (unsigned)pl.npanels);
        k_group_flags<<<grid, 256, 0, s>>>(pl.rowptr.p, pl.idx.p, ntransects, ncell, pl.panel_cells, vec, gpp, flags.p);
        count_launch();
    }
    exclusive_scan(flags.p, pos.p, ng, tmp, s);
    int64_t total = 0;
    NFX_CUDA(cudaMemcpyAsync(&total, pos.p + ng, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaStreamSynchronize(s));
    pl.grp.ensure((size_t)std::max<int64_t>(total, 1));
    pl.grp_ptr.ensure((size_t)pl.npanels + 1);
    k_group_compact<<<nblk(std::max<int64_t>(ng, pl.npanels + 1), 256), 256, 0, s>>>(flags.p, pos.p, ng, gpp, pl.npanels,
                                                                                    pl.grp.p, pl.grp_ptr.p);
    count_launch();
    NFX_CUDA(cudaGetLastError());
    std::vector<int64_t> h_ptr((size_t)pl.npanels + 1);
    NFX_CUDA(cudaMemcpyAsync(h_ptr.data(), pl.grp_ptr.p, sizeof(int64_t) * h_ptr.size(), cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaStreamSynchronize(s));   // before the scratch buffers go
    int64_t mx = 0;
    for (int q = 0; q < pl.npanels; ++q) mx = std::max(mx, h_ptr[q + 1] - h_ptr[q]);
    pl.ngroups = total;
    pl.ngroups_all = ng;
    pl.max_grp_per_panel = (int)mx;
    pl.grp_vec = vec;
}

void build_panel_plan(PliDev& p, int order, int64_t panel_cells, cudaStream_t s) {
    NFX_REQUIRE(p.has_compact, "the flux path needs nfx_grid_set_cgrid_shape before computeWeights");
    PanelPlan& pl = p.plan[order];
    const Csr& c = p.csr[order][1];
    const int64_t ncell = p.grid->ncell;
    const int M = p.ntransects;
    const int npanels = (int)((ncell + panel_cells - 1) / panel_cells);
    NFX_REQUIRE(npanels >= 1 && npanels <= kMaxPanels, "panel plan: too many panels");
    pl.panel_cells = panel_cells;
    pl.npanels = npanels;
    pl.grp_vec = 0;
    const int64_t nrows = (int64_t)npanels * M;
    pl.rowptr.ensure((size_t)nrows + 1);
    if (M == 0 || c.nnz == 0) {
        NFX_CUDA(cudaMemsetAsync(pl.rowptr.p, 0, sizeof(int64_t) * (nrows + 1), s));
        pl.sr_ptr.ensure(1);
        pl.panel_sr.ensure((size_t)npanels + 1);
        pl.tr_ptr.ensure((size_t)M + 1);
        pl.tr_sr.ensure(1);
        NFX_CUDA(cudaMemsetAsync(pl.sr_ptr.p, 0, sizeof(int64_t), s));
        NFX_CUDA(cudaMemsetAsync(pl.panel_sr.p, 0, sizeof(int64_t) * (npanels + 1), s));
        NFX_CUDA(cudaMemsetAsync(pl.tr_ptr.p, 0, sizeof(int64_t) * (M + 1), s));
        pl.nnz = 0;
        pl.nsr = 0;
        pl.max_sr_per_panel = 0;
        pl.h_panel_sr.assign((size_t)npanels + 1, 0);
        pl.built = true;
        return;
    }
    DevBuf<int64_t> counts;
    counts.alloc((size_t)nrows);
    const size_t pr_smem = sizeof(int64_t) * kPanelRowsWarps * (size_t)npanels;
    k_panel_rows<false><<<nblk(M, kPanelRowsWarps), 32 * kPanelRowsWarps, pr_smem, s>>>(
        c.rowptr.p, c.idx.p, c.w, M, ncell, panel_cells, npanels, counts.p, nullptr, nullptr, nullptr);
    count_launch();
    NFX_CUDA(cudaGetLastError());
    // the index arrays are small (npanels*M rows): build them on the host
    std::vector<int64_t> h_cnt((size_t)nrows), h_rowptr((size_t)nrows + 1, 0);
    NFX_CUDA(cudaMemcpyAsync(h_cnt.data(), counts.p, sizeof(int64_t) * nrows, cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaStreamSynchronize(s));
    for (int64_t r = 0; r < nrows; ++r) h_rowptr[r + 1] = h_rowptr[r] + h_cnt[r];
    const int64_t nnz = h_rowptr[nrows];
    std::vector<int64_t> sr_ptr, panel_sr((size_t)npanels + 1, 0), tr_ptr((size_t)M + 1, 0), tr_sr;
    std::vector<std::vector<int64_t>> per_tr((size_t)M);
    int max_sr = 0;
    for (int q = 0; q < npanels; ++q) {
        panel_sr[q] = (int64_t)sr_ptr.size();
        for (int m = 0; m < M; ++m) {
            const int64_t a = h_rowptr[(int64_t)q * M + m], b = h_rowptr[(int64_t)q * M + m + 1];
            for (int64_t e = a; e < b; e += kSubRow) {
                per_tr[m].push_back((int64_t)sr_ptr.size());
                sr_ptr.push_back(e);
            }
        }
        max_sr = std::max<int>(max_sr, (int)((int64_t)sr_ptr.size() - panel_sr[q]));
    }
    panel_sr[npanels] = (int64_t)sr_ptr.size();
    const int64_t nsr = (int64_t)sr_ptr.size();
    sr_ptr.push_back(nnz);
    for (int m = 0; m < M; ++m) {
        tr_ptr[m + 1] = tr_ptr[m] + (int64_t)per_tr[m].size();
        tr_sr.insert(tr_sr.end(), per_tr[m].begin(), per_tr[m].end());
    }
    pl.nnz = nnz;
    pl.nsr = nsr;
    pl.max_sr_per_panel = max_sr;
    pl.h_panel_sr = panel_sr;
    pl.idx.ensure((size_t)std::max<int64_t>(nnz, 1));
    pl.w.ensure((size_t)std::max<int64_t>(nnz, 1));
    pl.sr_ptr.ensure((size_t)nsr + 1);
    pl.panel_sr.ensure((size_t)npanels + 1);
    pl.tr_ptr.ensure((size_t)M + 1);
    pl.tr_sr.ensure((size_t)std::max<int64_t>(nsr, 1));
    NFX_CUDA(cudaMemcpyAsync(pl.rowptr.p, h_rowptr.data(), sizeof(int64_t) * (nrows + 1), cudaMemcpyHostToDevice, s));
    NFX_CUDA(cudaMemcpyAsync(pl.sr_ptr.p, sr_ptr.data(), sizeof(int64_t) * (nsr + 1), cudaMemcpyHostToDevice, s));
    NFX_CUDA(cudaMemcpyAsync(pl.panel_sr.p, panel_sr.data(), sizeof(int64_t) * (npanels + 1), cudaMemcpyHostToDevice, s));
    NFX_CUDA(cudaMemcpyAsync(pl.tr_ptr.p, tr_ptr.data(), sizeof(int64_t) * (M + 1), cudaMemcpyHostToDevice, s));
    if (nsr > 0)
        NFX_CUDA(cudaMemcpyAsync(pl.tr_sr.p, tr_sr.data(), sizeof(int64_t) * nsr, cudaMemcpyHostToDevice, s));
    k_panel_rows<true><<<nblk(M, kPanelRowsWarps), 32 * kPanelRowsWarps, pr_smem, s>>>(
        c.rowptr.p, c.idx.p, c.w, M, ncell, panel_cells, npanels, nullptr, pl.rowptr.p, pl.idx.p, pl.w.p);
    count_launch();
    NFX_CUDA(cudaGetLastError());
    NFX_CUDA(cudaStreamSynchronize(s));   // the host vectors go out of scope
    pl.built = true;
}

// ---- arc lengths on the device (optional, NOT the parity path) -----------------------------------------
// arc[c, e] = great-circle length of edge e -> e+1 on the unit sphere from the haversine of the lon/lat
// DIFFERENCES: hav = sin^2(dlat/2) + cos(lat1) cos(lat2) sin^2(dlon/2), arc = 2 asin(sqrt(hav)) -- accurate to a
// few ulp for edges of any length, unlike the reference's arccos(a.b) (geo.py:24-27) whose rounding noise is
// ~1e-16/arc.  The parity path keeps the reference formula on the host (nemoflux_b200/geo.py); this kernel
// serves callers that want the metric factors fast (13 M cells in ~1 ms) and more accurate.
__global__ void k_arc_lengths(const double2* __restrict__ verts, int64_t ncell, double* __restrict__ arc) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncell * 4) return;
    const int64_t c = i >> 2;
    const int e = (int)(i & 3);
    const double2 p = verts[c * 4 + e], q = verts[c * 4 + ((e + 1) & 3)];
    const double d2r = 0.017453292519943295;
    const double sdl = sin(0.5 * (q.x - p.x) * d2r);
    const double sdp = sin(0.5 * (q.y - p.y) * d2r);
    const double hav = sdp * sdp + cos(p.y * d2r) * cos(q.y * d2r) * sdl * sdl;
    arc[i] = 2.0 * asin(fmin(1.0, sqrt(hav)));
}

// ---- host side --------------------------------------------------------------------------------------
void grid_upload_points(GridDev& g, int64_t ncells, const double* points_host) {
    NFX_REQUIRE(ncells > 0, "nfx_grid_set_points: ncells must be positive");
    NFX_REQUIRE(points_host != nullptr, "nfx_grid_set_points: points is NULL");
    NFX_REQUIRE(ncells * 4 < (int64_t)2147483647, "nfx_grid_set_points: ncells*4 must fit in int32");
    DevBuf<double> tmp;
    tmp.alloc((size_t)ncells * 12);
    NFX_CUDA(cudaMemcpy(tmp.p, points_host, sizeof(double) * (size_t)ncells * 12, cudaMemcpyHostToDevice));
    g.verts.alloc((size_t)ncells * 4);
    k_pack_points<<<nblk(ncells * 4, 256), 256>>>(tmp.p, g.verts.p, ncells * 4);
    count_launch();
    NFX_CUDA(cudaGetLastError());
    NFX_CUDA(cudaDeviceSynchronize());
    g.ncell = ncells;
    g.locator_built = false;
}

void grid_arc_lengths(GridDev& g, double* arc_dev, cudaStream_t s) {
    NFX_REQUIRE(g.ncell > 0 && arc_dev, "arcLengths: the grid has no points / NULL output");
    k_arc_lengths<<<nblk(g.ncell * 4, 256), 256, 0, s>>>(g.verts.p, g.ncell, arc_dev);
    count_launch();
    NFX_CUDA(cudaGetLastError());
}

void grid_build_locator(GridDev& g, cudaStream_t s) {
    if (g.locator_built) return;
    NFX_REQUIRE(g.ncell > 0, "buildLocator: the grid has no points");
    g.nl1 = (g.ncell + kFan - 1) / kFan;
    g.nl2 = (g.nl1 + kFan - 1) / kFan;
    g.nl3 = (g.nl2 + kFan - 1) / kFan;
    g.box1.alloc((size_t)g.nl1);
    g.box2.alloc((size_t)g.nl2);
    g.box3.alloc((size_t)g.nl3);
    k_build_box1<<<nblk(g.nl1 * 32, 256), 256, 0, s>>>(g.verts.p, g.ncell, g.box1.p, g.nl1);
    k_build_box2<<<nblk(g.nl2 * 32, 256), 256, 0, s>>>(g.box1.p, g.nl1, g.box2.p, g.nl2);
    k_build_box2<<<nblk(g.nl3 * 32, 256), 256, 0, s>>>(g.box2.p, g.nl2, g.box3.p, g.nl3);   // same reduction, one level up
    count_launch(3);
    NFX_CUDA(cudaGetLastError());
    {   // bounding box of the grid from the top level -> mean cell size (K1's estimate of the sub-segment count)
        std::vector<double4> top((size_t)g.nl3);
        NFX_CUDA(cudaMemcpyAsync(top.data(), g.box3.p, sizeof(double4) * g.nl3, cudaMemcpyDeviceToHost, s));
        NFX_CUDA(cudaStreamSynchronize(s));
        double x0 = 1.0e300, x1 = -1.0e300, y0 = 1.0e300, y1 = -1.0e300;
        for (const double4& b : top) {
            x0 = std::min(x0, b.x);
            x1 = std::max(x1, b.y);
            y0 = std::min(y0, b.z);
            y1 = std::max(y1, b.w);
        }
        const double area = (x1 - x0) * (y1 - y0);
        g.mean_cell = area > 0.0 ? std::sqrt(area / (double)g.ncell) : 0.0;
    }
    g.locator_built = true;
}

void pli_compute_weights(PliDev& p, int ntransects, const int* offsets, const double* xyz, int counterclock,
                         cudaStream_t s) {
    NFX_REQUIRE(p.grid != nullptr, "computeWeights: setGrid was not called");
    NFX_REQUIRE(p.locator_requested && p.grid->locator_built, "computeWeights: buildLocator was not called");
    NFX_REQUIRE(ntransects >= 0, "computeWeights: negative number of transects");
    NFX_REQUIRE(ntransects == 0 || (offsets && xyz), "computeWeights: NULL offsets/xyz");
    GridDev& g = *p.grid;
    const int nimg = p.period_x > 0.0 ? 3 : 1;

    // segments of all transects
    std::vector<SegIn> segs;
    std::vector<int32_t> seg_local;         // index of the segment inside its transect
    std::vector<int64_t> tr_seg_off(ntransects + 1, 0);
    for (int m = 0; m < ntransects; ++m) {
        NFX_REQUIRE(offsets[m + 1] >= offsets[m], "computeWeights: offsets must be non-decreasing");
        const int np = offsets[m + 1] - offsets[m];
        for (int q = 0; q + 1 < np; ++q) {
            const double* a = xyz + 3 * (size_t)(offsets[m] + q);
            segs.push_back(SegIn{a[0], a[1], a[3], a[4]});
            seg_local.push_back(q);
        }
        tr_seg_off[m + 1] = (int64_t)segs.size();
    }
    const int nseg = (int)segs.size();
    const int64_t nw = (int64_t)nseg * nimg * kPieces;   // warps of the traversal: (segment, image, piece)

    p.ntransects = ntransects;
    p.nsub = 0;
    p.nmap = 0;
    p.h_sub_offsets.assign(ntransects + 1, 0);
    p.h_map_offsets.assign(ntransects + 1, 0);
    p.has_compact = (g.ny > 0 && g.nx > 0);
    p.plan[0].built = p.plan[1].built = false;
    p.class_ntiles = -1;
    for (int o = 0; o < 2; ++o)
        for (int l = 0; l < 2; ++l) p.csr[o][l].nnz = 0;
    p.sub_offsets.ensure(ntransects + 1);
    p.map_offsets.ensure(ntransects + 1);
    if (nseg == 0) {
        NFX_CUDA(cudaMemsetAsync(p.sub_offsets.p, 0, sizeof(int64_t) * (ntransects + 1), s));
        NFX_CUDA(cudaMemsetAsync(p.map_offsets.p, 0, sizeof(int64_t) * (ntransects + 1), s));
        for (int o = 0; o < 2; ++o)
            for (int l = 0; l < 2; ++l) {
                p.csr[o][l].rowptr.ensure(ntransects + 1);
                NFX_CUDA(cudaMemsetAsync(p.csr[o][l].rowptr.p, 0, sizeof(int64_t) * (ntransects + 1), s));
            }
        NFX_CUDA(cudaStreamSynchronize(s));
        return;
    }

    // temporaries come from the handle's scratch arena: (1) the per-segment arrays, sized now; (2) after the count
    // pass the arena is grown once for the per-sub-segment arrays (76 bytes each) and the small arrays are re-taken
    DevBuf<int64_t>& d_tmp = p.scan_tmp;
    // record list of the count pass (see RecList): sized from the previous call on this handle, else from the
    // lengths of the segments over the mean cell size; too small = the fill pass traverses again, nothing else
    int64_t rec_slots = 0;
    {
        double est = 0.0;
        if (p.nsub_hint > 0) {
            est = 1.25 * (double)p.nsub_hint;
        } else if (g.mean_cell > 0.0) {
            for (const SegIn& sg : segs)
                est += 1.2 * (std::fabs(sg.p1x - sg.p0x) + std::fabs(sg.p1y - sg.p0y)) / g.mean_cell + 2.0;
        }
        est += (double)kRecChunk * (double)(nw / 2 + 1);          // partly filled chunks
        if (est * 28.0 <= 1.0e9) rec_slots = ((int64_t)est + kRecChunk - 1) / kRecChunk * kRecChunk;
    }
    const size_t small_bytes = 256 * 16 + sizeof(SegIn) * nseg + sizeof(int32_t) * 2 * (size_t)nseg +
                               sizeof(int64_t) * (2 * (size_t)nw + (size_t)nseg + 2) + 28 * (size_t)rec_slots + 8;
    p.scratch.ensure(std::max(small_bytes, p.scratch_hint));   // the size the previous call ended with: no regrowth
    Arena ar{p.scratch.p, p.scratch.n, 0};
    auto d_segs = ar.take<SegIn>(nseg);
    auto d_seg_local = ar.take<int32_t>(nseg);
    auto d_counts = ar.take<int64_t>((size_t)nw);
    auto d_off = ar.take<int64_t>((size_t)nw + 1);
    auto rec_n = ar.take<unsigned long long>(1);
    auto rec_w = ar.take<int32_t>((size_t)rec_slots);
    auto rec_i = ar.take<int32_t>((size_t)rec_slots);
    auto rec_c = ar.take<int32_t>((size_t)rec_slots);
    auto rec_ta = ar.take<double>((size_t)rec_slots);
    auto rec_tb = ar.take<double>((size_t)rec_slots);
    NFX_CUDA(cudaMemcpyAsync(d_segs.p, segs.data(), sizeof(SegIn) * nseg, cudaMemcpyHostToDevice, s));
    NFX_CUDA(cudaMemcpyAsync(d_seg_local.p, seg_local.data(), sizeof(int32_t) * nseg, cudaMemcpyHostToDevice, s));
    NFX_CUDA(cudaMemsetAsync(rec_n.p, 0, sizeof(unsigned long long), s));
    RecList rec{rec_n.p, rec_slots / kRecChunk, rec_w.p, rec_i.p, rec_c.p, rec_ta.p, rec_tb.p};

    // count (and record)
    const unsigned tb = nblk(nw * 32, 128);
    k1_traverse<false><<<tb, 128, 0, s>>>(g.verts.p, g.ncell, g.box1.p, g.nl1, g.box2.p, g.nl2, g.box3.p, g.nl3, d_segs.p, nseg, nimg,
                                         p.period_x, d_counts.p, nullptr, nullptr, nullptr, nullptr, nullptr, rec);
    count_launch();
    NFX_CUDA(cudaGetLastError());
    exclusive_scan(d_counts.p, d_off.p, nw, d_tmp, s);
    std::vector<int64_t> h_off((size_t)nw + 1);
    unsigned long long h_chunks = 0;
    NFX_CUDA(cudaMemcpyAsync(h_off.data(), d_off.p, sizeof(int64_t) * (nw + 1), cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaMemcpyAsync(&h_chunks, rec_n.p, sizeof h_chunks, cudaMemcpyDeviceToHost, s));
    NFX_CUDA(cudaStreamSynchronize(s));
    const int64_t nsub = h_off[nw];
    p.nsub = nsub;
    p.nsub_hint = nsub;
    const bool rec_ok = rec.cap_chunks > 0 && (int64_t)h_chunks <= rec.cap_chunks;

    // per-segment / per-transect offsets
    std::vector<int64_t> h_seg_off(nseg + 1);
    int64_t max_seg = 0;
    for (int q = 0; q <= nseg; ++q) h_seg_off[q] = h_off[(size_t)q * nimg * kPieces];
    for (int q = 0; q < nseg; ++q) max_seg = std::max(max_seg, h_seg_off[q + 1] - h_seg_off[q]);
    int64_t max_tr = 0;
    for (int m = 0; m <= ntransects; ++m) p.h_sub_offsets[m] = h_seg_off[tr_seg_off[m]];
    for (int m = 0; m < ntransects; ++m) max_tr = std::max(max_tr, p.h_sub_offsets[m + 1] - p.h_sub_offsets[m]);
    NFX_CUDA(cudaMemcpyAsync(p.sub_offsets.p, p.h_sub_offsets.data(), sizeof(int64_t) * (ntransects + 1),
                             cudaMemcpyHostToDevice, s));

    const size_t ns = (size_t)std::max<int64_t>(nsub, 1);
    p.cell.ensure(ns);
    p.seg.ensure(ns);
    p.img.ensure(ns);
    p.ta.ensure(ns);
    p.tb.ensure(ns);
    p.coeff.ensure(ns);
    p.xia.ensure(2 * ns);
    p.xib.ensure(2 * ns);
    p.w.ensure(4 * ns);

    if (p.scratch.n < small_bytes + 256 * 16 + 76 * ns + 8) {
        // grow: the small arrays move to the new buffer (the stream is idle: h_off was just read back)
        DevBuf<unsigned char> bigger;
        bigger.alloc(small_bytes + 256 * 16 + 76 * ns + 8);
        NFX_CUDA(cudaMemcpyAsync(bigger.p, p.scratch.p, ar.used, cudaMemcpyDeviceToDevice, s));
        NFX_CUDA(cudaStreamSynchronize(s));
        std::swap(bigger.p, p.scratch.p);
        std::swap(bigger.n, p.scratch.n);
        std::swap(bigger.raw, p.scratch.raw);
        const size_t used = ar.used;
        ar = Arena{p.scratch.p, p.scratch.n, used};
        auto rebase = [&](auto& view) {   // same offset in the new buffer (bigger.p is the old one after the swap)
            using PT = decltype(view.p);
            view.p = reinterpret_cast<PT>(p.scratch.p + ((unsigned char*)view.p - bigger.p));
        };
        rebase(d_segs);
        rebase(d_seg_local);
        rebase(d_counts);
        rebase(d_off);
        rebase(rec_n);
        rebase(rec_w);
        rebase(rec_i);
        rebase(rec_c);
        rebase(rec_ta);
        rebase(rec_tb);
        rec = RecList{rec_n.p, rec.cap_chunks, rec_w.p, rec_i.p, rec_c.p, rec_ta.p, rec_tb.p};
    }
    auto d_seg_off = ar.take<int64_t>(nseg + 1);
    NFX_CUDA(cudaMemcpyAsync(d_seg_off.p, h_seg_off.data(), sizeof(int64_t) * (nseg + 1), cudaMemcpyHostToDevice, s));

    if (nsub > 0) {
        // fill
        const size_t mark = ar.used;
        auto r_cell = ar.take<int32_t>(ns);
        auto r_img = ar.take<int32_t>(ns);
        auto seg_global = ar.take<int32_t>(ns);
        auto r_ta = ar.take<double>(ns);
        auto r_tb = ar.take<double>(ns);
        auto kb = ar.take<int64_t>(ns);
        auto perm = ar.take<int64_t>(ns);
        if (rec_ok) {   // the count pass recorded every hit: scatter instead of a second traversal
            const int64_t nslots = (int64_t)h_chunks * kRecChunk;
            if (nslots > 0)
                k_scatter_records<<<nblk(nslots, 256), 256, 0, s>>>(rec, nslots, d_off.p, nimg, r_cell.p, r_img.p, r_ta.p,
                                                                   r_tb.p);
        } else {
            k1_traverse<true><<<tb, 128, 0, s>>>(g.verts.p, g.ncell, g.box1.p, g.nl1, g.box2.p, g.nl2, g.box3.p, g.nl3,
                                                d_segs.p, nseg, nimg, p.period_x, nullptr, d_off.p, r_cell.p, r_img.p,
                                                r_ta.p, r_tb.p, RecList{nullptr, 0, nullptr, nullptr, nullptr, nullptr,
                                                                        nullptr});
        }
        // sort inside each segment by (ta, cell, image)
        k_make_sort1_key<<<nblk(nsub, 256), 256, 0, s>>>(r_cell.p, r_img.p, nsub, kb.p);
        auto ska = ar.take<double>(ns);
        auto skb = ar.take<int64_t>(ns);
        sort_in_groups<true>(r_ta.p, kb.p, d_seg_off.p, nseg, max_seg, ska.p, skb.p, perm.p, s);
        k_apply_sort1<<<nblk(nsub, 256), 256, 0, s>>>(perm.p, nsub, r_cell.p, r_img.p, r_ta.p, r_tb.p, p.cell.p, p.img.p,
                                                      p.ta.p, p.tb.p);
        // segment ids: local (reported) and global (index into segs)
        k_fill_seg_ids<<<nseg, 128, 0, s>>>(d_seg_off.p, nseg, d_seg_local.p, p.seg.p);
        k_fill_seg_ids<<<nseg, 128, 0, s>>>(d_seg_off.p, nseg, nullptr, seg_global.p);   // nullptr: the index itself
        k1_weights<<<nblk(nsub, 128), 128, 0, s>>>(g.verts.p, d_segs.p, seg_global.p, d_seg_off.p, p.cell.p, p.img.p,
                                                  p.ta.p, p.tb.p, nsub, p.period_x, counterclock, p.coeff.p, p.xia.p,
                                                  p.xib.p, p.w.p);
        count_launch(6);
        NFX_CUDA(cudaGetLastError());

        // mint map view: sort inside each transect by (cell, emission index), merge equal cells
        auto flags = ar.take<int64_t>(ns);
        auto uidx = ar.take<int64_t>(ns + 1);
        k_make_sort2_key<<<nblk(nsub, 256), 256, 0, s>>>(p.cell.p, nsub, kb.p);
        sort_in_groups<false>(nullptr, kb.p, p.sub_offsets.p, ntransects, max_tr, nullptr, skb.p, perm.p, s);
        k_run_flags<<<nblk(nsub, 256), 256, 0, s>>>(perm.p, p.cell.p, p.sub_offsets.p, ntransects, nsub, flags.p);
        count_launch(2);
        exclusive_scan(flags.p, uidx.p, nsub, d_tmp, s);
        int64_t nuniq = 0;
        NFX_CUDA(cudaMemcpyAsync(&nuniq, uidx.p + nsub, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        NFX_CUDA(cudaStreamSynchronize(s));
        p.nmap = 4 * nuniq;
        p.map_keys.ensure((size_t)p.nmap);
        p.map_w.ensure((size_t)p.nmap);
        k_map_fill<<<nblk(nsub, 256), 256, 0, s>>>(perm.p, p.cell.p, p.w.p, flags.p, uidx.p, nsub, p.map_keys.p,
                                                   p.map_w.p);
        k_map_offsets<<<nblk(ntransects + 1, 256), 256, 0, s>>>(p.sub_offsets.p, ntransects, uidx.p, p.map_offsets.p);
        count_launch(2);
        NFX_CUDA(cudaGetLastError());
        NFX_CUDA(cudaMemcpyAsync(p.h_map_offsets.data(), p.map_offsets.p, sizeof(int64_t) * (ntransects + 1),
                                 cudaMemcpyDeviceToHost, s));

        // CSR lists for K3
        // order LIST: 4 entries per sub-segment in emission order
        {
            ar.used = mark;   // everything taken since `mark` is dead in stream order: reuse the space
            auto lkeys = ar.take<int64_t>(4 * ns);
            k_list_keys<<<nblk(4 * nsub, 256), 256, 0, s>>>(p.cell.p, nsub, lkeys.p);
            for (int l = 0; l < 2; ++l) {
                Csr& c = p.csr[NFX_ORDER_LIST][l];
                c.nnz = 4 * nsub;
                c.w = p.w.p;
                c.rowptr.ensure(ntransects + 1);
                c.idx.ensure(4 * ns);
                k_scale_offsets<<<nblk(ntransects + 1, 256), 256, 0, s>>>(p.sub_offsets.p, ntransects + 1, 4, c.rowptr.p);
            }
            k_csr_from_keys<<<nblk(4 * nsub, 256), 256, 0, s>>>(lkeys.p, 4 * nsub, g.ny, g.nx,
                                                               p.csr[NFX_ORDER_LIST][0].idx.p,
                                                               p.has_compact ? p.csr[NFX_ORDER_LIST][1].idx.p : nullptr);
            count_launch(4);
            NFX_CUDA(cudaGetLastError());
        }
        // order MAP
        for (int l = 0; l < 2; ++l) {
            Csr& c = p.csr[NFX_ORDER_MAP][l];
            c.nnz = p.nmap;
            c.w = p.map_w.p;
            c.rowptr.ensure(ntransects + 1);
            c.idx.ensure((size_t)std::max<int64_t>(p.nmap, 1));
            NFX_CUDA(cudaMemcpyAsync(c.rowptr.p, p.map_offsets.p, sizeof(int64_t) * (ntransects + 1),
                                     cudaMemcpyDeviceToDevice, s));
        }
        k_csr_from_keys<<<nblk(p.nmap, 256), 256, 0, s>>>(p.map_keys.p, p.nmap, g.ny, g.nx,
                                                         p.csr[NFX_ORDER_MAP][0].idx.p,
                                                         p.has_compact ? p.csr[NFX_ORDER_MAP][1].idx.p : nullptr);
        count_launch();
        NFX_CUDA(cudaGetLastError());
        NFX_CUDA(cudaStreamSynchronize(s));
    } else {
        NFX_CUDA(cudaMemsetAsync(p.map_offsets.p, 0, sizeof(int64_t) * (ntransects + 1), s));
        for (int o = 0; o < 2; ++o)
            for (int l = 0; l < 2; ++l) {
                p.csr[o][l].rowptr.ensure(ntransects + 1);
                NFX_CUDA(cudaMemsetAsync(p.csr[o][l].rowptr.p, 0, sizeof(int64_t) * (ntransects + 1), s));
            }
        NFX_CUDA(cudaStreamSynchronize(s));
    }
    // the arena is kept for the next call unless it is large (ORCA12 with 1024 transects: 1.2 GB)
    p.scratch_hint = p.scratch.n;
    if (p.scratch.n > ((size_t)256 << 20)) {
        NFX_CUDA(cudaStreamSynchronize(s));
        p.scratch.release();
    }
}

}  // namespace nfx
