// iqr.cuh -- KissICP::iqr_processing (L/src/sensors/lidar/icp.cpp:88-124) + outlier::IQR / median
// (L/include/common.hpp:22-63) executed by ONE CTA of BLOCK threads (keypoint clouds are 1e3..1e5 points): squared
// ranges, the <= 4 order statistics outlier::IQR needs (medians of the lower and upper halves of the sorted ranges) by
// an 8-pass MSB radix select over the IEEE bit patterns (non-negative doubles order like unsigned integers), Tukey
// bounds with IQR_TUCHEY = 1.25 (common.hpp:15), then an order-preserving compaction of the inliers.
#pragma once
#include "compact.cuh"

namespace limu {

struct IqrSmem {
    int hist[4][256];
    unsigned long long prefix[4];
    int rank[4];
    int ws[32];
    int total;
};

template <int BLOCK>
__device__ __forceinline__ void iqr_block(IqrSmem &sm, const double *__restrict__ xyz, int n, double *__restrict__ d2, double *__restrict__ out,
                                          int *out_count, double *bounds) {
    const int tid = threadIdx.x;
    if (n <= 0) { if (tid == 0) *out_count = 0; return; }
    for (int i = tid; i < n; i += BLOCK) {
        const double x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
        d2[i] = x * x + y * y + z * z;   // icp.cpp:97-100
    }
    double q1, q3, iqr;
    const int half = n / 2, m = half, u0 = half + n % 2;
    if (n == 1) {
        __syncthreads();
        q1 = 0.0; q3 = d2[0]; iqr = d2[0];   // common.hpp:49-52
    } else {
        if (tid < 4) {
            const int lo = (m % 2 == 0) ? m / 2 - 1 : m / 2, hi = m / 2;   // median(): common.hpp:22-38
            sm.rank[tid] = (tid & 1 ? hi : lo) + (tid >= 2 ? u0 : 0);
            sm.prefix[tid] = 0ull;
        }
        for (int pass = 0; pass < 8; ++pass) {
            const int shift = 56 - 8 * pass;
            for (int b = tid; b < 4 * 256; b += BLOCK) (&sm.hist[0][0])[b] = 0;
            __syncthreads();
            for (int i = tid; i < n; i += BLOCK) {
                const unsigned long long bits = (unsigned long long)__double_as_longlong(d2[i]);
                const unsigned long long hi_bits = pass == 0 ? 0ull : (bits >> (shift + 8));
                const int digit = (int)((bits >> shift) & 0xFF);
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (hi_bits == sm.prefix[t]) atomicAdd(&sm.hist[t][digit], 1);
            }
            __syncthreads();
            const int warp = tid >> 5, lane = tid & 31;
            if (warp < 4) {
                int c[8], sum = 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) { c[k] = sm.hist[warp][lane * 8 + k]; sum += c[k]; }
                int incl = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += v; }
                int cum = incl - sum;
                const int r = sm.rank[warp];
                __syncwarp();
                if (r >= cum && r < incl) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        if (r < cum + c[k]) { sm.prefix[warp] = (sm.prefix[warp] << 8) | (unsigned long long)(lane * 8 + k); sm.rank[warp] = r - cum; break; }
                        cum += c[k];
                    }
                }
            }
            __syncthreads();
        }
        const double v0 = __longlong_as_double((long long)sm.prefix[0]), v1 = __longlong_as_double((long long)sm.prefix[1]);
        const double v2 = __longlong_as_double((long long)sm.prefix[2]), v3 = __longlong_as_double((long long)sm.prefix[3]);
        q1 = (m % 2 == 0) ? (v0 + v1) / 2.0 : v1;
        q3 = (m % 2 == 0) ? (v2 + v3) / 2.0 : v3;
        iqr = q3 - q1;
    }
    const double low = q1 - 1.25 * iqr, high = q3 + 1.25 * iqr;   // icp.cpp:104-105
    if (tid == 0 && bounds) { bounds[0] = low; bounds[1] = high; }
    int base = 0;
    for (int start = 0; start < n; start += BLOCK) {
        const int i = start + tid;
        const double d = i < n ? d2[i] : 0.0;
        const int f = i < n && d >= low && d <= high;   // icp.cpp:117
        const int r = block_exclusive_scan_flag(f, &sm.total, sm.ws);
        if (f) {
            out[3 * (size_t)(base + r)] = xyz[3 * (size_t)i];
            out[3 * (size_t)(base + r) + 1] = xyz[3 * (size_t)i + 1];
            out[3 * (size_t)(base + r) + 2] = xyz[3 * (size_t)i + 2];
        }
        base += sm.total;
        __syncthreads();
    }
    if (tid == 0) *out_count = base;
}

// ---- the same filter spread over the CTAs of the Gauss-Newton loop (used by the fused frame kernel in its latency shape) ----
// The one-CTA radix select above costs ~25 us per scan for ~2.3 k keypoints (eight dependent passes). Here each of those CTAs copies the
// squared ranges into its shared memory and its warps rank their share of the elements by counting (#smaller, ties by index -> unique
// ranks); the <= 4 elements whose rank is one of the wanted order statistics publish their value. After one barrier among those CTAs,
// every one of them derives the Tukey bounds and the inlier index list from its own shared copy (iqr_local_compact), and CTA 0 writes
// the keypoints out later (iqr_write_out). Same values as the select above (an order statistic is an order statistic), so the filtered
// cloud is bit-identical.
constexpr int IQR_GRID_MAX = 4096;        // capacity of the copy every CTA keeps in STATIC shared memory
constexpr int IQR_GRID_MAX_DYN = 16384;   // ... in dynamic shared memory, for launches whose hint announces more candidates (8192 or 16384 of them)

template <int BLOCK>
__device__ __forceinline__ void iqr_grid_select(double *sd2 /* shared, IQR_GRID_MAX */, const double *__restrict__ xyz, int n, double *sel /* global, 4 */,
                                                int nblocks /* CTAs 0..nblocks-1 share the ranking (0: the whole grid) */) {
    // eight candidates per thread and round, all 24 loads in flight before the first product: one candidate per round cost one L2 round trip
    // per 256 candidates (5 of the 7 us of this phase at 2.5 k candidates, 15 us at 7.4 k)
    constexpr int FB = 8;
    for (int i0 = threadIdx.x; i0 < n; i0 += BLOCK * FB) {
        double x[FB], y[FB], z[FB];
#pragma unroll
        for (int u = 0; u < FB; ++u) {
            const int i = i0 + u * BLOCK;
            const size_t k = 3 * (size_t)(i < n ? i : n - 1);
            x[u] = xyz[k]; y[u] = xyz[k + 1]; z[u] = xyz[k + 2];
        }
#pragma unroll
        for (int u = 0; u < FB; ++u) {
            const int i = i0 + u * BLOCK;
            if (i < n) sd2[i] = x[u] * x[u] + y[u] * y[u] + z[u] * z[u];   // icp.cpp:97-100
        }
    }
    __syncthreads();
    const int half = n / 2, m = half, u0 = half + n % 2;
    const int lo = (m % 2 == 0) ? m / 2 - 1 : m / 2, hi = m / 2;   // median(): common.hpp:22-38
    const int r0 = lo, r1 = hi, r2 = lo + u0, r3 = hi + u0;
    const int lane = threadIdx.x & 31;
    const int gwarp = blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5), nwarps = (nblocks > 0 ? nblocks : (int)gridDim.x) * (BLOCK / 32);
    // A warp ranks FOUR candidates at a time: one shared-memory load per comparison partner feeds four comparisons (the one-candidate
    // loop spent ~1.6 us per candidate on the latency of its 81 dependent load/compare rounds).
    for (int i0 = gwarp * 4; i0 < n; i0 += nwarps * 4) {   // warp-uniform trip count
        double d[4];
        int c[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { d[k] = sd2[i0 + k < n ? i0 + k : n - 1]; c[k] = 0; }
#pragma unroll 4
        for (int j = lane; j < n; j += 32) {
            const double e = sd2[j];
#pragma unroll
            for (int k = 0; k < 4; ++k) c[k] += (e < d[k] || (e == d[k] && j < i0 + k)) ? 1 : 0;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = __reduce_add_sync(0xFFFFFFFFu, c[k]);
            if (lane == 0 && i0 + k < n) {
                if (r == r0) sel[0] = d[k];
                if (r == r1) sel[1] = d[k];
                if (r == r2) sel[2] = d[k];
                if (r == r3) sel[3] = d[k];
            }
        }
    }
}

// Tukey bounds from the four order statistics, inlier flags and the order-preserving INDEX list, by one CTA in its own shared memory in a
// single pass (IQR_GRID_MAX / BLOCK consecutive candidates per thread, one block scan): every CTA that runs the Gauss-Newton loop derives
// the keypoint list itself, so nobody waits for CTA 0 to compact it (icp.cpp:103-121; same bounds and comparisons as iqr_block).
// Returns the keypoint count.
template <int BLOCK, int PER = IQR_GRID_MAX / BLOCK /* candidates per thread: capacity = BLOCK * PER */>
__device__ __forceinline__ int iqr_local_compact(int *ws /* shared, 32 */, int *total /* shared */, const double *sd2, int n0, const double *sel,
                                                 unsigned short *qidx /* shared, BLOCK * PER */) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m = n0 / 2;
    const double v0 = __ldcg(sel), v1 = __ldcg(sel + 1), v2 = __ldcg(sel + 2), v3 = __ldcg(sel + 3);
    const double q1 = (m % 2 == 0) ? (v0 + v1) / 2.0 : v1;
    const double q3 = (m % 2 == 0) ? (v2 + v3) / 2.0 : v3;
    const double iqr = q3 - q1;
    const double low = q1 - 1.25 * iqr, high = q3 + 1.25 * iqr;   // icp.cpp:104-105
    static_assert((PER & (PER - 1)) == 0 && PER <= 64, "candidates per thread: a power of two, one flag bit each");
    unsigned long long f = 0;
    int cnt = 0;
    constexpr int UNROLL = PER > 16 ? 8 : PER;   // (fully unrolled, the 32 / 64-candidate variants want every register the launch bounds allow)
#pragma unroll UNROLL
    for (int v = 0; v < PER; ++v) {
        const int u = (v + tid) & (PER - 1);                       // rotated visiting order: the lanes of a warp read different banks
        const int i = tid * PER + u;
        const double d = i < n0 ? sd2[i] : 0.0;
        const bool in = i < n0 && d >= low && d <= high;          // icp.cpp:117
        f |= (in ? 1ull : 0ull) << u;
        cnt += in ? 1 : 0;
    }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) ws[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int v = lane < BLOCK / 32 ? ws[lane] : 0;
        int wi = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, wi, o); if (lane >= o) wi += t; }
        ws[lane] = wi - v;
        if (lane == 31) *total = wi;
    }
    __syncthreads();
    int pos = ws[warp] + incl - cnt;
#pragma unroll UNROLL
    for (int u = 0; u < PER; ++u) {
        if (f & (1ull << u)) {
            const int i = tid * PER + u;
            qidx[pos] = (unsigned short)i;
            ++pos;
        }
    }
    const int n = *total;
    __syncthreads();
    return n;
}

// The keypoint cloud and its count for the host, written by ONE CTA from its index list -- after the Gauss-Newton loop, off everybody's
// critical path (inside the compaction, 16 dependent load -> store rounds of CTA 0 held up the first row exchange of every scan by ~10 us).
template <int BLOCK>
__device__ __forceinline__ void iqr_write_out(const unsigned short *qidx, const double *__restrict__ xyz, int n, double *__restrict__ out, int *out_count, int tid) {
    // tid in [0, BLOCK): the caller may leave some of the CTA's threads out. Four points per round, their loads in flight together.
    for (int p0 = tid; p0 < n; p0 += 4 * BLOCK) {
        double v[4][3];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * BLOCK;
            if (p < n) { const size_t i = qidx[p]; v[u][0] = xyz[3 * i]; v[u][1] = xyz[3 * i + 1]; v[u][2] = xyz[3 * i + 2]; }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int p = p0 + u * BLOCK;
            if (p < n) { out[3 * (size_t)p] = v[u][0]; out[3 * (size_t)p + 1] = v[u][1]; out[3 * (size_t)p + 2] = v[u][2]; }
        }
    }
    if (tid == 0) *out_count = n;
}

}  // namespace limu
