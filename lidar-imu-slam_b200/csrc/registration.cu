// registration.cu -- correspondence search + point-to-point residual/Jacobian + normal-equation
// reduction + the Gauss-Newton loop, fused into ONE persistent cooperative kernel.
// Replaces (L/ = env_ws/src/limu):
//   VoxelHashMap::get_correspondences / get_closest_neighbour  L/src/sensors/lidar/helpers/voxel_hash_map.cpp:64-130
//   lidar::align_clouds                                        L/src/sensors/lidar/helpers/registration.cpp:43-92
//   lidar::ICP                                                 registration.cpp:94-130
//
// Per iteration the reference materialises two correspondence vectors, reduces 42-double tuples with
// tbb::parallel_reduce, solves 6x6 on the host and rewrites the source cloud. Here every query thread
// does lookup -> gate -> weight -> 16 FP64 partial sums in registers (J = [I | -hat(s)] makes H and g
// functions of sum w, w s, w s s^T, w r, w s x r); warps shuffle-reduce, CTAs write one partial row,
// a grid barrier publishes them, and every CTA redundantly folds the rows in a fixed order and runs
// the identical LDLT / exp / log on one thread, so the next iteration starts without any host or
// second-barrier round trip. Sums are FP64 throughout; the fold order is fixed -> run-to-run deterministic.
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "grid_sync.cuh"
#include "icp_args.cuh"
#include "iqr.cuh"

namespace limu {

constexpr int ICP_BLOCK = 256;
#ifndef LIMU_BW_CTAS
#define LIMU_BW_CTAS 2   // CTAs per SM of the bandwidth shape (register cap 65536 / (256 * LIMU_BW_CTAS)); measured 2 > 3 > 4 (profiles/r2f_*)
#endif
constexpr int NS = 20;   // 16 sums + ncorr + ncand + nmiss + pad
constexpr int NSP = 32;  // opt-in point-to-plane variant: 21 (upper triangle of H) + 6 (g) + ncorr + ncand + nmiss + 2 pad

}  // namespace limu
LIMU_TRACE_RING(limu_debug_trace_reg)
namespace limu {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    return v;
}

// The 16 sums one gated correspondence adds to (registration.cpp:46-58,75-76); zeros when gated out. A gated-out query's
// coordinates are replaced by zeros too: weight 0 times a NaN or infinite source would be NaN and poison the normal equations.
__device__ __forceinline__ void contribution(double *c, const V3 &s_in, const V3 &t_in, double d2, double th, bool on) {
    const V3 s = on ? s_in : V3{0.0, 0.0, 0.0}, t = on ? t_in : V3{0.0, 0.0, 0.0};
    const double rx = s.x - t.x, ry = s.y - t.y, rz = s.z - t.z;       // residual = source - target (:48)
    const double den = th + d2;
    const double w = on ? (th * th) / (den * den) : 0.0;                // :57-58
    const double wx = w * s.x, wy = w * s.y, wz = w * s.z;
    c[0] = w;
    c[1] = wx; c[2] = wy; c[3] = wz;
    c[4] = wx * s.x; c[5] = wx * s.y; c[6] = wx * s.z;
    c[7] = wy * s.y; c[8] = wy * s.z; c[9] = wz * s.z;
    c[10] = w * rx; c[11] = w * ry; c[12] = w * rz;
    c[13] = w * (s.y * rz - s.z * ry);
    c[14] = w * (s.z * rx - s.x * rz);
    c[15] = w * (s.x * ry - s.y * rx);
}

// Warp reduce-scatter of 16 values per lane: after five exchange steps lane L holds the warp total of
// value L>>1 (both lanes of a pair hold it). 16 double shuffles per 32 queries instead of 16 x 5, and each
// lane carries ONE running FP64 accumulator instead of 16 (registers are what bounds occupancy here).
// The exchange pattern is fixed, so sums are run-to-run deterministic.
__device__ __forceinline__ double warp_reduce_scatter16(const double *c) {
    const int lane = threadIdx.x & 31;
    double d[8], e[4], f[2];
    const bool u16 = lane & 16, u8 = lane & 8, u4 = lane & 4, u2 = lane & 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) d[i] = (u16 ? c[i + 8] : c[i]) + __shfl_xor_sync(0xFFFFFFFFu, u16 ? c[i] : c[i + 8], 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) e[i] = (u8 ? d[i + 4] : d[i]) + __shfl_xor_sync(0xFFFFFFFFu, u8 ? d[i] : d[i + 4], 8);
#pragma unroll
    for (int i = 0; i < 2; ++i) f[i] = (u4 ? e[i + 2] : e[i]) + __shfl_xor_sync(0xFFFFFFFFu, u4 ? e[i] : e[i + 2], 4);
    const double g = (u2 ? f[1] : f[0]) + __shfl_xor_sync(0xFFFFFFFFu, u2 ? f[0] : f[1], 2);
    return g + __shfl_xor_sync(0xFFFFFFFFu, g, 1);
}

// ---- opt-in point-to-plane variant LIMU_ICP_PLANE (SURVEY section 8f N2; defined by the C oracle's plane_step) ------------
// One correspondence with plane normal n: e = n.(s - t), w = th^2/(th + e^2)^2, a = [n ; s x n] (the reference's perturbation
// model: J_point = [I | -hat(s)], registration.cpp:46-54), H += w a a^T (21 upper-triangle sums, row-major), g += w a e (6),
// plus the three counters as doubles: 32 values, one per lane after the reduce-scatter.
__device__ __forceinline__ void contribution_plane(double *c, const V3 &s, const V3 &t, const double *n, double th, bool on, int ncand, bool miss, bool lead) {
    const double e = (n[0] * (s.x - t.x) + n[1] * (s.y - t.y)) + n[2] * (s.z - t.z);
    const double den = th + e * e;
    const double w = on ? (th * th) / (den * den) : 0.0;
    const double a[6] = {n[0], n[1], n[2], s.y * n[2] - s.z * n[1], s.z * n[0] - s.x * n[2], s.x * n[1] - s.y * n[0]};
    int k = 0;
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        const double wa = w * a[r];
#pragma unroll
        for (int q = r; q < 6; ++q) c[k++] = wa * a[q];
    }
#pragma unroll
    for (int r = 0; r < 6; ++r) c[21 + r] = (w * a[r]) * e;
    c[27] = on ? 1.0 : 0.0;
    c[28] = lead ? (double)ncand : 0.0;
    c[29] = miss ? 1.0 : 0.0;
    c[30] = c[31] = 0.0;
}
// Warp reduce-scatter of 32 values per lane: lane L ends up with the warp total of value L (fixed exchange pattern).
__device__ __forceinline__ double warp_reduce_scatter32(const double *c) {
    const int lane = threadIdx.x & 31;
    double d[16], e[8], f[4], g[2];
    const bool u16 = lane & 16, u8 = lane & 8, u4 = lane & 4, u2 = lane & 2, u1 = lane & 1;
#pragma unroll
    for (int i = 0; i < 16; ++i) d[i] = (u16 ? c[i + 16] : c[i]) + __shfl_xor_sync(0xFFFFFFFFu, u16 ? c[i] : c[i + 16], 16);
#pragma unroll
    for (int i = 0; i < 8; ++i) e[i] = (u8 ? d[i + 8] : d[i]) + __shfl_xor_sync(0xFFFFFFFFu, u8 ? d[i] : d[i + 8], 8);
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = (u4 ? e[i + 4] : e[i]) + __shfl_xor_sync(0xFFFFFFFFu, u4 ? e[i] : e[i + 4], 4);
#pragma unroll
    for (int i = 0; i < 2; ++i) g[i] = (u2 ? f[i + 2] : f[i]) + __shfl_xor_sync(0xFFFFFFFFu, u2 ? f[i] : f[i + 2], 2);
    return (u1 ? g[1] : g[0]) + __shfl_xor_sync(0xFFFFFFFFu, u1 ? g[0] : g[1], 1);
}
constexpr double PLANE_PRIOR = 1.0, PLANE_PRIOR_ARM2 = 100.0;   // the oracle's LO_PLANE_PRIOR, LO_PLANE_PRIOR_ARM2: D = diag(mu x 3, mu rho^2 x 3)
// S[0..20] = upper triangle of H row-major, S[21..26] = g.
__device__ __forceinline__ void expand_plane_equations(const double *S, double *H, double *g) {
    int k = 0;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int q = r; q < 6; ++q) { H[6 * r + q] = S[k]; H[6 * q + r] = S[k]; ++k; }
#pragma unroll
    for (int r = 0; r < 6; ++r) g[r] = S[21 + r];
}

// Legacy-style accumulation used by the stand-alone align kernel (16 accumulators per thread).
__device__ __forceinline__ void accumulate(double *a, const V3 &s, const V3 &t, double d2, double th) {
    double c[16];
    contribution(c, s, t, d2, th, true);
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] += c[k];
}

// Block-level reduction of NS values per thread into row[NS] (fixed tree -> deterministic).
__device__ __forceinline__ void block_reduce_row(double *a, double *smem /* [ICP_BLOCK/32][NS] */, double *row) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NS; ++k) {
        const double v = warp_sum(a[k]);
        if (lane == 0) smem[warp * NS + k] = v;
    }
    __syncthreads();
    if (threadIdx.x < NS) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < ICP_BLOCK / 32; ++w) v += smem[w * NS + threadIdx.x];
        row[threadIdx.x] = v;
    }
}

// Cooperative candidate scan (VoxelBlock::get_closest_point, voxel_block.cpp:87-105): the warp works as four groups
// of eight lanes; in step t group g scans the voxel of ITS lane t. Eight lanes read ranks r..r+7 of the x / y / z rows
// = three 64-byte coalesced segments (instead of 32 scattered 8-byte loads per instruction), each lane keeps its best
// (d2, rank) and a 3-step butterfly leaves the lexicographic minimum -- smallest distance, then lowest rank = "first
// minimum wins" -- in every lane of the group. ROUNDS = ceil(cap / 8) is a template parameter so every load of a step
// is unconditional and can be issued before the first one is consumed (ROUNDS == 0: generic loop for cap > 24).
template <int ROUNDS>
__device__ __forceinline__ void coop_scan(const MapView &m, const V3 &s, int slot, int count, int lane, double &my_d2, int &my_rank) {
    const int l8 = lane & 7;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const double qx = __shfl_sync(0xFFFFFFFFu, s.x, t, 8), qy = __shfl_sync(0xFFFFFFFFu, s.y, t, 8), qz = __shfl_sync(0xFFFFFFFFu, s.z, t, 8);
        const int qslot = __shfl_sync(0xFFFFFFFFu, slot, t, 8);
        const int qcount = qslot >= 0 ? __shfl_sync(0xFFFFFFFFu, count, t, 8) : (__shfl_sync(0xFFFFFFFFu, count, t, 8), 0);
        const double *bx = voxel_rows(m, (unsigned int)(qslot >= 0 ? qslot : 0)), *by = bx + m.capp, *bz = by + m.capp;
        double bd = 1.7976931348623157e308;
        int br = 0x7FFFFFFF;
        if (ROUNDS > 0) {
            double x[ROUNDS > 0 ? ROUNDS : 1], y[ROUNDS > 0 ? ROUNDS : 1], z[ROUNDS > 0 ? ROUNDS : 1];
#pragma unroll
            for (int k = 0; k < ROUNDS; ++k) {   // out-of-range ranks re-read rank l8 (always inside the block) and are ignored below
                const int r = l8 + 8 * k, rr = r < qcount ? r : l8;
                x[k] = *(bx + rr); y[k] = *(by + rr); z[k] = *(bz + rr);
            }
#pragma unroll
            for (int k = 0; k < ROUNDS; ++k) {
                const int r = l8 + 8 * k;
                const double d = sqnorm3(qx - x[k], qy - y[k], qz - z[k]);
                if (r < qcount && d < bd) { bd = d; br = r; }
            }
        } else {
            for (int r = l8; r < qcount; r += 8) {
                const double d = sqnorm3(qx - *(bx + r), qy - *(by + r), qz - *(bz + r));
                if (d < bd) { bd = d; br = r; }
            }
        }
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            const double od = __shfl_xor_sync(0xFFFFFFFFu, bd, o);
            const int orr = __shfl_xor_sync(0xFFFFFFFFu, br, o);
            if (od < bd || (od == bd && orr < br)) { bd = od; br = orr; }
        }
        if (l8 == t) { my_d2 = bd; my_rank = br == 0x7FFFFFFF ? -1 : br; }
    }
}

// One pass over this warp's share of the queries: transform, locate, scan, gate, weight, accumulate.
// NN27: the opt-in neighbour rule LIMU_NN_27 (nearest point of the 27-cell neighbourhood, voxel_map.cuh) instead of the reference's.
template <bool NN27, bool PLANE>
__device__ __forceinline__ void icp_query_pass(const IcpArgs &A, const volatile double *Pv, const double *in, int64_t n, int64_t wbase, int64_t wstride,
                                               int lane, double &acc, int &ncorr, int &ncand, int &nmiss) {
    for (int64_t base = wbase; base < n; base += wstride) {
        const int64_t q = base + lane;
        const bool on = q < n;
        V3 s{0.0, 0.0, 0.0};
        int slot = -1, count = 0, own = 1;
        if (on) {
            // j == 0: source = init_guess * points (:102-103); later: source <- estimate * source (:119),
            // applied lazily at the next visit
            const Pose P{Pv[0], Pv[1], Pv[2], Pv[3], Pv[4], Pv[5], Pv[6]};
            s = apply(P, V3{in[3 * q], in[3 * q + 1], in[3 * q + 2]});
            A.work[3 * q] = s.x; A.work[3 * q + 1] = s.y; A.work[3 * q + 2] = s.z;
            if (!NN27) slot = map_locate(A.map, s, &count, &own);   // which voxel answers (own, else farthest/latest of the 27)
        }
        double my_d2 = 0.0;
        int my_rank = -1;
        if (NN27) {
            if (on) {
                const Nearest nn = map_closest27(A.map, s);
                slot = nn.slot; my_rank = nn.rank; count = nn.ncand; own = nn.own;
                my_d2 = sqnorm3(nn.x - s.x, nn.y - s.y, nn.z - s.z);
            }
        } else if (A.coop_scan) {
            if (A.map.cap <= 8) coop_scan<1>(A.map, s, slot, count, lane, my_d2, my_rank);
            else if (A.map.cap <= 16) coop_scan<2>(A.map, s, slot, count, lane, my_d2, my_rank);
            else if (A.map.cap <= 24) coop_scan<3>(A.map, s, slot, count, lane, my_d2, my_rank);
            else coop_scan<0>(A.map, s, slot, count, lane, my_d2, my_rank);
        } else if (slot >= 0) {
            // latency shape (a few thousand keypoint queries): every lane scans its own voxel, one L2 round trip per
            // four candidates instead of eight dependent group steps
            Nearest nn;
            block_closest(A.map, slot, count, s, nn);
            my_rank = nn.rank;
            my_d2 = sqnorm3(nn.x - s.x, nn.y - s.y, nn.z - s.z);
        }
        V3 tg{0.0, 0.0, 0.0};   // nothing found -> (0,0,0), range-tested like a real point (voxel_hash_map.cpp:98-99,118-124)
        if (my_rank >= 0) {
            const double *bx = voxel_rows(A.map, (unsigned int)slot);
            tg = V3{*(bx + my_rank), *(bx + A.map.capp + my_rank), *(bx + 2 * A.map.capp + my_rank)};
        }
        const double d2 = my_rank >= 0 ? my_d2 : sqnorm3(tg.x - s.x, tg.y - s.y, tg.z - s.z);   // (found - point).squaredNorm() :120
        const bool gate = on && d2 < A.tau_sq;
        if (PLANE) {
            double nrm[3] = {0.0, 0.0, 0.0};
            bool planar = false;
            if (gate && my_rank >= 0) planar = voxel_normal(A.map, slot, meta_count(load_slot(slot_at(A.map, (unsigned int)slot)).y), nrm) != 0;
            double c[32];
            contribution_plane(c, s, tg, nrm, A.th, planar, count, on && !own, on);
            acc += warp_reduce_scatter32(c);
        } else {
            double c[16];
            contribution(c, s, tg, d2, A.th, gate);
            acc += warp_reduce_scatter16(c);
            ncorr += gate ? 1 : 0;
            ncand += count;
            nmiss += (on && !own) ? 1 : 0;
        }
    }
}

// Lane l8 of a query's eight lanes owns sums 2*l8 and 2*l8+1 of the 16 (same expressions, same operation order as contribution()):
// every lane knows s, t and d2 once the lookup is done, so the eight lanes of a group produce the 16 values without any exchange and
// each keeps two running FP64 accumulators for the whole pass (SIMT: the redundant weight is free).
__device__ __forceinline__ void contribution_pair(int l8, const V3 &s, const V3 &t, double d2, double th, bool on, double &c0, double &c1) {
    const double rx = s.x - t.x, ry = s.y - t.y, rz = s.z - t.z;       // residual = source - target (:48)
    const double den = th + d2;
    const double w = on ? (th * th) / (den * den) : 0.0;                // :57-58
    const double wx = w * s.x, wy = w * s.y, wz = w * s.z;
    switch (l8) {
        case 0: c0 = w; c1 = wx; break;
        case 1: c0 = wy; c1 = wz; break;
        case 2: c0 = wx * s.x; c1 = wx * s.y; break;
        case 3: c0 = wx * s.z; c1 = wy * s.y; break;
        case 4: c0 = wy * s.z; c1 = wz * s.z; break;
        case 5: c0 = w * rx; c1 = w * ry; break;
        case 6: c0 = w * rz; c1 = w * (s.y * rz - s.z * ry); break;
        default: c0 = w * (s.z * rx - s.x * rz); c1 = w * (s.x * ry - s.y * rx); break;
    }
}

struct PlaneMemo { int slot, planar; double n[3]; };   // slot < 0: nothing remembered
// One pass over this warp's share of the queries with eight lanes per query (four queries per warp and step), see group8_closest.
// On return lane L holds the warp total of sum index L>>1 (the layout of warp_reduce_scatter16) in `acc`.
template <bool NN27, bool PLANE, int ROUNDS>
__device__ __forceinline__ void icp_query_pass_grouped(const IcpArgs &A, const volatile double *Pv, const double *in, const unsigned short *qidx, int64_t n, int64_t gbase,
                                                       int64_t gstride, int lane, double &acc, int &ncorr, int &ncand, int &nmiss, QueryMemo *memo, PlaneMemo *pmemo) {
    const int l8 = lane & 7;
    const unsigned gmask = 0xFFu << (lane & 24);
    const int64_t wfirst = gbase - (lane >> 3);   // first group of this warp: the four groups of a warp iterate together
    double a0 = 0.0, a1 = 0.0;                    // reference rules: sums 2*l8 and 2*l8+1 over this group's queries
    for (int64_t q0 = wfirst; q0 < n; q0 += gstride) {
        const int64_t q = q0 + (lane >> 3);
        const bool on = q < n;
        V3 s{0.0, 0.0, 0.0}, tg{0.0, 0.0, 0.0};
        int slot = -1, count = 0, own = 1, my_rank = -1;
        double d2 = 0.0;
        if (on) {
            const Pose P{Pv[0], Pv[1], Pv[2], Pv[3], Pv[4], Pv[5], Pv[6]};
            const size_t qi = qidx ? (size_t)qidx[q] : (size_t)q;   // first iteration of a fused frame: keypoint q is IQR candidate qidx[q]
            s = apply(P, V3{in[3 * qi], in[3 * qi + 1], in[3 * qi + 2]});
            if (l8 == 0) { A.work[3 * q] = s.x; A.work[3 * q + 1] = s.y; A.work[3 * q + 2] = s.z; }
            if (NN27) {
                group8_closest27(A.map, s, gmask, l8, slot, count, own, d2, my_rank);
                if (my_rank >= 0) {
                    const double *bx = voxel_rows(A.map, (unsigned int)slot);
                    tg = V3{ldm(bx + my_rank), ldm(bx + A.map.capp + my_rank), ldm(bx + 2 * A.map.capp + my_rank)};
                }
            } else {
                group8_closest<ROUNDS>(A.map, s, gmask, l8, slot, count, own, d2, my_rank, tg, q0 == wfirst ? memo : nullptr);   // (the memo belongs to the first query this group serves in a pass)
            }
            if (my_rank < 0) d2 = sqnorm3(tg.x - s.x, tg.y - s.y, tg.z - s.z);   // nothing found -> (0,0,0), range-tested like a real point
        }
        const bool lead = on && l8 == 0;
        if (PLANE) {
            const bool gate = lead && d2 < A.tau_sq;
            double nrm[3] = {0.0, 0.0, 0.0};
            bool planar = false;   // the group's leading lane fits the plane of the matched voxel (sequential sums: bit-identical to the oracle)
            if (gate && my_rank >= 0) {
                // the plane of a voxel does not change inside a launch: the fit (two passes over the voxel's points + 15 Jacobi rotations,
                // the longest serial stretch of an iteration) is kept for the voxel this group's first query matched last time
                if (q0 == wfirst && pmemo->slot == slot) {
                    planar = pmemo->planar != 0; nrm[0] = pmemo->n[0]; nrm[1] = pmemo->n[1]; nrm[2] = pmemo->n[2];
                } else {
                    planar = voxel_normal(A.map, slot, meta_count(load_slot(slot_at(A.map, (unsigned int)slot)).y), nrm) != 0;
                    if (q0 == wfirst) { pmemo->slot = slot; pmemo->planar = planar ? 1 : 0; pmemo->n[0] = nrm[0]; pmemo->n[1] = nrm[1]; pmemo->n[2] = nrm[2]; }
                }
            }
            double c[32];
            contribution_plane(c, s, tg, nrm, A.th, planar, count, lead && !own, lead);
            acc += warp_reduce_scatter32(c);
        } else {
            const bool gate = on && d2 < A.tau_sq;   // known to all eight lanes
            if (gate) {
                double c0, c1;
                contribution_pair(l8, s, tg, d2, A.th, true, c0, c1);
                a0 += c0; a1 += c1;
            }
            ncorr += (gate && l8 == 0) ? 1 : 0;
            ncand += lead ? count : 0;
            nmiss += (lead && !own) ? 1 : 0;
        }
    }
    if (!PLANE) {
        // four groups per warp -> warp totals, then into the reduce-scatter layout the row code expects (lane L: sum L>>1)
        a0 += __shfl_xor_sync(0xFFFFFFFFu, a0, 8); a1 += __shfl_xor_sync(0xFFFFFFFFu, a1, 8);
        a0 += __shfl_xor_sync(0xFFFFFFFFu, a0, 16); a1 += __shfl_xor_sync(0xFFFFFFFFu, a1, 16);
        const int k = lane >> 1;
        const double v0 = __shfl_sync(0xFFFFFFFFu, a0, k >> 1), v1 = __shfl_sync(0xFFFFFFFFu, a1, k >> 1);
        acc += (k & 1) ? v1 : v0;
    }
}

// The bandwidth shape's pass (kernel mode: millions of queries against a map far larger than L2). Everything that is per-query scalar work
// -- transform, the three FP64 index divisions, key packing and hashing, and later residual, weight and the 16 products -- runs with ONE
// lane per query, i.e. one warp instruction serves 32 queries (eight lanes per query for ALL of it made the pass FP64-issue bound:
// 805 us instead of 630 us per iteration at 4 M queries). Only the memory part is cooperative: in step t the eight lanes of a group
// take over the query of the group's lane t, fetch the voxel block -- header and candidates in ONE round trip -- scan it and hand the
// winner back to lane t (group8_closest_at).
template <int ROUNDS>
__device__ __forceinline__ void icp_query_pass_coop(const IcpArgs &A, const volatile double *Pv, const double *in, int64_t n, int64_t wbase, int64_t wstride,
                                                    int lane, double &acc, int &ncorr, int &ncand, int &nmiss) {
    const int l8 = lane & 7;
    const unsigned gmask = 0xFFu << (lane & 24);
    for (int64_t base = wbase; base < n; base += wstride) {
        const int64_t q = base + lane;
        const bool on = q < n;
        V3 s{0.0, 0.0, 0.0};
        int kx = 0, ky = 0, kz = 0, inr = 0;
        unsigned long long key = 0ull;
        unsigned int h = 0u;
        if (on) {
            const Pose P{Pv[0], Pv[1], Pv[2], Pv[3], Pv[4], Pv[5], Pv[6]};
            s = apply(P, V3{in[3 * q], in[3 * q + 1], in[3 * q + 2]});
            A.work[3 * q] = s.x; A.work[3 * q + 1] = s.y; A.work[3 * q + 2] = s.z;
            kx = vox_index(A.map, s.x); ky = vox_index(A.map, s.y); kz = vox_index(A.map, s.z);
            inr = key_in_range(kx, ky, kz) ? 1 : 0;
            key = pack_key(kx, ky, kz);
            h = inr ? slot_of(key, A.map.shift) : 0u;
        }
        double my_d2 = 0.0;
        int my_rank = -1, my_count = 0, my_own = 1;
        V3 tg{0.0, 0.0, 0.0};
#pragma unroll 1
        for (int t = 0; t < 8; ++t) {
            const V3 qp{__shfl_sync(0xFFFFFFFFu, s.x, t, 8), __shfl_sync(0xFFFFFFFFu, s.y, t, 8), __shfl_sync(0xFFFFFFFFu, s.z, t, 8)};
            const int qx = __shfl_sync(0xFFFFFFFFu, kx, t, 8), qy = __shfl_sync(0xFFFFFFFFu, ky, t, 8), qz = __shfl_sync(0xFFFFFFFFu, kz, t, 8);
            const int qin = __shfl_sync(0xFFFFFFFFu, inr, t, 8);
            const unsigned long long qkey = __shfl_sync(0xFFFFFFFFu, key, t, 8);
            const unsigned int qh = __shfl_sync(0xFFFFFFFFu, h, t, 8);
            int slot, count, own, rank;
            double d2;
            V3 tt;
            group8_closest_at<ROUNDS>(A.map, qp, qx, qy, qz, qin != 0, qkey, qh, gmask, l8, slot, count, own, d2, rank, tt);
            if (l8 == t) { my_d2 = d2; my_rank = rank; my_count = count; my_own = own; tg = tt; }
        }
        const double d2 = my_rank >= 0 ? my_d2 : sqnorm3(tg.x - s.x, tg.y - s.y, tg.z - s.z);   // nothing found -> (0,0,0), range-tested like a real point
        const bool gate = on && d2 < A.tau_sq;
        double c[16];
        contribution(c, s, tg, d2, A.th, gate);
        acc += warp_reduce_scatter16(c);
        ncorr += gate ? 1 : 0;
        ncand += on ? my_count : 0;
        nmiss += (on && !my_own) ? 1 : 0;
    }
}

// ---- staged pass of the bandwidth shape ------------------------------------------------------------------------------------------------
// What bounds kernel mode is memory-level parallelism: a warp that waits for the ~1 us of an HBM round trip with four voxel blocks in
// flight (registers hold the candidates) leaves the SM with ~50 KB in flight at best, and every displaced voxel adds a dependent trip.
// Here the voxel blocks go from HBM to SHARED memory with cp.async (LDGSTS, 16 bytes per lane: ONE warp instruction moves one whole
// 384/512-byte block, header included, no registers involved), eight blocks per commit group, double-buffered per warp: while the warp
// scans one group of eight blocks out of shared memory, the next eight (4 KB) are in flight.
//   1. one lane per query: transform, voxel index, hash, and map_locate (header loads, probing, 26-cell fallback) -- 32 queries per
//      warp instruction, 32 independent chains in flight;
//   2. four steps of eight blocks: stage -> wait -> the four lanes of a quad scan the block of their lane t from shared memory
//      (ranks l4, l4+4, ...), butterfly for the lexicographic minimum of (d^2, rank), winner's point by shuffle;
//   3. one lane per query again: residual, weight, the 16 products, one reduce-scatter per 32 queries.
constexpr int STAGE_MAX_STRIDE = 64;                        // doubles per block this path handles (max_points_per_voxel <= 20)
constexpr int STAGE_SLOT = STAGE_MAX_STRIDE + 2;            // + 16 bytes: the four groups of a warp read different banks
constexpr int STAGE_WARP_DOUBLES = 2 * 8 * STAGE_SLOT;      // two buffers of eight blocks per query warp (8448 bytes)
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc) {
    const unsigned int sa = (unsigned int)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Step t of a batch: the eight quads of a warp serve the queries of lanes 4i + t (i = quad). Their eight blocks are one commit group.
__device__ __forceinline__ void stage_step(const IcpArgs &A, double *stage, int t, const double *blk_ptr, int lane) {
    double *buf = stage + (t & 1) * 8 * STAGE_SLOT;
    const int chunks = A.map.stride >> 1;                   // 16-byte chunks per block
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const unsigned long long p = __shfl_sync(0xFFFFFFFFu, (unsigned long long)blk_ptr, 4 * i + t);
        if (p && lane < chunks) cp_async16(buf + i * STAGE_SLOT + 2 * lane, reinterpret_cast<const double *>(p) + 2 * lane);
    }
    cp_async_commit();
}

// one lane per query: running source point and the voxel that answers it
struct StagedQuery {
    V3 s;
    int slot, count, own, on;
};
__device__ __forceinline__ V3 staged_load_raw(const double *in, int64_t base, int lane, int64_t n) {
    const int64_t q = base + lane;
    return q < n ? V3{in[3 * q], in[3 * q + 1], in[3 * q + 2]} : V3{0.0, 0.0, 0.0};
}
__device__ __forceinline__ StagedQuery staged_prepare(const IcpArgs &A, const Pose &P, const V3 &raw, int64_t base, int lane, int64_t n) {
    StagedQuery c;
    const int64_t q = base + lane;
    c.on = q < n ? 1 : 0;
    c.s = V3{0.0, 0.0, 0.0};
    c.slot = -1; c.count = 0; c.own = 1;
    if (c.on) {
        // j == 0: source = init_guess * points (:102-103); later: source <- estimate * source (:119), applied lazily at this visit
        c.s = apply(P, raw);
        A.work[3 * q] = c.s.x; A.work[3 * q + 1] = c.s.y; A.work[3 * q + 2] = c.s.z;
        c.slot = map_locate(A.map, c.s, &c.count, &c.own);   // which voxel answers (own, else farthest/latest of the 27)
    }
    return c;
}

// Software pipeline over the batches of 32 queries a warp visits: while the eight-block groups of batch k are in flight / being scanned,
// the warp already transforms and locates batch k+1 (its header loads overlap the copies) and has the raw points of batch k+2 on the way.
// FOUR lanes scan a block (quad q = lane / 4 serves the query of its lane t in step t = 0..3): measured, the pass is bound by issued
// instructions, not by HBM (a cap-10 map with half the bytes took the same time), and four steps of eight quads cost about half the
// shuffles, butterflies and loop overhead of eight steps of four octets for the same k-bar distance evaluations.
__device__ __forceinline__ void icp_query_pass_staged(const IcpArgs &A, const volatile double *Pv, const double *in, int64_t n, int64_t wbase, int64_t wstride,
                                                      int lane, double *stage, double &acc, int &ncorr, int &ncand, int &nmiss) {
    const int l4 = lane & 3, quad = lane >> 2, capp = A.map.capp;
    const unsigned qmask = 0xFu << (lane & 28);
    if (wbase >= n) return;   // warp-uniform
    const Pose P{Pv[0], Pv[1], Pv[2], Pv[3], Pv[4], Pv[5], Pv[6]};
    StagedQuery cur = staged_prepare(A, P, staged_load_raw(in, wbase, lane, n), wbase, lane, n);
    V3 raw_next = staged_load_raw(in, wbase + wstride, lane, n);
    for (int64_t base = wbase; base < n; base += wstride) {
        const double *blk_ptr = cur.slot >= 0 ? A.map.blk + (size_t)cur.slot * (size_t)A.map.stride : nullptr;
        __syncwarp();
        stage_step(A, stage, 0, blk_ptr, lane);
        stage_step(A, stage, 1, blk_ptr, lane);
        const V3 raw_after = staged_load_raw(in, base + 2 * wstride, lane, n);
        const StagedQuery nxt = staged_prepare(A, P, raw_next, base + wstride, lane, n);   // all lanes off when base + wstride >= n
        raw_next = raw_after;
        double my_d2 = 0.0;
        int my_rank = -1;
        V3 tg{0.0, 0.0, 0.0};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (t < 3) cp_async_wait<1>(); else cp_async_wait<0>();   // the blocks of step t have landed (one younger group may still be in flight)
            __syncwarp();
            const double qx = __shfl_sync(0xFFFFFFFFu, cur.s.x, t, 4), qy = __shfl_sync(0xFFFFFFFFu, cur.s.y, t, 4), qz = __shfl_sync(0xFFFFFFFFu, cur.s.z, t, 4);
            const int qslot = __shfl_sync(0xFFFFFFFFu, cur.slot, t, 4), qcount = __shfl_sync(0xFFFFFFFFu, cur.count, t, 4);
            const double *bx = stage + ((t & 1) * 8 + quad) * STAGE_SLOT + 2, *by = bx + capp, *bz = by + capp;
            double bd2 = 1.7976931348623157e308, tx = 0.0, ty = 0.0, tz = 0.0;
            int br = 0x7FFFFFFF;
            if (qslot >= 0) {
                for (int r = l4; r < qcount; r += 4) {      // VoxelBlock::get_closest_point (voxel_block.cpp:87-105): ascending ranks, strict '<'
                    const double x = bx[r], y = by[r], z = bz[r];
                    const double d = sqnorm3(qx - x, qy - y, qz - z);
                    if (d < bd2) { bd2 = d; br = r; tx = x; ty = y; tz = z; }
                }
            }
#pragma unroll
            for (int o = 2; o > 0; o >>= 1) {               // lexicographic minimum of (d^2, rank) = "first minimum wins"
                const double od = __shfl_xor_sync(qmask, bd2, o);
                const int orr = __shfl_xor_sync(qmask, br, o);
                if (od < bd2 || (od == bd2 && orr < br)) { bd2 = od; br = orr; }
            }
            const int src = br == 0x7FFFFFFF ? 0 : (br & 3);   // the winner's point sits in lane (rank & 3) of the quad
            tx = __shfl_sync(qmask, tx, src, 4); ty = __shfl_sync(qmask, ty, src, 4); tz = __shfl_sync(qmask, tz, src, 4);
            if (l4 == t && br != 0x7FFFFFFF) { my_d2 = bd2; my_rank = br; tg = V3{tx, ty, tz}; }
            __syncwarp();                                   // everybody is done with this buffer: refill it
            if (t + 2 < 4) stage_step(A, stage, t + 2, blk_ptr, lane);
        }
        const double d2 = my_rank >= 0 ? my_d2 : sqnorm3(tg.x - cur.s.x, tg.y - cur.s.y, tg.z - cur.s.z);   // nothing found -> (0,0,0), range-tested like a real point
        const bool gate = cur.on && d2 < A.tau_sq;
        double c[16];
        contribution(c, cur.s, tg, d2, A.th, gate);
        acc += warp_reduce_scatter16(c);
        ncorr += gate ? 1 : 0;
        ncand += cur.on ? cur.count : 0;
        nmiss += (cur.on && !cur.own) ? 1 : 0;
        cur = nxt;
    }
}

#ifdef LIMU_ICP_PHASE_TIMING
// developer build only (tools/icp_phase_timing.py, tools/frame_phase_timing.py): %globaltimer stamps of CTA 0 / thread 0
__device__ unsigned long long g_frame_marks[72];   // [24 + j]: clock of CTA 0 / warp 0 at the start of round j of the Gauss-Newton loop (j < 48)
#define FT_MARK(k) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && ((k) >= 8 || threadIdx.x == 0)) { unsigned long long _t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t)); g_frame_marks[k] = _t; } } while (0)
// SM cycle counter of CTA 0 (one SM: the marks of different warps are comparable): any lane 0 / lane 0 of warp w
#define IQ_MARK(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_frame_marks[k] = (unsigned long long)clock64(); } while (0)
// (stamped in iteration 2 of the Gauss-Newton loop; marks 13 / 14 = the tail of iteration 2, which runs during loop round 3)
#define CW_MARK(k, w) do { if (blockIdx.x == 0 && warp == (w) && lane == 0 && j == (((k) == 13 || (k) == 14) ? 3 : 2)) g_frame_marks[k] = (unsigned long long)clock64(); } while (0)
#define ROUND_MARK() do { if (blockIdx.x == 0 && threadIdx.x == 0 && j < 48) g_frame_marks[24 + j] = (unsigned long long)clock64(); } while (0)
__device__ unsigned int g_warp_pass[160][8];   // SM cycles every warp of the loop spent in its pass of round 3
__device__ unsigned long long g_cta_marks[4][160];   // globaltimer of every CTA of the loop in round 3: [0] round start, [1] S1 (its pass is over), [2] all rows folded, [3] S2
#define WARP_PASS(t0) do { if (lane == 0 && j == 3 && blockIdx.x < 160) g_warp_pass[blockIdx.x][warp] = (unsigned int)(clock64() - (t0)) & 0xFFFFFFu; } while (0)
#define CTA_MARK(k) do { if (threadIdx.x == 0 && j == 3 && blockIdx.x < 160) { unsigned long long _t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t)); g_cta_marks[k][blockIdx.x] = _t; } } while (0)
extern "C" int limu_debug_warp_pass(unsigned int out[1280]) { return cudaMemcpyFromSymbol(out, g_warp_pass, sizeof(unsigned int) * 1280) == cudaSuccess ? 0 : -1; }
extern "C" int limu_debug_cta_marks(double out[640]) {
    unsigned long long h[640];
    if (cudaMemcpyFromSymbol(h, g_cta_marks, sizeof h) != cudaSuccess) return -1;
    for (int k = 0; k < 640; ++k) out[k] = (double)h[k];
    return 0;
}
#else
#define FT_MARK(k) do {} while (0)
#define IQ_MARK(k) do {} while (0)
#define CW_MARK(k, w) do {} while (0)
#define ROUND_MARK() do {} while (0)
#define CTA_MARK(k) do {} while (0)
#define WARP_PASS(t0) do {} while (0)
#endif

// local_map.update(down_sampled, new_pose) (icp.cpp:81; voxel_hash_map.cpp:138-144) inside a frame kernel: transform + capped ordered insert
// (two passes separated by a grid barrier) + eviction around the new position. Every CTA of the grid takes part (those that sat out the
// Gauss-Newton loop join here); everybody reads the new pose that CTA 0 published in A.out. E: 7 doubles of shared memory.
// The next scan deskews with delta_pose(poses[N-2], poses[N-1]) = log(last^-1 * new) (deskew.cpp:14): left on the device for a k_voxelize
// that sits behind this kernel in the stream. One thread (~3 us of scalar code).
__device__ __forceinline__ void publish_twist(const IcpArgs &A, const Pose &np) {
    if (A.twist_out) {
        double tw[6];
        se3_log(mul(inverse(Pose{A.last_pose[0], A.last_pose[1], A.last_pose[2], A.last_pose[3], A.last_pose[4], A.last_pose[5], A.last_pose[6]}), np), tw);
#pragma unroll
        for (int k = 0; k < 6; ++k) A.twist_out[k] = tw[k];
    }
}

template <int BLOCK, bool FUSED = true>
__device__ __forceinline__ void frame_update_epilogue(const IcpArgs &A, GridSync &gs, double *E) {
    if (FUSED) gs.sync();   // (a launch of its own starts behind the kernel that wrote the pose)
    if (threadIdx.x < 7) E[threadIdx.x] = __ldcg(A.out + threadIdx.x);
    __syncthreads();
    const Pose np = pose_load(E);
    // Fused launch: one thread of the LAST CTA publishes the twist while the grid inserts -- on CTA 0's thread 0, in front of the barrier
    // above, it held up every CTA.
    if (FUSED && blockIdx.x == gridDim.x - 1 && threadIdx.x == BLOCK - 1) publish_twist(A, np);
    const int64_t nd = (int64_t)__ldcg(A.upd_n);
    const int64_t gtid = (int64_t)blockIdx.x * BLOCK + threadIdx.x, gthreads = (int64_t)gridDim.x * BLOCK;
    for (int64_t base = (int64_t)blockIdx.x * BLOCK; base < nd; base += gthreads) {   // whole warps stay converged for the ballot
        const int64_t i = base + threadIdx.x;
        bool claimed = false;
        unsigned int slot = PEND_NONE;
        if (i < nd) {
            const V3 w = apply(np, V3{A.upd_down[3 * i], A.upd_down[3 * i + 1], A.upd_down[3 * i + 2]});
            A.upd_world[3 * i] = w.x; A.upd_world[3 * i + 1] = w.y; A.upd_world[3 * i + 2] = w.z;
            A.upd_pslot[i] = slot = insert_claim_one(A.map, w, (unsigned int)i, A.upd_birth_base, A.status, &claimed);
        }
        insert_account(claimed, slot, A.upd_counters, A.map);
    }
    gs.sync();
    FT_MARK(3);
    LIMU_TRACE(21);
    for (int64_t i = gtid; i < nd; i += gthreads)
        insert_place_one(A.map, V3{A.upd_world[3 * i], A.upd_world[3 * i + 1], A.upd_world[3 * i + 2]}, (unsigned int)i, __ldcg(A.upd_pslot + i));
    gs.sync();
    FT_MARK(4);
    LIMU_TRACE(22);
    // eviction (remove_points_from_far, voxel_hash_map.cpp:146-171) over the dense list of voxels (V entries, 4 B + one 16 B slot each)
    // instead of the C table slots: a scan that evicts nothing used to read the whole 16 MB slot array.
    // The voxel test needs the key only: the sweep streams the list's key words (coalesced) and touches the block of a far voxel alone --
    // a map of 2.6 M voxels spread over a 4 GB block array took 110 us per scan to visit header by header.
    const int64_t used = (int64_t)__ldcg(A.upd_counters + 3);
    const int ovx = vox_index(A.map, np.tx), ovy = vox_index(A.map, np.ty), ovz = vox_index(A.map, np.tz);
    for (int64_t i0 = gtid; i0 < used; i0 += 4 * gthreads) {
        unsigned long long key[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t idx = i0 + (int64_t)u * gthreads;
            key[u] = idx < used ? __ldcg(A.map.live_key + idx) : KEY_TOMB;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            remove_far_entry(A.map, i0 + (int64_t)u * gthreads, key[u], ovx, ovy, ovz, np.tx, np.ty, np.tz, A.upd_max_distance, A.upd_counters);
    }
}

// x = H^-1 (-g) from the 16 sums (registration.cpp:90), one thread. Kept out of line: its live registers (~90 on the ldlt6_solve
// fallback) would otherwise compete with the query pass of the bandwidth build for the registers its LIMU_BW_CTAS CTAs per SM allow.
static __device__ __noinline__ void solve_normal_equations(const double *S, double *x_out) {
    double x[6];
    solve_point_to_point(S, x);
#pragma unroll
    for (int k = 0; k < 6; ++k) x_out[k] = x[k];
}

// ---- row exchange without a barrier ("LL" protocol) ---------------------------------------------------------------------------------------
// Every CTA of the loop needs every CTA's row of sums. A global-memory barrier + fold cost ~3.5 us per iteration (atomic arrive, release
// fence, acquire polling, then the loads). Instead each 8-byte word a CTA publishes carries its own validity: a double travels as two
// words {low 32 bits | stamp}, {high 32 bits | stamp} (aligned 8-byte accesses are single-copy atomic), written with one 16-byte store;
// readers request all the rows they fold at once and simply re-request the words whose stamp is not this iteration's yet. No fence, no
// atomic, no separate arrival: store -> L2 -> load. Two buffers alternate by iteration parity (a CTA can only be one iteration ahead
// of the slowest: it needs everybody's row j+1 before it can write row j+2).
__device__ __forceinline__ void ll_store(unsigned long long *slot /* 16-byte aligned pair */, double v, unsigned int stamp) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v), st = (unsigned long long)stamp << 32;
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(slot), "l"((bits & 0xFFFFFFFFull) | st), "l"((bits >> 32) | st) : "memory");
}
__device__ __forceinline__ bool ll_load(const unsigned long long *slot, unsigned int stamp, double &v) {
    unsigned long long lo, hi;
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(slot) : "memory");
    v = __longlong_as_double((long long)((lo & 0xFFFFFFFFull) | (hi << 32)));
    return (unsigned int)(lo >> 32) == stamp && (unsigned int)(hi >> 32) == stamp;
}

// SHAPE 0 = latency build (a few thousand keypoints: one CTA per SM at most, so the compiler may use up to 255 registers and the serial
// Gauss-Newton solve stays out of local memory); SHAPE 1 = bandwidth build for kernel mode (millions of queries against a map far larger
// than L2): LIMU_BW_CTAS CTAs per SM, voxel blocks staged through shared memory (icp_query_pass_staged), the solve out of line.
// the index-list compaction for the larger candidate capacities, out of line: unrolled 32 / 64 times inside the loop kernel it took that kernel
// from 140 to 255 registers
static __device__ __noinline__ int iqr_local_compact_dyn(int cap, int *ws, int *total, const double *sd2, int n0, const double *sel, unsigned short *qidx) {
    if (cap <= 8192) return iqr_local_compact<ICP_BLOCK, 8192 / ICP_BLOCK>(ws, total, sd2, n0, sel, qidx);
    return iqr_local_compact<ICP_BLOCK, IQR_GRID_MAX_DYN / ICP_BLOCK>(ws, total, sd2, n0, sel, qidx);
}

template <int SHAPE, bool NN27, bool PLANE>
static __global__ void __launch_bounds__(ICP_BLOCK, SHAPE == 0 ? 1 : LIMU_BW_CTAS) k_icp_persistent(const IcpArgs A) {
    constexpr int NSX = PLANE ? NSP : NS;              // doubles per partial row
    constexpr int I_NCORR = PLANE ? 27 : 16;           // where the three counters sit in a row
    __shared__ double red[(ICP_BLOCK / 32) * 32];
    __shared__ double S[NSX];
    __shared__ double E[7], Tinit[7], Ticp[7], xs[8];
    __shared__ int done;
    __shared__ int verdict;   // on the iteration just solved: 1 converged, 0 not, 2 too close to call from the twist itself (see below)
    __shared__ int comm_dead;
    __shared__ IqrSmem iqr_sm;
    GridSync gs{A.barrier, 0u, gridDim.x};
    GridSync gs_icp{A.barrier_icp, 0u, (unsigned int)A.icp_blocks};
    const bool icp_member = (int)blockIdx.x < A.icp_blocks;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    FT_MARK(0);
    LIMU_TRACE(1);
    __shared__ unsigned short qidx_static[SHAPE == 0 ? IQR_GRID_MAX : 1];
    extern __shared__ __align__(16) double stage_smem[];
    // more than IQR_GRID_MAX candidates announced (~7 k at configs[2]): the two lists live in dynamic shared memory -- the one-CTA select
    // behind a whole-grid barrier that such scans used to fall back to took 61 us per scan
    const bool iqr_dyn = SHAPE == 0 && A.iqr_cap > IQR_GRID_MAX;
    unsigned short *qidx_s = iqr_dyn ? reinterpret_cast<unsigned short *>(stage_smem + A.iqr_cap) : qidx_static;
    int n_keypoints = -1;   // >= 0: the keypoints are IQR candidates qidx_s[0 .. n_keypoints) (known to the CTAs of the Gauss-Newton loop)
    if (A.iqr_in) {   // KissICP::iqr_processing (icp.cpp:88-124, :133)
        // Latency shape: only the CTAs that will run the Gauss-Newton loop take part. They rank their share of the ~2.5 k squared ranges by
        // counting and meet at THEIR barrier (the leading CTAs of a launch start first; the whole-grid barrier also waits for the last CTA to
        // be scheduled); then each of them derives bounds, flags and the keypoint index list in its own shared memory, so nobody waits for
        // CTA 0 to compact (CTA 0 also writes the keypoints out for the host). The bandwidth shape keeps the one-CTA select.
        __shared__ double iqr_sd2_static[SHAPE == 0 ? IQR_GRID_MAX : 1];
        double *iqr_sd2 = iqr_dyn ? stage_smem : iqr_sd2_static;
        const int n0 = __ldcg(A.iqr_n);
        if (SHAPE == 0 && n0 > 1 && n0 <= (iqr_dyn ? A.iqr_cap : IQR_GRID_MAX)) {   // uniform across the grid
            if (icp_member) {
                IQ_MARK(16);
                iqr_grid_select<ICP_BLOCK>(iqr_sd2, A.iqr_in, n0, A.iqr_d2, A.icp_blocks);
                IQ_MARK(17);
                gs_icp.sync();
                IQ_MARK(18);
                if (!iqr_dyn) n_keypoints = iqr_local_compact<ICP_BLOCK>(iqr_sm.ws, &iqr_sm.total, iqr_sd2, n0, A.iqr_d2, qidx_s);
                else n_keypoints = iqr_local_compact_dyn(A.iqr_cap, iqr_sm.ws, &iqr_sm.total, iqr_sd2, n0, A.iqr_d2, qidx_s);
                IQ_MARK(19);
            }
        } else {
            if (blockIdx.x == 0) iqr_block<ICP_BLOCK>(iqr_sm, A.iqr_in, *A.iqr_n, A.iqr_d2, A.iqr_out, A.iqr_count, nullptr);
            gs.sync();
        }
    }
    FT_MARK(1);
    LIMU_TRACE(2);
    const int64_t n = n_keypoints >= 0 ? (int64_t)n_keypoints : (A.n_dev ? (int64_t)__ldcg(A.n_dev) : A.n_max);
    const bool run_icp = !(__ldcg(A.map_counters) == 0ull || A.max_iter <= 0);   // ICP :99-100: empty map -> init_guess
    if (threadIdx.x < 7) { Tinit[threadIdx.x] = A.init_pose[threadIdx.x]; Ticp[threadIdx.x] = threadIdx.x == 3 ? 1.0 : 0.0; }
    if (threadIdx.x < NSX) S[threadIdx.x] = 0.0;
    if (threadIdx.x == 0) { comm_dead = 0; verdict = 0; done = 0; }
    __syncthreads();
    // Warps 0..QW-1 own the queries; the last warp is the SOLVER warp: it has no queries, solves the normal equations once the rows
    // are folded, publishes the estimate -- and then finishes T_icp, log(estimate) and the convergence test WHILE the query warps are
    // already in the next pass (the ~2 us of SE3 product + log leave the critical path of the iteration; a pass made after the
    // converging iteration is simply dropped).
    constexpr int QW = ICP_BLOCK / 32 - 1;
    const int64_t wbase = ((int64_t)blockIdx.x * QW + warp) * 32, wstride = (int64_t)A.icp_blocks * QW * 32;
    int j = 0;
    int converged = 0;
    PlaneMemo pmemo;  // (latency shape, point-to-plane variant: the plane fitted to the voxel this lane's query matched in the previous iteration)
    pmemo.slot = -1; pmemo.planar = 0; pmemo.n[0] = pmemo.n[1] = pmemo.n[2] = 0.0;
    QueryMemo memo;   // (latency shape, reference rules: what this lane's group found for its query in the previous iteration)
    memo.own = -1; memo.kx = memo.ky = memo.kz = 0; memo.slot = -1; memo.count = 0;
    if (run_icp && icp_member) for (;;) {
        const bool no_more = j >= A.max_iter;   // nothing left to do but wait for the verdict on iteration j-1
        ROUND_MARK();
        CTA_MARK(0);
        if (warp < QW) {
            if (!no_more) {
                CW_MARK(6, 0);
#ifdef LIMU_ICP_PHASE_TIMING
                const long long wp0 = clock64();
#endif
                double acc = 0.0;            // lane L: running total of sum index L>>1
                int ncorr = 0, ncand = 0, nmiss = 0;
                const volatile double *Pv = j == 0 ? Tinit : E;   // re-read per batch: keeps 14 registers free across the lookup
                const double *in = j == 0 ? (n_keypoints >= 0 ? A.iqr_in : A.points) : A.work;
                const unsigned short *qi0 = (j == 0 && n_keypoints >= 0) ? qidx_s : nullptr;
                if (SHAPE == 1 && !NN27 && !PLANE && A.stage_doubles > 0) {   // bandwidth shape: voxel blocks staged through shared memory
                    icp_query_pass_staged(A, Pv, in, n, wbase, wstride, lane, stage_smem + (size_t)warp * STAGE_WARP_DOUBLES, acc, ncorr, ncand, nmiss);
                } else if (SHAPE == 1 && !NN27 && !PLANE) {     // ... or, for blocks too large to stage, fetched by eight lanes into registers
                    if (A.map.cap <= 8) icp_query_pass_coop<1>(A, Pv, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
                    else if (A.map.cap <= 16) icp_query_pass_coop<2>(A, Pv, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
                    else icp_query_pass_coop<3>(A, Pv, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
                } else if (SHAPE == 0) {                 // latency shape: eight lanes per query
                    if (A.map.cap <= 8) icp_query_pass_grouped<NN27, PLANE, 1>(A, Pv, in, qi0, n, wbase / 8 + (lane >> 3), wstride / 8, lane, acc, ncorr, ncand, nmiss, &memo, &pmemo);
                    else if (A.map.cap <= 16) icp_query_pass_grouped<NN27, PLANE, 2>(A, Pv, in, qi0, n, wbase / 8 + (lane >> 3), wstride / 8, lane, acc, ncorr, ncand, nmiss, &memo, &pmemo);
                    else icp_query_pass_grouped<NN27, PLANE, 3>(A, Pv, in, qi0, n, wbase / 8 + (lane >> 3), wstride / 8, lane, acc, ncorr, ncand, nmiss, &memo, &pmemo);
                } else {
                    icp_query_pass<NN27, PLANE>(A, Pv, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
                }
                CW_MARK(7, 0);
#ifdef LIMU_ICP_PHASE_TIMING
                WARP_PASS(wp0);
#endif
                if (PLANE) {
                    red[warp * 32 + lane] = acc;   // lane L of every warp holds sum L (27 sums + 3 counters + 2 zeros)
                } else {                           // 16 sums (even lanes hold them) + 3 counters
                    ncorr = __reduce_add_sync(0xFFFFFFFFu, ncorr);
                    ncand = __reduce_add_sync(0xFFFFFFFFu, ncand);
                    nmiss = __reduce_add_sync(0xFFFFFFFFu, nmiss);
                    red[warp * 32 + lane] = (lane & 1) ? (lane == 1 ? (double)ncorr : lane == 3 ? (double)ncand : lane == 5 ? (double)nmiss : 0.0) : acc;
                }
            }
        } else if (j > 0) {
            // tail of iteration j-1, overlapped with pass j: T_icp = estimate * T_icp (:122) on lane 0, |log(estimate)| < eps (:124) on lane 1
            CW_MARK(13, QW);
            const Pose est = pose_load(E);
            if (lane == 0) pose_store(mul(est, pose_load(Ticp)), Ticp);
            if (lane == 1 && verdict == 2) {
                double lg[6];
                se3_log(est, lg);
                done = norm6(lg) < A.eps;
            }
            if (blockIdx.x == 0 && lane == 2) {   // traces of iteration j-1 (S still holds its sums)
                if (A.est_trace) pose_store(est, A.est_trace + 7 * (size_t)(j - 1));
                if (A.ncorr_trace) A.ncorr_trace[j - 1] = (long long)S[I_NCORR];
                if (A.hg_trace) {
                    double H[36], g[6];
                    if (PLANE) expand_plane_equations(S, H, g);
                    else expand_normal_equations(S, H, g);
                    double *o = A.hg_trace + 42 * (size_t)(j - 1);
                    for (int k = 0; k < 36; ++k) o[k] = H[k];
                    for (int k = 0; k < 6; ++k) o[36 + k] = g[k];
                }
            }
            CW_MARK(14, QW);
        }
        __syncthreads();   // S1: CTA partial sums of pass j, and the verdict on iteration j-1
        CW_MARK(11, 0);
        CTA_MARK(1);
        if (j > 0 && verdict == 2 && done) { converged = 1; break; }   // (the pass just made belongs to an iteration that does not exist)
        if (no_more) break;
        const unsigned int stamp = 0x80000000u | ((A.ll_stamp_base + (unsigned int)j) & 0x7FFFFFFFu);
        unsigned long long *rows = reinterpret_cast<unsigned long long *>(A.partials) + (size_t)(j & 1) * A.icp_blocks * (2 * NSX);
        if (threadIdx.x < NSX) {   // CTA row, fixed order over the query warps; published word by word with its stamp
            const int src_lane = PLANE ? (int)threadIdx.x : (threadIdx.x < 16 ? 2 * (int)threadIdx.x : 2 * ((int)threadIdx.x - 16) + 1);
            double v = 0.0;
#pragma unroll
            for (int w = 0; w < QW; ++w) v += red[w * 32 + src_lane];
            ll_store(rows + ((size_t)blockIdx.x * NSX + threadIdx.x) * 2, v, stamp);
        }
        __syncthreads();           // (red is reused below)
        CW_MARK(12, 0);
        // fold the rows in a fixed order: lane = column, warp g sums rows g, g+8, ...; up to 16 rows per warp are requested at once and
        // re-requested until their stamp says they are this iteration's, then one thread per column adds the 8 warp partials.
        {
            double acc = 0.0;
            constexpr int G = ICP_BLOCK / 32;
            for (int b0 = warp; b0 < A.icp_blocks; b0 += 16 * G) {   // CTA-uniform trip count
                double v[16];
                unsigned int pending = 0u;
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    v[k] = 0.0;
                    if (lane < NSX && b0 + k * G < A.icp_blocks) pending |= 1u << k;
                }
                unsigned int spins = 0u;
                while (pending) {
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        if (pending & (1u << k)) {
                            double x;
                            if (ll_load(rows + ((size_t)(b0 + k * G) * NSX + lane) * 2, stamp, x)) { v[k] = x; pending &= ~(1u << k); }
                        }
                    }
                    if (++spins > (1u << 24)) __trap();   // a CTA of the loop never published its row: fail loudly instead of hanging the device
                }
#pragma unroll
                for (int k = 0; k < 16; ++k) acc += v[k];
            }
            red[warp * 32 + lane] = acc;
            __syncthreads();
            if (threadIdx.x < NSX) {
                double v = 0.0;
#pragma unroll
                for (int w = 0; w < ICP_BLOCK / 32; ++w) v += red[w * 32 + threadIdx.x];
                S[threadIdx.x] = v;
            }
        }
        __syncthreads();
        CTA_MARK(2);
        if (!PLANE && A.nranks > 1) {
            // Fused exchange: CTA 0 stores this rank's row into EVERY rank's mailbox (its own included) over NVLink, then a
            // system-scope release of the stamp; every CTA of every rank then waits for all stamps in its LOCAL mailbox and
            // adds the rows in rank order -- the same order everywhere, so all ranks solve bit-identical normal equations
            // and take identical convergence decisions. No host, no NCCL launch, no second grid barrier.
            const unsigned long long seq = A.stamp_base + (unsigned long long)j, stamp = seq + 1ull;
            const size_t par = (size_t)(seq % MBOX_RING) * MBOX_MAX_RANKS * MBOX_ROW;
            if (blockIdx.x == 0) {
                if (threadIdx.x < NS) {
                    const double v = S[threadIdx.x];
                    for (int r = 0; r < A.nranks; ++r) A.mbox_peer[r][par + (size_t)A.rank * MBOX_ROW + threadIdx.x] = v;
                }
                __threadfence_system();
                __syncthreads();
                if (threadIdx.x < A.nranks) {
                    unsigned long long *flag = reinterpret_cast<unsigned long long *>(A.mbox_peer[threadIdx.x] + par + (size_t)A.rank * MBOX_ROW + NS);
                    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(stamp) : "memory");
                }
            }
            if (threadIdx.x < A.nranks) {
                const unsigned long long *flag = reinterpret_cast<const unsigned long long *>(A.mbox_local + par + (size_t)threadIdx.x * MBOX_ROW + NS);
                unsigned long long v, t0, t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                do {
                    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t1 - t0 > 2000000000ull) { *A.comm_error = 1; comm_dead = 1; break; }   // 2 s: a peer never arrived
                } while (v < stamp);
            }
            __syncthreads();
            if (comm_dead) break;   // every CTA of this rank times out the same way; the host reports LIMU_ERR_COMM
            if (threadIdx.x < NS) {
                double v = 0.0;
                for (int r = 0; r < A.nranks; ++r) v += *reinterpret_cast<const volatile double *>(A.mbox_local + par + (size_t)r * MBOX_ROW + threadIdx.x);
                S[threadIdx.x] = v;
            }
            __syncthreads();
        }
        if (warp == QW) {
            // normal equations -> twist -> estimate: the critical path of the iteration
            CW_MARK(8, QW);
            if (lane == 0) {   // (one thread from the sums to the verdict: lanes of one warp would take turns anyway)
                double x[6];
                if (SHAPE == 1 && !PLANE) {
                    solve_normal_equations(S, xs);                // out of line: the bandwidth build has no registers to spare
#pragma unroll
                    for (int k = 0; k < 6; ++k) x[k] = xs[k];
                } else if (!PLANE) {
                    solve_point_to_point(S, x);                   // JTJ.ldlt().solve(-JTr) :90, by the Schur complement of its w I block
                } else {
                    // point-to-plane: weak prior on the initial guess (oracle: lo_icp), x = LDLT(H + D).solve(-(g + D log(T_icp))) -- a map
                    // that offers only a handful of planar voxels does not determine six degrees of freedom, and the plain step runs away.
                    // (T_icp is this lane's own: it folded the previous estimate into it in the tail above.)
                    double H[36], g[6], xi[6];
                    expand_plane_equations(S, H, g);
                    se3_log(pose_load(Ticp), xi);
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        H[7 * k] += PLANE_PRIOR; H[7 * (k + 3)] += PLANE_PRIOR * PLANE_PRIOR_ARM2;
                        g[k] = -(S[21 + k] + PLANE_PRIOR * xi[k]);
                        g[k + 3] = -(S[24 + k] + (PLANE_PRIOR * PLANE_PRIOR_ARM2) * xi[k + 3]);
                    }
                    ldlt6_solve(H, g, x);
                }
                CW_MARK(9, QW);
                pose_store(se3_exp_gn(x), E);                     // estimate = SE3::exp(x) (vector6d_to_mat4d :91)
                // Convergence from the twist itself (gn_verdict): unless it is too close to call, the verdict is known NOW and the loop need
                // not make one more pass just to learn that it was over; otherwise the tail takes the logarithm, as the reference does.
                verdict = gn_verdict(x, A.eps);
            }
            __syncwarp();
            CW_MARK(10, QW);
        }
        __syncthreads();   // S2: the estimate is visible to the query warps
        CW_MARK(15, 0);
        CTA_MARK(3);
        ++j;
        if (verdict == 1) {   // iteration j-1 converged: finish its bookkeeping (the tail above, without a pass beside it) and leave
            if (warp == QW) {
                const Pose est = pose_load(E);
                if (lane == 0) pose_store(mul(est, pose_load(Ticp)), Ticp);
                if (blockIdx.x == 0 && lane == 2) {
                    if (A.est_trace) pose_store(est, A.est_trace + 7 * (size_t)(j - 1));
                    if (A.ncorr_trace) A.ncorr_trace[j - 1] = (long long)S[I_NCORR];
                    if (A.hg_trace) {
                        double H[36], g[6];
                        if (PLANE) expand_plane_equations(S, H, g);
                        else expand_normal_equations(S, H, g);
                        double *o = A.hg_trace + 42 * (size_t)(j - 1);
                        for (int k = 0; k < 36; ++k) o[k] = H[k];
                        for (int k = 0; k < 6; ++k) o[36 + k] = g[k];
                    }
                }
            }
            converged = 1;
            __syncthreads();
            break;
        }
    }
    FT_MARK(2);
    LIMU_TRACE(3);
    // new_pose = T_icp * init_guess (:129); with an empty map the loop did not run and this is init_guess itself (:99-100). What follows is
    // CTA 0's: in a launch without the map-update epilogue (pipelined odometry) the next scan's k_voxelize sits behind this kernel in the
    // stream, so its tail is kept short: thread 0 takes the pose, warp 0 leaves the result block in pinned host memory, then thread 0
    // takes the deskew twist while warps 1.. write the keypoints out.
    if (blockIdx.x == 0) {
        if (threadIdx.x == 0) {
            const Pose np = run_icp ? mul(pose_load(Ticp), pose_load(Tinit)) : pose_load(Tinit);
            pose_store(np, A.out);
            A.out[7] = (double)j; A.out[8] = (double)converged; A.out[9] = S[I_NCORR]; A.out[10] = S[I_NCORR + 1]; A.out[11] = S[I_NCORR + 2]; A.out[12] = (double)n;
            if (A.host_res && n_keypoints >= 0) *A.iqr_count = n_keypoints;   // (part of the result block that leaves below; the warps that write the cloud out store it again)
            if (!A.upd_down && A.loop_flag) {
                // the map update of this scan, on another stream, is released by this flag: the pose is in memory, the loop's reads of the map are over
                __threadfence();
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(A.loop_flag), "r"(A.loop_seq) : "memory");
            }
        }
        if (A.host_res && threadIdx.x < 32) {
            // Result block -> pinned host memory as ONE 256-byte store of warp 0, FIRST (the stores take a microsecond or two to cross PCIe,
            // and a kernel is not over before they have): words 0..29 data, 30 = XOR of the others, 31 = this launch's sequence number.
            // No system-scope fence: the host accepts the block when the sequence number is the one it waits for AND the checksum holds,
            // so a torn read is simply read again. (The keypoint CLOUD is complete when the kernel is: a host that wants it waits for that.)
            __syncwarp();
            unsigned long long w = 0ull;
            if ((int)threadIdx.x < A.res_doubles && threadIdx.x < 30) w = (unsigned long long)__double_as_longlong(__ldcg(A.res_block + threadIdx.x));
            if (threadIdx.x == 31) w = (unsigned long long)A.loop_seq;
            unsigned long long x = threadIdx.x == 30 ? 0ull : w;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
            if (threadIdx.x == 30) w = x;
            reinterpret_cast<volatile unsigned long long *>(A.host_res)[threadIdx.x] = w;
        }
        if (threadIdx.x == 0 && !A.upd_down) publish_twist(A, pose_load(A.out));   // (~3 us of scalar code beside the cloud being written out)
        if (n_keypoints >= 0) {   // keypoints for the host
            if (A.host_res) { if (threadIdx.x >= 32) iqr_write_out<ICP_BLOCK - 32>(qidx_s, A.iqr_in, n_keypoints, A.iqr_out, A.iqr_count, (int)threadIdx.x - 32); }
            else iqr_write_out<ICP_BLOCK>(qidx_s, A.iqr_in, n_keypoints, A.iqr_out, A.iqr_count, (int)threadIdx.x);
        }
    }
    if (A.upd_down) frame_update_epilogue<ICP_BLOCK>(A, gs, E);
    FT_MARK(5);
    LIMU_TRACE(4);
    // the last CTA out re-arms the barrier for the next launch
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(A.exit_count, 1u) == gridDim.x - 1) { *A.barrier = 0u; *A.barrier_icp = 0u; *A.exit_count = 0u; __threadfence(); }
    }
}

// local_map.update(down_sampled, new_pose) as a launch of its own (pipelined odometry: the Gauss-Newton loop of a scan is launched before the
// caller has confirmed that scan, its map update only afterwards). Two CTAs' worth of registers at most, so that it fits beside the next
// scan's k_voxelize.
// at most 64 registers (256 threads x 4): the CTA has to fit into the 16 K registers k_voxelize_lean (1024 x 48) leaves on the SM -- at 72 the two kernels took
// turns on every SM instead of running beside each other (-10 % scans/s)
static __global__ void __launch_bounds__(ICP_BLOCK, 4) k_frame_update(const IcpArgs A) {
    __shared__ double E[7];
    GridSync gs{A.barrier, 0u, gridDim.x};
    LIMU_TRACE(20);
    frame_update_epilogue<ICP_BLOCK, false>(A, gs, E);
    __syncthreads();
    LIMU_TRACE(23);
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(A.exit_count, 1u) == gridDim.x - 1) { *A.barrier = 0u; *A.exit_count = 0u; __threadfence(); }
    }
}

int frame_update_device(limu_map *m, IcpArgs A) {
    limu_ctx *c = m->ctx;
    A.map = m->view();
    if (!A.barrier) A.barrier = reinterpret_cast<unsigned int *>(c->d_small.as<double>() + 56);
    A.exit_count = A.barrier + 1;
    A.upd_counters = m->counters.as<unsigned long long>();
    if (!A.status) A.status = c->d_status;
    A.upd_capacity = (long long)m->capacity; A.upd_max_distance = m->max_distance;
    void *args[] = {&A};
    LIMU_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_frame_update, dim3(c->sm_count), dim3(ICP_BLOCK), args, 0, c->stream));
    LIMU_LAUNCHED();
    return LIMU_OK;
}

// ---- stand-alone align_clouds -------------------------------------------------------------------------
static __global__ void __launch_bounds__(ICP_BLOCK) k_align_partial(const double *__restrict__ src, const double *__restrict__ tgt, int64_t n, double th,
                                                                   double *partials) {
    __shared__ double red[(ICP_BLOCK / 32) * NS];
    double acc[NS];
#pragma unroll
    for (int k = 0; k < NS; ++k) acc[k] = 0.0;
    for (int64_t q = (int64_t)blockIdx.x * ICP_BLOCK + threadIdx.x; q < n; q += (int64_t)gridDim.x * ICP_BLOCK) {
        const V3 s{src[3 * q], src[3 * q + 1], src[3 * q + 2]}, t{tgt[3 * q], tgt[3 * q + 1], tgt[3 * q + 2]};
        accumulate(acc, s, t, sqnorm3(s.x - t.x, s.y - t.y, s.z - t.z), th);
        acc[16] += 1.0;
    }
    block_reduce_row(acc, red, partials + (size_t)blockIdx.x * NS);
}
static __global__ void k_align_solve(const double *partials, int nblocks, double *out /* H36 g6 x6 pose7 */) {
    __shared__ double S[NS];
    if (threadIdx.x < NS) {
        double v = 0.0;
        for (int b = 0; b < nblocks; ++b) v += partials[(size_t)b * NS + threadIdx.x];
        S[threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double H[36], g[6], ng[6], x[6];
        expand_normal_equations(S, H, g);
        for (int k = 0; k < 6; ++k) ng[k] = -g[k];
        ldlt6_solve(H, ng, x);
        for (int k = 0; k < 36; ++k) out[k] = H[k];
        for (int k = 0; k < 6; ++k) { out[36 + k] = g[k]; out[42 + k] = x[k]; }
        pose_store(se3_exp(x), out + 48);
    }
}

static int g_icp_blocks_per_sm = 0;

static int icp_partial_rows(limu_ctx *c) { return c->sm_count * 4; }   // >= the largest grid of any shape

int icp_partials_reserve(limu_ctx *c, DevBuf &rows, cudaStream_t s) {   // (value, stamp) word pairs of NS_MAX doubles, two rows per CTA
    const void *before = rows.p;
    LIMU_TRY(rows.reserve((size_t)2 * icp_partial_rows(c) * NS_MAX * 16 + 256, s));
    if (rows.p != before) LIMU_CUDA_TRY(cudaMemsetAsync(rows.p, 0, rows.bytes, s));
    return LIMU_OK;
}

int icp_device(limu_map *m, IcpArgs A, int64_t n_hint, int icp_mode, bool sharded, cudaStream_t stream) {
    limu_ctx *c = m->ctx;
    sharded = sharded && c->comm && c->comm->nranks > 1;   // point-sharded call: fused peer exchange
    const bool nn27 = (icp_mode & LIMU_ICP_NN27) != 0, plane = (icp_mode & LIMU_ICP_PLANE) != 0;
    const bool grouped = n_hint <= 16384 && m->cap <= 64;   // latency shape: eight lanes per query, one CTA per SM
    // bandwidth shape with the reference's rules: voxel blocks are staged through dynamic shared memory (two buffers of eight blocks per query warp)
    size_t stage_bytes = (!grouped && !nn27 && !plane && block_stride(m->cap) <= STAGE_MAX_STRIDE) ? (size_t)(ICP_BLOCK / 32 - 1) * STAGE_WARP_DOUBLES * sizeof(double) : 0;
    // latency shape with the IQR filter in front: the candidates (a few per cent more than the keypoints the hint counts) are ranked by the whole
    // grid out of a copy in every CTA's shared memory -- static up to IQR_GRID_MAX of them, dynamic (8192 or 16384) when the hint announces more
    int iqr_cap = IQR_GRID_MAX;
    if (grouped && A.iqr_in && n_hint + n_hint / 8 + 64 > IQR_GRID_MAX) {
        iqr_cap = (n_hint + n_hint / 8 + 64 <= 8192) ? 8192 : IQR_GRID_MAX_DYN;
        stage_bytes = (size_t)iqr_cap * (sizeof(double) + sizeof(unsigned short));
        static bool iqr_attr_set = false;
        if (!iqr_attr_set) {
            const void *lat[4] = {(const void *)k_icp_persistent<0, false, false>, (const void *)k_icp_persistent<0, false, true>, (const void *)k_icp_persistent<0, true, false>,
                                  (const void *)k_icp_persistent<0, true, true>};
            for (const void *f : lat) LIMU_CUDA_TRY(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, IQR_GRID_MAX_DYN * 10));
            iqr_attr_set = true;
        }
    }
    static bool stage_attr_set[64] = {};
    if (stage_bytes && !stage_attr_set[c->device & 63]) {
        LIMU_CUDA_TRY(cudaFuncSetAttribute(k_icp_persistent<1, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stage_bytes));
        stage_attr_set[c->device & 63] = true;
    }
    if (!grouped) {
        int b = 0;
        LIMU_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, nn27 || plane ? (const void *)k_icp_persistent<1, true, true> : (const void *)k_icp_persistent<1, false, false>,
                                                                    ICP_BLOCK, stage_bytes));
        g_icp_blocks_per_sm = std::max(1, b);
    }
    // queries per CTA: 7 query warps (the eighth warp is the solver warp); eight lanes per query in the latency shape, one in the bandwidth shape
    const bool lanes8 = grouped;
    const int64_t want = std::max<int64_t>(1, div_up(std::max<int64_t>(n_hint, 1) * (lanes8 ? 8 : 1), ICP_BLOCK - 32));
    // Pipelined path: a k_gate thread may already sit on an SM, waiting for THIS launch, when its CTAs are placed -- and an SM that runs a
    // kernel without shared memory is not handed a CTA that needs a different shared-memory carve-out until it has drained. A cooperative
    // grid that needs every SM of the GPU would then wait for the gate and the gate for the grid (until the gate's 5 s give-up; seen with
    // ~7 k keypoints per scan = 148 CTAs, configs[2]). Such launches leave GATE_SLACK_SMS SMs free.
    const int sms = A.loop_flag ? std::max(1, c->sm_count - GATE_SLACK_SMS) : c->sm_count;
    int grid = (int)std::min<int64_t>(want, (int64_t)sms * (grouped ? 1 : std::min(g_icp_blocks_per_sm, LIMU_BW_CTAS)));
    grid = (int)std::min<int64_t>(grid, (int64_t)icp_partial_rows(c));
    const int icp_blocks = grid;   // the Gauss-Newton loop is latency bound at keypoint counts: it runs on the leading CTAs only
    if (A.upd_down) grid = std::max(grid, c->sm_count);   // the insert and the eviction sweep want one CTA per SM
    A.map = m->view();
    A.map_counters = m->counters.as<unsigned long long>();
    A.ll_stamp_base = c->ll_seq;
    c->ll_seq = (c->ll_seq + (unsigned int)std::max(A.max_iter, 0) + 2u) & 0x7FFFFFFFu;
    // grid barrier + exit counter live in the context's zero-initialised small area; the last CTA out re-arms them
    if (!A.barrier) A.barrier = reinterpret_cast<unsigned int *>(c->d_small.as<double>() + 56);
    A.exit_count = A.barrier + 1;
    A.barrier_icp = A.barrier + 2;
    A.icp_blocks = icp_blocks;
    A.coop_scan = n_hint >= 32768 ? 1 : 0;
    A.grouped = grouped ? 1 : 0;
    A.stage_doubles = grouped ? 0 : (int)(stage_bytes / sizeof(double));
    A.iqr_cap = iqr_cap;
    A.nranks = 1; A.rank = 0;
    if (!A.status) A.status = c->d_status;
    if (sharded) {
        limu_comm *cm = c->comm;
        A.nranks = cm->nranks; A.rank = cm->rank; A.mbox_local = cm->mbox_local; A.comm_error = cm->d_error;
        for (int r = 0; r < cm->nranks; ++r) A.mbox_peer[r] = cm->mbox_peer[r];
        A.stamp_base = cm->stamp_base;   // advanced by the iterations this call executes once they are known (icp_common)
    }
    A.upd_counters = m->counters.as<unsigned long long>();
    A.upd_capacity = (long long)m->capacity; A.upd_max_distance = m->max_distance;
    void *args[] = {&A};
    if (!stream) stream = c->stream;
    if (c->profiling) { LIMU_CUDA_TRY(cudaEventRecord(c->ev[LIMU_STAGE_ICP][0], stream)); c->ev_used[LIMU_STAGE_ICP] = true; }
    if (plane && sharded) { set_error("the point-to-plane variant is not available in the point-sharded loop"); return LIMU_ERR_INVALID; }
    const void *fns[2][2][2] = {{{(const void *)k_icp_persistent<0, false, false>, (const void *)k_icp_persistent<0, false, true>},
                                 {(const void *)k_icp_persistent<0, true, false>, (const void *)k_icp_persistent<0, true, true>}},
                                {{(const void *)k_icp_persistent<1, false, false>, (const void *)k_icp_persistent<1, false, true>},
                                 {(const void *)k_icp_persistent<1, true, false>, (const void *)k_icp_persistent<1, true, true>}}};
    const void *fn = fns[grouped ? 0 : 1][nn27 ? 1 : 0][plane ? 1 : 0];
    LIMU_CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(ICP_BLOCK), args, stage_bytes, stream));
    LIMU_LAUNCHED();
    if (c->profiling) LIMU_CUDA_TRY(cudaEventRecord(c->ev[LIMU_STAGE_ICP][1], stream));
    return LIMU_OK;
}

// ---- multi-hypothesis registration: K Gauss-Newton loops of the latency shape in one launch --------------------------------------------
// Relocalization runs ICP of one scan against one map from a grid of initial guesses and keeps the best. One loop of the latency shape
// leaves most of the GPU idle (a few thousand keypoints on ~72 CTAs), so here every hypothesis is run by a GROUP of G CTAs with the
// loop's own device functions (query pass and memo, LDLT / Schur solve, se3_exp_gn, gn_verdict, stamped row exchange), and a persistent
// cooperative grid of as many groups as are co-resident takes the hypotheses in waves (group g serves hypotheses g, g + groups, ...).
// G depends on the query count only, so a hypothesis's sums -- and its result -- do not depend on K or on its place in the list.
constexpr int MULTI_STEPS = 16;        // query steps of a warp per pass that G aims at (G = ceil(8 n / (224 MULTI_STEPS)), 1 ... 8)
constexpr int MULTI_OUT = 12;          // doubles per hypothesis: pose 7, iterations, converged, inliers, sum of d^2, pad
constexpr int MULTI_MAX_G = ICP_BLOCK / 32;   // one row per warp in the fold below

int icp_multi_group_ctas(int64_t n) {
    return (int)std::min<int64_t>(MULTI_MAX_G, std::max<int64_t>(1, div_up(std::max<int64_t>(n, 1) * 8, (int64_t)(ICP_BLOCK - 32) * MULTI_STEPS)));
}

struct MultiArgs {
    IcpArgs A;                 // map, points, tau_sq, th, max_iter, eps, partials, ll_stamp_base, map_counters; work = groups x n x 3
    const double *guesses;     // k x 7
    double *out;               // k x MULTI_OUT
    int k, group_ctas;
};

// Fitness of a converged hypothesis: correspondences of its final working cloud under the loop's neighbour rule and tau^2 test, counted and
// their squared distances summed by the group's leading lane (transform: the cloud still needs the last estimate applied).
template <bool NN27, int ROUNDS>
__device__ __forceinline__ void fitness_pass_grouped(const IcpArgs &A, const volatile double *Pv, const double *in, bool transform, int64_t n, int64_t gbase,
                                                     int64_t gstride, int lane, int &inliers, double &d2sum) {
    const int l8 = lane & 7;
    const unsigned gmask = 0xFFu << (lane & 24);
    for (int64_t q0 = gbase - (lane >> 3); q0 < n; q0 += gstride) {
        const int64_t q = q0 + (lane >> 3);
        if (q >= n) continue;   // group-uniform
        const Pose P{Pv[0], Pv[1], Pv[2], Pv[3], Pv[4], Pv[5], Pv[6]};
        const V3 raw{in[3 * q], in[3 * q + 1], in[3 * q + 2]};
        const V3 s = transform ? apply(P, raw) : raw;
        V3 tg{0.0, 0.0, 0.0};
        int slot = -1, count = 0, own = 1, rank = -1;
        double d2 = 0.0;
        if (NN27) group8_closest27(A.map, s, gmask, l8, slot, count, own, d2, rank);
        else group8_closest<ROUNDS>(A.map, s, gmask, l8, slot, count, own, d2, rank, tg);
        if (rank < 0) d2 = sqnorm3(s.x, s.y, s.z);   // nothing found -> (0,0,0), range-tested like a real point
        if (l8 == 0 && d2 < A.tau_sq) { ++inliers; d2sum += d2; }
    }
}

// Publish this CTA's row (thread t < NS holds column t as `mine`) with the exchange's stamp, then fold the G rows of the group: warp g
// reads row g, thread t adds the eight warp values in warp order -- the order of the loop kernel's fold for a grid of G <= 8 CTAs.
__device__ __forceinline__ void multi_exchange(unsigned long long *rows, int G, int rank, unsigned int stamp, double mine, double *red, double *S) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < NS) ll_store(rows + ((size_t)rank * NS + threadIdx.x) * 2, mine, stamp);
    double v = 0.0;
    if (warp < G && lane < NS) {
        unsigned int spins = 0u;
        while (!ll_load(rows + ((size_t)warp * NS + lane) * 2, stamp, v))
            if (++spins > (1u << 24)) __trap();   // a CTA of the group never published its row: fail loudly instead of hanging the device
    }
    __syncthreads();   // (every reader of red is done)
    red[warp * 32 + lane] = 0.0 + v;
    __syncthreads();
    if (threadIdx.x < NS) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < ICP_BLOCK / 32; ++w) s += red[w * 32 + threadIdx.x];
        S[threadIdx.x] = s;
    }
    __syncthreads();
}

template <bool NN27>
static __global__ void __launch_bounds__(ICP_BLOCK, 2) k_icp_multi(const MultiArgs M) {
    constexpr int QW = ICP_BLOCK / 32 - 1;   // query warps; the last warp is the solver warp, as in k_icp_persistent
    __shared__ double red[(ICP_BLOCK / 32) * 32];
    __shared__ double S[NS];
    __shared__ double E[7], Tinit[7], Ticp[7];
    __shared__ int done, verdict;
    const int G = M.group_ctas, grp = (int)blockIdx.x / G, rank = (int)blockIdx.x % G, groups = (int)gridDim.x / G;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t n = M.A.n_max;
    IcpArgs A = M.A;
    A.work = M.A.work + (size_t)grp * 3 * (size_t)n;   // this group's working cloud
    unsigned long long *rows0 = reinterpret_cast<unsigned long long *>(A.partials) + (size_t)grp * 2 * G * NS * 2;   // two parities of G rows
    const int64_t gbase = (((int64_t)rank * QW + warp) * 32) / 8 + (lane >> 3), gstride = (int64_t)G * QW * 4;
    const bool run_icp = !(__ldcg(A.map_counters) == 0ull || A.max_iter <= 0);   // ICP :99-100: empty map -> init_guess
    unsigned int x = 0u;   // exchanges this group made so far: its stamps never repeat across the hypotheses it serves
    QueryMemo memo;        // (keyed by voxel index: the map does not change inside the launch, so it stays valid from one hypothesis to the next)
    memo.own = -1; memo.kx = memo.ky = memo.kz = 0; memo.slot = -1; memo.count = 0;
    for (int h = grp; h < M.k; h += groups) {
        __syncthreads();   // the previous hypothesis is finished with the shared state
        if (threadIdx.x < 7) { Tinit[threadIdx.x] = M.guesses[7 * (size_t)h + threadIdx.x]; Ticp[threadIdx.x] = threadIdx.x == 3 ? 1.0 : 0.0; }
        if (threadIdx.x < NS) S[threadIdx.x] = 0.0;
        if (threadIdx.x == 0) { verdict = 0; done = 0; }
        __syncthreads();
        int j = 0, converged = 0;
        bool fresh = false;   // the working cloud already holds the final estimate applied (a pass was made after the converging iteration)
        if (run_icp) for (;;) {
            const bool no_more = j >= A.max_iter;
            if (warp < QW) {
                if (!no_more) {
                    double acc = 0.0;
                    int ncorr = 0, ncand = 0, nmiss = 0;   // (statistics of the single loop; not reported per hypothesis)
                    const volatile double *Pv = j == 0 ? Tinit : E;
                    const double *in = j == 0 ? A.points : A.work;
                    if (A.map.cap <= 8) icp_query_pass_grouped<NN27, false, 1>(A, Pv, in, nullptr, n, gbase, gstride, lane, acc, ncorr, ncand, nmiss, &memo, nullptr);
                    else if (A.map.cap <= 16) icp_query_pass_grouped<NN27, false, 2>(A, Pv, in, nullptr, n, gbase, gstride, lane, acc, ncorr, ncand, nmiss, &memo, nullptr);
                    else icp_query_pass_grouped<NN27, false, 3>(A, Pv, in, nullptr, n, gbase, gstride, lane, acc, ncorr, ncand, nmiss, &memo, nullptr);
                    red[warp * 32 + lane] = (lane & 1) ? 0.0 : acc;   // lane 2i holds sum i
                }
            } else if (j > 0) {
                // tail of iteration j-1, overlapped with pass j: T_icp = estimate * T_icp (:122), |log(estimate)| < eps (:124) when the twist left it open
                const Pose est = pose_load(E);
                if (lane == 0) pose_store(mul(est, pose_load(Ticp)), Ticp);
                if (lane == 1 && verdict == 2) {
                    double lg[6];
                    se3_log(est, lg);
                    done = norm6(lg) < A.eps;
                }
            }
            __syncthreads();
            if (j > 0 && verdict == 2 && done) { converged = 1; fresh = !no_more; break; }
            if (no_more) break;
            double mine = 0.0;
            if (threadIdx.x < NS) {   // the CTA row in the loop kernel's layout: 16 sums from the even lanes (the counters stay zero)
                const int src_lane = threadIdx.x < 16 ? 2 * (int)threadIdx.x : 2 * ((int)threadIdx.x - 16) + 1;
#pragma unroll
                for (int w = 0; w < QW; ++w) mine += red[w * 32 + src_lane];
            }
            const unsigned int stamp = 0x80000000u | ((A.ll_stamp_base + x) & 0x7FFFFFFFu);
            multi_exchange(rows0 + (size_t)(x & 1u) * G * NS * 2, G, rank, stamp, mine, red, S);
            ++x;
            if (warp == QW && lane == 0) {
                double xv[6];
                solve_point_to_point(S, xv);
                pose_store(se3_exp_gn(xv), E);
                verdict = gn_verdict(xv, A.eps);
            }
            __syncthreads();
            ++j;
            if (verdict == 1) {
                if (warp == QW && lane == 0) pose_store(mul(pose_load(E), pose_load(Ticp)), Ticp);
                converged = 1;
                __syncthreads();
                break;
            }
        }
        // fitness over src_after: points * init_guess when the loop did not run, else the working cloud (plus the last estimate unless applied)
        int inliers = 0;
        double d2sum = 0.0;
        if (warp < QW) {
            const volatile double *Pv = run_icp ? E : Tinit;
            const double *in = run_icp ? A.work : A.points;
            if (NN27 || A.map.cap <= 8) fitness_pass_grouped<NN27, 1>(A, Pv, in, !fresh, n, gbase, gstride, lane, inliers, d2sum);
            else if (A.map.cap <= 16) fitness_pass_grouped<NN27, 2>(A, Pv, in, !fresh, n, gbase, gstride, lane, inliers, d2sum);
            else fitness_pass_grouped<NN27, 3>(A, Pv, in, !fresh, n, gbase, gstride, lane, inliers, d2sum);
            inliers = __reduce_add_sync(0xFFFFFFFFu, inliers);
            d2sum = warp_sum(d2sum);
        }
        if (lane == 0) { red[warp * 32] = (double)inliers; red[warp * 32 + 1] = d2sum; }
        __syncthreads();
        double mine = 0.0;
        if (threadIdx.x < 2) {
#pragma unroll
            for (int w = 0; w < QW; ++w) mine += red[w * 32 + threadIdx.x];
        }
        const unsigned int stamp = 0x80000000u | ((A.ll_stamp_base + x) & 0x7FFFFFFFu);
        multi_exchange(rows0 + (size_t)(x & 1u) * G * NS * 2, G, rank, stamp, mine, red, S);
        ++x;
        if (rank == 0 && threadIdx.x == 0) {
            double *o = M.out + (size_t)h * MULTI_OUT;
            pose_store(run_icp ? mul(pose_load(Ticp), pose_load(Tinit)) : pose_load(Tinit), o);   // new_pose = T_icp * init_guess (:129)
            o[7] = (double)j; o[8] = (double)converged; o[9] = S[0]; o[10] = S[1];
        }
    }
}

// Fitness of one hypothesis of the bandwidth shape (the loop kernel run once per guess): src_after is rebuilt from the points by the guess
// and the estimates of the loop's iterations applied in turn, as the loop applied them; one thread per query; block rows folded on the host.
template <bool NN27>
static __global__ void __launch_bounds__(ICP_BLOCK) k_icp_fitness(const MapView map, const double *points, int64_t n, const double *poses, int nposes,
                                                                   double tau_sq, double *rows /* [grid][2]: inliers, sum of d^2 */) {
    __shared__ double red[2][ICP_BLOCK / 32];
    double inliers = 0.0, d2sum = 0.0;
    for (int64_t q = (int64_t)blockIdx.x * ICP_BLOCK + threadIdx.x; q < n; q += (int64_t)gridDim.x * ICP_BLOCK) {
        V3 s{points[3 * q], points[3 * q + 1], points[3 * q + 2]};
        for (int p = 0; p < nposes; ++p) s = apply(pose_load(poses + 7 * p), s);
        Nearest nn;
        nn.rank = -1;
        if (NN27) {
            nn = map_closest27(map, s);
        } else {
            int count = 0, own = 1;
            const int slot = map_locate(map, s, &count, &own);
            if (slot >= 0) block_closest(map, slot, count, s, nn);
        }
        const double d2 = nn.rank >= 0 ? sqnorm3(nn.x - s.x, nn.y - s.y, nn.z - s.z) : sqnorm3(s.x, s.y, s.z);
        if (d2 < tau_sq) { inliers += 1.0; d2sum += d2; }
    }
    inliers = warp_sum(inliers);   // fixed trees: warp, then warps in order
    d2sum = warp_sum(d2sum);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = inliers; red[1][threadIdx.x >> 5] = d2sum; }
    __syncthreads();
    if (threadIdx.x < 2) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < ICP_BLOCK / 32; ++w) v += red[threadIdx.x][w];
        rows[2 * (size_t)blockIdx.x + threadIdx.x] = v;
    }
}

// ---- pose scoring and global relocalization: the fitness of k_icp_multi at millions of poses, without a Gauss-Newton loop --------------
// Where the poses come from: a list (7 doubles each), or the planar grid of limu_relocalize -- candidate p = (l * ny + j) * nx + i is
// center * {q = (0, 0, sin(t_l / 2), cos(t_l / 2)), t = (x_i, y_j, 0)}, built where it is scored, so a grid never exists in memory.
struct PoseSource {
    const double *list;   // k x 7, or null: the grid
    double center[7];
    const double *yaw;    // nyaw x 2: sin(t_l / 2), cos(t_l / 2) (host libm: the table is tiny)
    int64_t nx, ny;
    double step_xy;
    __device__ __forceinline__ Pose at(int64_t p) const {
        if (list) return pose_load(list + 7 * p);
        const int64_t i = p % nx, r = p / nx, j = r % ny, l = r / ny;
        const double x = ((double)i - 0.5 * (double)(nx - 1)) * step_xy, y = ((double)j - 0.5 * (double)(ny - 1)) * step_xy;
        return mul(pose_load(center), Pose{0.0, 0.0, yaw[2 * l], yaw[2 * l + 1], x, y, 0.0});
    }
};

constexpr int SCORE_BLOCK = 256;

// One warp per pose (a persistent grid of warps takes poses p, p + warps, ...), one lane per query: the points moved by the pose, the
// correspondence test of k_icp_multi's fitness under the loop's neighbour rule (map_locate + block_closest / map_closest27, any cap), and a
// per-pose reduction inside the warp -- so a pose's sums depend on n only, never on k, on the pose's place in the list or on the grid.
// (Eight lanes per query, as in fitness_pass_grouped, was measured slower overall: DESIGN.md section 9.)
// hist (optional): histogram of the inlier counts (n + 1 bins) for the selection of limu_relocalize.
template <bool NN27>
static __global__ void __launch_bounds__(SCORE_BLOCK) k_score_poses(const MapView map, const double *points, int64_t n, const PoseSource src,
                                                                    int64_t k, double tau_sq, int64_t *inliers_out, double *rms_out,
                                                                    unsigned long long *hist) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (SCORE_BLOCK / 32);
    for (int64_t p = (int64_t)blockIdx.x * (SCORE_BLOCK / 32) + (threadIdx.x >> 5); p < k; p += warps) {   // warp-uniform
        const Pose P = src.at(p);
        long long inl = 0;
        double d2sum = 0.0;
        for (int64_t q = lane; q < n; q += 32) {
            const V3 s = apply(P, V3{points[3 * q], points[3 * q + 1], points[3 * q + 2]});
            Nearest nn;
            nn.rank = -1;
            if (NN27) {
                nn = map_closest27(map, s);
            } else {
                int count = 0, own = 1;
                const int slot = map_locate(map, s, &count, &own);
                if (slot >= 0) block_closest(map, slot, count, s, nn);
            }
            const double d2 = nn.rank >= 0 ? sqnorm3(nn.x - s.x, nn.y - s.y, nn.z - s.z) : sqnorm3(s.x, s.y, s.z);   // nothing found -> (0,0,0)
            if (d2 < tau_sq) { ++inl; d2sum += d2; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) inl += __shfl_down_sync(0xFFFFFFFFu, inl, o);
        d2sum = warp_sum(d2sum);
        if (lane == 0) {
            inliers_out[p] = inl;
            rms_out[p] = inl > 0 ? sqrt(d2sum / (double)inl) : 0.0;   // limu_icp_multi's expression
            if (hist) atomicAdd(hist + inl, 1ull);
        }
    }
}

// Exact top-M of limu_relocalize by (inliers desc, rms asc, index asc). The inlier histogram gives the class T the M-th candidate falls in;
// inside that class the order is that of the 128-bit key (rms bits, index) -- rms >= 0, so its bits order like the values -- and a radix
// select fixes that key's top `digits` bytes, eight bits per pass over the candidates: a candidate of class T is taken when its key's top
// bytes are <= the prefix found (Sel::mh / ml mask them).
struct Sel {
    int64_t T;
    unsigned long long mh, ml, ph, pl;
};
__device__ __forceinline__ bool sel_taken(const Sel &S, int64_t inl, double rms, int64_t p) {
    if (inl != S.T) return inl > S.T;
    const unsigned long long h = (unsigned long long)__double_as_longlong(rms) & S.mh, l = (unsigned long long)p & S.ml;
    return h < S.ph || (h == S.ph && l <= S.pl);
}
// Histogram of key byte `digit` (0: the top byte of the rms bits ... 15: the low byte of the index) over the class-T candidates whose
// decided bytes equal the prefix.
static __global__ void __launch_bounds__(256) k_select_digit(const int64_t *inliers, const double *rms, int64_t k, const Sel S, int digit,
                                                             unsigned long long *hist256) {
    __shared__ unsigned int h[256];
    h[threadIdx.x] = 0u;
    __syncthreads();
    for (int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x; p < k; p += (int64_t)gridDim.x * 256) {
        if (inliers[p] != S.T) continue;
        const unsigned long long hi = (unsigned long long)__double_as_longlong(rms[p]), lo = (unsigned long long)p;
        if ((hi & S.mh) != S.ph || (lo & S.ml) != S.pl) continue;
        const unsigned int d = (unsigned int)((digit < 8 ? hi >> (56 - 8 * digit) : lo >> (56 - 8 * (digit - 8))) & 255u);
        atomicAdd(&h[d], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(hist256 + threadIdx.x, (unsigned long long)h[threadIdx.x]);
}
// The selected candidates as (index, inliers, rms bits), in no particular order (the host sorts at most 4096 of them).
static __global__ void __launch_bounds__(256) k_select_gather(const int64_t *inliers, const double *rms, int64_t k, const Sel S,
                                                              unsigned long long *count, int64_t cap, long long *rec) {
    for (int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x; p < k; p += (int64_t)gridDim.x * 256) {
        if (!sel_taken(S, inliers[p], rms[p], p)) continue;
        const unsigned long long at = atomicAdd(count, 1ull);
        if ((int64_t)at < cap) { rec[3 * at] = p; rec[3 * at + 1] = inliers[p]; rec[3 * at + 2] = __double_as_longlong(rms[p]); }
    }
}
// The poses of m grid candidates, by index.
static __global__ void k_grid_poses(const PoseSource src, const int64_t *index, int m, double *poses) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) pose_store(src.at(index[i]), poses + 7 * (size_t)i);
}

#ifdef LIMU_ICP_PHASE_TIMING
extern "C" int limu_debug_frame_marks(double out[72]) {
    unsigned long long h[72];
    if (cudaMemcpyFromSymbol(h, g_frame_marks, sizeof h) != cudaSuccess) return -1;
    for (int k = 0; k < 72; ++k) out[k] = (double)h[k];
    return 0;
}
#endif

// ---- un-fused baseline for the sharded loop: step kernel -> fold kernel -> ncclAllReduce -> solve kernel, host in the loop ----
static __global__ void __launch_bounds__(ICP_BLOCK, LIMU_BW_CTAS) k_icp_step(const IcpArgs A, const double *state /* E at +24 */, int first, double *rows) {
    __shared__ double red[(ICP_BLOCK / 32) * 32];
    __shared__ double Pose7[7];
    const int64_t n = A.n_max;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < 7) Pose7[threadIdx.x] = first ? A.init_pose[threadIdx.x] : state[24 + threadIdx.x];
    __syncthreads();
    double acc = 0.0;
    int ncorr = 0, ncand = 0, nmiss = 0;
    const int64_t wbase = ((int64_t)blockIdx.x * (ICP_BLOCK / 32) + warp) * 32, wstride = (int64_t)A.icp_blocks * ICP_BLOCK;
    const double *in = first ? A.points : A.work;
    if (A.map.cap <= 8) icp_query_pass_coop<1>(A, Pose7, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
    else if (A.map.cap <= 16) icp_query_pass_coop<2>(A, Pose7, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
    else icp_query_pass_coop<3>(A, Pose7, in, n, wbase, wstride, lane, acc, ncorr, ncand, nmiss);
    ncorr = __reduce_add_sync(0xFFFFFFFFu, ncorr);
    ncand = __reduce_add_sync(0xFFFFFFFFu, ncand);
    nmiss = __reduce_add_sync(0xFFFFFFFFu, nmiss);
    red[warp * 32 + lane] = (lane & 1) ? (lane == 1 ? (double)ncorr : lane == 3 ? (double)ncand : lane == 5 ? (double)nmiss : 0.0) : acc;
    __syncthreads();
    if (threadIdx.x < NS) {
        const int src_lane = threadIdx.x < 16 ? 2 * threadIdx.x : 2 * (threadIdx.x - 16) + 1;
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < ICP_BLOCK / 32; ++w) v += red[w * 32 + src_lane];
        rows[(size_t)blockIdx.x * NS + threadIdx.x] = v;
    }
}
static __global__ void k_icp_fold_rows(const double *rows, int nblocks, double *sums) {
    if (threadIdx.x < NS) {
        double v = 0.0;
        for (int b = 0; b < nblocks; ++b) v += rows[(size_t)b * NS + threadIdx.x];
        sums[threadIdx.x] = v;
    }
}
static __global__ void k_icp_solve_step(double *state, double eps, int first) {
    if (threadIdx.x != 0) return;
    double H[36], g[6], x[6], lg[6];
    expand_normal_equations(state, H, g);
#pragma unroll
    for (int k = 0; k < 6; ++k) g[k] = -g[k];
    ldlt6_solve(H, g, x);
    const Pose est = se3_exp(x);
    const Pose Ticp = first ? pose_identity() : pose_load(state + 32);
    pose_store(mul(est, Ticp), state + 32);
    pose_store(est, state + 24);
    se3_log(est, lg);
    state[40] = norm6(lg) < eps ? 1.0 : 0.0;
    state[41] = first ? 1.0 : state[41] + 1.0;
}

typedef int (*nccl_allreduce_fn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
int comm_nccl_allreduce_sum_f64(limu_ctx *c, double *buf, size_t count);   // comm.cu

static int icp_sharded_nccl(limu_map *m, const double *points_dev, int64_t n, const double init_guess[7], double tau, double th, int max_iter,
                            double eps, double pose_out[7], limu_icp_stats *stats) {
    limu_ctx *c = m->ctx;
    limu_comm *cm = c->comm;
    const int rows = icp_partial_rows(c);
    LIMU_TRY(c->tmp4.reserve((size_t)std::max<int64_t>(n, 1) * 24, c->stream));
    LIMU_TRY(c->tmp5.reserve((size_t)rows * NS * 8 + 256, c->stream));
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(div_up(std::max<int64_t>(n, 1), ICP_BLOCK), rows));
    IcpArgs A;
    memset(&A, 0, sizeof A);
    A.map = m->view(); A.points = points_dev; A.work = c->tmp4.as<double>(); A.n_max = n;
    for (int k = 0; k < 7; ++k) A.init_pose[k] = init_guess[k];
    A.tau_sq = tau * tau; A.th = th; A.coop_scan = n >= 32768 ? 1 : 0; A.nranks = 1;
    A.icp_blocks = grid;   // k_icp_step strides its queries by icp_blocks * ICP_BLOCK (left at 0 this loop never ended: the "NCCL hang" of round 1)
    double *state = cm->d_state;
    double *h = static_cast<double *>(c->h_pinned) + 256;
    int64_t nv = 0;
    LIMU_TRY(limu_map_size(m, &nv, nullptr));
    if (nv == 0 || max_iter <= 0) { for (int k = 0; k < 7; ++k) pose_out[k] = init_guess[k]; if (stats) memset(stats, 0, sizeof *stats); return LIMU_OK; }
    int j = 0, done = 0;
    for (; j < max_iter && !done; ++j) {
        k_icp_step<<<grid, ICP_BLOCK, 0, c->stream>>>(A, state, j == 0 ? 1 : 0, c->tmp5.as<double>());
        LIMU_LAUNCHED();
        k_icp_fold_rows<<<1, 32, 0, c->stream>>>(c->tmp5.as<double>(), grid, state);
        LIMU_LAUNCHED();
        LIMU_TRY(comm_nccl_allreduce_sum_f64(c, state, NS));
        k_icp_solve_step<<<1, 32, 0, c->stream>>>(state, eps, j == 0 ? 1 : 0);
        LIMU_LAUNCHED();
        LIMU_CUDA_TRY(cudaMemcpyAsync(h, state, 48 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
        done = h[40] != 0.0;
    }
    const Pose out = mul(pose_load(h + 32), pose_load(init_guess));
    pose_store(out, pose_out);
    if (stats) { stats->iterations = j; stats->converged = done; stats->last_ncorr = (int64_t)h[16]; stats->mean_candidates = h[17]; stats->miss_fraction = h[18]; }
    return check_status(c);
}

}  // namespace limu

using namespace limu;

static int icp_common(limu_map *m, const double *points_dev, int64_t n, const double init_guess[7], double tau, double th, int max_iter, double eps,
                      double pose_out[7], limu_icp_stats *stats, double *est_trace, int64_t *ncorr_trace, double *hg_trace, bool sharded = false,
                      int icp_mode = 0) {
    limu_ctx *c = m->ctx;
    LIMU_TRY(c->tmp4.reserve((size_t)std::max<int64_t>(n, 1) * 24, c->stream));                 // working cloud
    LIMU_TRY(icp_partials_reserve(c, c->ll_rows, c->stream));
    const bool tr = est_trace || ncorr_trace || hg_trace;
    const size_t it = (size_t)std::max(max_iter, 1);
    if (tr) LIMU_TRY(c->tmp3.reserve(it * (7 + 1 + 42) * 8, c->stream));
    double *out13 = c->d_small.as<double>() + 16;
    double *d_est = tr ? c->tmp3.as<double>() : nullptr;
    long long *d_nc = tr ? reinterpret_cast<long long *>(d_est + it * 7) : nullptr;
    double *d_hg = tr ? d_est + it * 8 : nullptr;
    IcpArgs A;
    memset(&A, 0, sizeof A);
    A.points = points_dev; A.work = c->tmp4.as<double>(); A.n_max = n;
    for (int k = 0; k < 7; ++k) A.init_pose[k] = init_guess[k];
    A.tau_sq = tau * tau; A.th = th; A.max_iter = max_iter; A.eps = eps;
    A.partials = c->ll_rows.as<double>(); A.out = out13;
    A.est_trace = d_est; A.ncorr_trace = d_nc; A.hg_trace = d_hg;
    LIMU_TRY(icp_device(m, A, n, icp_mode, sharded && max_iter >= 0, nullptr));   // (a negative iteration count exchanges nothing)
    double *h = static_cast<double *>(c->h_pinned) + 16;
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, out13, 13 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    for (int k = 0; k < 7; ++k) pose_out[k] = h[k];
    const int iters = (int)h[7];
    if (stats) {   // in a sharded call the counters are global sums; the caller divides by the global query count
        stats->iterations = iters; stats->converged = (int)h[8]; stats->last_ncorr = (int64_t)h[9];
        stats->mean_candidates = sharded ? h[10] : (n > 0 ? h[10] / (double)n : 0.0);
        stats->miss_fraction = sharded ? h[11] : (n > 0 ? h[11] / (double)n : 0.0);
    }
    if (sharded && c->comm && c->comm->nranks > 1) {
        c->comm->stamp_base += (unsigned long long)iters;   // identical on every rank: all ranks solve the same equations
        int err = 0;
        LIMU_CUDA_TRY(cudaMemcpy(&err, c->comm->d_error, sizeof(int), cudaMemcpyDeviceToHost));
        if (err) { set_error("limu_icp_sharded: a peer rank did not reach the exchange within 2 s"); cudaMemset(c->comm->d_error, 0, sizeof(int)); return LIMU_ERR_COMM; }
    }
    if (tr && iters > 0) {
        if (est_trace) LIMU_CUDA_TRY(cudaMemcpyAsync(est_trace, d_est, (size_t)iters * 56, cudaMemcpyDeviceToHost, c->stream));
        if (ncorr_trace) LIMU_CUDA_TRY(cudaMemcpyAsync(ncorr_trace, d_nc, (size_t)iters * 8, cudaMemcpyDeviceToHost, c->stream));
        if (hg_trace) LIMU_CUDA_TRY(cudaMemcpyAsync(hg_trace, d_hg, (size_t)iters * 42 * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    return check_status(c);
}

// All k hypotheses of the latency shape in one cooperative launch; guesses: k x 7 doubles (device); res: k x MULTI_OUT doubles (host).
static int icp_multi_grouped(limu_map *m, int64_t n, const double *guesses, int k, double tau, double th, int max_iter, double eps, bool nn27, double *res) {
    limu_ctx *c = m->ctx;
    const int G = icp_multi_group_ctas(n);
    const void *fn = nn27 ? (const void *)k_icp_multi<true> : (const void *)k_icp_multi<false>;
    int per_sm = 0;
    LIMU_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, ICP_BLOCK, 0));
    // every CTA spins on the rows of its group, so the whole grid must be co-resident -- with GATE_SLACK_SMS SMs left for the k_gate threads
    // of a pipelined odometry handle that may sit on the GPU when this grid is placed (DESIGN section 4, "A launch that needs every SM")
    const int resident = std::min(std::max(per_sm, 1) * std::max(1, c->sm_count - GATE_SLACK_SMS), icp_partial_rows(c));
    const int groups = std::max(1, std::min(k, resident / G));
    LIMU_TRY(c->tmp4.reserve((size_t)groups * (size_t)std::max<int64_t>(n, 1) * 24, c->stream));   // one working cloud per running group
    LIMU_TRY(icp_partials_reserve(c, c->ll_rows, c->stream));
    LIMU_TRY(c->tmp3.reserve((size_t)k * MULTI_OUT * sizeof(double), c->stream));
    MultiArgs M;
    memset(&M, 0, sizeof M);
    IcpArgs &A = M.A;
    A.map = m->view(); A.map_counters = m->counters.as<unsigned long long>();
    A.points = c->in0.as<double>(); A.work = c->tmp4.as<double>(); A.n_max = n;
    A.tau_sq = tau * tau; A.th = th; A.max_iter = max_iter; A.eps = eps;
    A.partials = c->ll_rows.as<double>();
    A.ll_stamp_base = c->ll_seq;
    const unsigned int waves = (unsigned int)div_up(k, groups);   // a group makes at most max_iter + 1 exchanges per hypothesis (the last: its fitness)
    c->ll_seq = (c->ll_seq + waves * ((unsigned int)std::max(max_iter, 0) + 1u) + 2u) & 0x7FFFFFFFu;
    M.guesses = guesses; M.out = c->tmp3.as<double>(); M.k = k; M.group_ctas = G;
    void *args[] = {&M};
    LIMU_CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(groups * G), dim3(ICP_BLOCK), args, 0, c->stream));
    LIMU_LAUNCHED();
    LIMU_CUDA_TRY(cudaMemcpyAsync(res, M.out, (size_t)k * MULTI_OUT * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

// One hypothesis outside the latency shape: the loop kernel itself (its estimates traced), then the fitness of src_after.
static int icp_multi_single(limu_map *m, int64_t n, const double guess[7], double tau, double th, int max_iter, double eps, int icp_mode, double *res) {
    limu_ctx *c = m->ctx;
    std::vector<double> poses(7 * ((size_t)std::max(max_iter, 1) + 1));
    std::copy(guess, guess + 7, poses.begin());
    limu_icp_stats st;
    LIMU_TRY(icp_common(m, c->in0.as<double>(), n, guess, tau, th, max_iter, eps, res, &st, poses.data() + 7, nullptr, nullptr, false, icp_mode));
    const int grid = std::max(1, std::min(div_up(n, ICP_BLOCK), c->sm_count * 4));   // depends on n only: the fold order is the same for every guess
    LIMU_TRY(stage_in(c, c->tmp5, poses.data(), (size_t)(st.iterations + 1) * 7 * sizeof(double)));
    LIMU_TRY(c->tmp2.reserve((size_t)grid * 2 * sizeof(double), c->stream));
    if (icp_mode & LIMU_ICP_NN27)
        k_icp_fitness<true><<<grid, ICP_BLOCK, 0, c->stream>>>(m->view(), c->in0.as<double>(), n, c->tmp5.as<double>(), st.iterations + 1, tau * tau, c->tmp2.as<double>());
    else
        k_icp_fitness<false><<<grid, ICP_BLOCK, 0, c->stream>>>(m->view(), c->in0.as<double>(), n, c->tmp5.as<double>(), st.iterations + 1, tau * tau, c->tmp2.as<double>());
    LIMU_LAUNCHED();
    std::vector<double> rows((size_t)grid * 2);
    LIMU_CUDA_TRY(cudaMemcpyAsync(rows.data(), c->tmp2.p, rows.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LIMU_TRY(check_status(c));
    double inl = 0.0, d2 = 0.0;
    for (int b = 0; b < grid; ++b) { inl += rows[2 * b]; d2 += rows[2 * b + 1]; }
    res[7] = st.iterations; res[8] = st.converged; res[9] = inl; res[10] = d2;
    return LIMU_OK;
}

// limu_icp_multi on the scan in c->in0 from k guesses, given on the host and optionally already on the device (guesses_dev).
static int icp_multi_run(limu_map *m, int64_t n, const double *guesses, const double *guesses_dev, int k, double tau, double th, int max_iter,
                         double eps, int icp_mode, double *poses_out, limu_icp_hypothesis *out, int32_t *best) {
    limu_ctx *c = m->ctx;
    std::vector<double> res((size_t)k * MULTI_OUT);
    if (n <= 16384 && m->cap <= 64) {   // the latency shape, as icp_device would choose it for one hypothesis
        if (!guesses_dev) {
            LIMU_TRY(stage_in(c, c->tmp5, guesses, (size_t)k * 7 * sizeof(double)));
            guesses_dev = c->tmp5.as<double>();
        }
        LIMU_TRY(icp_multi_grouped(m, n, guesses_dev, k, tau, th, max_iter, eps, (icp_mode & LIMU_ICP_NN27) != 0, res.data()));
    } else {
        for (int h = 0; h < k; ++h)
            LIMU_TRY(icp_multi_single(m, n, guesses + 7 * (size_t)h, tau, th, max_iter, eps, icp_mode, res.data() + (size_t)h * MULTI_OUT));
    }
    for (int h = 0; h < k; ++h) {   // best: most inliers, then the smaller rms, then the lower index
        const double *r = res.data() + (size_t)h * MULTI_OUT;
        const int64_t inl = (int64_t)r[9];
        const double rms = inl > 0 ? sqrt(r[10] / (double)inl) : 0.0;
        std::copy(r, r + 7, poses_out + 7 * (size_t)h);
        if (out) { out[h].iterations = (int32_t)r[7]; out[h].converged = (int32_t)r[8]; out[h].inliers = inl; out[h].rms = rms; }
        if (best) {
            const double *b = *best >= 0 ? res.data() + (size_t)*best * MULTI_OUT : nullptr;
            const int64_t binl = b ? (int64_t)b[9] : -1;
            const double brms = b && binl > 0 ? sqrt(b[10] / (double)binl) : 0.0;
            if (!b || inl > binl || (inl == binl && rms < brms)) *best = h;
        }
    }
    return LIMU_OK;
}

// Scores k poses of `src` against the scan in c->in0: inliers into c->tmp0, rms into c->tmp1 (k each); hist: see k_score_poses.
static int score_poses_device(limu_map *m, int64_t n, const PoseSource &src, int64_t k, double tau, bool nn27, unsigned long long *hist) {
    limu_ctx *c = m->ctx;
    LIMU_TRY(c->tmp0.reserve((size_t)k * sizeof(int64_t), c->stream));
    LIMU_TRY(c->tmp1.reserve((size_t)k * sizeof(double), c->stream));
    const void *fn = nn27 ? (const void *)k_score_poses<true> : (const void *)k_score_poses<false>;
    int per_sm = 0;
    LIMU_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, SCORE_BLOCK, 0));
    const int64_t blocks = std::max<int64_t>(1, std::min<int64_t>((k + SCORE_BLOCK / 32 - 1) / (SCORE_BLOCK / 32), (int64_t)std::max(per_sm, 1) * c->sm_count));
    const MapView view = m->view();
    const double *points = c->in0.as<double>();
    const double tau_sq = tau * tau;
    int64_t *inl = c->tmp0.as<int64_t>();
    double *rms = c->tmp1.as<double>();
    void *args[] = {(void *)&view, (void *)&points, (void *)&n, (void *)&src, (void *)&k, (void *)&tau_sq, (void *)&inl, (void *)&rms, (void *)&hist};
    LIMU_CUDA_TRY(cudaLaunchKernel(fn, dim3((unsigned int)blocks), dim3(SCORE_BLOCK), args, 0, c->stream));
    LIMU_LAUNCHED();
    return LIMU_OK;
}

// Size of the allocation DevBuf::reserve would make for `want` bytes (0: none).
static size_t reserve_growth(const DevBuf &b, size_t want) {
    if (want <= b.bytes) return 0;
    size_t nb = b.bytes ? b.bytes : 256;
    while (nb < want) {
        if (nb > SIZE_MAX / 2) return SIZE_MAX;
        nb *= 2;
    }
    return nb;
}

// limu_relocalize's candidate scores for a grid of k candidates: LIMU_ERR_NOMEM when they do not fit the device.
static int reserve_scores(limu_ctx *c, int64_t k) {
    size_t fr = 0, total = 0;
    LIMU_CUDA_TRY(cudaMemGetInfo(&fr, &total));
    const bool fits = (uint64_t)k <= SIZE_MAX / 8 && [&] {
        const size_t a = reserve_growth(c->tmp0, (size_t)k * 8), b = reserve_growth(c->tmp1, (size_t)k * 8);
        // (reserve allocates before it frees: tmp0's new block, then tmp1's with tmp0's old block back)
        return a <= fr && b <= fr - a + (a ? c->tmp0.bytes : 0);
    }();
    if (!fits) { set_error("limu_relocalize: the scores of %lld candidates (16 bytes each) do not fit in device memory", (long long)k); return LIMU_ERR_NOMEM; }
    LIMU_TRY(c->tmp0.reserve((size_t)k * 8, c->stream));
    return c->tmp1.reserve((size_t)k * 8, c->stream);
}

extern "C" {

int limu_icp_multi(limu_map *m, const double *xyz, int64_t n, const double *init_guesses, int32_t k, double max_corresp_dist, double kernel,
                   int icp_max_iteration, double est_threshold, int32_t icp_mode, double *poses_out, limu_icp_hypothesis *out, int32_t *best) {
    LIMU_REQUIRE(m && n >= 0 && (n == 0 || xyz) && k >= 0 && (k == 0 || (init_guesses && poses_out)), "limu_icp_multi: bad arguments");
    LIMU_REQUIRE((icp_mode & ~(LIMU_ICP_NN27 | LIMU_ICP_PLANE)) == 0, "limu_icp_multi: unknown icp_mode bits");
    LIMU_REQUIRE(!(icp_mode & LIMU_ICP_PLANE), "limu_icp_multi: the point-to-plane variant is not available in the multi-hypothesis loop");
    if (best) *best = -1;
    if (k == 0) return LIMU_OK;
    LIMU_TRY(bind(m->ctx));
    LIMU_TRY(stage_in(m->ctx, m->ctx->in0, xyz, (size_t)n * 24));
    return icp_multi_run(m, n, init_guesses, nullptr, k, max_corresp_dist, kernel, icp_max_iteration, est_threshold, icp_mode, poses_out, out, best);
}

int limu_map_score_poses(limu_map *m, const double *xyz, int64_t n, const double *poses, int64_t k, double max_corresp_dist, int32_t icp_mode,
                         int64_t *inliers, double *rms) {
    LIMU_REQUIRE(m && n >= 0 && (n == 0 || xyz) && k >= 0 && (k == 0 || (poses && inliers && rms)), "limu_map_score_poses: bad arguments");
    LIMU_REQUIRE((icp_mode & ~(LIMU_ICP_NN27 | LIMU_ICP_PLANE)) == 0, "limu_map_score_poses: unknown icp_mode bits");
    LIMU_REQUIRE(!(icp_mode & LIMU_ICP_PLANE), "limu_map_score_poses: point-to-plane scoring is not available");
    if (k == 0) return LIMU_OK;
    limu_ctx *c = m->ctx;
    LIMU_TRY(bind(c));
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    LIMU_TRY(stage_in(c, c->tmp5, poses, (size_t)k * 7 * sizeof(double)));
    PoseSource src;
    memset(&src, 0, sizeof src);
    src.list = c->tmp5.as<double>();
    LIMU_TRY(score_poses_device(m, n, src, k, max_corresp_dist, (icp_mode & LIMU_ICP_NN27) != 0, nullptr));
    LIMU_CUDA_TRY(cudaMemcpyAsync(inliers, c->tmp0.p, (size_t)k * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaMemcpyAsync(rms, c->tmp1.p, (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    return check_status(c);
}

int limu_relocalize(limu_map *m, const double *xyz, int64_t n, const limu_reloc_grid *grid, int32_t n_refine, double max_corresp_dist, double kernel,
                    int icp_max_iteration, double est_threshold, int32_t icp_mode, limu_reloc_candidate *out, int32_t *n_out, int32_t *best) {
    LIMU_REQUIRE(m && grid && out && n >= 0 && (n == 0 || xyz), "limu_relocalize: bad arguments");
    LIMU_REQUIRE((icp_mode & ~(LIMU_ICP_NN27 | LIMU_ICP_PLANE)) == 0, "limu_relocalize: unknown icp_mode bits");
    LIMU_REQUIRE(!(icp_mode & LIMU_ICP_PLANE), "limu_relocalize: point-to-plane scoring is not available");
    LIMU_REQUIRE(n_refine >= 1 && n_refine <= 4096, "limu_relocalize: n_refine must be in 1 ... 4096");
    LIMU_REQUIRE(grid->nx >= 1 && grid->ny >= 1 && grid->nyaw >= 1, "limu_relocalize: every grid count must be >= 1");
    LIMU_REQUIRE(grid->step_xy > 0.0 && grid->step_yaw > 0.0, "limu_relocalize: the grid steps must be > 0");
    if (n_out) *n_out = 0;
    if (best) *best = -1;
    limu_ctx *c = m->ctx;
    LIMU_TRY(bind(c));
    const int64_t nxy = (int64_t)grid->nx * grid->ny;
    if (nxy > INT64_MAX / grid->nyaw) { set_error("limu_relocalize: the grid has more than 2^63 candidates"); return LIMU_ERR_NOMEM; }
    const int64_t K = nxy * grid->nyaw;
    const int M = (int)std::min<int64_t>(n_refine, K);
    LIMU_TRY(reserve_scores(c, K));
    LIMU_TRY(stage_in(c, c->in0, xyz, (size_t)n * 24));
    // out2: yaw table (2 nyaw doubles), then the selected indices in ranking order (M), then their coarse poses (7 M)
    std::vector<double> yaw(2 * (size_t)grid->nyaw);
    for (int l = 0; l < grid->nyaw; ++l) {
        const double t = ((double)l - 0.5 * (double)(grid->nyaw - 1)) * grid->step_yaw;
        yaw[2 * l] = sin(t / 2.0); yaw[2 * l + 1] = cos(t / 2.0);
    }
    LIMU_TRY(c->out2.reserve((yaw.size() + 8 * (size_t)M) * 8, c->stream));
    LIMU_CUDA_TRY(cudaMemcpyAsync(c->out2.p, yaw.data(), yaw.size() * 8, cudaMemcpyHostToDevice, c->stream));
    int64_t *d_index = reinterpret_cast<int64_t *>(c->out2.as<double>() + yaw.size());
    double *d_poses = c->out2.as<double>() + yaw.size() + M;
    PoseSource src;
    memset(&src, 0, sizeof src);
    std::copy(grid->center, grid->center + 7, src.center);
    src.yaw = c->out2.as<double>(); src.nx = grid->nx; src.ny = grid->ny; src.step_xy = grid->step_xy;
    // out0: inlier histogram (n + 1), digit histogram (256), gather counter; out1: the gathered records (3 M)
    LIMU_TRY(c->out0.reserve(((size_t)n + 1 + 256 + 1) * 8, c->stream));
    LIMU_TRY(c->out1.reserve((size_t)M * 3 * 8, c->stream));
    unsigned long long *hist = c->out0.as<unsigned long long>(), *hist256 = hist + n + 1, *count = hist256 + 256;
    LIMU_CUDA_TRY(cudaMemsetAsync(hist, 0, ((size_t)n + 1) * 8, c->stream));
    LIMU_TRY(score_poses_device(m, n, src, K, max_corresp_dist, (icp_mode & LIMU_ICP_NN27) != 0, hist));
    std::vector<unsigned long long> h((size_t)n + 1);
    LIMU_CUDA_TRY(cudaMemcpyAsync(h.data(), hist, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    LIMU_TRY(check_status(c));
    // the class of the M-th candidate, and how many of it are taken
    Sel S;
    memset(&S, 0, sizeof S);
    int64_t above = 0;
    for (S.T = n; above + (int64_t)h[S.T] < M; --S.T) above += (int64_t)h[S.T];
    uint64_t need = (uint64_t)(M - above);
    const int sel_blocks = (int)std::max<int64_t>(1, std::min<int64_t>((K + 255) / 256, (int64_t)c->sm_count * 8));
    if (need < h[S.T]) {
        unsigned long long hd[256];
        for (int digit = 0; digit < 16; ++digit) {
            const int shift = digit < 8 ? 56 - 8 * digit : 56 - 8 * (digit - 8);
            unsigned long long &mask = digit < 8 ? S.mh : S.ml, &prefix = digit < 8 ? S.ph : S.pl;
            if (digit >= 8 && ((uint64_t)(K - 1) >> shift) == 0) { mask |= 0xFFull << shift; continue; }   // an index byte that is 0 for every candidate
            LIMU_CUDA_TRY(cudaMemsetAsync(hist256, 0, 256 * 8, c->stream));
            k_select_digit<<<sel_blocks, 256, 0, c->stream>>>(c->tmp0.as<int64_t>(), c->tmp1.as<double>(), K, S, digit, hist256);
            LIMU_LAUNCHED();
            LIMU_CUDA_TRY(cudaMemcpyAsync(hd, hist256, sizeof hd, cudaMemcpyDeviceToHost, c->stream));
            LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
            int d = 0;
            while (hd[d] < need) need -= hd[d++];   // (d < 256: the candidates left hold at least `need`)
            mask |= 0xFFull << shift;
            prefix |= (unsigned long long)d << shift;
            if (hd[d] == need) break;   // every candidate of this byte value is taken
        }
    }
    LIMU_CUDA_TRY(cudaMemsetAsync(count, 0, 8, c->stream));
    k_select_gather<<<sel_blocks, 256, 0, c->stream>>>(c->tmp0.as<int64_t>(), c->tmp1.as<double>(), K, S, count, M, c->out1.as<long long>());
    LIMU_LAUNCHED();
    std::vector<long long> rec(3 * (size_t)M);
    unsigned long long got = 0;
    LIMU_CUDA_TRY(cudaMemcpyAsync(&got, count, 8, cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaMemcpyAsync(rec.data(), c->out1.p, rec.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (got != (unsigned long long)M) { set_error("limu_relocalize: selected %llu candidates instead of %d", got, M); return LIMU_ERR_CUDA; }
    std::vector<int> order(M);
    for (int i = 0; i < M; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) {   // inliers desc, rms asc (its bits order like the values), index asc
        const long long *x = &rec[3 * (size_t)a], *y = &rec[3 * (size_t)b];
        if (x[1] != y[1]) return x[1] > y[1];
        if (x[2] != y[2]) return (unsigned long long)x[2] < (unsigned long long)y[2];
        return x[0] < y[0];
    });
    std::vector<int64_t> index(M);
    for (int i = 0; i < M; ++i) index[i] = rec[3 * (size_t)order[i]];
    LIMU_CUDA_TRY(cudaMemcpyAsync(d_index, index.data(), (size_t)M * 8, cudaMemcpyHostToDevice, c->stream));
    k_grid_poses<<<div_up(M, 128), 128, 0, c->stream>>>(src, d_index, M, d_poses);
    LIMU_LAUNCHED();
    std::vector<double> coarse(7 * (size_t)M), refined(7 * (size_t)M);
    LIMU_CUDA_TRY(cudaMemcpyAsync(coarse.data(), d_poses, coarse.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    LIMU_TRY(check_status(c));
    std::vector<limu_icp_hypothesis> hyp(M);
    int32_t b = -1;
    LIMU_TRY(icp_multi_run(m, n, coarse.data(), d_poses, M, max_corresp_dist, kernel, icp_max_iteration, est_threshold, icp_mode, refined.data(), hyp.data(), &b));
    for (int i = 0; i < M; ++i) {
        const long long *r = &rec[3 * (size_t)order[i]];
        limu_reloc_candidate &o = out[i];
        o.index = r[0];
        std::copy(&coarse[7 * (size_t)i], &coarse[7 * (size_t)i] + 7, o.coarse_pose);
        o.coarse_inliers = r[1];
        memcpy(&o.coarse_rms, &r[2], 8);
        std::copy(&refined[7 * (size_t)i], &refined[7 * (size_t)i] + 7, o.pose);
        o.icp = hyp[i];
    }
    if (n_out) *n_out = M;
    if (best) *best = b;
    return LIMU_OK;
}

int limu_icp(limu_map *m, const double *xyz, int64_t n, const double init_guess[7], double max_corresp_dist, double kernel, int icp_max_iteration,
             double est_threshold, double pose_out[7], limu_icp_stats *stats, double *est_trace, int64_t *ncorr_trace, double *hg_trace) {
    LIMU_REQUIRE(m && init_guess && pose_out && n >= 0 && (n == 0 || xyz), "limu_icp: bad arguments");
    LIMU_TRY(bind(m->ctx));
    LIMU_TRY(stage_in(m->ctx, m->ctx->in0, xyz, (size_t)n * 24));
    return icp_common(m, m->ctx->in0.as<double>(), n, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, pose_out, stats,
                      est_trace, ncorr_trace, hg_trace);
}

int limu_icp_ex(limu_map *m, const double *xyz, int64_t n, const double init_guess[7], double max_corresp_dist, double kernel, int icp_max_iteration,
                double est_threshold, int32_t icp_mode, double pose_out[7], limu_icp_stats *stats, double *est_trace, int64_t *ncorr_trace, double *hg_trace) {
    LIMU_REQUIRE(m && init_guess && pose_out && n >= 0 && (n == 0 || xyz), "limu_icp_ex: bad arguments");
    LIMU_REQUIRE((icp_mode & ~(LIMU_ICP_NN27 | LIMU_ICP_PLANE)) == 0, "limu_icp_ex: unknown icp_mode bits");
    LIMU_TRY(bind(m->ctx));
    LIMU_TRY(stage_in(m->ctx, m->ctx->in0, xyz, (size_t)n * 24));
    return icp_common(m, m->ctx->in0.as<double>(), n, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, pose_out, stats,
                      est_trace, ncorr_trace, hg_trace, false, icp_mode);
}

int limu_icp_dev(limu_map *m, const double *xyz_dev, int64_t n, const double init_guess[7], double max_corresp_dist, double kernel,
                 int icp_max_iteration, double est_threshold, double pose_out[7], limu_icp_stats *stats) {
    LIMU_REQUIRE(m && init_guess && pose_out && n >= 0 && (n == 0 || xyz_dev), "limu_icp_dev: bad arguments");
    LIMU_TRY(bind(m->ctx));
    return icp_common(m, xyz_dev, n, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, pose_out, stats, nullptr, nullptr, nullptr);
}

int limu_icp_sharded_dev(limu_map *m, const double *xyz_dev, int64_t n_local, const double init_guess[7], double max_corresp_dist, double kernel,
                         int icp_max_iteration, double est_threshold, int mode, double pose_out[7], limu_icp_stats *stats) {
    LIMU_REQUIRE(m && init_guess && pose_out && n_local >= 0 && (n_local == 0 || xyz_dev), "limu_icp_sharded_dev: bad arguments");
    LIMU_TRY(bind(m->ctx));
    LIMU_REQUIRE(m->ctx->comm, "limu_icp_sharded_dev: call limu_comm_create / limu_comm_connect first");
    if (mode == LIMU_SHARD_NCCL) {
        LIMU_REQUIRE(m->ctx->comm->nccl_comm, "limu_icp_sharded_dev: NCCL baseline requested but limu_comm_nccl_init was not called");
        return icp_sharded_nccl(m, xyz_dev, n_local, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, pose_out, stats);
    }
    return icp_common(m, xyz_dev, n_local, init_guess, max_corresp_dist, kernel, icp_max_iteration, est_threshold, pose_out, stats, nullptr, nullptr, nullptr, true);
}

int limu_align(limu_ctx *c, const double *src, const double *tgt, int64_t n, double th, double H[36], double g[6], double x[6], double pose_out[7]) {
    LIMU_TRY(bind(c));
    LIMU_REQUIRE(n >= 0 && (n == 0 || (src && tgt)), "limu_align: bad arguments");
    LIMU_TRY(stage_in(c, c->in0, src, (size_t)n * 24));
    LIMU_TRY(stage_in(c, c->in1, tgt, (size_t)n * 24));
    const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(div_up(n, ICP_BLOCK), (int64_t)c->sm_count * 4));
    LIMU_TRY(c->tmp5.reserve((size_t)blocks * NS * 8 + 64 * 8, c->stream));
    double *partials = c->tmp5.as<double>();
    double *out = c->d_small.as<double>() + 128;
    k_align_partial<<<blocks, ICP_BLOCK, 0, c->stream>>>(c->in0.as<double>(), c->in1.as<double>(), n, th, partials);
    LIMU_LAUNCHED();
    k_align_solve<<<1, 32, 0, c->stream>>>(partials, blocks, out);
    LIMU_LAUNCHED();
    double *h = static_cast<double *>(c->h_pinned) + 128;
    LIMU_CUDA_TRY(cudaMemcpyAsync(h, out, 55 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LIMU_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (H) memcpy(H, h, 36 * 8);
    if (g) memcpy(g, h + 36, 6 * 8);
    if (x) memcpy(x, h + 42, 6 * 8);
    if (pose_out) memcpy(pose_out, h + 48, 7 * 8);
    return check_status(c);
}

}  // extern "C"
