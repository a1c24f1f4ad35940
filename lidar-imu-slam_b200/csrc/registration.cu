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
#include "iqr.cuh"
#include "voxel_map.cuh"

namespace limu {

constexpr int ICP_BLOCK = 256;
#ifndef LIMU_BW_CTAS
#define LIMU_BW_CTAS 2   // CTAs per SM of the bandwidth shape (register cap 65536 / (256 * LIMU_BW_CTAS)); measured 2 > 3 > 4 (profiles/r2f_*)
#endif
constexpr int NS = 20;   // 16 sums + ncorr + ncand + nmiss + pad
constexpr int NSP = 32;  // opt-in point-to-plane variant: 21 (upper triangle of H) + 6 (g) + ncorr + ncand + nmiss + 2 pad
constexpr int NS_MAX = 32;
constexpr int MBOX_MAX_RANKS = 8, MBOX_ROW = 24, MBOX_RING = 4;   // mailbox row: NS doubles + stamp + pad; ring of 4 exchange slots

}  // namespace limu
#include "frame_fusion.cuh"
LIMU_TRACE_RING(limu_debug_trace_reg)
namespace limu {

struct IcpArgs {
    MapView map;
    const unsigned long long *map_counters;   // [0] = live voxels (empty map -> return init_guess, registration.cpp:99-100)
    const double *points;       // n x 3, sensor frame (read only)
    double *work;               // n x 3, running source cloud
    int64_t n_max;
    const int *n_dev;
    double init_pose[7];        // init_guess, by value (no staging copy per call)
    double tau_sq;              // max_corresp_dist^2 (voxel_hash_map.cpp:112)
    double th;                  // kernel (registration.cpp:57-58)
    int max_iter;
    double eps;
    double *partials;           // [2][icp_blocks][NSX] (value, stamp) word pairs: the per-CTA rows of an iteration, self-validating (see ll_* below)
    unsigned int ll_stamp_base; // stamps of this launch are 0x80000000 | ((ll_stamp_base + iteration) & 0x7FFFFFFF): never 0, never reused soon
    unsigned int *barrier;      // zeroed before launch
    double *out;                // [0..6] pose, [7] iterations, [8] converged, [9] ncorr, [10] ncand, [11] nmiss, [12] n
    int grouped;                // 1: eight lanes per query (latency shape: a few thousand keypoints)
    int stage_doubles;          // > 0: the launch carries dynamic shared memory for the staged pass of the bandwidth shape
    int iqr_cap;                // latency shape: candidates the grid-wide IQR ranking can hold per CTA: IQR_GRID_MAX (static shared memory), or 8192 / 16384
                                // (the launch then carries iqr_cap * 10 bytes of dynamic shared memory: squared ranges + index list)
    int coop_scan;              // 1: sub-warp cooperative candidate scan (bandwidth shape); 0: one lane per query (latency shape)
    // point-sharded multi-GPU (SURVEY section 8e): every rank owns a contiguous shard of the queries and a full replica of
    // the map; per iteration the ranks exchange their NS-double row through peer-mapped mailboxes (NVLink stores).
    int nranks, rank;
    double *mbox_local;         // [MBOX_RING][MAX_RANKS][MBOX_ROW] in this rank's memory
    double *mbox_peer[8];       // the same buffer of every rank (peer mappings; [rank] == mbox_local)
    unsigned long long stamp_base;   // exchanges completed by earlier calls: iteration j of this call is exchange number stamp_base + j, its
                                     // stamp is that number + 1 and its ring slot that number mod MBOX_RING (contiguous ACROSS calls, so a rank
                                     // that is already in the next call can never overwrite a slot a slower peer is still reading)
    int *comm_error;            // set to 1 if a peer did not show up in time
    // ---- fused frame mode (odometry.cu): optional IQR prologue and local_map.update epilogue in the same launch ----
    const double *iqr_in;       // src0 (after the two downsampling stages); nullptr = no prologue
    const int *iqr_n;           // its count (device)
    double *iqr_d2;             // scratch, one double per point
    double *iqr_out;            // filtered keypoints (== points); count written to iqr_count
    int *iqr_count;
    const double *upd_down;     // downsampled scan (sensor frame); nullptr = no epilogue
    const int *upd_n;           // its count (device)
    double *upd_world;          // transformed copy
    unsigned int *upd_pslot;
    unsigned long long *upd_counters;   // map counters (writable)
    unsigned long long upd_birth_base;
    long long upd_capacity;     // C
    double upd_max_distance;
    DevStatus *status;
    unsigned int *exit_count;   // last CTA out resets the barrier words (no memset per launch)
    unsigned int *barrier_icp;  // barrier of the leading `icp_blocks` CTAs that run the Gauss-Newton loop
    int icp_blocks;
    double *twist_out;          // see FrameFusion
    double last_pose[7];
    unsigned int *loop_flag;    // non-null: set to loop_seq (release, GPU scope) once the pose of this launch is in memory and its reads of the map are over (what k_gate waits for)
    unsigned int loop_seq;
    double *host_res;           // non-null: pinned host memory; CTA 0 copies the handle's result block (res_block, res_doubles) there when the
    const double *res_block;    // launch is over and then stores loop_seq into word 31 (system scope): the host reads its pose without a copy
    int res_doubles;            // engine round trip in the stream, and the next kernel of the stream starts right behind this one
    double *est_trace;          // optional [max_iter][7]
    long long *ncorr_trace;     // optional [max_iter]
    double *hg_trace;           // optional [max_iter][42]
};

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
#define CT_MARK(k) do { if (blockIdx.x == 0 && lane == 0 && j == (((k) == 13 || (k) == 14) ? 3 : 2)) g_frame_marks[k] = (unsigned long long)clock64(); } while (0)
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
#define CT_MARK(k) do {} while (0)
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

// x = LDLT(H).solve(-g) from the 16 sums (registration.cpp:90), one thread. Kept out of line: its ~90 live registers would otherwise
// compete with the query pass of the cluster kernel for the 128 registers a 512-thread CTA allows.
static __device__ __noinline__ void solve_normal_equations(const double *S, double *x_out) {
    double H[36], g[6], x[6];
    expand_normal_equations(S, H, g);
#pragma unroll
    for (int k = 0; k < 6; ++k) g[k] = -g[k];
    ldlt6_solve(H, g, x);
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
            if (lane == 0) {
                if (SHAPE == 1 && !PLANE) {
                    solve_normal_equations(S, xs);                // out of line: the bandwidth build has no registers to spare
                } else {
                    double H[36], g[6], x[6];
                    if (PLANE) expand_plane_equations(S, H, g);
                    else expand_normal_equations(S, H, g);
#pragma unroll
                    for (int k = 0; k < 6; ++k) g[k] = -g[k];
                    if (PLANE) {
                        // point-to-plane: weak prior on the initial guess (oracle: lo_icp), x = LDLT(H + D).solve(-(g + D log(T_icp))) -- a map
                        // that offers only a handful of planar voxels does not determine six degrees of freedom, and the plain step runs away.
                        // (T_icp is this lane's own: it folded the previous estimate into it in the tail above.)
                        double xi[6];
                        se3_log(pose_load(Ticp), xi);
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            H[7 * k] += PLANE_PRIOR; H[7 * (k + 3)] += PLANE_PRIOR * PLANE_PRIOR_ARM2;
                            g[k] = -(S[21 + k] + PLANE_PRIOR * xi[k]);
                            g[k + 3] = -(S[24 + k] + (PLANE_PRIOR * PLANE_PRIOR_ARM2) * xi[k + 3]);
                        }
                    }
                    ldlt6_solve(H, g, x);                         // JTJ.ldlt().solve(-JTr) :90
#pragma unroll
                    for (int k = 0; k < 6; ++k) xs[k] = x[k];
                }
                CW_MARK(9, QW);
            }
            __syncwarp();
            // estimate = SE3::exp(x) (vector6d_to_mat4d :91): rotation half on lane 0, translation half on lane 1
            if (lane == 0) { double th_; se3_exp_rotation(xs, E, &th_); }
            if (lane == 1) se3_exp_translation(xs, E + 4);
            // Convergence, |log(estimate)| < eps (:124), from the twist itself: log(exp(x)) is x up to rounding (rotation below pi), so
            // unless |x| lies within 1e-6 eps of eps -- or the rotation is large -- the verdict is known NOW and the loop need not make
            // one more pass just to learn that it was over. Too close to call: the tail takes the logarithm, as the reference does.
            if (lane == 2) {
                const double nx = norm6(xs), nw = sqrt(xs[3] * xs[3] + xs[4] * xs[4] + xs[5] * xs[5]);
                verdict = !(nw < 3.0) ? 2 : (nx < A.eps * (1.0 - 1e-6) ? 1 : (nx > A.eps * (1.0 + 1e-6) ? 0 : 2));
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

int frame_update_device(limu_map *m, const FrameFusion &fuse, const double *pose_dev) {
    limu_ctx *c = m->ctx;
    IcpArgs A;
    memset(&A, 0, sizeof A);
    A.map = m->view();
    A.out = const_cast<double *>(pose_dev);
    A.barrier = fuse.barrier ? fuse.barrier + 4 : reinterpret_cast<unsigned int *>(c->d_small.as<double>() + 56);   // (its own words: another handle's loop may be running)
    A.exit_count = A.barrier + 1;
    A.upd_down = fuse.upd_down; A.upd_n = fuse.upd_n; A.upd_world = fuse.upd_world; A.upd_pslot = fuse.upd_pslot;
    A.upd_counters = m->counters.as<unsigned long long>(); A.upd_birth_base = fuse.upd_birth_base;
    A.status = fuse.status ? fuse.status : c->d_status;
    A.upd_capacity = (long long)m->capacity; A.upd_max_distance = m->max_distance;
    void *args[] = {&A};
    LIMU_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_frame_update, dim3(c->sm_count), dim3(ICP_BLOCK), args, 0, c->stream));
    LIMU_LAUNCHED();
    return LIMU_OK;
}

// ============================================================================================================================
// Cluster latency shape of the frame kernel (pipeline mode, the reference's registration rules): the Gauss-Newton loop of one scan
// runs on ONE 16-CTA thread-block cluster instead of ~72 CTAs that meet at a global-memory barrier.
//   * two lanes per query (pair_closest): 15 query warps x 16 pairs x 16 CTAs = 3 840 keypoints per pass, so a scan's ~2.4 k keypoints
//     are ONE pass and every query lives in the registers of its lane pair for the whole loop (no working cloud in memory);
//   * the common lookup is one L2 round trip (home slot + candidates requested together; the matched point comes back by shuffle);
//   * the 16 CTA rows are exchanged through distributed shared memory: each CTA stores its 20-double row into every CTA's shared
//     memory and a hardware cluster barrier (~0.2 us) replaces the global barrier + L2 fold (~3.5 us);
//   * warp 0 of every CTA is a solver warp without queries: it folds the rows, solves (redundantly, bit-identically in all 16 CTAs),
//     publishes the estimate, and finishes T_icp / log / the convergence test WHILE the query warps already run the next pass
//     (a pass made after the converging iteration is simply dropped);
//   * the IQR filter needs one grid barrier: the order statistics are ranked grid-wide, then every loop CTA derives bounds, flags and
//     the compacted index list in its own shared memory (CTA 0 also writes the keypoints out for the host).
// The other clusters of the grid only take part in the grid-wide phases (IQR ranking, map insert, eviction).
constexpr int CL_THREADS = 512, CL_SIZE = 16, CL_QWARPS = CL_THREADS / 32 - 1, CL_QPC = CL_QWARPS * 16, CL_QPP = CL_SIZE * CL_QPC;

struct ClusterSmem {
    double sd2[IQR_GRID_MAX];                 // squared ranges of the IQR candidates
    unsigned short qidx[IQR_GRID_MAX];        // source index of keypoint q (after the IQR filter)
    double red[CL_THREADS / 32][32];          // per-warp partial sums of one pass
    double rows[2][CL_SIZE][NS];              // the 16 CTA rows of an iteration (written by the peers through DSMEM), double-buffered
    double S[NS];
    double E[8], Tinit[8], Ticp[8], x[8];
    int ws[32];
    int total, done, pad0, pad1;
    IqrSmem iqr;                              // one-CTA select for candidate clouds beyond IQR_GRID_MAX
};

__device__ __forceinline__ unsigned int cluster_ctarank() { unsigned int r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned int cluster_nctarank() { unsigned int r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void dsmem_store_f64(const double *local_smem, unsigned int cta, double v) {
    const unsigned int la = (unsigned int)__cvta_generic_to_shared(local_smem);
    unsigned int ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(la), "r"(cta));
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(ra), "d"(v) : "memory");
}

template <int ROUNDS>   // candidate ranks per lane of a query pair: max_points_per_voxel <= 2 * ROUNDS
static __global__ void __launch_bounds__(CL_THREADS, 1) k_frame_cluster(const IcpArgs A) {
    extern __shared__ __align__(16) unsigned char cl_raw[];
    ClusterSmem &sm = *reinterpret_cast<ClusterSmem *>(cl_raw);
    GridSync gs{A.barrier, 0u, gridDim.x};
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, l2 = lane & 1;
    const unsigned int crank = cluster_ctarank();
    const bool loop_cta = blockIdx.x < CL_SIZE;   // cluster 0 (1-D cluster of CL_SIZE CTAs) runs the Gauss-Newton loop
    FT_MARK(0);
    // ---- KissICP::iqr_processing (icp.cpp:88-124, :133): exactly one grid barrier -------------------------------------------------
    const int n0 = __ldcg(A.iqr_n);
    const bool small = n0 <= IQR_GRID_MAX;     // uniform across the grid
    int n = 0;                                 // keypoints (known to the loop CTAs)
    bool compacted_here = false;               // the keypoints are IQR candidates sm.qidx[0 .. n)
    if (small && n0 > 1) {
        iqr_grid_select<CL_THREADS>(sm.sd2, A.iqr_in, n0, A.iqr_d2);
        gs.sync();
        if (loop_cta) { n = iqr_local_compact<CL_THREADS>(sm.ws, &sm.total, sm.sd2, n0, A.iqr_d2, sm.qidx); compacted_here = true; }
    } else if (small) {                        // 0 or 1 candidate: outlier::IQR keeps a single value (common.hpp:49-52)
        if (threadIdx.x == 0) {
            sm.qidx[0] = 0;
            if (blockIdx.x == 0) {
                if (n0 == 1) { A.iqr_out[0] = A.iqr_in[0]; A.iqr_out[1] = A.iqr_in[1]; A.iqr_out[2] = A.iqr_in[2]; }
                *A.iqr_count = n0;
            }
        }
        n = n0;
        gs.sync();
    } else {
        if (blockIdx.x == 0) iqr_block<CL_THREADS>(sm.iqr, A.iqr_in, n0, A.iqr_d2, A.iqr_out, A.iqr_count, nullptr);
        gs.sync();
        n = __ldcg(A.iqr_count);
    }
    FT_MARK(1);
    const bool run_icp = !(__ldcg(A.map_counters) == 0ull || A.max_iter <= 0);   // ICP :99-100: empty map -> init_guess
    if (threadIdx.x < 7) { sm.Tinit[threadIdx.x] = A.init_pose[threadIdx.x]; sm.Ticp[threadIdx.x] = threadIdx.x == 3 ? 1.0 : 0.0; }
    if (threadIdx.x < NS) sm.S[threadIdx.x] = 0.0;
    if (threadIdx.x == 0) sm.done = 0;
    __syncthreads();
    int j = 0, converged = 0;
    if (loop_cta && run_icp) {
        const bool single = small && n <= CL_QPP;            // one pass: the running source point stays in the pair's registers
        const int64_t pair0 = (int64_t)crank * CL_QPC + (int64_t)(warp - 1) * 16 + (lane >> 1);
        V3 s_reg{0.0, 0.0, 0.0};
        for (;;) {
            const bool no_more = j >= A.max_iter;             // only wait for the tail of iteration j-1
            if (warp > 0) {
                if (!no_more) {
                    CW_MARK(11, 1);
                    double acc = 0.0;                         // lane L: running total of sum index L>>1
                    int ncorr = 0, ncand = 0, nmiss = 0;
                    const volatile double *Pv = j == 0 ? sm.Tinit : sm.E;
                    for (int64_t base = 0; base < n; base += CL_QPP) {
                        const int64_t q = base + pair0;
                        const bool on = q < n;
                        V3 s{0.0, 0.0, 0.0};
                        if (on) {
                            const Pose P{Pv[0], Pv[1], Pv[2], Pv[3], Pv[4], Pv[5], Pv[6]};
                            V3 p;
                            if (j == 0) {   // source = init_guess * points (:102-103); the keypoints are the IQR inliers of src0
                                const size_t i = small ? (size_t)sm.qidx[q] : (size_t)q;
                                const double *src = small ? A.iqr_in : A.iqr_out;
                                p = V3{src[3 * i], src[3 * i + 1], src[3 * i + 2]};
                            } else if (single) {
                                p = s_reg;                    // source <- estimate * source (:119), applied at the next visit
                            } else {
                                p = V3{A.work[3 * q], A.work[3 * q + 1], A.work[3 * q + 2]};
                            }
                            s = apply(P, p);
                            if (single) s_reg = s;
                            else if (l2 == 0) { A.work[3 * q] = s.x; A.work[3 * q + 1] = s.y; A.work[3 * q + 2] = s.z; }
                        }
                        int count, own, my_rank;
                        double d2;
                        V3 tg;
                        pair_closest<ROUNDS>(A.map, s, l2, count, own, d2, tg, my_rank);
                        if (my_rank < 0) d2 = sqnorm3(tg.x - s.x, tg.y - s.y, tg.z - s.z);   // nothing found -> (0,0,0), range-tested like a real point
                        const bool lead = on && l2 == 0;
                        const bool gate = lead && d2 < A.tau_sq;
                        double c[16];
                        contribution(c, s, tg, d2, A.th, gate);
                        acc += warp_reduce_scatter16(c);
                        ncorr += gate ? 1 : 0;
                        ncand += lead ? count : 0;
                        nmiss += (lead && !own) ? 1 : 0;
                    }
                    CW_MARK(12, 1);
                    ncorr = __reduce_add_sync(0xFFFFFFFFu, ncorr);
                    ncand = __reduce_add_sync(0xFFFFFFFFu, ncand);
                    nmiss = __reduce_add_sync(0xFFFFFFFFu, nmiss);
                    sm.red[warp][lane] = (lane & 1) ? (lane == 1 ? (double)ncorr : lane == 3 ? (double)ncand : lane == 5 ? (double)nmiss : 0.0) : acc;
                }
            } else if (j > 0) {
                // tail of iteration j-1 on the solver warp, overlapped with pass j: T_icp = estimate * T_icp (:122) on lane 0,
                // |log(estimate)| < eps (:124) on lane 1
                CW_MARK(13, 0);
                const Pose est = pose_load(sm.E);
                if (lane == 0) pose_store(mul(est, pose_load(sm.Ticp)), sm.Ticp);
                if (lane == 1) {
                    double lg[6];
                    se3_log(est, lg);
                    sm.done = norm6(lg) < A.eps;
                }
                CW_MARK(14, 0);
            }
            __syncthreads();                                  // S1: partial sums of pass j and the verdict on iteration j-1
            if (j > 0 && sm.done) { converged = 1; break; }   // (the pass just made belongs to an iteration that does not exist)
            if (no_more) break;
            CT_MARK(6);
            const int par = j & 1;
            if (warp == 0 && lane < NS) {
                // CTA row (fixed order over the query warps), stored into every CTA of the cluster
                const int src_lane = lane < 16 ? 2 * lane : 2 * (lane - 16) + 1;
                double v = 0.0;
#pragma unroll
                for (int w = 1; w <= CL_QWARPS; ++w) v += sm.red[w][src_lane];
#pragma unroll
                for (unsigned int r = 0; r < (unsigned int)CL_SIZE; ++r) dsmem_store_f64(&sm.rows[par][crank][lane], r, v);
            }
            cluster_arrive_release();
            cluster_wait_acquire();
            CT_MARK(7);
            if (warp == 0) {
                if (lane < NS) {
                    double v = 0.0;
#pragma unroll
                    for (int r = 0; r < CL_SIZE; ++r) v += sm.rows[par][r][lane];
                    sm.S[lane] = v;
                }
                __syncwarp();
                CT_MARK(8);
                if (lane == 0) solve_normal_equations(sm.S, sm.x);   // JTJ.ldlt().solve(-JTr) :90
                __syncwarp();
                CT_MARK(9);
                // estimate = SE3::exp(x) (vector6d_to_mat4d :91): rotation half on lane 0, translation half on lane 1
                if (lane == 0) { double th_; se3_exp_rotation(sm.x, sm.E, &th_); }
                if (lane == 1) se3_exp_translation(sm.x, sm.E + 4);
                __syncwarp();
                CT_MARK(10);
            }
            __syncthreads();                                  // S2: the estimate is visible to the query warps
            ++j;
        }
    }
    FT_MARK(2);
    if (blockIdx.x == 0 && compacted_here) iqr_write_out<CL_THREADS>(sm.qidx, A.iqr_in, n, A.iqr_out, A.iqr_count, (int)threadIdx.x);   // keypoints for the host
    // new_pose = T_icp * init_guess (:129); with an empty map the loop did not run and this is init_guess itself (:99-100)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const Pose np = run_icp ? mul(pose_load(sm.Ticp), pose_load(sm.Tinit)) : pose_load(sm.Tinit);
        pose_store(np, A.out);
        A.out[7] = (double)j; A.out[8] = (double)converged; A.out[9] = sm.S[16]; A.out[10] = sm.S[17]; A.out[11] = sm.S[18]; A.out[12] = (double)n;
    }
    if (A.upd_down) frame_update_epilogue<CL_THREADS>(A, gs, sm.E);
    FT_MARK(5);
    // no CTA of a cluster may exit while a peer can still store into its shared memory: the last DSMEM store precedes the last cluster
    // barrier of the loop, and every loop CTA passes the grid barriers above after it. The last CTA out re-arms the grid barrier.
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(A.exit_count, 1u) == gridDim.x - 1) { *A.barrier = 0u; *A.barrier_icp = 0u; *A.exit_count = 0u; __threadfence(); }
    }
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

// ---- launch of the cluster latency shape -----------------------------------------------------------------------------------------
// Per device: 0 = not probed yet, -1 = unavailable (the classic kernel is used), > 0 = clusters of CL_SIZE CTAs that can be co-resident.
static int g_cluster_state[64] = {};
static int g_cluster_coop[64] = {};   // 1: launched with the cooperative attribute as well
static int launch_frame_cluster(limu_ctx *c, IcpArgs &A, int cap) {
    const int dev = c->device & 63;
    if (g_cluster_state[dev] < 0) return LIMU_ERR_CUDA;
    const void *fn = cap <= 10 ? (const void *)k_frame_cluster<5> : (const void *)k_frame_cluster<10>;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.blockDim = dim3(CL_THREADS);
    cfg.dynamicSmemBytes = sizeof(ClusterSmem);
    cfg.stream = c->stream;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL_SIZE; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeCooperative;
    at[1].val.cooperative = 1;
    cfg.attrs = at;
    if (g_cluster_state[dev] == 0) {
        g_cluster_state[dev] = -1;
        const void *both[2] = {(const void *)k_frame_cluster<5>, (const void *)k_frame_cluster<10>};
        for (const void *f : both) {
            if (cudaFuncSetAttribute(f, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess ||
                cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ClusterSmem)) != cudaSuccess) { (void)cudaGetLastError(); return LIMU_ERR_CUDA; }
        }
        int ncl = 0;
        cfg.gridDim = dim3(CL_SIZE * 8);
        cfg.numAttrs = 1;
        if (cudaOccupancyMaxActiveClusters(&ncl, fn, &cfg) != cudaSuccess || ncl < 1) { (void)cudaGetLastError(); return LIMU_ERR_CUDA; }
        g_cluster_state[dev] = std::min(ncl, 8);
        g_cluster_coop[dev] = 1;
    }
    cfg.gridDim = dim3(CL_SIZE * g_cluster_state[dev]);
    void *args[] = {&A};
    cfg.numAttrs = g_cluster_coop[dev] ? 2 : 1;
    cudaError_t e = cudaLaunchKernelExC(&cfg, fn, args);
    if (e != cudaSuccess && g_cluster_coop[dev]) {   // cooperative + cluster refused: the grid fits by construction (cudaOccupancyMaxActiveClusters), launch it plainly
        (void)cudaGetLastError();
        g_cluster_coop[dev] = 0;
        cfg.numAttrs = 1;
        e = cudaLaunchKernelExC(&cfg, fn, args);
    }
    if (e != cudaSuccess) { (void)cudaGetLastError(); g_cluster_state[dev] = -1; return LIMU_ERR_CUDA; }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return LIMU_OK;
}

static int g_icp_blocks_per_sm = 0;

// Enqueue the persistent ICP kernel. All pointers are device memory; `out13` receives pose + stats.
int icp_device(limu_map *m, const double *points_dev, double *work_dev, int64_t n_max, const int *n_dev, const double *init_pose_host,
               double tau, double th, int max_iter, double eps, double *partials_dev, size_t partial_rows, double *out13_dev, int64_t n_hint,
               double *est_trace_dev, long long *ncorr_trace_dev, double *hg_trace_dev, int max_iter_all_ranks, const FrameFusion *fuse, int icp_mode) {
    limu_ctx *c = m->ctx;
    const bool nn27 = (icp_mode & LIMU_ICP_NN27) != 0, plane = (icp_mode & LIMU_ICP_PLANE) != 0;
    const bool grouped = n_hint <= 16384 && m->cap <= 64;   // latency shape: eight lanes per query, one CTA per SM
    // bandwidth shape with the reference's rules: voxel blocks are staged through dynamic shared memory (two buffers of eight blocks per query warp)
    size_t stage_bytes = (!grouped && !nn27 && !plane && block_stride(m->cap) <= STAGE_MAX_STRIDE) ? (size_t)(ICP_BLOCK / 32 - 1) * STAGE_WARP_DOUBLES * sizeof(double) : 0;
    // latency shape with the IQR filter in front: the candidates (a few per cent more than the keypoints the hint counts) are ranked by the whole
    // grid out of a copy in every CTA's shared memory -- static up to IQR_GRID_MAX of them, dynamic (8192 or 16384) when the hint announces more
    int iqr_cap = IQR_GRID_MAX;
    if (grouped && fuse && fuse->iqr_in && n_hint + n_hint / 8 + 64 > IQR_GRID_MAX) {
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
    const int sms = (fuse && fuse->loop_flag) ? std::max(1, c->sm_count - GATE_SLACK_SMS) : c->sm_count;
    int grid = (int)std::min<int64_t>(want, (int64_t)sms * (grouped ? 1 : std::min(g_icp_blocks_per_sm, LIMU_BW_CTAS)));
    grid = (int)std::min<int64_t>(grid, (int64_t)partial_rows);
    const int icp_blocks = grid;   // the Gauss-Newton loop is latency bound at keypoint counts: it runs on the leading CTAs only
    if (fuse && fuse->upd_down) grid = std::max(grid, c->sm_count);   // the insert and the eviction sweep want one CTA per SM
    IcpArgs A;
    memset(&A, 0, sizeof A);
    A.map = m->view();
    A.map_counters = m->counters.as<unsigned long long>();
    A.points = points_dev; A.work = work_dev; A.n_max = n_max; A.n_dev = n_dev;
    for (int k = 0; k < 7; ++k) A.init_pose[k] = init_pose_host[k];
    A.tau_sq = tau * tau; A.th = th; A.max_iter = max_iter; A.eps = eps;
    A.partials = partials_dev; A.out = out13_dev;
    A.ll_stamp_base = c->ll_seq;
    c->ll_seq = (c->ll_seq + (unsigned int)std::max(max_iter, 0) + 2u) & 0x7FFFFFFFu;
    // grid barrier + exit counter live in the context's zero-initialised small area; the last CTA out re-arms them
    A.barrier = (fuse && fuse->barrier) ? fuse->barrier : reinterpret_cast<unsigned int *>(c->d_small.as<double>() + 56);
    A.exit_count = A.barrier + 1;
    A.barrier_icp = A.barrier + 2;
    A.icp_blocks = icp_blocks;
    A.est_trace = est_trace_dev; A.ncorr_trace = ncorr_trace_dev; A.hg_trace = hg_trace_dev;
    A.coop_scan = n_hint >= 32768 ? 1 : 0;
    A.grouped = grouped ? 1 : 0;
    A.stage_doubles = grouped ? 0 : (int)(stage_bytes / sizeof(double));
    A.iqr_cap = iqr_cap;
    A.nranks = 1; A.rank = 0;
    A.status = c->d_status;
    if (max_iter_all_ranks >= 0 && c->comm && c->comm->nranks > 1) {   // point-sharded call: fused peer exchange
        limu_comm *cm = c->comm;
        A.nranks = cm->nranks; A.rank = cm->rank; A.mbox_local = cm->mbox_local; A.comm_error = cm->d_error;
        for (int r = 0; r < cm->nranks; ++r) A.mbox_peer[r] = cm->mbox_peer[r];
        A.stamp_base = cm->stamp_base;   // advanced by the iterations this call executes once they are known (icp_common)
    }
    if (fuse) {
        A.iqr_in = fuse->iqr_in; A.iqr_n = fuse->iqr_n; A.iqr_d2 = fuse->iqr_d2; A.iqr_out = fuse->iqr_out; A.iqr_count = fuse->iqr_count;
        A.upd_down = fuse->upd_down; A.upd_n = fuse->upd_n; A.upd_world = fuse->upd_world; A.upd_pslot = fuse->upd_pslot;
        A.upd_counters = m->counters.as<unsigned long long>(); A.upd_birth_base = fuse->upd_birth_base;
        if (fuse->status) A.status = fuse->status;
        A.upd_capacity = (long long)m->capacity; A.upd_max_distance = m->max_distance;
        A.twist_out = fuse->twist_out;
        A.loop_flag = fuse->loop_flag; A.loop_seq = fuse->loop_seq;
        A.host_res = fuse->host_res; A.res_block = fuse->res_block; A.res_doubles = fuse->res_doubles;
        for (int k = 0; k < 7; ++k) A.last_pose[k] = fuse->last_pose[k];
    }
    void *args[] = {&A};
    cudaStream_t stream = (fuse && fuse->stream) ? fuse->stream : c->stream;
    if (c->profiling) { LIMU_CUDA_TRY(cudaEventRecord(c->ev[LIMU_STAGE_ICP][0], stream)); c->ev_used[LIMU_STAGE_ICP] = true; }
    // pipeline mode with the reference's rules: the cluster latency shape (falls back to the classic kernel where clusters of 16 cannot be launched)
    if (fuse && fuse->iqr_in && fuse->upd_down && icp_mode == 0 && A.nranks == 1 && !est_trace_dev && !ncorr_trace_dev && !hg_trace_dev && m->cap <= 20 &&
        n_hint <= CL_QPP && fuse->allow_cluster && launch_frame_cluster(c, A, m->cap) == LIMU_OK) {
        LIMU_TRY(prof_end(c, LIMU_STAGE_ICP));
        return LIMU_OK;
    }
    if (plane && max_iter_all_ranks >= 0 && c->comm && c->comm->nranks > 1) { set_error("the point-to-plane variant is not available in the point-sharded loop"); return LIMU_ERR_INVALID; }
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

int icp_partial_rows(limu_ctx *c) { return c->sm_count * 4; }   // >= the largest grid of any shape

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
    const int rows = icp_partial_rows(c);
    LIMU_TRY(c->tmp4.reserve((size_t)std::max<int64_t>(n, 1) * 24, c->stream));                 // working cloud
    {   // partial rows: (value, stamp) word pairs; a fresh allocation must not hold anything that looks like a stamp
        const void *before = c->ll_rows.p;
        LIMU_TRY(c->ll_rows.reserve((size_t)2 * rows * NS_MAX * 16 + 256, c->stream));
        if (c->ll_rows.p != before) LIMU_CUDA_TRY(cudaMemsetAsync(c->ll_rows.p, 0, c->ll_rows.bytes, c->stream));
    }
    const bool tr = est_trace || ncorr_trace || hg_trace;
    const size_t it = (size_t)std::max(max_iter, 1);
    if (tr) LIMU_TRY(c->tmp3.reserve(it * (7 + 1 + 42) * 8, c->stream));
    double *partials = c->ll_rows.as<double>();
    double *out13 = c->d_small.as<double>() + 16;
    double *d_est = tr ? c->tmp3.as<double>() : nullptr;
    long long *d_nc = tr ? reinterpret_cast<long long *>(d_est + it * 7) : nullptr;
    double *d_hg = tr ? d_est + it * 8 : nullptr;
    LIMU_TRY(icp_device(m, points_dev, c->tmp4.as<double>(), n, nullptr, init_guess, tau, th, max_iter, eps, partials, (size_t)rows, out13, n,
                        d_est, d_nc, d_hg, sharded ? max_iter : -1, nullptr, icp_mode));
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

extern "C" {

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
