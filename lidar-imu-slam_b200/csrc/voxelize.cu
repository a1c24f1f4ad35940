// voxelize.cu -- KissICP::deskew_scan + KissICP::voxelize's two downsampling stages as ONE persistent cooperative
// kernel (L/src/sensors/lidar/icp.cpp:36-47, :9-30, :126-131; helpers/deskew.cpp:10-28).
//
// The stand-alone stages (ops.cu) cost 13 launches + 2 memsets per scan, each a few microseconds of work on 128k points;
// here the phases are separated by grid barriers instead of kernel boundaries:
//   P1 deskew/widen -> frame[], stage-1 claim
//   P2 stage-1 winner flags, per-tile counts, ordered scatter of the winners -> down[], stage-2 claim
//   P3 (un-claim the stage-1 table) stage-2 winner flags, per-tile counts, ordered scatter -> src0[]
// Inside P2 / P3 a tile does not wait at a grid barrier for the counts of the tiles before it: every count is published as ONE 8-byte word
// {launch epoch | count}, and a tile simply re-reads the words of its predecessors until they carry this launch's epoch (tiles are handed
// out in increasing order and all CTAs are co-resident, so every predecessor is finished or in progress). Two grid barriers per scan, not four.
// The scan-local hash tables are left CLEAN instead of being cleared at the start (6 MB of stores and a grid barrier per scan): every
// claimed slot is remembered per point, so the stage-1 table is un-claimed in P4 (nobody reads it after P3) and the stage-2 table of
// this launch is un-claimed by the NEXT launch, which works on the other of two stage-2 tables.
// "First point per voxel wins, output in first-occurrence order" (icp.cpp:13-27 + the oracle's ordered map) becomes:
// atomicMin of the input index per voxel, then a stable compaction over VX_BLOCK-point tiles.
#include <stdlib.h>

#include <algorithm>

#include "compact.cuh"
#include "grid_sync.cuh"
#include "ops.cuh"
#include "voxel_map.cuh"

LIMU_TRACE_RING(limu_debug_trace_vox)

namespace limu {

#ifndef LIMU_VX_BLOCK
#define LIMU_VX_BLOCK 1024   // one fat CTA per SM: a grid barrier is paid per ARRIVING CTA (atomics on one word serialise at ~4 ns each: 592 CTAs of 256 -> 148 of 1024)
#endif
constexpr int VX_BLOCK = LIMU_VX_BLOCK;
// The pipelined odometry path (odometry.cu) runs the NEXT scan's launch beside the current scan's map update: 1024 threads x 64 registers
// are a whole register file, so that launch uses half-size CTAs (one per SM) and leaves room for the update kernel's CTA.
constexpr int VX_BLOCK_BESIDE = 512;
constexpr int VX_TILE = 1024;            // points per tile in both shapes (1024 x 1 and 512 x 2)
static_assert(VX_BLOCK == VX_TILE, "the full-size launch handles one point per thread");

struct VoxelizeArgs {
    const void *raw;            // mode 0: float4 {x,y,z,t}; mode 1: records `stride` bytes apart + ts; mode 2: double xyz (already a frame)
    const double *ts;
    int mode, stride, deskew;
    double twist[6];            // by value, read when deskew != 0
    const double *twist_dev;    // non-null: the twist is left in device memory by the previous scan's loop kernel
    int64_t n;
    double vs1, vs2;            // 0.5 v and 1.5 v (icp.cpp:129-130)
    double *frame, *down, *src0;
    unsigned long long *keys1, *keys2;
    unsigned int *min1, *min2, *pslot1, *pslot2;
    unsigned long long *keys2_prev;   // the stage-2 table (and claimed slots) of the previous launch: un-claimed here
    unsigned int *min2_prev, *pslot2_prev;
    int *nd_prev, *nd_this;           // how many stage-2 claims the previous launch made / this launch makes
    unsigned int mask1, mask2;
    int shift1, shift2;
    unsigned long long *tile1, *tile2;   // per-tile survivor counts of the two stages: {epoch << 32 | count}
    unsigned int epoch;                  // of this launch (never 0; the words are zero after a reset)
    int *counts;                // [0] n_down, [1] n_src0
    unsigned int *barrier;      // [0] grid barrier, [1] exit counter; zero at rest (the last CTA out re-arms them, no memset per launch)
    DevStatus *st;
    DevStatus *st_next;         // non-null: the status word of the NEXT launch of this pipeline (two words alternate); zeroed late in this launch
};

// Claim the voxel of p in a scan-local table and note `index` as a candidate for its first point (atomicMin). Split in two so that a thread
// with several points has all their first probes in flight together: claim_issue sends ONE compare-and-swap per point (it both finds and
// claims: the slot is the voxel's if it was empty or already held the key), claim_finish looks at the answer and walks on in the rare case
// of a collision.
struct Claim {
    unsigned long long key, cur;
    unsigned int s;
    bool valid;
};
__device__ __forceinline__ Claim claim_issue(unsigned long long *keys, int shift, const V3 &p, double vs, bool active, DevStatus *st) {
    Claim c;
    c.valid = false; c.key = KEY_EMPTY; c.cur = KEY_EMPTY; c.s = 0u;
    if (active) {
        const int kx = vox_index(p.x, vs), ky = vox_index(p.y, vs), kz = vox_index(p.z, vs);
        // NaN: the reference's (int) cast gives INT_MIN on x86-64 (cvttsd2si), and so does vox_index: far outside the packed range
        if (!key_in_range(kx, ky, kz)) st->key_range = 1;
        else {
            c.valid = true;
            c.key = pack_key(kx, ky, kz);
            c.s = slot_of(c.key, shift);
            c.cur = atomicCAS(&keys[c.s], KEY_EMPTY, c.key);
        }
    }
    return c;
}
__device__ __forceinline__ unsigned int claim_finish(const Claim &c, unsigned long long *keys, unsigned int *minidx, unsigned int mask, unsigned int index, DevStatus *st) {
    if (!c.valid) return PEND_NONE;
    unsigned int s = c.s;
    unsigned long long cur = c.cur;
    for (unsigned int probes = 0; probes <= mask; ++probes) {
        if (cur == KEY_EMPTY || cur == c.key) { atomicMin(&minidx[s], index); return s; }
        s = (s + 1) & mask;
        cur = atomicCAS(&keys[s], KEY_EMPTY, c.key);
    }
    st->table_full = 1;
    return PEND_NONE;
}

// exclusive prefix of small per-thread counts over the CTA (thread order); *total = their sum
__device__ __forceinline__ int block_exclusive_scan_count(int c, int *total, int *warp_sums /* 32 ints shared */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        const int v = lane < nw ? warp_sums[lane] : 0;
        int wi = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, wi, o); if (lane >= o) wi += t; }
        warp_sums[lane] = wi - v;
        if (lane == 31) *total = wi;
    }
    __syncthreads();
    return warp_sums[warp] + incl - c;
}

// exclusive prefix of tile counts: sum of counts[0..tile) computed by the whole CTA; a word is re-read until it is this launch's
template <int BLOCK>
__device__ __forceinline__ int tile_base(const unsigned long long *words, int tile, unsigned int epoch, int *ws /* 32 ints */) {
    int part = 0;
    for (int b = threadIdx.x; b < tile; b += BLOCK) {
        unsigned long long w;
        do {
            asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(words + b) : "memory");
        } while ((unsigned int)(w >> 32) != epoch);
        part += (int)(unsigned int)w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xFFFFFFFFu, part, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = part;
    __syncthreads();
    int v = 0;
#pragma unroll
    for (int w = 0; w < BLOCK / 32; ++w) v += ws[w];
    __syncthreads();
    return v;
}
__device__ __forceinline__ void tile_publish(unsigned long long *word, unsigned int epoch, int count) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(word), "l"(((unsigned long long)epoch << 32) | (unsigned int)count) : "memory");
}

#ifdef LIMU_ICP_PHASE_TIMING
__device__ unsigned long long g_vox_marks[8];   // globaltimer of thread 0 of CTA 0: start, after each of the two grid barriers, end
#define VX_MARK(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long _t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t)); g_vox_marks[k] = _t; } } while (0)
#else
#define VX_MARK(k) do {} while (0)
#endif

// BLOCK threads handle tiles of VX_TILE = BLOCK * ITEMS consecutive points, ITEMS per thread: the full-size launch is 1024 x 1, the launch
// that runs beside the map update 512 x 2 -- half the registers per SM, the same tiles, and a thread's two claims in flight together.
template <int BLOCK, int ITEMS>
__device__ __forceinline__ void voxelize_body(const VoxelizeArgs &A) {
    constexpr int TILE = BLOCK * ITEMS;
    __shared__ int ws[32];
    __shared__ int total;
    GridSync gs{A.barrier, 0u, gridDim.x};
    const int64_t n = A.n;
    const int64_t gtid = (int64_t)blockIdx.x * BLOCK + threadIdx.x, gthreads = (int64_t)gridDim.x * BLOCK;
    const int ntiles = (int)((n + TILE - 1) / TILE);
    VX_MARK(0);
    LIMU_TRACE(10);
    // un-claim what the previous launch left in ITS stage-2 table (this launch uses the other one): no barrier needed
    {
        const int ndp = __ldcg(A.nd_prev);
        for (int64_t j = gtid; j < ndp; j += gthreads) {
            const unsigned int sl = __ldcg(A.pslot2_prev + j);
            if (sl != PEND_NONE) { A.keys2_prev[sl] = KEY_EMPTY; A.min2_prev[sl] = PEND_NONE; }
        }
    }
    // P1: frame[i] = deskewed / widened point (icp.cpp:36-47, deskew.cpp:18-26); stage-1 claim at 0.5 v
    {
        double tw[6];
        if (A.deskew) {
#pragma unroll
            for (int k = 0; k < 6; ++k) tw[k] = A.twist[k];
            if (A.twist_dev) {
#pragma unroll
                for (int k = 0; k < 6; ++k) tw[k] = __ldcg(A.twist_dev + k);
            }
        }
        for (int64_t i0 = gtid; i0 < n; i0 += (int64_t)ITEMS * gthreads) {
            V3 p[ITEMS];
            Claim c[ITEMS];
#pragma unroll
            for (int u = 0; u < ITEMS; ++u) {
                const int64_t i = i0 + (int64_t)u * gthreads;
                const bool on = i < n;
                double t = 0.0;
                p[u] = V3{0.0, 0.0, 0.0};
                if (on) {
                    if (A.mode == 0) {
                        const float4 q = __ldg(reinterpret_cast<const float4 *>(A.raw) + i);
                        p[u] = V3{(double)q.x, (double)q.y, (double)q.z};
                        t = (double)q.w;
                    } else if (A.mode == 1) {
                        const float *q = reinterpret_cast<const float *>(static_cast<const unsigned char *>(A.raw) + (size_t)i * A.stride);
                        p[u] = V3{(double)q[0], (double)q[1], (double)q[2]};
                        if (A.deskew) t = A.ts[i];
                    } else {
                        const double *q = static_cast<const double *>(A.raw) + 3 * i;
                        p[u] = V3{q[0], q[1], q[2]};
                    }
                    if (A.deskew) {
                        const double s = t - 0.5;   // mid_pose_timestamp, deskew.hpp:12
                        double st[6];
#pragma unroll
                        for (int k = 0; k < 6; ++k) st[k] = s * tw[k];
                        p[u] = apply(se3_exp(st), p[u]);
                    }
                    A.frame[3 * i] = p[u].x; A.frame[3 * i + 1] = p[u].y; A.frame[3 * i + 2] = p[u].z;
                }
                c[u] = claim_issue(A.keys1, A.shift1, p[u], A.vs1, on, A.st);
            }
#pragma unroll
            for (int u = 0; u < ITEMS; ++u) {
                const int64_t i = i0 + (int64_t)u * gthreads;
                if (i < n) A.pslot1[i] = claim_finish(c[u], A.keys1, A.min1, A.mask1, (unsigned int)i, A.st);
            }
        }
    }
    gs.sync();
    VX_MARK(1);
    LIMU_TRACE(11);
    // P2: a point survives stage 1 iff it holds its voxel's smallest input index. Per tile: flags, count (published), ordered scatter
    // -> down[]; each winner immediately claims its 1.5 v voxel with its OUTPUT index. A thread owns ITEMS consecutive points of the tile.
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t e0 = (int64_t)tile * TILE + (int64_t)threadIdx.x * ITEMS;
        int f[ITEMS], cnt = 0;
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
            const int64_t i = e0 + u;
            f[u] = 0;
            if (i < n) { const unsigned int s = A.pslot1[i]; f[u] = s != PEND_NONE && __ldcg(A.min1 + s) == (unsigned int)i; }
            cnt += f[u];
        }
        const int r = block_exclusive_scan_count(cnt, &total, ws);
        if (threadIdx.x == 0) tile_publish(A.tile1 + tile, A.epoch, total);
        const int base = tile_base<BLOCK>(A.tile1, tile, A.epoch, ws);
        V3 p[ITEMS];
        Claim c[ITEMS];
        int j = base + r;
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
            const int64_t i = e0 + u;
            p[u] = V3{0.0, 0.0, 0.0};
            if (f[u]) {
                p[u] = V3{A.frame[3 * i], A.frame[3 * i + 1], A.frame[3 * i + 2]};
                A.down[3 * (size_t)(j + (u ? f[0] : 0))] = p[u].x; A.down[3 * (size_t)(j + (u ? f[0] : 0)) + 1] = p[u].y; A.down[3 * (size_t)(j + (u ? f[0] : 0)) + 2] = p[u].z;
            }
            c[u] = claim_issue(A.keys2, A.shift2, p[u], A.vs2, f[u] != 0, A.st);
        }
#pragma unroll
        for (int u = 0; u < ITEMS; ++u)
            if (f[u]) { const int jj = j + (u ? f[0] : 0); A.pslot2[jj] = claim_finish(c[u], A.keys2, A.min2, A.mask2, (unsigned int)jj, A.st); }
        if (tile == ntiles - 1 && threadIdx.x == 0) { A.counts[0] = base + total; *A.nd_this = base + total; }
        __syncthreads();
    }
    if (ntiles == 0 && gtid == 0) { A.counts[0] = 0; *A.nd_this = 0; }
    gs.sync();
    VX_MARK(2);
    LIMU_TRACE(12);
    if (gtid == 0 && A.st_next) *A.st_next = DevStatus{0, 0, {0, 0}};   // (its last reader, the result copy of the previous scan, is long done)
    // the stage-1 table was last read in P2: un-claim it for the next launch
    for (int64_t i = gtid; i < n; i += gthreads) {
        const unsigned int sl = A.pslot1[i];
        if (sl != PEND_NONE) { A.keys1[sl] = KEY_EMPTY; A.min1[sl] = PEND_NONE; }
    }
    // P3: the same flag -> count -> scatter over down[] for stage 2
    const int nd = __ldcg(A.counts);
    const int ntiles2 = (nd + TILE - 1) / TILE;
    for (int tile = blockIdx.x; tile < ntiles2; tile += gridDim.x) {
        const int e0 = tile * TILE + (int)threadIdx.x * ITEMS;
        int f[ITEMS], cnt = 0;
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
            const int j = e0 + u;
            f[u] = 0;
            if (j < nd) { const unsigned int s = __ldcg(A.pslot2 + j); f[u] = s != PEND_NONE && __ldcg(A.min2 + s) == (unsigned int)j; }
            cnt += f[u];
        }
        const int r = block_exclusive_scan_count(cnt, &total, ws);
        if (threadIdx.x == 0) tile_publish(A.tile2 + tile, A.epoch, total);
        const int base = tile_base<BLOCK>(A.tile2, tile, A.epoch, ws);
#pragma unroll
        for (int u = 0; u < ITEMS; ++u)
            if (f[u]) {
                const size_t k = (size_t)(base + r + (u ? f[0] : 0)), j = (size_t)(e0 + u);
                A.src0[3 * k] = __ldcg(A.down + 3 * j); A.src0[3 * k + 1] = __ldcg(A.down + 3 * j + 1); A.src0[3 * k + 2] = __ldcg(A.down + 3 * j + 2);
            }
        if (tile == ntiles2 - 1 && threadIdx.x == 0) A.counts[1] = base + total;
        __syncthreads();
    }
    if (ntiles2 == 0 && gtid == 0) A.counts[1] = 0;
    // every CTA has left the last barrier before it gets here, so the last one out can re-arm it for the next launch
    __syncthreads();
    VX_MARK(3);
    LIMU_TRACE(13);
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(A.barrier + 1, 1u) == gridDim.x - 1) { A.barrier[0] = 0u; A.barrier[1] = 0u; __threadfence(); }
    }
}
// The three launch shapes: full (alone on the GPU: 1024 threads x 64 registers = a whole register file), half (512 x 2 points) and lean
// (1024 x 1 at 48 registers, a few spills) -- the latter two leave 16 K registers per SM to the map update's CTA that runs beside them.
static __global__ void __launch_bounds__(VX_BLOCK, 1) k_voxelize_full(const VoxelizeArgs A) { voxelize_body<VX_BLOCK, 1>(A); }
static __global__ void __launch_bounds__(VX_BLOCK_BESIDE, 2) k_voxelize_half(const VoxelizeArgs A) { voxelize_body<VX_BLOCK_BESIDE, VX_TILE / VX_BLOCK_BESIDE>(A); }
static __global__ void __maxnreg__(48) k_voxelize_lean(const VoxelizeArgs A) { voxelize_body<VX_BLOCK, 1>(A); }

// One thread that waits until a frame kernel launched EARLIER on another stream has published the pose of its scan (the flag carries that
// launch's sequence number): the stream it sits in -- the next scan's k_voxelize behind it -- is released the moment the Gauss-Newton loop is
// over instead of when that kernel and the map update behind it have finished. A single thread holds no resource anybody waits for, so the
// wait cannot deadlock; after 5 s (the awaited kernel is gone) it gives up and lets the error surface on the host.
static __global__ void k_gate(const unsigned int *flag, unsigned int seq) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (unsigned int spins = 1;; ++spins) {   // (no __nanosleep: its granularity is microseconds, and one thread polling costs nothing)
        unsigned int v;
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int)(v - seq) >= 0) break;
        if ((spins & 1023u) == 0u) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 5000000000ull) break;
        }
    }
    LIMU_TRACE(30);
}
int gate_device(cudaStream_t s, const unsigned int *flag, unsigned int seq) {
    static bool hinted = false;
    if (!hinted) {   // ask for the largest shared-memory carve-out: the SM the gate sits on can then take CTAs of the kernels it waits for without draining first
        if (cudaFuncSetAttribute(k_gate, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess) (void)cudaGetLastError();
        hinted = true;
    }
    k_gate<<<1, 1, 0, s>>>(flag, seq);
    LIMU_LAUNCHED();
    return LIMU_OK;
}

#ifdef LIMU_ICP_PHASE_TIMING
extern "C" int limu_debug_vox_marks(double out[8]) {
    unsigned long long h[8];
    if (cudaMemcpyFromSymbol(h, g_vox_marks, sizeof h) != cudaSuccess) return -1;
    for (int k = 0; k < 8; ++k) out[k] = (double)h[k];
    return 0;
}
#endif

static int g_vx_blocks_per_sm = 0;

static int64_t pow2_slots(int64_t n) { int64_t p = 1024; while (p < 2 * n) p <<= 1; return p; }

// Enqueue the fused kernel. raw/ts/twist are device pointers; outputs: frame (n x 3), down, src0, counts[0..1].
int voxelize_device(limu_ctx *c, VoxelizeScratch &sc, const void *raw_dev, int mode, int stride, const double *ts_dev, int deskew, const double *twist_host,
                    int64_t n, double v, double *frame_dev, double *down_dev, double *src0_dev, int *counts_dev, const double *twist_dev, DevStatus *own_status, int *status_used,
                    cudaStream_t stream, bool beside) {
    if (!stream) stream = c->stream;
    if (n <= 0) {
        LIMU_CUDA_TRY(cudaMemsetAsync(counts_dev, 0, 2 * sizeof(int), stream));
        if (own_status) {   // the word this (empty) launch reports into must read clean; the rotation moves on as for any launch
            const int w = sc.st_word;
            sc.st_word = (w + 1) % 3;
            LIMU_CUDA_TRY(cudaMemsetAsync(own_status + w, 0, sizeof(DevStatus), stream));
            LIMU_CUDA_TRY(cudaMemsetAsync(own_status + sc.st_word, 0, sizeof(DevStatus), stream));
            if (status_used) *status_used = w;
        } else if (status_used) *status_used = 0;
        return LIMU_OK;
    }
    if (g_vx_blocks_per_sm == 0) {
        int b = 0;
        LIMU_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_voxelize_full, VX_BLOCK, 0));
        g_vx_blocks_per_sm = std::max(1, std::min(b, 1024 / VX_BLOCK));
    }
    const int64_t C1 = pow2_slots(n), C2 = pow2_slots(n);
    int lg = 0;
    while ((int64_t(1) << lg) < C1) ++lg;
    const int ntiles = div_up(n, VX_TILE);
    {   // three tables [u64 key x cap | u32 min-index x cap] at offsets fixed by the ALLOCATED capacity (claimed slots are remembered as indices), all-ones
        // = clean at rest. Whenever one of the buffers is re-allocated the memory of what the previous launch claimed is gone: start over clean.
        bool reset = false;
        if (C1 > sc.cap_slots) {
            int64_t cap = sc.cap_slots ? sc.cap_slots : 1024;
            while (cap < C1) cap <<= 1;
            LIMU_TRY(sc.table.reserve((size_t)cap * 12 * 3, stream));
            sc.cap_slots = cap;
            reset = true;
        }
        const void *before = sc.pslot.p;
        LIMU_TRY(sc.pslot.reserve((size_t)n * 4 * 3, stream));   // pslot1 | pslot2 of the two parities
        if (sc.pslot.p != before) reset = true;
        sc.pslot_n = (int64_t)(sc.pslot.bytes / 12);
        // [16 ints: barrier words 0-1, stage-2 claim counts of the two parities 4-5 | per-tile count words of the two stages]; the kernel keeps
        // the barrier words at zero, and a count word is only believed when it carries the epoch of the launch that reads it
        before = sc.tiles.p;
        LIMU_TRY(sc.tiles.reserve((size_t)ntiles * 16 + 128, stream));
        if (sc.tiles.p != before) reset = true;
        if (reset) {
            LIMU_CUDA_TRY(cudaMemsetAsync(sc.table.p, 0xFF, (size_t)sc.cap_slots * 12 * 3, stream));
            LIMU_CUDA_TRY(cudaMemsetAsync(sc.tiles.p, 0, sc.tiles.bytes, stream));
        }
    }
    const int par = sc.parity;
    sc.parity ^= 1;
    VoxelizeArgs A;
    A.raw = raw_dev; A.ts = ts_dev; A.mode = mode; A.stride = stride; A.deskew = deskew; A.n = n;
    for (int k = 0; k < 6; ++k) A.twist[k] = (deskew && twist_host) ? twist_host[k] : 0.0;
    A.twist_dev = deskew ? twist_dev : nullptr;
    A.vs1 = v * 0.5; A.vs2 = v * 1.5;
    A.frame = frame_dev; A.down = down_dev; A.src0 = src0_dev;
    {
        unsigned char *base = sc.table.as<unsigned char>();
        const size_t tb = (size_t)sc.cap_slots * 12;   // bytes per table
        auto keys_of = [&](int t) { return reinterpret_cast<unsigned long long *>(base + tb * t); };
        auto min_of = [&](int t) { return reinterpret_cast<unsigned int *>(base + tb * t + (size_t)sc.cap_slots * 8); };
        A.keys1 = keys_of(0); A.min1 = min_of(0);
        A.keys2 = keys_of(1 + par); A.min2 = min_of(1 + par);
        A.keys2_prev = keys_of(1 + (par ^ 1)); A.min2_prev = min_of(1 + (par ^ 1));
    }
    A.mask1 = (unsigned int)(C1 - 1); A.mask2 = (unsigned int)(C2 - 1); A.shift1 = A.shift2 = 64 - lg;
    A.pslot1 = sc.pslot.as<unsigned int>();
    A.pslot2 = A.pslot1 + sc.pslot_n * (1 + par);
    A.pslot2_prev = A.pslot1 + sc.pslot_n * (1 + (par ^ 1));
    A.barrier = sc.tiles.as<unsigned int>();
    A.nd_this = sc.tiles.as<int>() + 4 + par;
    A.nd_prev = sc.tiles.as<int>() + 4 + (par ^ 1);
    A.tile1 = reinterpret_cast<unsigned long long *>(sc.tiles.as<int>() + 16); A.tile2 = A.tile1 + ntiles;
    if (++sc.epoch == 0u) sc.epoch = 1u;
    A.epoch = sc.epoch;
    A.counts = counts_dev;
    // own_status: three DevStatus words in rotation; this launch reports into word w and zeroes word w+1 (the next launch's) late. Three, not
    // two: in the pipelined path launch k+1 runs before the result copy of scan k has read launch k's word.
    const int w = sc.st_word;
    if (own_status) sc.st_word = (w + 1) % 3;
    A.st = own_status ? own_status + w : c->d_status;
    A.st_next = own_status ? own_status + sc.st_word : nullptr;
    if (status_used) *status_used = w;
    // beside the map update (pipelined path) the grid leaves GATE_SLACK_SMS SMs free: the NEXT scan's k_gate may become resident before every
    // CTA of this cooperative launch has been placed, and this launch sits in front of the loop that gate waits for (see icp_device)
    const int grid = (int)std::min<int64_t>(ntiles, beside ? (int64_t)std::max(1, c->sm_count - GATE_SLACK_SMS) : (int64_t)c->sm_count * g_vx_blocks_per_sm);
    void *args[] = {&A};
    static const int beside_shape = getenv("LIMU_VX_BESIDE") ? atoi(getenv("LIMU_VX_BESIDE")) : 1;   // 1: lean (measured 2.6 % more scans/s than half, profiles/r2_voxelize_beside_ab.json), 0: half
    if (beside && beside_shape == 1) LIMU_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_voxelize_lean, dim3(grid), dim3(VX_BLOCK), args, 0, stream));
    else if (beside) LIMU_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_voxelize_half, dim3(grid), dim3(VX_BLOCK_BESIDE), args, 0, stream));
    else LIMU_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)k_voxelize_full, dim3(grid), dim3(VX_BLOCK), args, 0, stream));
    LIMU_LAUNCHED();
    return LIMU_OK;
}

}  // namespace limu
