// voxelize.cu -- KissICP::deskew_scan + KissICP::voxelize's two downsampling stages as ONE persistent cooperative
// kernel (L/src/sensors/lidar/icp.cpp:36-47, :9-30, :126-131; helpers/deskew.cpp:10-28).
//
// The stand-alone stages (ops.cu) cost 13 launches + 2 memsets per scan, each a few microseconds of work on 128k points;
// here the phases are separated by grid barriers instead of kernel boundaries:
//   P1 deskew/widen -> frame[], stage-1 claim (the IMU variant: limu_deskew_imu's compensation of each record, imu_compensate.cuh)
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
#include <algorithm>

#include "compact.cuh"
#include "grid_sync.cuh"
#include "imu_compensate.cuh"
#include "ops.cuh"
#include "voxel_map.cuh"

LIMU_TRACE_RING(limu_debug_trace_vox)

namespace limu {

// Threads per CTA and points per tile (one point per thread). One fat CTA per SM: a grid barrier is paid per ARRIVING CTA (atomics on one
// word serialise at ~4 ns each: 592 CTAs of 256 -> 148 of 1024).
constexpr int VX_BLOCK = 1024;
// Deskew transforms one tile keeps in shared memory (one per run of equal timestamps; 3.5 KB). The bench scan has at most 19 runs in a tile;
// 64 leaves room for sensors with fewer beams per firing (a 16-beam sensor: 64 runs).
constexpr int VX_RUNS = 64;

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
// The parameters of the IMU variant (mode 3): a struct of their own, so the parameter block of the other kernels stays as it is.
// The pose table is read from global memory with ordinary loads, served by L1 (a warp's points mostly share their head row). Not staged in
// shared memory: the kernel keeps a small shared-memory footprint (132 B; the plain variants' 4 KB run table included), and so the carve-out
// next to k_gate (DESIGN section 4).
struct VoxelizeImuArgs : VoxelizeArgs {
    ImuDeskew imu;
};

// Claim the voxel of p in a scan-local table and note `index` as a candidate for its first point (atomicMin). Each probe is ONE
// compare-and-swap that both finds and claims: the slot is the voxel's if it was empty or already held the key. Returns the slot, or
// PEND_NONE for a key out of range or a full table (both reported in *st).
__device__ __forceinline__ unsigned int claim(unsigned long long *keys, unsigned int *minidx, int shift, unsigned int mask, const V3 &p, double vs,
                                              unsigned int index, DevStatus *st) {
    const int kx = vox_index(p.x, vs), ky = vox_index(p.y, vs), kz = vox_index(p.z, vs);
    // NaN: the reference's (int) cast gives INT_MIN on x86-64 (cvttsd2si), and so does vox_index: far outside the packed range
    if (!key_in_range(kx, ky, kz)) { st->key_range = 1; return PEND_NONE; }
    const unsigned long long key = pack_key(kx, ky, kz);
    unsigned int s = slot_of(key, shift);
    for (unsigned int probes = 0; probes <= mask; ++probes) {
        const unsigned long long cur = atomicCAS(&keys[s], KEY_EMPTY, key);
        if (cur == KEY_EMPTY || cur == key) { atomicMin(&minidx[s], index); return s; }
        s = (s + 1) & mask;
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

// The motion of a point fired at time t: SE3::exp((t - mid_pose_timestamp) * twist) (deskew.cpp:18-26, deskew.hpp:12).
__device__ __forceinline__ Pose deskew_motion(double t, const double *tw) {
    const double s = t - 0.5;
    double st[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) st[k] = s * tw[k];
    return se3_exp(st);
}

// VX_BLOCK threads handle tiles of VX_BLOCK consecutive points, one point per thread. IMU: the variant of mode 3 (Args = VoxelizeImuArgs).
template <bool IMU, class Args>
__device__ __forceinline__ void voxelize_body(const Args &A) {
    __shared__ int ws[32];
    __shared__ int total;
    GridSync gs{A.barrier, 0u, gridDim.x};
    const int64_t n = A.n;
    const int64_t gtid = (int64_t)blockIdx.x * VX_BLOCK + threadIdx.x, gthreads = (int64_t)gridDim.x * VX_BLOCK;
    const int ntiles = (int)((n + VX_BLOCK - 1) / VX_BLOCK);
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
    if constexpr (IMU) {
        for (int64_t i = gtid; i < n; i += gthreads) {
            const unsigned char *r = static_cast<const unsigned char *>(A.raw) + (size_t)i * A.stride;
            const float *q = reinterpret_cast<const float *>(r);
            float xyz[3] = {q[0], q[1], q[2]};
            imu_deskew_point(A.imu.table, A.imu.M, i, imu_point_time(r, A.imu.toff), A.imu.rot_end, A.imu.pos_lidar_end, A.imu.p_il, xyz);
            const V3 p{(double)xyz[0], (double)xyz[1], (double)xyz[2]};   // the float write-back, widened (ekf.cpp:451-468)
            A.frame[3 * i] = p.x; A.frame[3 * i + 1] = p.y; A.frame[3 * i + 2] = p.z;
            A.pslot1[i] = claim(A.keys1, A.min1, A.shift1, A.mask1, p, A.vs1, (unsigned int)i, A.st);
        }
    } else {
        // the twist in shared memory, not in 12 registers across the loop (k_voxelize_lean has 48)
        __shared__ double tw[6];
        if (A.deskew && threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < 6; ++k) tw[k] = A.twist_dev ? __ldcg(A.twist_dev + k) : A.twist[k];
        }
        // One tile of VX_BLOCK points per CTA pass (the points the grid-stride loop gave this thread), with a CTA-uniform trip count: the
        // deskew transform is a function of the timestamp alone, and a spinning LiDAR fires all beams of one azimuth step at the same time
        // (64 beams per timestamp in the bench scan: ~16 distinct times per tile). So each run of equal timestamps BITS in a tile gets ONE
        // se3_exp, in a shared table, and every point applies its run's pose: the same operations on the same operands as the per-point
        // computation, hence bit-identical frames. Equal bits, not equal values: NaN, +-0 and denormals group deterministically. A tile
        // with more than VX_RUNS runs (per-point times, unsorted clouds) takes the per-point path; the branch is CTA-uniform.
        __shared__ unsigned long long last_t[VX_BLOCK / 32];   // bits of each warp's last timestamp
        __shared__ Pose runs[VX_RUNS];                         // the run's timestamp (in .qx) until its pose replaces it
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int64_t i = (int64_t)tile * VX_BLOCK + threadIdx.x;
            const bool live = i < n;
            // the timestamp first, the point after its transform is known: p is not live across se3_exp
            double t = 0.0;
            if (live && A.deskew) t = A.mode == 0 ? (double)__ldg(reinterpret_cast<const float4 *>(A.raw) + i).w : A.mode == 1 ? A.ts[i] : 0.0;
            Pose T{};
            if (A.deskew) {
                const unsigned long long tb = (unsigned long long)__double_as_longlong(t);
                unsigned long long prev = __shfl_up_sync(0xFFFFFFFFu, tb, 1);
                if (lane == 31) last_t[warp] = tb;
                __syncthreads();
                if (lane == 0 && warp > 0) prev = last_t[warp - 1];
                const int head = live && (threadIdx.x == 0 || tb != prev);
                const int run = block_exclusive_scan_count(head, &total, ws) + head - 1;   // (thread 0 of a tile is live: run >= 0 for live points)
                // one se3_exp site for both branches (two copies of its FP64 state would not fit k_voxelize_lean's 48 registers): with the
                // table, thread r computes the pose of run r; without it, every point its own
                const bool table = total <= VX_RUNS;
                if (table && head) runs[run].qx = t;
                if (table) __syncthreads();
                const bool mine = table ? (int)threadIdx.x < total : live;
                if (mine) T = deskew_motion(table ? runs[threadIdx.x].qx : t, tw);
                if (table) {
                    if (mine) runs[threadIdx.x] = T;
                    __syncthreads();
                    if (live) T = runs[run];
                }
            }
            if (live) {
                V3 p;
                if (A.mode == 0) {
                    const float4 q = __ldg(reinterpret_cast<const float4 *>(A.raw) + i);
                    p = V3{(double)q.x, (double)q.y, (double)q.z};
                } else if (A.mode == 1) {
                    const float *q = reinterpret_cast<const float *>(static_cast<const unsigned char *>(A.raw) + (size_t)i * A.stride);
                    p = V3{(double)q[0], (double)q[1], (double)q[2]};
                } else {
                    const double *q = static_cast<const double *>(A.raw) + 3 * i;
                    p = V3{q[0], q[1], q[2]};
                }
                if (A.deskew) p = apply(T, p);
                A.frame[3 * i] = p.x; A.frame[3 * i + 1] = p.y; A.frame[3 * i + 2] = p.z;
                A.pslot1[i] = claim(A.keys1, A.min1, A.shift1, A.mask1, p, A.vs1, (unsigned int)i, A.st);
            }
        }
    }
    gs.sync();
    VX_MARK(1);
    LIMU_TRACE(11);
    // P2: a point survives stage 1 iff it holds its voxel's smallest input index. Per tile: flags, count (published), ordered scatter
    // -> down[]; each winner immediately claims its 1.5 v voxel with its OUTPUT index.
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t i = (int64_t)tile * VX_BLOCK + threadIdx.x;
        int f = 0;
        if (i < n) { const unsigned int s = A.pslot1[i]; f = s != PEND_NONE && __ldcg(A.min1 + s) == (unsigned int)i; }
        const int r = block_exclusive_scan_count(f, &total, ws);
        if (threadIdx.x == 0) tile_publish(A.tile1 + tile, A.epoch, total);
        const int base = tile_base<VX_BLOCK>(A.tile1, tile, A.epoch, ws);
        if (f) {
            const int j = base + r;
            const V3 p{A.frame[3 * i], A.frame[3 * i + 1], A.frame[3 * i + 2]};
            A.down[3 * (size_t)j] = p.x; A.down[3 * (size_t)j + 1] = p.y; A.down[3 * (size_t)j + 2] = p.z;
            A.pslot2[j] = claim(A.keys2, A.min2, A.shift2, A.mask2, p, A.vs2, (unsigned int)j, A.st);
        }
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
    const int ntiles2 = (nd + VX_BLOCK - 1) / VX_BLOCK;
    for (int tile = blockIdx.x; tile < ntiles2; tile += gridDim.x) {
        const int j = tile * VX_BLOCK + (int)threadIdx.x;
        int f = 0;
        if (j < nd) { const unsigned int s = __ldcg(A.pslot2 + j); f = s != PEND_NONE && __ldcg(A.min2 + s) == (unsigned int)j; }
        const int r = block_exclusive_scan_count(f, &total, ws);
        if (threadIdx.x == 0) tile_publish(A.tile2 + tile, A.epoch, total);
        const int base = tile_base<VX_BLOCK>(A.tile2, tile, A.epoch, ws);
        if (f) {
            const size_t k = (size_t)(base + r);
            A.src0[3 * k] = __ldcg(A.down + 3 * (size_t)j); A.src0[3 * k + 1] = __ldcg(A.down + 3 * (size_t)j + 1); A.src0[3 * k + 2] = __ldcg(A.down + 3 * (size_t)j + 2);
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
// The two launch shapes: full (alone on the GPU: 1024 threads x 64 registers = a whole register file) and lean (48 registers, a few
// spills), which leaves 16 K registers per SM to the map update's CTA that runs beside it in the pipelined odometry path (odometry.cu).
static __global__ void __launch_bounds__(VX_BLOCK, 1) k_voxelize_full(const VoxelizeArgs A) { voxelize_body<false>(A); }
static __global__ void __maxnreg__(48) k_voxelize_lean(const VoxelizeArgs A) { voxelize_body<false>(A); }
static __global__ void __launch_bounds__(VX_BLOCK, 1) k_voxelize_imu_full(const VoxelizeImuArgs A) { voxelize_body<true>(A); }
static __global__ void __maxnreg__(48) k_voxelize_imu_lean(const VoxelizeImuArgs A) { voxelize_body<true>(A); }

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

// Enqueue the fused kernel. outputs: frame (n x 3), down, src0, counts[0..1].
int voxelize_device(limu_ctx *c, VoxelizeScratch &sc, const Scan &scan, int deskew, const double *twist_host, double v, double *frame_dev, double *down_dev,
                    double *src0_dev, int *counts_dev, const double *twist_dev, DevStatus *own_status, int *status_used, cudaStream_t stream, bool beside) {
    if (!stream) stream = c->stream;
    if (scan.layout == SCAN_IMU && !scan.imu) { set_error("voxelize_device: an IMU scan without IMU deskew arguments"); return LIMU_ERR_INVALID; }
    const int64_t n = scan.n;
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
    const int ntiles = div_up(n, VX_BLOCK);
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
    VoxelizeImuArgs X;
    VoxelizeArgs &A = X;
    A.raw = scan.ptr; A.ts = scan.ts; A.mode = scan.layout; A.stride = scan.stride; A.deskew = deskew; A.n = n;
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
    const void *fn = beside ? (const void *)k_voxelize_lean : (const void *)k_voxelize_full;
    if (scan.layout == SCAN_IMU) {
        const ImuCall &a = *scan.imu;
        X.imu.table = scan.imu_table; X.imu.M = a.M; X.imu.toff = a.toff;
        memcpy(X.imu.rot_end, a.rot_end, sizeof a.rot_end); memcpy(X.imu.pos_lidar_end, a.pos_lidar_end, sizeof a.pos_lidar_end); memcpy(X.imu.p_il, a.p_il, sizeof a.p_il);
        args[0] = &X;
        fn = beside ? (const void *)k_voxelize_imu_lean : (const void *)k_voxelize_imu_full;
    }
    LIMU_CUDA_TRY(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(VX_BLOCK), args, 0, stream));
    LIMU_LAUNCHED();
    return LIMU_OK;
}

}  // namespace limu
