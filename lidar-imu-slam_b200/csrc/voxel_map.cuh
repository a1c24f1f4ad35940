// voxel_map.cuh -- device view of the GPU-resident voxel hash map and the lookups kernels inline.
//
// Replaces lidar::VoxelHashMap + lidar::VoxelBlock (L/include/limu/sensors/lidar/helpers/
// voxel_hash_map.hpp:14-48, voxel_block.hpp:13-56): tsl::robin_map<Voxel, VoxelBlock> whose blocks hold
// one heap node per point becomes ONE open-addressing table in HBM:
//
//   blk[C*stride]   one 128-byte-aligned BLOCK per table slot, header first:
//                          {u64 packed (i,j,k) key, u64 meta = birth << 13 | count}, then three rows x[capp] y[capp] z[capp]
//                          (structure-of-arrays INSIDE a voxel, capp = cap rounded up to 4), padded to a multiple of 128 B
//                          (cap 10 -> 384 B, cap 20 -> 512 B). C = power of two, load <= 0.5. birth = creation sequence of the
//                          voxel (= the reference container's address order, used only by the 27-cell fallback tie-break,
//                          voxel_hash_map.cpp:81-101). Key, count and points of a voxel are ONE contiguous object: a hit costs
//                          one DRAM page / one L2 round trip, and the candidates can be requested together with the header.
//   pend[C*cap]      4 B  per point slot: insert scratch (sorted pending input indices), all-ones at rest
//   live[C]          4 B  dense list of the slots that ever became a voxel since the last rebuild (append order; an
//                          erased voxel leaves its entry behind and its slot reads KEY_TOMB): the eviction sweep
//                          walks this list (V entries) instead of the C table slots. Length = counters[3].
//
// One 16-byte load answers "is this my voxel, how many points does it hold, and how old is it"; the points follow in the same block.
#pragma once
#include "common.cuh"

namespace limu {

constexpr unsigned long long KEY_EMPTY = 0xFFFFFFFFFFFFFFFFull;
constexpr unsigned long long KEY_TOMB = 0xFFFFFFFFFFFFFFFEull;
constexpr unsigned long long META_NONE = 0xFFFFFFFFFFFFFFFFull;
constexpr int META_COUNT_BITS = 13;                       // max_points_per_voxel <= 4096 < 2^13
constexpr unsigned long long META_COUNT_MASK = (1ull << META_COUNT_BITS) - 1ull;
constexpr unsigned int PEND_NONE = 0xFFFFFFFFu;
constexpr int KEY_BIAS = 1 << 20;  // voxel indices in (-2^20, 2^20) pack into 3 x 21 bits

struct __align__(16) Slot {
    unsigned long long key;
    unsigned long long meta;   // birth << 13 | count
};
__host__ __device__ __forceinline__ int meta_count(unsigned long long meta) { return (int)(meta & META_COUNT_MASK); }
__host__ __device__ __forceinline__ unsigned long long meta_birth(unsigned long long meta) { return meta >> META_COUNT_BITS; }

struct MapView {
    double *blk;         // C blocks of `stride` doubles: 2 header words (Slot) + 3 rows of capp doubles + padding
    unsigned int *pend;
    unsigned int *live;  // dense list of used slots (live + erased), counters[3] entries
    unsigned long long *live_key;   // the packed voxel key of live[i] (KEY_TOMB once the voxel has been erased): the eviction sweep streams these 8-byte words
                                    // instead of one scattered block header per voxel
    unsigned int mask;   // C - 1
    int shift;           // 64 - log2(C)
    int cap;
    int capp;            // cap rounded up to a multiple of 4: row length of the per-voxel SoA block
    int stride;          // doubles per block: 2 + 3*capp rounded up to 16 (= 128 B)
    double vox;
    double inv_vox;      // 1/vox when vox is a power of two (then p * inv_vox == p / vox bit for bit and the FP64 division subroutine is avoided), else 0
};
__host__ __device__ __forceinline__ int cap_padded(int cap) { return (cap + 3) & ~3; }
__host__ __device__ __forceinline__ int block_stride(int cap) { return (2 + 3 * cap_padded(cap) + 15) & ~15; }
// header of table slot `slot`, and the row pointers of its voxel: x = base, y = base + capp, z = base + 2*capp
__host__ __device__ __forceinline__ Slot *slot_at(const MapView &m, unsigned int slot) { return reinterpret_cast<Slot *>(m.blk + (size_t)slot * (size_t)m.stride); }
__device__ __forceinline__ double *voxel_rows(const MapView &m, unsigned int slot) { return m.blk + (size_t)slot * (size_t)m.stride + 2; }

// utils::get_vox_index, calculation_helpers.cpp:142-147: IEEE double division, truncation toward zero, with the x86-64 semantics of
// the reference's (int) cast (cvttsd2si): a NaN quotient, or one whose truncation leaves int32, gives INT_MIN. cvt.rzi alone would give 0
// for NaN (aliasing a real voxel) and saturate beyond int32. INT_MIN lies outside the packed key range, so lookups see "absent" and the
// entries that make keys report LIMU_ERR_KEY_RANGE without a test of their own.
constexpr int VOX_INDEX_INVALID = -2147483647 - 1;
__device__ __forceinline__ int vox_trunc(double q) {
    // |q| >= 2^31: the saturated -2^31 is INT_MIN already, +2^31 and beyond become INT_MIN; NaN fails the compare
    return fabs(q) < 2147483648.0 ? __double2int_rz(q) : VOX_INDEX_INVALID;
}
__device__ __forceinline__ int vox_index(double p, double v) { return vox_trunc(p / v); }
__device__ __forceinline__ int vox_index(const MapView &m, double p) { return vox_trunc(m.inv_vox != 0.0 ? p * m.inv_vox : p / m.vox); }

__device__ __forceinline__ bool key_in_range(int x, int y, int z) {
    return (unsigned)(x + KEY_BIAS - 1) < (unsigned)(2 * KEY_BIAS - 1) && (unsigned)(y + KEY_BIAS - 1) < (unsigned)(2 * KEY_BIAS - 1) &&
           (unsigned)(z + KEY_BIAS - 1) < (unsigned)(2 * KEY_BIAS - 1);
}
__device__ __forceinline__ unsigned long long pack_key(int x, int y, int z) {
    return ((unsigned long long)(unsigned)(x + KEY_BIAS) << 42) | ((unsigned long long)(unsigned)(y + KEY_BIAS) << 21) |
           (unsigned long long)(unsigned)(z + KEY_BIAS);
}
__host__ __device__ __forceinline__ void unpack_key(unsigned long long k, int &x, int &y, int &z) {
    x = (int)((k >> 42) & 0x1FFFFF) - KEY_BIAS;
    y = (int)((k >> 21) & 0x1FFFFF) - KEY_BIAS;
    z = (int)(k & 0x1FFFFF) - KEY_BIAS;
}
// Fibonacci hashing of the packed key; the top log2(C) bits index the table.
__device__ __forceinline__ unsigned int slot_of(unsigned long long key, int shift) {
    return (unsigned int)((key * 0x9E3779B97F4A7C15ull) >> shift);
}

// Map data is read with plain (coherent, L1-cached) loads, not ld.global.nc: the fused frame kernel WRITES slots and points
// in its insert / eviction epilogue after the Gauss-Newton loop has read them, so the read-only-for-the-kernel-lifetime
// contract of the non-coherent path does not hold there.
__device__ __forceinline__ ulonglong2 load_slot(const Slot *s) { return *reinterpret_cast<const ulonglong2 *>(s); }
__device__ __forceinline__ double ldm(const double *p) { return *p; }

// Read-only lookup. Returns slot index or -1; count of the voxel in *count.
__device__ __forceinline__ int map_find(const MapView &m, unsigned long long key, int *count) {
    unsigned int s = slot_of(key, m.shift);
    for (;;) {
        const ulonglong2 v = load_slot(slot_at(m, s));
        if (v.x == key) { *count = meta_count(v.y); return (int)s; }
        if (v.x == KEY_EMPTY) return -1;
        s = (s + 1) & m.mask;
    }
}

// 27-neighbourhood offsets by |delta|^2 class.
__device__ constexpr signed char NB_CORNERS[8][3] = {{-1, -1, -1}, {-1, -1, 1}, {-1, 1, -1}, {-1, 1, 1}, {1, -1, -1}, {1, -1, 1}, {1, 1, -1}, {1, 1, 1}};
__device__ constexpr signed char NB_EDGES[12][3] = {{-1, -1, 0}, {-1, 1, 0}, {1, -1, 0}, {1, 1, 0}, {-1, 0, -1}, {-1, 0, 1},
                                                    {1, 0, -1},  {1, 0, 1},  {0, -1, -1}, {0, -1, 1}, {0, 1, -1}, {0, 1, 1}};
// faces are padded to 8 entries (two chunks of four); the padding repeats real faces, which is harmless for a maximum
__device__ constexpr signed char NB_FACES[8][3] = {{-1, 0, 0}, {1, 0, 0}, {0, -1, 0}, {0, 1, 0}, {0, 0, -1}, {0, 0, 1}, {0, 0, -1}, {0, 0, 1}};

struct Nearest {
    double x, y, z;   // matched map point, or (0,0,0) when nothing was found
    int slot;         // table slot of the matched voxel, -1 if none
    int rank;         // position of the match inside its voxel, -1 if none
    int ncand;        // points compared
    int own;          // 1 if the query's own voxel was present
};

// VoxelBlock::get_closest_point, voxel_block.cpp:87-105: linear scan, strict '<', first minimum wins.
// One-thread-per-query form: candidates are fetched four at a time (one 32 B sector per row) and compared in order.
__device__ __forceinline__ void block_closest(const MapView &m, int slot, int count, const V3 &p, Nearest &r) {
    const double *bx = voxel_rows(m, (unsigned int)slot), *by = bx + m.capp, *bz = by + m.capp;
    double best = 1.7976931348623157e308;
    r.rank = -1;
    for (int base = 0; base < count; base += 4) {   // rows are padded to a multiple of 4, so the loads stay in bounds
        double cx[4], cy[4], cz[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { cx[k] = ldm(bx + base + k); cy[k] = ldm(by + base + k); cz[k] = ldm(bz + base + k); }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double d = sqnorm3(p.x - cx[k], p.y - cy[k], p.z - cz[k]);
            if (base + k < count && d < best) { best = d; r.rank = base + k; r.x = cx[k]; r.y = cy[k]; r.z = cz[k]; }
        }
    }
    r.ncand = count;
}

// Step 1 of the lookup: WHICH voxel answers the query (rules (a)/(b) below). Returns its slot (or -1), its count,
// and whether it is the query's own voxel.
__device__ __forceinline__ int map_locate(const MapView &m, const V3 &p, int *count_out, int *own_out) {
    const int kx = vox_index(m, p.x), ky = vox_index(m, p.y), kz = vox_index(m, p.z);
    *own_out = 0;
    *count_out = 0;
    if (key_in_range(kx, ky, kz)) {
        int count = 0;
        const int s = map_find(m, pack_key(kx, ky, kz), &count);
        if (s >= 0) { *own_out = 1; *count_out = count; return s; }
    }
    // Fallback (b): the winner is the occupied neighbour with the largest (|delta|^2, birth). Visit the
    // three distance classes in decreasing |delta|^2 -- 8 corners (3), 12 edges (2), 6 faces (1) -- and stop
    // after the first class with an occupied cell. Cells are probed four at a time: the four 16-byte home-slot
    // loads are issued before any is consumed, and each answers key, birth and count at once.
    int best_slot = -1;
    unsigned long long best_meta = 0;
#define LIMU_PROBE_CHUNK(TABLE, FIRST)                                                                      \
    {                                                                                                       \
        ulonglong2 got[4];                                                                                  \
        _Pragma("unroll") for (int c = 0; c < 4; ++c) {                                                     \
            const int x = kx + TABLE[FIRST + c][0], y = ky + TABLE[FIRST + c][1], z = kz + TABLE[FIRST + c][2]; \
            got[c] = key_in_range(x, y, z) ? load_slot(slot_at(m, slot_of(pack_key(x, y, z), m.shift))) : make_ulonglong2(KEY_EMPTY, 0ull); \
        }                                                                                                   \
        _Pragma("unroll") for (int c = 0; c < 4; ++c) {                                                     \
            ulonglong2 v = got[c];                                                                          \
            if (v.x != KEY_EMPTY) {                                                                         \
                const unsigned long long want = pack_key(kx + TABLE[FIRST + c][0], ky + TABLE[FIRST + c][1], kz + TABLE[FIRST + c][2]); \
                unsigned int s = slot_of(want, m.shift);                                                    \
                while (v.x != want && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); } \
                if (v.x == want && (best_slot < 0 || v.y > best_meta)) { best_meta = v.y; best_slot = (int)s; } \
            }                                                                                               \
        }                                                                                                   \
    }
    LIMU_PROBE_CHUNK(NB_CORNERS, 0)
    LIMU_PROBE_CHUNK(NB_CORNERS, 4)
    if (best_slot < 0) {
        LIMU_PROBE_CHUNK(NB_EDGES, 0)
        LIMU_PROBE_CHUNK(NB_EDGES, 4)
        LIMU_PROBE_CHUNK(NB_EDGES, 8)
    }
    if (best_slot < 0) {
        LIMU_PROBE_CHUNK(NB_FACES, 0)
        LIMU_PROBE_CHUNK(NB_FACES, 4)
    }
#undef LIMU_PROBE_CHUNK
    if (best_slot >= 0) *count_out = meta_count(best_meta);   // births are unique, so comparing meta compared birth
    return best_slot;
}

// VoxelHashMap::get_closest_neighbour, voxel_hash_map.cpp:64-102:
//  (a) own voxel present            -> closest point inside it only (:71-73)
//  (b) else the top of a max-heap on (|delta index|^2, block address) over the occupied cells of the
//      27-neighbourhood (:76-96,101) = the FARTHEST occupied cell, ties to the later-created voxel
//  (c) nothing                      -> (0,0,0) (:98-99)
__device__ __forceinline__ Nearest map_closest(const MapView &m, const V3 &p) {
    Nearest r;
    r.x = r.y = r.z = 0.0; r.rank = -1; r.ncand = 0;
    int count;
    r.slot = map_locate(m, p, &count, &r.own);
    if (r.slot >= 0) {
        block_closest(m, r.slot, count, p, r);
        if (r.rank < 0) { r.x = r.y = r.z = 0.0; }
    }
    return r;
}

// The 26 neighbour offsets in one table (corners, edges, faces) for the group-cooperative fallback below.
__device__ constexpr signed char NB_ALL[26][3] = {
    {-1, -1, -1}, {-1, -1, 1}, {-1, 1, -1}, {-1, 1, 1}, {1, -1, -1}, {1, -1, 1}, {1, 1, -1}, {1, 1, 1},
    {-1, -1, 0}, {-1, 1, 0}, {1, -1, 0}, {1, 1, 0}, {-1, 0, -1}, {-1, 0, 1}, {1, 0, -1}, {1, 0, 1}, {0, -1, -1}, {0, -1, 1}, {0, 1, -1}, {0, 1, 1},
    {-1, 0, 0}, {1, 0, 0}, {0, -1, 0}, {0, 1, 0}, {0, 0, -1}, {0, 0, 1}};

// Group-cooperative lookup: EIGHT lanes serve one query (both shapes of the fused registration kernel: a few thousand keypoints per
// iteration, latency bound -- and millions of queries against a map far larger than L2, bandwidth bound).
// The common case -- the query's own voxel exists and sits in its home slot -- is ONE round trip: the block header (key, count, birth:
// the same address for all eight lanes, one broadcast load) and this lane's candidate ranks l8, l8+8, ... of the same block are requested
// together, before the key comparison can say whether they will be used; header and points are one contiguous object. A displaced voxel
// costs dependent probes; an absent one the 26-cell fallback: lane l probes neighbours l, l+8, l+16, l+24 at once and a 3-step butterfly
// picks the lexicographic maximum of (|delta|^2, birth) = the reference's max-heap top (voxel_hash_map.cpp:81-101). A second butterfly
// picks the lexicographic minimum of (d^2, rank) = "first minimum wins" (voxel_block.cpp:87-105) and the winning lane hands its point
// to the group by shuffle. Every lane of the group returns the result. ROUNDS*8 >= cap keeps the whole scan in registers.
template <int ROUNDS>
__device__ __forceinline__ void group8_load(const MapView &m, unsigned int slot, int l8, double *cx, double *cy, double *cz) {
    const double *bx = voxel_rows(m, slot), *by = bx + m.capp, *bz = by + m.capp;
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {   // ranks beyond the row re-read rank l8 & 3 (always inside the block) and are ignored by the scan
        const int r = l8 + 8 * k, rr = r < m.capp ? r : (l8 & 3);
        cx[k] = ldm(bx + rr); cy[k] = ldm(by + rr); cz[k] = ldm(bz + rr);
    }
}
template <int ROUNDS>
__device__ __forceinline__ void group8_scan(const V3 &p, int l8, int count, const double *cx, const double *cy, const double *cz, double &bd2, int &br, double &tx,
                                            double &ty, double &tz) {
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
        const int r = l8 + 8 * k;
        const double d = sqnorm3(p.x - cx[k], p.y - cy[k], p.z - cz[k]);
        if (r < count && d < bd2) { bd2 = d; br = r; tx = cx[k]; ty = cy[k]; tz = cz[k]; }
    }
}
// The rare part of the lookup, kept out of line so that its registers (four 16-byte probes in flight per lane) do not weigh on the hot
// path: the home slot `h` holds ANOTHER voxel (collision: probe on) or nothing. If the query's own voxel is not in the table, fall back
// to the 26 neighbours: lane l probes cells l, l+8, l+16, l+24 at once and a 3-step butterfly picks the lexicographic maximum of
// (|delta|^2, birth) = the reference's max-heap top (voxel_hash_map.cpp:81-101). Group-uniform; returns the slot (or -1).
struct MapProbe { double *blk; unsigned int mask; int shift, stride; };   // what probing needs of a MapView, passed BY VALUE (a reference to the
                                                                          // kernel's parameter block would force a local copy of all of it)
// the home slots of this lane's four neighbour cells l8, l8+8, l8+16, l8+24 of the 26 (issued together: one round trip)
__device__ __forceinline__ void group8_probe_neighbours(const MapView &m, int kx, int ky, int kz, int l8, ulonglong2 *got) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = l8 + 8 * u;
        got[u] = make_ulonglong2(KEY_EMPTY, 0ull);
        if (c < 26) {
            const int x = kx + NB_ALL[c][0], y = ky + NB_ALL[c][1], z = kz + NB_ALL[c][2];
            if (key_in_range(x, y, z)) got[u] = load_slot(slot_at(m, slot_of(pack_key(x, y, z), m.shift)));
        }
    }
}
// The rare part: the home slot `h` holds ANOTHER voxel (collision: probe on) or nothing; if the query's own voxel is not in the table, the
// fallback over the neighbour probes `got`. Group-uniform; returns the slot (or -1).
__device__ __forceinline__ int group8_resolve_core(const MapView &m, int kx, int ky, int kz, bool inr, unsigned long long key, unsigned int h, ulonglong2 sv,
                                                   const ulonglong2 *got, unsigned gmask, int l8, int *count_out, int *own_out) {
    *own_out = 0;
    *count_out = 0;
    if (inr) {
        unsigned int s = h;
        ulonglong2 v = sv;
        while (v.x != key && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); }
        if (v.x == key) { *count_out = meta_count(v.y); *own_out = 1; return (int)s; }
    }
    int bd = -1, bslot = -1;
    unsigned long long bmeta = 0ull;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = l8 + 8 * u;
        ulonglong2 v = got[u];
        if (c < 26 && v.x != KEY_EMPTY) {
            const unsigned long long want = pack_key(kx + NB_ALL[c][0], ky + NB_ALL[c][1], kz + NB_ALL[c][2]);
            unsigned int s = slot_of(want, m.shift);
            while (v.x != want && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); }
            if (v.x == want) {
                const int d = c < 8 ? 3 : (c < 20 ? 2 : 1);
                if (d > bd || (d == bd && v.y > bmeta)) { bd = d; bmeta = v.y; bslot = (int)s; }
            }
        }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        const int od = __shfl_xor_sync(gmask, bd, o), os = __shfl_xor_sync(gmask, bslot, o);
        const unsigned long long om = __shfl_xor_sync(gmask, bmeta, o);
        if (od > bd || (od == bd && om > bmeta)) { bd = od; bmeta = om; bslot = os; }
    }
    if (bslot >= 0) *count_out = meta_count(bmeta);
    return bslot;
}
// ... kept out of line where registers are scarce (bandwidth shape: the four 16-byte probes in flight per lane must not weigh on the hot path)
static __device__ __noinline__ int group8_resolve_rare(MapProbe mp, int kx, int ky, int kz, bool inr, unsigned long long key, unsigned int h, ulonglong2 sv,
                                                      unsigned gmask, int l8, int *count_out, int *own_out) {
    MapView m;
    m.blk = mp.blk; m.mask = mp.mask; m.shift = mp.shift; m.stride = mp.stride;
    ulonglong2 got[4];
    group8_probe_neighbours(m, kx, ky, kz, l8, got);
    return group8_resolve_core(m, kx, ky, kz, inr, key, h, sv, got, gmask, l8, count_out, own_out);
}

// Core: the query's voxel index (kx, ky, kz), whether it is inside the packed key range (inr), its packed key and home slot h are given
// (the bandwidth shape computes them with ONE lane per query and hands them to the group by shuffle).
// PREFETCH_NB (latency shape, registers to spare): the 26 neighbour probes are requested together with the home block, so an absent voxel
// costs two round trips (probes, then the neighbour's candidates) instead of three -- the slowest query of an iteration sets its pace.
// known: the caller has resolved this voxel index before (slot_out / count_out / own_out hold the answer, the map has not changed since):
// straight to the candidates of that block, one round trip whatever the voxel's situation was.
template <int ROUNDS, bool PREFETCH_NB = false>
__device__ __forceinline__ void group8_closest_at(const MapView &m, const V3 &p, int kx, int ky, int kz, bool inr, unsigned long long key, unsigned int h,
                                                  unsigned gmask, int l8, int &slot_out, int &count_out, int &own_out, double &d2_out, int &rank_out, V3 &t_out,
                                                  bool known = false) {
    double bd2 = 1.7976931348623157e308, tx = 0.0, ty = 0.0, tz = 0.0;
    int br = 0x7FFFFFFF, slot, count, own;
    if (known) {
        slot = slot_out; count = count_out; own = own_out;
        if (slot >= 0) {
            double cx[ROUNDS], cy[ROUNDS], cz[ROUNDS];
            group8_load<ROUNDS>(m, (unsigned int)slot, l8, cx, cy, cz);
            group8_scan<ROUNDS>(p, l8, count, cx, cy, cz, bd2, br, tx, ty, tz);
        }
    } else {   // the one round trip of the common case: header and this lane's candidate ranks of the home block, requested together
        const ulonglong2 sv = load_slot(slot_at(m, h));
        double cx[ROUNDS], cy[ROUNDS], cz[ROUNDS];
        group8_load<ROUNDS>(m, h, l8, cx, cy, cz);
        ulonglong2 got[PREFETCH_NB ? 4 : 1];
        if (PREFETCH_NB) group8_probe_neighbours(m, kx, ky, kz, l8, got);
        if (inr && sv.x == key) {
            slot = (int)h; count = meta_count(sv.y); own = 1;
        } else if (PREFETCH_NB) {
            slot = group8_resolve_core(m, kx, ky, kz, inr, key, h, sv, got, gmask, l8, &count, &own);
            if (slot >= 0) group8_load<ROUNDS>(m, (unsigned int)slot, l8, cx, cy, cz);
        } else {   // group-uniform: all eight lanes saw the same header
            slot = group8_resolve_rare(MapProbe{m.blk, m.mask, m.shift, m.stride}, kx, ky, kz, inr, key, h, sv, gmask, l8, &count, &own);
            if (slot >= 0) group8_load<ROUNDS>(m, (unsigned int)slot, l8, cx, cy, cz);   // displaced or neighbour voxel: its candidates are a second trip
        }
        if (slot >= 0) group8_scan<ROUNDS>(p, l8, count, cx, cy, cz, bd2, br, tx, ty, tz);
    }
    if (slot >= 0 && count > 8 * ROUNDS) {   // max_points_per_voxel beyond the register-resident part (cap > 24)
        const double *bx = voxel_rows(m, (unsigned int)slot), *by = bx + m.capp, *bz = by + m.capp;
        for (int r = l8 + 8 * ROUNDS; r < count; r += 8) {
            const double x = ldm(bx + r), y = ldm(by + r), z = ldm(bz + r);
            const double d = sqnorm3(p.x - x, p.y - y, p.z - z);
            if (d < bd2) { bd2 = d; br = r; tx = x; ty = y; tz = z; }
        }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(gmask, bd2, o);
        const int orr = __shfl_xor_sync(gmask, br, o);
        if (od < bd2 || (od == bd2 && orr < br)) { bd2 = od; br = orr; }
    }
    {   // the winner's point: lane (rank & 7) of the group holds it
        const int src = (br == 0x7FFFFFFF ? 0 : (br & 7));
        tx = __shfl_sync(gmask, tx, src, 8); ty = __shfl_sync(gmask, ty, src, 8); tz = __shfl_sync(gmask, tz, src, 8);
    }
    slot_out = slot; count_out = count; own_out = own; d2_out = bd2; rank_out = br == 0x7FFFFFFF ? -1 : br;
    t_out = br == 0x7FFFFFFF ? V3{0.0, 0.0, 0.0} : V3{tx, ty, tz};   // nothing found -> (0,0,0)
}
// What a group remembers about the query it serves in every iteration of a Gauss-Newton loop: the voxel index it resolved last time and
// the answer. The map does not change inside a launch and an iteration moves a point by less and less, so from the second iteration on
// nearly every lookup -- in particular the slow kind, an absent voxel answered by a neighbour after two more round trips -- is a repeat.
// (Measured alternatives, profiles/r2_latency_loop_lookup_variants.json: repeats and first-time lookups in ONE instruction stream, and
//  neighbour probes requested together with the home block on first-time lookups, both made the rare warp faster -- 3.5 -> 2.9 us --
//  and every other warp slower -- 1.45 -> 1.7 us; scans/s went down.)
struct QueryMemo {
    int kx, ky, kz;
    int slot, count, own;   // own < 0: nothing remembered
};
template <int ROUNDS>
__device__ __forceinline__ void group8_closest(const MapView &m, const V3 &p, unsigned gmask, int l8, int &slot_out, int &count_out, int &own_out,
                                               double &d2_out, int &rank_out, V3 &t_out, QueryMemo *memo = nullptr) {
    const int kx = vox_index(m, p.x), ky = vox_index(m, p.y), kz = vox_index(m, p.z);
    if (memo && memo->own >= 0 && memo->kx == kx && memo->ky == ky && memo->kz == kz) {   // group-uniform
        slot_out = memo->slot; count_out = memo->count; own_out = memo->own;
        group8_closest_at<ROUNDS, false>(m, p, kx, ky, kz, false, 0ull, 0u, gmask, l8, slot_out, count_out, own_out, d2_out, rank_out, t_out, true);
        return;
    }
    const bool inr = key_in_range(kx, ky, kz);
    const unsigned long long key = pack_key(kx, ky, kz);
    // (PREFETCH_NB was measured in the pipeline's latency shape: the absent-voxel path got shorter, but the four extra probes and their key
    //  arithmetic on EVERY query cost more than they saved -- 9.2 vs 8.7 us per iteration -- so it stays off)
    group8_closest_at<ROUNDS, false>(m, p, kx, ky, kz, inr, key, inr ? slot_of(key, m.shift) : 0u, gmask, l8, slot_out, count_out, own_out, d2_out, rank_out, t_out);
    if (memo) { memo->kx = kx; memo->ky = ky; memo->kz = kz; memo->slot = slot_out; memo->count = count_out; memo->own = own_out; }
}

// Pair-cooperative lookup for the cluster latency shape (registration.cu, k_frame_cluster): TWO lanes serve one query, so that one
// 16-CTA cluster covers a whole keypoint cloud in a single pass. The common case -- the query's own voxel exists and sits in its home
// slot (the pipeline's table is sparse: ~6 % load) -- costs ONE L2 round trip: the home slot and this lane's candidate ranks l2, l2+2, ...
// of the home slot's block are requested together, before the key comparison can say whether they will be used. A displaced or absent
// voxel falls back to dependent loads: linear probing, or the 26-cell fallback of get_closest_neighbour with 13 cells per lane.
// Same decisions as map_locate + block_closest: first minimum in storage order wins (lexicographic minimum of (d^2, rank)).
// Every lane of the warp must call this (the pair exchanges are warp-wide shuffles); lanes without a query pass any point and ignore the result.
template <int ROUNDS>
__device__ __forceinline__ void pair_load_candidates(const MapView &m, unsigned int slot, int l2, double *cx, double *cy, double *cz) {
    const double *bx = voxel_rows(m, slot), *by = bx + m.capp, *bz = by + m.capp;
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {   // ranks beyond the row re-read rank l2 (always inside the block) and are ignored by the caller
        const int r = l2 + 2 * k, rr = r < m.capp ? r : l2;
        cx[k] = ldm(bx + rr); cy[k] = ldm(by + rr); cz[k] = ldm(bz + rr);
    }
}
// this lane's share of VoxelBlock::get_closest_point (voxel_block.cpp:87-105): ranks l2, l2+2, ... in ascending order, strict '<'
template <int ROUNDS>
__device__ __forceinline__ void pair_scan(const V3 &p, int l2, int count, const double *cx, const double *cy, const double *cz, double &bd2, int &br, double &tx,
                                          double &ty, double &tz) {
#pragma unroll
    for (int k = 0; k < ROUNDS; ++k) {
        const int r = l2 + 2 * k;
        const double d = sqnorm3(p.x - cx[k], p.y - cy[k], p.z - cz[k]);
        if (r < count && d < bd2) { bd2 = d; br = r; tx = cx[k]; ty = cy[k]; tz = cz[k]; }
    }
}
template <int ROUNDS>
__device__ __forceinline__ void pair_closest(const MapView &m, const V3 &p, int l2, int &count_out, int &own_out, double &d2_out, V3 &t_out, int &rank_out) {
    const int kx = vox_index(m, p.x), ky = vox_index(m, p.y), kz = vox_index(m, p.z);
    const bool inr = key_in_range(kx, ky, kz);
    const unsigned long long key = pack_key(kx, ky, kz);
    const unsigned int h = inr ? slot_of(key, m.shift) : 0u;
    double bd2 = 1.7976931348623157e308, tx = 0.0, ty = 0.0, tz = 0.0;
    int br = 0x7FFFFFFF, slot = -1, count = 0;
    own_out = 0;
    {   // the one round trip of the common case; the prefetched candidates are consumed right here, so that their registers are free
        // again before the fallback below puts its probes in flight
        const ulonglong2 sv = load_slot(slot_at(m, h));
        double cx[ROUNDS], cy[ROUNDS], cz[ROUNDS];
        pair_load_candidates<ROUNDS>(m, h, l2, cx, cy, cz);
        if (inr) {
            unsigned int s = h;
            ulonglong2 v = sv;
            while (v.x != key && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); }
            if (v.x == key) { slot = (int)s; count = meta_count(v.y); own_out = 1; }
        }
        if (slot >= 0) {
            if ((unsigned int)slot != h) pair_load_candidates<ROUNDS>(m, (unsigned int)slot, l2, cx, cy, cz);   // displaced by a collision: second trip
            pair_scan<ROUNDS>(p, l2, count, cx, cy, cz, bd2, br, tx, ty, tz);
        }
    }
    // fallback (voxel_hash_map.cpp:76-101): the occupied neighbour with the largest (|delta|^2 class, birth); lane l2 probes cells l2, l2+2, ...
    int bd = -1, bslot = -1;
    unsigned long long bmeta = 0ull;
    if (slot < 0) {
        ulonglong2 got[13];
#pragma unroll
        for (int u = 0; u < 13; ++u) {
            const int c = l2 + 2 * u;
            const int x = kx + NB_ALL[c][0], y = ky + NB_ALL[c][1], z = kz + NB_ALL[c][2];
            got[u] = key_in_range(x, y, z) ? load_slot(slot_at(m, slot_of(pack_key(x, y, z), m.shift))) : make_ulonglong2(KEY_EMPTY, 0ull);
        }
#pragma unroll
        for (int u = 0; u < 13; ++u) {
            const int c = l2 + 2 * u;
            ulonglong2 v = got[u];
            if (v.x != KEY_EMPTY) {
                const unsigned long long want = pack_key(kx + NB_ALL[c][0], ky + NB_ALL[c][1], kz + NB_ALL[c][2]);
                unsigned int s = slot_of(want, m.shift);
                while (v.x != want && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); }
                if (v.x == want) {
                    const int d = c < 8 ? 3 : (c < 20 ? 2 : 1);
                    if (d > bd || (d == bd && v.y > bmeta)) { bd = d; bmeta = v.y; bslot = (int)s; }
                }
            }
        }
    }
    {   // both lanes of the pair agree on the winner (warp-wide exchange; pairs that did not search carry bd = -1 on both lanes)
        const int od = __shfl_xor_sync(0xFFFFFFFFu, bd, 1), os = __shfl_xor_sync(0xFFFFFFFFu, bslot, 1);
        const unsigned long long om = __shfl_xor_sync(0xFFFFFFFFu, bmeta, 1);
        if (od > bd || (od == bd && om > bmeta)) { bd = od; bmeta = om; bslot = os; }
    }
    if (slot < 0 && bslot >= 0) {   // neighbour voxel: its candidates are a second trip
        slot = bslot; count = meta_count(bmeta);
        double cx[ROUNDS], cy[ROUNDS], cz[ROUNDS];
        pair_load_candidates<ROUNDS>(m, (unsigned int)slot, l2, cx, cy, cz);
        pair_scan<ROUNDS>(p, l2, count, cx, cy, cz, bd2, br, tx, ty, tz);
    }
    {
        const double od = __shfl_xor_sync(0xFFFFFFFFu, bd2, 1), ox = __shfl_xor_sync(0xFFFFFFFFu, tx, 1), oy = __shfl_xor_sync(0xFFFFFFFFu, ty, 1),
                     oz = __shfl_xor_sync(0xFFFFFFFFu, tz, 1);
        const int orr = __shfl_xor_sync(0xFFFFFFFFu, br, 1);
        if (od < bd2 || (od == bd2 && orr < br)) { bd2 = od; br = orr; tx = ox; ty = oy; tz = oz; }
    }
    count_out = count; d2_out = bd2; rank_out = br == 0x7FFFFFFF ? -1 : br;
    t_out = V3{tx, ty, tz};   // (0,0,0) when nothing was found
}

// ---- opt-in neighbour rule LIMU_NN_27 (SURVEY section 8f N2; no counterpart in the reference) -----------------------------
// What the north star literally names and upstream KISS-ICP does: the NEAREST stored point over all 27 cells of the
// query's neighbourhood (the reference only looks into the query's own voxel when it exists, voxel_hash_map.cpp:71-73).
// Defined order: cells c = (dx+1)*9 + (dy+1)*3 + (dz+1) for dx, dy, dz in -1..1 (x outermost), points in storage order,
// strict '<' -- the first minimum in (cell, rank) order wins, so the result is the lexicographic minimum of (d^2, c, rank)
// and any evaluation order gives the same answer. Nothing stored in the 27 cells -> (0,0,0) like rule (c) above.
__device__ __forceinline__ Nearest map_closest27(const MapView &m, const V3 &p) {
    Nearest r;
    r.x = r.y = r.z = 0.0; r.rank = -1; r.ncand = 0; r.slot = -1; r.own = 0;
    const int kx = vox_index(m, p.x), ky = vox_index(m, p.y), kz = vox_index(m, p.z);
    double best = 1.7976931348623157e308;
    for (int dx = -1; dx <= 1; ++dx) {
        ulonglong2 got[9];
#pragma unroll
        for (int c = 0; c < 9; ++c) {   // nine home-slot loads in flight
            const int x = kx + dx, y = ky + (c / 3 - 1), z = kz + (c % 3 - 1);
            got[c] = key_in_range(x, y, z) ? load_slot(slot_at(m, slot_of(pack_key(x, y, z), m.shift))) : make_ulonglong2(KEY_EMPTY, 0ull);
        }
#pragma unroll
        for (int c = 0; c < 9; ++c) {
            ulonglong2 v = got[c];
            if (v.x == KEY_EMPTY) continue;
            const unsigned long long want = pack_key(kx + dx, ky + (c / 3 - 1), kz + (c % 3 - 1));
            unsigned int s = slot_of(want, m.shift);
            while (v.x != want && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); }
            if (v.x != want) continue;
            if (dx == 0 && c == 4) r.own = 1;
            const int count = meta_count(v.y);
            const double *bx = voxel_rows(m, s), *by = bx + m.capp, *bz = by + m.capp;
            for (int k = 0; k < count; ++k) {
                const double cx = ldm(bx + k), cy = ldm(by + k), cz = ldm(bz + k);
                const double d = sqnorm3(p.x - cx, p.y - cy, p.z - cz);
                if (d < best) { best = d; r.rank = k; r.slot = (int)s; r.x = cx; r.y = cy; r.z = cz; }
            }
            r.ncand += count;
        }
    }
    return r;
}

// The same rule with eight lanes per query (latency shape): lane l probes cells l, l+8, l+16 (and 24..26), scans the
// points of the cells it found, and a 3-step butterfly takes the lexicographic minimum of (d^2, cell, rank).
__device__ __forceinline__ void group8_closest27(const MapView &m, const V3 &p, unsigned gmask, int l8, int &slot_out, int &count_out, int &own_out,
                                                 double &d2_out, int &rank_out) {
    const int kx = vox_index(m, p.x), ky = vox_index(m, p.y), kz = vox_index(m, p.z);
    ulonglong2 got[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = l8 + 8 * u;
        got[u] = make_ulonglong2(KEY_EMPTY, 0ull);
        if (c < 27) {
            const int x = kx + (c / 9 - 1), y = ky + ((c / 3) % 3 - 1), z = kz + (c % 3 - 1);
            if (key_in_range(x, y, z)) got[u] = load_slot(slot_at(m, slot_of(pack_key(x, y, z), m.shift)));
        }
    }
    double bd2 = 1.7976931348623157e308;
    int bc = 0x7FFFFFFF, br = 0x7FFFFFFF, bslot = -1, ncand = 0, own = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        const int c = l8 + 8 * u;
        ulonglong2 v = got[u];
        if (c < 27 && v.x != KEY_EMPTY) {
            const unsigned long long want = pack_key(kx + (c / 9 - 1), ky + ((c / 3) % 3 - 1), kz + (c % 3 - 1));
            unsigned int s = slot_of(want, m.shift);
            while (v.x != want && v.x != KEY_EMPTY) { s = (s + 1) & m.mask; v = load_slot(slot_at(m, s)); }
            if (v.x == want) {
                if (c == 13) own = 1;
                const int count = meta_count(v.y);
                const double *bx = voxel_rows(m, s), *by = bx + m.capp, *bz = by + m.capp;
                for (int k = 0; k < count; ++k) {   // cells and ranks are visited in increasing order: strict '<' keeps the first minimum
                    const double d = sqnorm3(p.x - ldm(bx + k), p.y - ldm(by + k), p.z - ldm(bz + k));
                    if (d < bd2) { bd2 = d; bc = c; br = k; bslot = (int)s; }
                }
                ncand += count;
            }
        }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(gmask, bd2, o);
        const int oc = __shfl_xor_sync(gmask, bc, o), orr = __shfl_xor_sync(gmask, br, o), os = __shfl_xor_sync(gmask, bslot, o);
        ncand += __shfl_xor_sync(gmask, ncand, o);
        own |= __shfl_xor_sync(gmask, own, o);
        if (od < bd2 || (od == bd2 && (oc < bc || (oc == bc && orr < br)))) { bd2 = od; bc = oc; br = orr; bslot = os; }
    }
    slot_out = bslot; count_out = ncand; own_out = own; d2_out = bd2; rank_out = bslot >= 0 ? br : -1;
}

// ---- opt-in point-to-plane residual LIMU_ICP_PLANE (SURVEY section 8f N2; no counterpart in the reference) -----------------
// Plane of a correspondence = plane of the matched point's VOXEL: with c >= 5 stored points, mean mu and scatter
// S = sum (p-mu)(p-mu)^T, the normal is the eigenvector of S's smallest eigenvalue by 5 cyclic Jacobi sweeps (only + - * /
// sqrt in a fixed order, compiled without FMA: bit-identical to the C oracle's voxel_normal). Planar when
// l_min <= 0.04 l_mid; otherwise (or with < 5 points) the correspondence is dropped. Returns 1 and the normal if planar.
constexpr int PLANE_MIN_POINTS = 5;
constexpr double PLANE_RATIO = 0.04;
__device__ __forceinline__ int voxel_normal(const MapView &m, int slot, int c, double *nrm) {
    if (c < PLANE_MIN_POINTS) return 0;
    const double *bx = voxel_rows(m, (unsigned int)slot), *by = bx + m.capp, *bz = by + m.capp;
    double mx = 0.0, my = 0.0, mz = 0.0;
    for (int r = 0; r < c; ++r) { mx += ldm(bx + r); my += ldm(by + r); mz += ldm(bz + r); }
    mx /= (double)c; my /= (double)c; mz /= (double)c;
    double a00 = 0.0, a01 = 0.0, a02 = 0.0, a11 = 0.0, a12 = 0.0, a22 = 0.0;
    for (int r = 0; r < c; ++r) {
        const double dx = ldm(bx + r) - mx, dy = ldm(by + r) - my, dz = ldm(bz + r) - mz;
        a00 += dx * dx; a01 += dx * dy; a02 += dx * dz; a11 += dy * dy; a12 += dy * dz; a22 += dz * dz;
    }
    double v00 = 1.0, v01 = 0.0, v02 = 0.0, v10 = 0.0, v11 = 1.0, v12 = 0.0, v20 = 0.0, v21 = 0.0, v22 = 1.0;
    // One Jacobi rotation in the (p,q) plane; o is the third index. App/Aqq/Apq: the pivot block; Aop/Aoq: the other two entries;
    // Vxp/Vxq: the eigenvector columns p and q.
#define LIMU_JACOBI(App, Aqq, Apq, Aop, Aoq, V0p, V0q, V1p, V1q, V2p, V2q)                                   \
    if (Apq != 0.0) {                                                                                       \
        const double theta = (Aqq - App) / (2.0 * Apq);                                                     \
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));           \
        const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;                                             \
        const double app = App, aqq = Aqq, aop = Aop, aoq = Aoq;                                            \
        App = app - t * Apq; Aqq = aqq + t * Apq; Apq = 0.0;                                                \
        Aop = cs * aop - sn * aoq; Aoq = sn * aop + cs * aoq;                                               \
        double vp, vq;                                                                                      \
        vp = V0p; vq = V0q; V0p = cs * vp - sn * vq; V0q = sn * vp + cs * vq;                               \
        vp = V1p; vq = V1q; V1p = cs * vp - sn * vq; V1q = sn * vp + cs * vq;                               \
        vp = V2p; vq = V2q; V2p = cs * vp - sn * vq; V2q = sn * vp + cs * vq;                               \
    }
#pragma unroll 1
    for (int sweep = 0; sweep < 5; ++sweep) {
        LIMU_JACOBI(a00, a11, a01, a02, a12, v00, v01, v10, v11, v20, v21)   // (p,q) = (0,1), o = 2: A[2][0], A[2][1]
        LIMU_JACOBI(a00, a22, a02, a01, a12, v00, v02, v10, v12, v20, v22)   // (0,2), o = 1: A[1][0], A[1][2]
        LIMU_JACOBI(a11, a22, a12, a01, a02, v01, v02, v11, v12, v21, v22)   // (1,2), o = 0: A[0][1], A[0][2]
    }
#undef LIMU_JACOBI
    int lo = 0;
    double l_lo = a00;
    if (a11 < l_lo) { lo = 1; l_lo = a11; }
    if (a22 < l_lo) { lo = 2; l_lo = a22; }
    const double l1 = lo == 0 ? a11 : (lo == 1 ? a22 : a00), l2 = lo == 0 ? a22 : (lo == 1 ? a00 : a11);
    const double mid = l1 < l2 ? l1 : l2;
    if (!(mid > 0.0) || !(l_lo <= PLANE_RATIO * mid)) return 0;
    nrm[0] = lo == 0 ? v00 : (lo == 1 ? v01 : v02);
    nrm[1] = lo == 0 ? v10 : (lo == 1 ? v11 : v12);
    nrm[2] = lo == 0 ? v20 : (lo == 1 ? v21 : v22);
    return 1;
}

// ---- insertion / eviction, one element per call (used by the stand-alone kernels and the fused frame kernel) -------
// Pass 1 of insert_points (voxel_hash_map.cpp:12-62) for input point `i` of the batch:
//   - voxel key (get_vox_index), claim-or-find its slot (64-bit CAS on the packed key),
//   - meta = min(meta, (base + i) << 13): a fresh slot (meta all-ones) becomes {birth = first input index that named
//     the voxel, count 0}; an existing voxel's meta is smaller and stays untouched,
//   - sorted insertion of i into the voxel's pending list pend[slot*cap + count .. slot*cap + cap): each position keeps
//     the minimum it has seen and passes the loser on (atomicMin chain), so when the pass ends the list holds the
//     (cap - count) smallest input indices in ascending order -- exactly the points a serial "append until full" loop
//     (voxel_block.cpp:68-73) would have kept. Returns the slot (PEND_NONE on failure).
__device__ __forceinline__ unsigned int insert_claim_one(const MapView &m, const V3 &p, unsigned int i, unsigned long long birth_base, DevStatus *st, bool *claimed) {
    const int kx = vox_index(m, p.x), ky = vox_index(m, p.y), kz = vox_index(m, p.z);
    unsigned int slot = PEND_NONE;
    if (!key_in_range(kx, ky, kz)) { st->key_range = 1; return slot; }   // (NaN gives INT_MIN: out of range)
    const unsigned long long key = pack_key(kx, ky, kz);
    unsigned int s = slot_of(key, m.shift);
    for (unsigned int probes = 0; probes <= m.mask; ++probes) {
        unsigned long long cur = __ldcg(&slot_at(m, (unsigned int)s)->key);
        if (cur == KEY_EMPTY) {
            cur = atomicCAS(&slot_at(m, (unsigned int)s)->key, KEY_EMPTY, key);
            if (cur == KEY_EMPTY) { *claimed = true; cur = key; }
        }
        if (cur == key) { slot = s; break; }
        s = (s + 1) & m.mask;
    }
    if (slot == PEND_NONE) { st->table_full = 1; return slot; }
    const unsigned long long mine = (birth_base + (unsigned long long)i) << META_COUNT_BITS;
    const unsigned long long old = atomicMin(&slot_at(m, (unsigned int)slot)->meta, mine);
    const int count = meta_count(old < mine ? old : mine);   // only pass 2 changes counts
    unsigned int x = i;
    unsigned int *list = m.pend + (size_t)slot * m.cap;
    for (int r = count; r < m.cap; ++r) {
        const unsigned int prev = atomicMin(&list[r], x);
        if (prev == PEND_NONE) break;
        if (prev > x) x = prev;
    }
    return slot;
}
// warp-aggregated occupancy accounting + append of the new voxels' slots to the dense live list (call with the whole
// warp converged; `slot` is what insert_claim_one returned)
__device__ __forceinline__ void insert_account(bool claimed, unsigned int slot, unsigned long long *counters, const MapView &m) {
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, claimed);
    if (!bal) return;   // warp-uniform
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) {
        atomicAdd(&counters[0], (unsigned long long)__popc(bal));          // live voxels
        base = atomicAdd(&counters[3], (unsigned long long)__popc(bal));   // used slots (live + tombstones) = length of the live list
    }
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (claimed) {
        const unsigned long long at = base + (unsigned long long)__popc(bal & ((1u << lane) - 1u));
        m.live[at] = slot;
        m.live_key[at] = __ldcg(&slot_at(m, slot)->key);   // (this thread's own compare-and-swap put it there)
    }
}
// Pass 2: the point looks for its own index in its voxel's pending list; position r IS its storage rank (the list
// started at the old count). Winners store their coordinates and clear the entry.
__device__ __forceinline__ void insert_place_one(const MapView &m, const V3 &p, unsigned int i, unsigned int slot) {
    if (slot == PEND_NONE) return;
    unsigned int *list = m.pend + (size_t)slot * m.cap;
    for (int r = 0; r < m.cap; ++r) {
        if (__ldcg(list + r) == i) {
            double *d = voxel_rows(m, slot);
            d[r] = p.x; d[m.capp + r] = p.y; d[2 * m.capp + r] = p.z;
            list[r] = PEND_NONE;
            atomicAdd(&slot_at(m, (unsigned int)slot)->meta, 1ull);
            break;
        }
    }
}
// remove_points_from_far (voxel_hash_map.cpp:146-171) as it executes under null locks, for slot s: voxels whose INDEX
// distance^2 to the origin voxel exceeds max_distance^2 (units as written, :148,:160) drop their points farther than
// max_distance metres from origin, order preserved (voxel_block.cpp:107-118); empty voxels are erased (tombstoned).
// the voxel test of :160 on a packed key (origin voxel ovx/ovy/ovz). Vector3i::squaredNorm() is int arithmetic: the difference and
// the sum of squares wrap modulo 2^32, so a voxel ~46 341 or more indices away can pass for a near one and survive. Reproduced on
// purpose (map contents stay bit-exact with the reference), in unsigned arithmetic so that the wrap is defined behaviour.
__device__ __forceinline__ bool voxel_is_far(unsigned long long key, int ovx, int ovy, int ovz, double max_sq) {
    int x, y, z;
    unpack_key(key, x, y, z);
    const unsigned dx = (unsigned)x - (unsigned)ovx, dy = (unsigned)y - (unsigned)ovy, dz = (unsigned)z - (unsigned)ovz;
    const int d2 = (int)(dx * dx + dy * dy + dz * dz);
    return (double)d2 > max_sq;
}
// returns true when the voxel was erased
__device__ __forceinline__ bool remove_far_one(const MapView &m, int64_t s, double ox, double oy, double oz, double max_distance, unsigned long long *counters) {
    const unsigned long long key = slot_at(m, (unsigned int)s)->key;
    if (key >= KEY_TOMB) return false;
    const double max_sq = max_distance * max_distance;
    if (!voxel_is_far(key, vox_index(m, ox), vox_index(m, oy), vox_index(m, oz), max_sq)) return false;
    double *px = voxel_rows(m, (unsigned int)s), *py = px + m.capp, *pz = py + m.capp;
    const unsigned long long meta = slot_at(m, (unsigned int)s)->meta;
    const int count = meta_count(meta);
    int w = 0;
    for (int r = 0; r < count; ++r) {
        const double ax = px[r], ay = py[r], az = pz[r];
        if (!(sqnorm3(ax - ox, ay - oy, az - oz) > max_sq)) {
            if (w != r) { px[w] = ax; py[w] = ay; pz[w] = az; }
            ++w;
        }
    }
    if (w != count) slot_at(m, (unsigned int)s)->meta = (meta & ~META_COUNT_MASK) | (unsigned long long)w;
    if (w == 0) {
        slot_at(m, (unsigned int)s)->key = KEY_TOMB;
        slot_at(m, (unsigned int)s)->meta = META_NONE;
        atomicAdd(&counters[0], ~0ull);  // --live
        atomicAdd(&counters[1], 1ull);   // ++tombstones
        return true;
    }
    return false;
}
// entry i of the dense live list: its key decides (one coalesced 8-byte word); only a far voxel's block is touched
__device__ __forceinline__ void remove_far_entry(const MapView &m, int64_t i, unsigned long long key, int ovx, int ovy, int ovz, double ox, double oy, double oz,
                                                 double max_distance, unsigned long long *counters) {
    if (key >= KEY_TOMB || !voxel_is_far(key, ovx, ovy, ovz, max_distance * max_distance)) return;
    if (remove_far_one(m, (int64_t)__ldcg(m.live + i), ox, oy, oz, max_distance, counters)) m.live_key[i] = KEY_TOMB;
}

}  // namespace limu

// Host-side object behind the C handle.
struct limu_map {
    limu_ctx *ctx = nullptr;
    double vox_size = 1.0, max_distance = 100.0;
    int cap = 10;
    int64_t capacity = 0;          // C (slots), power of two
    limu::DevBuf blk, pend, live;
    limu::DevBuf counters;         // device: [0] n_live voxels, [1] n_tomb, [2] n_points, [3] n_used (live + tomb)
    uint64_t birth_base = 0;       // creation sequence offset of the next insert batch
    int64_t used_upper = 0;        // host upper bound on live + tomb slots
    cudaEvent_t readers_done = nullptr;   // set by an odometry handle that reads this map from another stream: entry points that change the map wait for it (not owned)
    uint64_t mutations = 0;        // bumped by every entry point of the C ABI that changes the map's contents (odometry.cu: a loop that ran ahead on an older map is dropped)
    limu::DevBuf pslot;            // per-point slot scratch of the current insert batch
    limu::DevBuf world;            // transformed copy for update(points, pose)
    limu::MapView view() const;
};

namespace limu {
int map_alloc(limu_map *m, int64_t capacity_slots);
int map_insert_device(limu_map *m, const double *xyz_dev, int64_t n, const int *n_dev /* optional device count */);
int map_remove_far_device(limu_map *m, const double *origin_dev3);
int map_maybe_grow(limu_map *m, int64_t incoming);
inline int map_wait_readers(limu_map *m) {
    if (m->readers_done) LIMU_CUDA_TRY(cudaStreamWaitEvent(m->ctx->stream, m->readers_done, 0));
    return LIMU_OK;
}
}  // namespace limu
