"""Independent numpy restatements of the integer/index work of the path (test infrastructure). They run at BASELINE's full
sizes in well under a second, where a pass of the serial C oracle per property would be slow; tests/test_np_restatement.py
pins them against the C oracle on CPU, tests/test_full_size.py uses them to check the CUDA path at 128k / 512k / 1.5M points."""
import numpy as np

BIAS = 1 << 20


def np_keys(xyz, s):
    """utils::get_vox_index (calculation_helpers.cpp:142-147): IEEE division, truncation toward zero."""
    return np.trunc(xyz / s).astype(np.int64)


def np_vox_index_x86(xyz, s):
    """get_vox_index as the reference's x86-64 build executes it: (int)(p / v) is cvttsd2si, which gives INT_MIN where the
    quotient is NaN or its truncation leaves int32."""
    q = np.asarray(xyz, np.float64) / s
    ok = (q > -2147483649.0) & (q < 2147483648.0)
    return np.where(ok, np.trunc(np.where(ok, q, 0.0)), -2147483648.0).astype(np.int32)


def np_remove_far(keys, counts, pts, origin, vox, max_distance):
    """VoxelHashMap::remove_points_from_far (voxel_hash_map.cpp:146-171) on a dump (keys [V,3] int32, counts [V], pts): a voxel whose
    Vector3i::squaredNorm() distance to the origin's voxel exceeds max_distance^2 drops its points farther than max_distance from
    origin (order kept) and disappears when none is left. squaredNorm is int arithmetic: the subtraction and the sum of squares wrap
    modulo 2^32 (a voxel ~46 341 indices away can survive). -> the dump after the eviction."""
    ov = np_vox_index_x86(np.asarray(origin, np.float64).reshape(1, 3), vox)[0]
    d = keys.astype(np.uint32) - ov.astype(np.uint32)
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]).view(np.int32)
    max_sq = float(max_distance) * float(max_distance)
    far_voxel = d2.astype(np.float64) > max_sq
    owner = np.repeat(np.arange(len(keys)), counts)
    a = pts - np.asarray(origin, np.float64)
    far_point = ((a[:, 0] * a[:, 0] + a[:, 1] * a[:, 1]) + a[:, 2] * a[:, 2]) > max_sq
    keep = ~(far_voxel[owner] & far_point)
    new_counts = np.bincount(owner[keep], minlength=len(keys)).astype(np.int32)
    alive = new_counts > 0
    return keys[alive], new_counts[alive], pts[keep]


def np_pack(k):
    return ((k[:, 0] + BIAS) << 42) | ((k[:, 1] + BIAS) << 21) | (k[:, 2] + BIAS)


def np_first_per_voxel(xyz, s):
    """voxel_downsample (icp.cpp:9-30): indices of the first point of every voxel, in input order."""
    _, first = np.unique(np_pack(np_keys(xyz, s)), return_index=True)
    return np.sort(first)


def np_iqr(xyz):
    """KissICP::iqr_processing + outlier::IQR (icp.cpp:88-124, common.hpp:22-63)."""
    d2 = (xyz[:, 0] * xyz[:, 0] + xyz[:, 1] * xyz[:, 1]) + xyz[:, 2] * xyz[:, 2]
    n = len(d2)
    if n == 0:
        return xyz
    a = np.sort(d2)

    def med(v):
        m = len(v)
        return (v[m // 2 - 1] + v[m // 2]) / 2.0 if m % 2 == 0 else v[m // 2]
    if n == 1:
        q1, q3, iqr = 0.0, a[0], a[0]
    else:
        half = n // 2
        q1, q3 = med(a[:half]), med(a[half + n % 2:])
        iqr = q3 - q1
    lo, hi = q1 - 1.25 * iqr, q3 + 1.25 * iqr
    return xyz[(d2 >= lo) & (d2 <= hi)]


def np_map_insert(xyz, vox, cap):
    """VoxelHashMap::insert_points on an empty map (voxel_hash_map.cpp:12-62, voxel_block.cpp:68-73): voxels in creation order
    (= order of first occurrence), each holding its first `cap` points in input order. -> (keys [V,3], counts [V], pts)."""
    packed = np_pack(np_keys(xyz, vox))
    uniq, first, inverse = np.unique(packed, return_index=True, return_inverse=True)
    creation_rank = np.empty(len(uniq), np.int64)
    creation_rank[np.argsort(first, kind="stable")] = np.arange(len(uniq))   # voxel -> position in creation order
    vpos = creation_rank[inverse]                                            # creation position of every point's voxel
    order = np.lexsort((np.arange(len(xyz)), vpos))                          # by voxel (creation order), then input order
    sv = vpos[order]
    start = np.flatnonzero(np.r_[True, sv[1:] != sv[:-1]])
    sizes = np.diff(np.r_[start, len(sv)])
    rank = np.arange(len(sv)) - np.repeat(start, sizes)
    keep = order[rank < cap]
    keys = np_keys(xyz[np.sort(first)], vox).astype(np.int32)
    return keys, np.minimum(sizes, cap).astype(np.int32), xyz[keep]


def np_closest(keys, counts, pts, q, vox):
    """VoxelHashMap::get_closest_neighbour (voxel_hash_map.cpp:64-102) by brute force over a dump (creation order):
    (a) the query's own voxel exists -> the first minimum of (p - q).squaredNorm() over its stored points, in storage order;
    (b) else the occupied neighbour of the 27 cells with the largest (|delta|^2, creation position) -- the reference's max-heap
        top, a later-created voxel wins ties;
    (c) else (0,0,0). -> (points [n,3], voxel keys [n,3] int32 (INT_MIN where none), ranks [n] int32 (-1 where none))."""
    q = np.asarray(q, np.float64).reshape(-1, 3)
    n, nv = len(q), len(keys)
    packed = np_pack(keys.astype(np.int64))
    order = np.argsort(packed, kind="stable")
    spacked = packed[order]

    def find(k):   # creation position of the voxel with key k (rows), -1 where absent
        p = np_pack(k)
        i = np.minimum(np.searchsorted(spacked, p), max(nv - 1, 0))
        return np.where((nv > 0) & (spacked[i] == p), order[i], -1) if nv else np.full(len(k), -1)

    kq = np_keys(q, vox)
    pos = find(kq)
    best_d = np.where(pos >= 0, 4, -1)                       # own voxel: beats every neighbour
    for dx in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dz in (-1, 0, 1):
                if dx == dy == dz == 0:
                    continue
                c = find(kq + np.array([dx, dy, dz]))
                d = dx * dx + dy * dy + dz * dz
                better = (c >= 0) & ((d > best_d) | ((d == best_d) & (c > pos)))
                pos = np.where(better, c, pos)
                best_d = np.where(better, d, best_d)
    start = np.r_[0, np.cumsum(counts)].astype(np.int64)
    out, rank = np.zeros((n, 3)), np.full(n, -1, np.int32)
    key = np.full((n, 3), np.iinfo(np.int32).min, np.int32)
    for v in np.unique(pos[pos >= 0]):
        b = pts[start[v]:start[v + 1]]
        every = np.flatnonzero(pos == v)
        step = max(1, 1 << 20 >> max(len(b).bit_length(), 1))
        for at in range(0, len(every), step):
            sel = every[at:at + step]
            dd = q[sel, None, :] - b[None, :, :]
            d2 = (dd[..., 0] * dd[..., 0] + dd[..., 1] * dd[..., 1]) + dd[..., 2] * dd[..., 2]
            r = np.argmin(d2, axis=1)                          # first minimum in storage order
            out[sel], rank[sel], key[sel] = b[r], r, keys[v]
    return out, key, rank
