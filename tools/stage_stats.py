"""How full are the (128-row tile, kernel offset) stages of k_conv_tc on the bench workload?  CPU only (numpy).

Motivation (DESIGN.md §7): a stage whose 128 output rows have no neighbour through offset k could be skipped; a row
order that clusters tracks could make stages either empty or dense.  This script counts, for the synthetic dune3d
batch bench.py uses, the live rows of every stage at every resolution level, for three row orders.

  python tools/stage_stats.py [events]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sparseeventid_b200 import data_transforms as T  # noqa: E402
from sparseeventid_b200 import synthetic as S  # noqa: E402


def pack(c):
    return (c[:, 3] << 48) | (c[:, 0] << 32) | (c[:, 1] << 16) | c[:, 2]


def spread3(x):
    x = x.astype(np.uint64) & np.uint64(0x1FFFFF)
    for s, m in ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3),
                 (2, 0x1249249249249249)):
        x = (x | (x << np.uint64(s))) & np.uint64(m)
    return x


def morton(c):
    return ((spread3(c[:, 0]) << np.uint64(2)) | (spread3(c[:, 1]) << np.uint64(1)) | spread3(c[:, 2])
            | (c[:, 3].astype(np.uint64) << np.uint64(58)))


def stage_counts(coords, tile=128):
    """live rows per (tile, offset) of the 3x3x3 submanifold rulebook of `coords` taken in the given row order"""
    n = coords.shape[0]
    keys = pack(coords)
    order = np.argsort(keys)
    skeys = keys[order]
    cnt = np.zeros(((n + tile - 1) // tile, 27), np.int64)
    k = 0
    for dx in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dz in (-1, 0, 1):
                q = coords.copy()
                q[:, 0] += dx; q[:, 1] += dy; q[:, 2] += dz
                ok = (q[:, :3] >= 0).all(1)
                qk = pack(q)
                pos = np.clip(np.searchsorted(skeys, qk), 0, n - 1)
                live = ok & (skeys[pos] == qk)
                np.add.at(cnt[:, k], np.nonzero(live)[0] // tile, 1)
                k += 1
    return cnt


def report(name, coords):
    cnt = stage_counts(coords)
    nz = cnt > 0
    print(f"  {name:26s} P/N {cnt.sum() / coords.shape[0]:5.2f}  stages {cnt.size:6d}  empty {1 - nz.mean():6.3f}  "
          f"live rows per non-empty stage: mean {cnt[nz].mean():5.1f}  <=8 rows {np.mean(cnt[nz] <= 8):.2f}  "
          f">=64 rows {np.mean(cnt[nz] >= 64):.2f}")


def main():
    events = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    coords, _, _ = T.larcvsparse_to_scnsparse_3d(S.larcv_batch_3d(events, seed=1234))
    coords = coords.astype(np.int64)
    _, first = np.unique(pack(coords), return_index=True)
    active = coords[np.sort(first)]                      # InputLayer order: first appearance
    for level in range(6):
        print(f"level {level}: {active.shape[0]} sites")
        report("first appearance (SCN)", active)
        report("sorted by (b,x,y,z) key", active[np.argsort(pack(active), kind="stable")])
        report("Morton order", active[np.argsort(morton(active), kind="stable")])
        coarse = active.copy()
        coarse[:, :3] //= 2
        _, first = np.unique(pack(coarse), return_index=True)
        active = coarse[np.sort(first)]                  # first appearance = what scn_strided_rulebook_hash produces


if __name__ == "__main__":
    main()
