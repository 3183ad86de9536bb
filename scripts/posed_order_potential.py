"""How much of the culled search's work a per-frame row order of the POSED cloud could save, on a skinned cloud dumped by
a real fit (bench.py --dump-outputs DIR writes DIR/skinned.npy; scripts/gpu_posed_order.py --dump DIR writes
skinned_headline.npy / skinned_late.npy).

The observed frames are regenerated from the benchmark's seed.  Rows are grouped into 256-point blocks (one warp of the
search) and targets into 32-point k-d leaves, as in RelaxationEngine(search="auto").  A (row block, target chunk) pair
must be evaluated iff the squared gap between the two boxes does not exceed the largest exact nearest-neighbour distance
of the block's rows or of the chunk's targets: the floor of any bound scheme (the engine's bounds are within ~1.3x of it,
profiles/r02_culling.md).  Printed per row grouping, the mean fraction over all frames:
    canonical k-d   one k-d order of the canonical cloud, shared by every frame (the engine today)
    posed STR       per frame, sort-tile-recursive on the skinned cloud as csrc/order.cu builds it: along the frame's
                    longest axis into slabs of 2048, each slab along the second axis into pieces of 512, each piece
                    along the third into leaves of 256 (8 x 4 x 2 at 16 384 points), on quantised coordinates
    posed k-d       per frame, a k-d order of the skinned cloud with 256-point leaves

    python scripts/posed_order_potential.py DIR/skinned.npy [more.npy ...] [--frames 64]
"""
import argparse
import os
import sys

import numpy as np
from scipy.spatial import cKDTree

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from reart_b200.synth import make_sequence                                               # noqa: E402
from scripts.culling_potential import kd_order                                           # noqa: E402

ROWS, COLS = 256, 32


def str_order(p):
    """csrc/order.cu in numpy: axes by decreasing extent (lower axis first on equal extents); per level the rows ordered by
    (segment, quantised coordinate, caller index) and cut into runs of 2048 / 512 / 256 from the front; every leaf in
    ascending caller index."""
    p = p.astype(np.float32)
    lo = p.min(0)
    ext = p.max(0) - lo
    axes = sorted(range(3), key=lambda a: (-ext[a], a))
    n = len(p)
    idx = np.arange(n)
    seg = np.zeros(n, np.int64)
    order = idx
    for a, cells, size in zip(axes, (4096, 512, 128), (2048, 512, 256)):
        e = ext[a]
        scale = np.float32(cells) / e if 0 < e < np.inf else np.float32(0)
        v = (p[:, a] - lo[a]) * np.float32(scale)
        q = np.where(v > 0, np.minimum(np.float32(cells - 1), np.floor(v)), 0).astype(np.int64)
        order = np.lexsort((idx, seg * cells + q))
        seg[order] = np.arange(n) // size
    return np.concatenate([np.sort(order[s:s + 256]) for s in range(0, n, 256)])


def evaluated_fraction(src, tgt, tgt_tree):
    """src [N,3] in the row grouping, tgt [M,3] in the target grouping: fraction of block pairs an exact bound keeps."""
    n, m = len(src) // ROWS * ROWS, len(tgt) // COLS * COLS
    sb, gb = src[:n].reshape(-1, ROWS, 3), tgt[:m].reshape(-1, COLS, 3)
    gap = np.maximum(0, np.maximum(sb.min(1)[:, None] - gb.max(1)[None], gb.min(1)[None] - sb.max(1)[:, None]))
    gap = (gap * gap).sum(-1)
    rows = (tgt_tree.query(src[:n])[0] ** 2).reshape(-1, ROWS).max(1)
    cols = (cKDTree(src).query(tgt[:m])[0] ** 2).reshape(-1, COLS).max(1)
    return float(((gap <= rows[:, None]) | (gap <= cols[None, :])).mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("skinned", nargs="+", help=".npy [T,N,3] skinned clouds in caller order")
    ap.add_argument("--frames", type=int, default=0, help="evaluate only the first F frames (0: all)")
    ap.add_argument("--parts", type=int, default=15)
    args = ap.parse_args()
    cache = {}
    for path in args.skinned:
        sk = np.load(path).astype(np.float32)
        T, N, _ = sk.shape
        if (T, N) not in cache:
            seq = make_sequence(T=T, N=N, P=args.parts, seed=2)
            cache[(T, N)] = (seq["cano"], seq["frames"])
        cano, frames = cache[(T, N)]
        canon = kd_order(cano, ROWS)
        nf = T if args.frames <= 0 else min(T, args.frames)
        res = {"canonical k-d": [], "posed STR": [], "posed k-d": []}
        for t in range(nf):
            g = frames[t][kd_order(frames[t], COLS)]
            tree = cKDTree(g)
            s = sk[t]
            res["canonical k-d"].append(evaluated_fraction(s[canon], g, tree))
            res["posed STR"].append(evaluated_fraction(s[str_order(s)], g, tree))
            res["posed k-d"].append(evaluated_fraction(s[kd_order(s, ROWS)], g, tree))
        base = np.mean(res["canonical k-d"])
        print(f"{path}: T={T} N={N}, {nf} frames")
        for k, v in res.items():
            print(f"  {k:14s} {np.mean(v):.3f}  (min {np.min(v):.3f}, max {np.max(v):.3f})  x{np.mean(v) / base:.2f} of canonical")


if __name__ == "__main__":
    main()
