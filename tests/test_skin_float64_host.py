"""CPU side of the skinning tests (tests/test_skin_float64_gpu.py): the launchers' variant selection mirrored in Python and
shown to be covered by the GPU test's parameter lists, the workspace offsets the GPU test reads the x-sorted copy from,
and the numpy reference of that copy on a hand-built block.  Needs the library built, no GPU."""
import numpy as np
import pytest

SMS = 148


def cdiv(a, b):
    return -(-a // b)


def rup(a, b):
    return cdiv(a, b) * b


# ------------------------------------------------------------------------------------------------ variant selection
def skin_fwd_fpb(T, N):
    """csrc/skin.cu launch_skin_fwd (no packed copy: n_pad = N):
    while (fpb > 1 && ceil_div(n_pad, kSkinThreads) * ceil_div(T, fpb) < 2 * 148) fpb /= 2;"""
    fpb = 8
    while fpb > 1 and cdiv(N, 128) * cdiv(T, fpb) < 2 * SMS:
        fpb //= 2
    return fpb


def skin_fwd_sorted_fpb(T, N):
    """csrc/skin.cu launch_skin_fwd_sorted, n_pad = round_up(N, 256) (capi.cu energy_pipeline):
    while (fpb > 1 && (n_pad / kSortBlock) * ceil_div(T, fpb) < 2 * 148) fpb /= 2;   fpb == 8: skin_fwd_sorted8_kernel"""
    fpb = 8
    while fpb > 1 and (rup(N, 256) // 256) * cdiv(T, fpb) < 2 * SMS:
        fpb //= 2
    return fpb


def skin_bwd_groups(T, N):
    """csrc/skin.cu skin_bwd_groups: while (chunks * groups < 3 * 148 && groups * 2 <= ntiles) groups *= 2;"""
    chunks, ntiles = cdiv(N, 128), cdiv(T, 8)
    g = 1
    while chunks * g < 3 * SMS and g * 2 <= ntiles:
        g *= 2
    return g


def tiles_per_group(T, N):
    """csrc/skin.cu launch_skin_bwd_p: tiles_per_group = ceil_div(ceil_div(T, kBwdFrames), groups)"""
    return cdiv(cdiv(T, 8), skin_bwd_groups(T, N))


def group_frames(T, N, g):
    """frames [lo, hi) of frame group g (empty when the group owns no tile): skin_bwd_fused_kernel's tile_lo / tile_hi"""
    tpg = tiles_per_group(T, N)
    lo, hi = g * tpg, min(g * tpg + tpg, cdiv(T, 8))
    return (8 * lo, min(T, 8 * hi)) if lo < hi else (0, 0)


def pmax(P):
    """csrc/skin.cu launch_skin_bwd: P <= 8 -> <8>, P <= 16 -> <16>, else <32> (P > 32: REART_ERR_UNSUPPORTED)"""
    return 8 if P <= 8 else 16 if P <= 16 else 32


# ------------------------------------------------------------------------------------------------ parameter lists
# weight classes: onehot (one non-zero, 1 +- a few ulps), two (exactly two non-zeros), dense (softmax rows),
# sparse (exact zeros, 0..P non-zeros per row, a few negative weights); scale multiplies coordinates and translations.
# (T, N, P, weights, scale) of the float64 forward test of reart_skin_fwd
FWD_SHAPES = [
    (64, 16384, 8, "onehot", 1.0),         # fpb 8
    (20, 8192, 9, "two", 1.0),             # fpb 4
    (20, 4096, 16, "dense", 1.0),          # fpb 2
    (3, 3001, 17, "sparse", 1.0),          # fpb 1
    (9, 129, 32, "dense", 1.0),
    (5, 1000, 1, "dense", 1.0),
    (7, 2000, 32, "sparse", 1024.0),       # the bound is relative
]
# (T, N, P, weights) of the producer test: skinned cloud and x-sorted copy of every producer, energy gradients
PRODUCER_SHAPES = [
    (64, 16384, 8, "onehot"),              # sorted8 (cfg3_16k), posed at its largest cloud
    (41, 16384, 16, "two"),                # sorted8, the last CTA row holds 1 frame
    (20, 16384, 32, "dense"),              # fpb 4
    (20, 8192, 9, "sparse"),               # fpb 2
    (3, 3001, 17, "onehot"),               # fpb 1
    (20, 8192, 4, "lattice"),              # fpb 2 on an integer lattice: many equal x in every block
    (64, 16384, 3, "lattice"),             # sorted8 on the lattice
    (2, 1, 1, "lattice"),
    (2, 255, 4, "lattice"),
    (3, 256, 2, "lattice"),
    (3, 257, 5, "lattice"),
]
# (T, N, P, weights, scale) of the float64 backward test of reart_skin_bwd
BWD_SHAPES = [
    (1, 5, 1, "onehot", 1.0),              # 1 group
    (9, 4096, 8, "two", 1.0),              # 2 groups
    (64, 16384, 9, "dense", 1.0),          # 4 groups
    (64, 1000, 16, "sparse", 1.0),         # 8 groups
    (200, 300, 17, "onehot", 1.0),         # 16 groups of 2 tiles: groups 13-15 own no tile
    (33, 127, 8, "two", 1.0),              # 4 groups of 2 tiles: group 3 owns no tile
    (7, 129, 32, "dense", 1.0),
    (15, 255, 32, "sparse", 1.0),
    (8, 2000, 16, "dense", 1024.0),
]
# raw clouds of reart_chamfer_bidir_fwd (pack_cloud_sorted_kernel), with explicit -0.0 / +0.0 x values
RAW_N = [1, 255, 256, 257, 1000]

P_EDGES = {1, 8, 9, 16, 17, 32}


def test_every_variant_is_covered():
    assert {skin_fwd_fpb(T, N) for T, N, *_ in FWD_SHAPES} == {1, 2, 4, 8}
    assert {skin_fwd_sorted_fpb(T, N) for T, N, *_ in PRODUCER_SHAPES} == {1, 2, 4, 8}
    assert any(skin_fwd_sorted_fpb(T, N) == 8 and T % 8 == 1 for T, N, *_ in PRODUCER_SHAPES)
    # the worked examples
    assert skin_fwd_sorted_fpb(64, 16384) == 8 and skin_fwd_sorted_fpb(41, 16384) == 8
    assert skin_fwd_sorted_fpb(20, 16384) == 4 and skin_fwd_sorted_fpb(20, 8192) == 2 and skin_fwd_sorted_fpb(3, 3001) == 1
    assert [skin_bwd_groups(T, N) for T, N in ((1, 5), (9, 4096), (64, 16384), (64, 1000), (200, 300))] == [1, 2, 4, 8, 16]
    assert tiles_per_group(200, 300) == 2
    assert [group_frames(200, 300, g) for g in (12, 13, 14, 15)] == [(192, 200), (0, 0), (0, 0), (0, 0)]
    assert {skin_bwd_groups(T, N) for T, N, *_ in BWD_SHAPES} >= {1, 2, 4, 8, 16}
    assert any(group_frames(T, N, skin_bwd_groups(T, N) - 1) == (0, 0) for T, N, *_ in BWD_SHAPES)
    assert {pmax(P) for _, _, P, *_ in BWD_SHAPES} == {8, 16, 32}
    assert {P for _, _, P, *_ in BWD_SHAPES} >= P_EDGES
    assert {P for _, _, P, *_ in FWD_SHAPES} | {P for _, _, P, _ in PRODUCER_SHAPES} >= P_EDGES
    assert {N % 128 for _, N, *_ in BWD_SHAPES} >= {0, 1, 127}
    assert {T % 8 for T, *_ in BWD_SHAPES} >= {0, 1, 7}
    assert {N for _, N, *_ in PRODUCER_SHAPES} >= {1, 255, 256, 257} and set(RAW_N) >= {1, 255, 256, 257}
    assert any(N % 256 and N > 256 for _, N, *_ in PRODUCER_SHAPES)
    weights = {w for *_, w, _ in FWD_SHAPES} | {w for *_, w in PRODUCER_SHAPES} | {w for *_, w, _ in BWD_SHAPES}
    assert weights >= {"onehot", "two", "dense", "sparse"}
    assert any(s != 1.0 for *_, s in FWD_SHAPES) and any(s != 1.0 for *_, s in BWD_SHAPES)


# ------------------------------------------------------------------------------------------------ workspace layout
def carve(sizes):
    """csrc/capi.cu Carver: every piece rounded up to 256 bytes from the workspace base -> byte offsets"""
    off, out = 0, []
    for nbytes in sizes:
        out.append(off)
        off += rup(nbytes, 256)
    return out, off


def energy_sorted_copy_layout(T, N, M):
    """(psrc, perm, xq) byte offsets in the workspace of the energy entries (capi.cu energy_pipeline):
    psrc = take<float>(T * n_pad_sorted * 3); ka = take<u64>(T * N); kb = take<u64>(T * M);
    gs only when g_skinned is null (the tests pass g_skinned); perm = take<uchar>(T * n_pad_sorted); xq = take<float>(xq_floats)"""
    n_pad = rup(N, 256)
    offs, end = carve([T * n_pad * 12, T * N * 8, T * M * 8, T * n_pad, T * (n_pad // 256) * 16 * 4])
    return dict(psrc=offs[0], perm=offs[3], xq=offs[4], end=end, n_pad=n_pad)


def chamfer_sorted_copy_layout(B, N, M):
    """(psrc, perm, xq) byte offsets in the workspace of reart_chamfer_bidir_fwd (capi.cu):
    psrc = take<float>(B * n_pad_sorted * 3); ptgt = take<float>(B * packed_floats_per_batch(M)); kf = take<u64>(B * N);
    kb = take<u64>(B * M); perm = take<uchar>(B * n_pad_sorted); xq = take<float>(xq_floats)"""
    n_pad = rup(N, 256)
    m_pad = rup(max(M, 1), 32)
    offs, end = carve([B * n_pad * 12, B * m_pad * 12, B * N * 8, B * M * 8, B * n_pad, B * (n_pad // 256) * 16 * 4])
    return dict(psrc=offs[0], perm=offs[4], xq=offs[5], end=end, n_pad=n_pad)


PRODUCER_M = 1024                          # targets of the energy calls


def test_workspace_mirrors_fit_inside_the_workspace_sizes():
    from reart_b200 import _lib
    L = _lib.lib()
    for T, N, *_ in PRODUCER_SHAPES:
        lay = energy_sorted_copy_layout(T, N, PRODUCER_M)
        assert lay["end"] <= L.reart_energy_workspace_bytes(T, N, PRODUCER_M), (T, N)
    for N in RAW_N:
        for B, M in ((2, 300), (1, N)):
            lay = chamfer_sorted_copy_layout(B, N, M)
            assert lay["end"] <= L.reart_chamfer_workspace_bytes(B, N, M), (B, N, M)


# ------------------------------------------------------------------------------------------------ sorted-copy reference
def orderable_bits(x):
    """common.cuh orderable_bits: u ^ (u >> 31 ? 0xffffffff : 0x80000000) -- -0.0 sorts before +0.0"""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return u ^ np.where(u >> 31, np.uint32(0xffffffff), np.uint32(0x80000000)).astype(np.uint32)


def sorted_blocks(rows, n_pad):
    """rows [T,N,3] float32 in the order the producer was given them -> (packed [T, n_pad * 3] float32, perm [T, n_pad] uint8,
    xq [T, n_pad / 256, 16] float32): per 256-row block sorted by (orderable_bits(x), offset in block), +INF padding,
    laid out [x0..x255 | (y,z) x 256] (common.cuh sorted_block_store), xq[k] = x at sorted position 16k + 15."""
    rows = np.asarray(rows, dtype=np.float32)
    T, N, _ = rows.shape
    pad = np.full((T, n_pad, 3), np.inf, dtype=np.float32)
    pad[:, :N] = rows
    nblk = n_pad // 256
    blk = pad.reshape(T, nblk, 256, 3)
    key = (orderable_bits(blk[..., 0]).astype(np.uint64) << np.uint64(32)) | np.arange(256, dtype=np.uint64)
    src = np.argsort(key, axis=-1)
    s = np.take_along_axis(blk, src[..., None], axis=2)                       # [T, nblk, 256, 3]
    packed = np.concatenate([s[..., 0], s[..., 1:].reshape(T, nblk, 512)], axis=-1).reshape(T, n_pad * 3)
    xq = s[..., 15::16, 0]
    return packed, src.astype(np.uint8).reshape(T, n_pad), np.ascontiguousarray(xq)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def test_sorted_blocks_on_a_hand_built_block():
    """One frame, 300 rows (two blocks, the second holding 44 rows and 212 padding rows): signed zeros, exact ties and
    padding land where the contract puts them."""
    rng = np.random.default_rng(0)
    rows = rng.integers(-3, 4, (1, 300, 3)).astype(np.float32)
    rows[0, :, 0] = np.float32(5.0)
    rows[0, 7, 0], rows[0, 3, 0] = np.float32(0.0), np.float32(-0.0)           # +0 at offset 7 BEFORE -0 at offset 3 ...
    rows[0, 11, 0], rows[0, 2, 0] = np.float32(-0.0), np.float32(0.0)
    rows[0, 100, 0] = rows[0, 50, 0] = np.float32(-1.0)                        # an exact tie: offset order
    rows[0, 260, 0] = np.float32(-np.inf)
    packed, perm, xq = sorted_blocks(rows, 512)
    x0 = packed[0, :256]
    # -1, -1 (offsets 50, 100), then -0.0 (3, 11), then +0.0 (2, 7), then the 5s in offset order
    assert list(perm[0, :6]) == [50, 100, 3, 11, 2, 7]
    assert list(bits(x0[2:6])) == [0x80000000, 0x80000000, 0, 0]
    assert np.all(x0[6:] == 5.0) and np.all(np.diff(perm[0, 6:256].astype(int)) > 0)
    # float sorting would tie -0.0 with +0.0 and keep them in offset order (2, 3, 7, 11)
    assert list(np.argsort(rows[0, :256, 0], kind="stable")[2:6]) == [2, 3, 7, 11]
    # (y, z) follow their x
    yz = packed[0, 256:768].reshape(256, 2)
    assert np.array_equal(yz, rows[0, perm[0, :256].astype(int), 1:])
    # second block: -inf first, 43 x = 5 rows, then 212 padding rows at +INF in x, y and z, in offset order
    b1 = packed[0, 768:1536]
    assert perm[0, 256] == 4 and b1[0] == -np.inf
    assert np.all(b1[1:44] == 5.0) and np.all(np.isinf(b1[44:256])) and np.all(b1[44:256] > 0)
    assert np.array_equal(perm[0, 256 + 44:].astype(int), np.arange(44, 256))
    assert np.all(np.isposinf(b1[256:].reshape(256, 2)[44:]))
    # the quantile index: x at sorted positions 15, 31, ..., 255
    assert np.array_equal(bits(xq[0, 0]), bits(x0[15::16])) and xq[0, 0, 0] == 5.0
    assert xq[0, 1, 1] == 5.0 and np.all(np.isposinf(xq[0, 1, 2:]))
