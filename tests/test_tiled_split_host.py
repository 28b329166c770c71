"""The split of one tiled canvas over ranks (fdsr_tiled_plan, include/fdsr.h): the library's partition and exchange plan
against a brute-force statement of the rule on the tile windows of tiled_oracle.tile_starts.  Host only: the plan
needs no context and no GPU."""
import numpy as np
import pytest

import tiled_oracle as TO
from fastdiffsr_b200 import Engine, FdsrError

SHAPES = [(1, 100, 140), (2, 61, 203)]   # neither H nor W a multiple of 8


def windows(B, H, W, tile, overlap):
    """(canvas, y0, x0) of every tile in global order, and the effective extents."""
    ys, tey, _ = TO.tile_starts(H, tile, overlap)
    xs, tex, _ = TO.tile_starts(W, tile, overlap)
    return np.array([(b, y, x) for b in range(B) for y in ys for x in xs]), tey, tex


def brute_plan(B, H, W, tile, overlap, world):
    """own[r] = (lo, hi); need[r][q] = sorted tiles of rank q whose windows intersect rank r's update region."""
    win, tey, tex = windows(B, H, W, tile, overlap)
    n = len(win)
    own = [(r * n // world, (r + 1) * n // world) for r in range(world)]
    b, y, x = win[:, 0], win[:, 1], win[:, 2]
    meets = ((b[:, None] == b[None, :]) & (np.abs(y[:, None] - y[None, :]) < tey)
             & (np.abs(x[:, None] - x[None, :]) < tex))
    need = [[None] * world for _ in range(world)]
    for r, (lo, hi) in enumerate(own):
        hit = meets[lo:hi].any(axis=0) if hi > lo else np.zeros(n, bool)
        for q, (qlo, qhi) in enumerate(own):
            need[r][q] = [] if q == r else [g for g in range(qlo, qhi) if hit[g]]
    return win, tey, tex, own, need


def as_range(tiles):
    return (tiles[0], tiles[-1] + 1) if tiles else (0, 0)


def update_mask(win, tey, tex, lo, hi, B, H, W):
    m = np.zeros((B, H, W), bool)
    for b, y, x in win[lo:hi]:
        m[b, y:y + tey, x:x + tex] = True
    return m


@pytest.mark.parametrize("overlap", [0, 16, 48])
@pytest.mark.parametrize("tile", [32, 64])
@pytest.mark.parametrize("B,H,W", SHAPES)
def test_plan_matches_rule(B, H, W, tile, overlap):
    win, tey, tex, _, _ = brute_plan(B, H, W, tile, overlap, 1)
    n = len(win)
    for world in range(1, 10):
        _, _, _, own, need = brute_plan(B, H, W, tile, overlap, world)
        plans = [Engine.tiled_plan(B, H, W, tile, overlap, world, r) for r in range(world)]
        covered = np.zeros(n, int)
        for r, p in enumerate(plans):
            assert p["n_tiles"] == n and p["te"] == (tey, tex)
            assert p["own"] == own[r], (world, r)
            covered[p["own"][0]:p["own"][1]] += 1
            for q in range(world):
                assert p["recv"][q] == as_range(need[r][q]), (world, r, q)
                assert p["recv"][q] == plans[q]["send"][r], (world, r, q)
                lo, hi = p["send"][q]
                assert hi == lo == 0 or p["own"][0] <= lo < hi <= p["own"][1], (world, r, q)   # only own slots leave
        assert (covered == 1).all(), world                                                   # the ranges partition
        # every tile that covers a pixel of U_r is owned or received by r
        owner = np.zeros((B, H, W), int) - 1
        for g in range(n - 1, -1, -1):                                 # the first covering tile in global order wins
            b, y, x = win[g]
            owner[b, y:y + tey, x:x + tex] = g
        pix_rank = np.zeros((B, H, W), int) - 1
        for r, p in enumerate(plans):
            lo, hi = p["own"]
            u = update_mask(win, tey, tex, lo, hi, B, H, W)
            avail = np.zeros(n, bool)
            avail[lo:hi] = True
            for rlo, rhi in p["recv"]:
                avail[rlo:rhi] = True
            for g in np.flatnonzero(~avail):
                b, y, x = win[g]
                assert not u[b, y:y + tey, x:x + tex].any(), (world, r, g)
            mine = (owner >= lo) & (owner < hi)
            assert not (mine & ~u).any()                                 # a rank writes only pixels it updates
            assert (pix_rank[mine] == -1).all()
            pix_rank[mine] = r
        assert (pix_rank >= 0).all()                                     # pixel owners partition the canvas


def test_heavy_overlap_needs_non_adjacent_ranks():
    """tile 64, overlap 48 (stride 16): a pixel lies under four tile rows, so a rank receives from ranks that are not
    its neighbours."""
    B, H, W, world = 1, 100, 140, 9
    far = [(r, q) for r in range(world) for q, (lo, hi) in enumerate(Engine.tiled_plan(B, H, W, 64, 48, world, r)["recv"])
           if hi > lo and abs(q - r) > 1]
    assert far


def test_more_ranks_than_tiles():
    plans = [Engine.tiled_plan(1, 64, 64, 64, 16, 3, r) for r in range(3)]
    assert [p["own"] for p in plans] == [(0, 0), (0, 0), (0, 1)]
    assert all(lo == hi == 0 for p in plans for lo, hi in p["send"] + p["recv"])


@pytest.mark.parametrize("world,rank", [(0, 0), (-1, 0), (2, 2), (2, -1), (3, 5)])
def test_bad_world_and_rank(world, rank):
    with pytest.raises(FdsrError, match="world|rank"):
        Engine.tiled_plan(1, 100, 140, 64, 16, world, rank)


def test_bad_arguments_and_capacity():
    import ctypes as C
    from fastdiffsr_b200 import _lib
    for args, msg in [((1, 100, 140, 60, 16), "multiples of 8"), ((0, 100, 140, 64, 16), "B must be"),
                      ((1, 7, 140, 64, 16), ">= 8"), ((1, 100, 140, 64, -1), "overlap")]:
        with pytest.raises(FdsrError, match=msg):
            Engine.tiled_plan(*args, 2, 0)
    lib = _lib.load()
    buf = (C.c_int64 * 12)()
    assert lib.fdsr_tiled_plan(1, 100, 140, 64, 64, 16, 2, 0, buf, 12) == -1          # 5 + 4 * 2 = 13 entries needed
    assert "cap" in lib.fdsr_global_error().decode()
    big = (C.c_int64 * 13)()
    assert lib.fdsr_tiled_plan(1, 100, 140, 64, 64, 16, 2, 0, big, 13) == 13
    assert lib.fdsr_tiled_plan(1, 100, 140, 64, 64, 16, 2, 0, None, 13) == -1
