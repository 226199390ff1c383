"""Polygon meshes for the tests: groups of adjacent real cells of a synthetic.make_plan plan merged into single cells.

HEC-RAS 2D meshes away from refinement regions are made of polygons with up to eight faces, so a real plan gives rows of
five to eight internal neighbours (ELL width W = 8); make_plan's quads and triangles never have more than four (W = 4).
Merging two quads gives a cell of 6 faces, three in an L or a line 8, four in a strip 10 (W = 12).  The merge keeps the
generator's conventions (see synthetic.py): real cells 0..n-1, ghosts n..F-1 in their old order, f1 always real with
max(f1) == n-1, flow > 0 leaves f1, dry cells never merged.  A merged cell holds the summed volume (fp64, rounded to f32),
plan area and the area-weighted centre; the edges inside a group are dropped and every other edge keeps its flow and
velocity, so continuity holds to f32 rounding.
"""
from __future__ import annotations

from dataclasses import replace
from typing import Sequence, Union

import numpy as np
import scipy.sparse as sp

from clearwater_riverine_b200.synthetic import SyntheticPlan, make_plan


def _neighbour_table(a: np.ndarray, b: np.ndarray, n: int) -> np.ndarray:
    """(n, D) neighbour ids of every real cell over the internal edges (a, b), padded with -1."""
    src = np.concatenate([a, b]); dst = np.concatenate([b, a])
    order = np.argsort(src, kind="stable")
    src, dst = src[order], dst[order]
    deg = np.bincount(src, minlength=n)
    ptr = np.concatenate([[0], np.cumsum(deg)])
    slot = np.arange(len(src)) - ptr[src]
    table = np.full((n, max(1, int(deg.max()))), -1, np.int64)
    table[src, slot] = dst
    return table


def _walk(nbr: np.ndarray, free: np.ndarray, seeds: np.ndarray, length: np.ndarray, rng) -> np.ndarray:
    """Self-avoiding random walks over free cells from `seeds`: (G, max length) members, -1 where a walk got stuck."""
    G, L = len(seeds), int(length.max())
    members = np.full((G, L), -1, np.int64)
    members[:, 0] = seeds
    tip = seeds.copy()
    alive = np.ones(G, bool)
    rows = np.arange(G)
    for j in range(1, L):
        cand = nbr[tip]
        valid = (cand >= 0) & free[np.maximum(cand, 0)]
        for i in range(j):
            valid &= cand != members[:, i:i + 1]
        r = np.where(valid, rng.random(cand.shape), -1.0)
        pick = cand[rows, r.argmax(1)]
        need = length > j
        grow = need & valid.any(1)
        alive &= ~need | grow
        members[grow, j] = pick[grow]
        tip = np.where(grow, pick, tip)
    members[~alive] = -1
    return members


def _parallel_pairs(label: np.ndarray, a: np.ndarray, b: np.ndarray):
    """Label pairs joined by more than one internal edge: (low label, high label) arrays."""
    la, lb = label[a], label[b]
    keep = la != lb
    lo, hi = np.minimum(la[keep], lb[keep]), np.maximum(la[keep], lb[keep])
    key = lo * (int(label.max()) + 1) + hi
    uk, cnt = np.unique(key, return_counts=True)
    dup = uk[cnt > 1]
    return dup // (int(label.max()) + 1), dup % (int(label.max()) + 1)


def group_sizes(sizes: Union[int, Sequence[int]], n_groups: int) -> np.ndarray:
    """The size of each of the n_groups groups: `sizes` taken in turn."""
    sizes = np.atleast_1d(np.asarray(sizes, np.int64))
    return sizes[np.arange(n_groups) % len(sizes)]


def merged_count(plan: SyntheticPlan, sizes, n_groups: int) -> int:
    """Real cells left after merge_cells(plan, sizes, n_groups): every group of s cells removes s - 1."""
    return plan.n_real - int((group_sizes(sizes, n_groups) - 1).sum())


def merge_cells(plan: SyntheticPlan, sizes: Union[int, Sequence[int]], n_groups: int, *, seed: int,
                interior_only: bool = False, allow_parallel: bool = False, max_rounds: int = 60) -> SyntheticPlan:
    """Merge n_groups groups of adjacent real cells into single polygon cells.  The i-th group has sizes[i % len(sizes)]
    cells (a self-avoiding walk: lines, Ls and zigzags), so the merged plan has exactly merged_count(...) real cells.
    Dry cells are never merged; interior_only keeps cells with a ghost edge out too.  Unless allow_parallel, a group
    that would put two faces between the same pair of cells is refused: no cell or group outside it may touch it through
    more than one face.  Groups are drawn in vectorised rounds; ValueError if n_groups cannot be placed."""
    rng = np.random.default_rng(seed)
    n, F = plan.n_real, plan.n_face
    f1 = plan.f1.astype(np.int64); f2 = plan.f2.astype(np.int64)
    internal = f2 < n
    a, b = f1[internal], f2[internal]
    nbr = _neighbour_table(a, b, n)
    eligible = np.ones(n, bool)
    eligible[plan.dry_cells] = False
    if interior_only:
        eligible[f1[~internal]] = False
    want = group_sizes(sizes, n_groups)
    need = {int(s): int((want == s).sum()) for s in np.unique(want)}
    if min(need) < 1:
        raise ValueError("group sizes must be >= 1")

    group_of = np.full(n, -1, np.int64)          # accepted group id per cell
    gsize = []                                   # size of each accepted group id (dissolved: 0)
    for _ in range(max_rounds):
        left = {s: c - sum(1 for g in gsize if g == s) for s, c in need.items()}
        todo = sum(left.values())
        if todo == 0:
            break
        free = eligible & (group_of < 0)
        pool = np.nonzero(free)[0]
        m = min(len(pool), 3 * todo + 64)
        if m == 0:
            break
        seeds = rng.choice(pool, size=m, replace=False)
        length = rng.choice(np.repeat(list(left), list(left.values())), size=m)
        members = _walk(nbr, free, seeds, length, rng)
        members = members[members[:, 0] >= 0]
        length = (members >= 0).sum(1)
        # candidates claiming the same cell: the first one (random order) keeps it
        cells = members.ravel()
        cand = np.repeat(np.arange(len(members)), members.shape[1])
        on = cells >= 0
        claim = np.full(n, len(members), np.int64)
        np.minimum.at(claim, cells[on], cand[on])
        ok = np.ones(len(members), bool)
        np.logical_and.at(ok, cand[on], claim[cells[on]] == cand[on])
        members, length = members[ok], length[ok]
        # keep only as many of each size as are still wanted
        keep = np.zeros(len(members), bool)
        for s, c in left.items():
            idx = np.nonzero(length == s)[0][:c]
            keep[idx] = True
        members, length = members[keep], length[keep]
        g0 = len(gsize)
        on = members >= 0
        group_of[members[on]] = g0 + np.nonzero(on)[0]
        gsize.extend(int(s) for s in length)
        if not allow_parallel:
            while True:                          # dissolve the newer group of every pair joined by two faces
                label = np.where(group_of >= 0, n + group_of, np.arange(n))
                lo, hi = _parallel_pairs(label, a, b)
                if len(hi) == 0:
                    break
                bad = np.unique(hi) - n          # hi is a group: the newer of two groups, or the group beside a cell
                assert np.all(bad >= g0)
                for g in bad:
                    gsize[g] = 0
                group_of[np.isin(group_of, bad)] = -1
    if sorted(g for g in gsize if g) != sorted(int(s) for s in want):
        raise ValueError(f"could not place {n_groups} groups of sizes {sorted(need)}")

    # new ids: groups and single cells ordered by their lowest old id
    rep = np.arange(n)
    grouped = group_of >= 0
    first = np.full(len(gsize), n, np.int64)
    np.minimum.at(first, group_of[grouped], np.nonzero(grouped)[0])
    rep[grouped] = first[group_of[grouped]]
    reps, new = np.unique(rep, return_inverse=True)
    nn = len(reps)
    ng = F - n
    keep_e = ~internal
    keep_e[internal] = new[a] != new[b]
    g1 = new[f1[keep_e]]
    g2 = np.where(f2[keep_e] < n, new[np.minimum(f2[keep_e], n - 1)], f2[keep_e] - n + nn)
    flow = plan.face_flow[:, keep_e].copy()
    vel = plan.edge_velocity[:, keep_e].copy()
    if g1.max() != nn - 1:                       # the reference defines nreal = max(f1): flip one edge onto cell n-1
        e = np.nonzero(g2 == nn - 1)[0][0]
        g1[e], g2[e] = g2[e], g1[e]
        flow[:, e] = -flow[:, e]
        vel[:, e] = -vel[:, e]
        vel[:, e][vel[:, e] == 0] = 0.0
    S = sp.csr_matrix((np.ones(n), (new, np.arange(n))), shape=(nn, n))
    volume = np.empty((plan.n_time, nn + ng), np.float32)
    volume[:, :nn] = (S @ plan.volume[:, :n].astype(np.float64).T).T.astype(np.float32)
    volume[:, nn:] = plan.volume[:, n:]
    area = plan.cell_area
    cell_area = np.concatenate([S @ area[:n], area[n:]])
    face_x = np.concatenate([(S @ (area[:n] * plan.face_x[:n])) / cell_area[:nn], plan.face_x[n:]])
    face_y = np.concatenate([(S @ (area[:n] * plan.face_y[:n])) / cell_area[:nn], plan.face_y[n:]])
    edge_id = np.cumsum(keep_e) - 1
    bfaces = {name: edge_id[faces] for name, faces in plan.boundary_faces.items()}
    return replace(plan, f1=g1.astype(np.int32), f2=g2.astype(np.int32), face_x=face_x, face_y=face_y,
                   face_flow=flow, edge_velocity=vel, volume=volume, n_real=nn, boundary_faces=bfaces,
                   dry_cells=np.sort(new[plan.dry_cells]), cell_area=cell_area)


def row_lengths(plan: SyntheticPlan) -> np.ndarray:
    """Internal neighbours of every real cell (the length of its matrix row without the diagonal)."""
    n = plan.n_real
    internal = plan.f2 < n
    return np.bincount(plan.f1[internal], minlength=n) + np.bincount(plan.f2[internal], minlength=n)


def ell_width(plan: SyntheticPlan) -> int:
    """The ELL width build_topology gives the plan: max(4, ceil(max row length / 4) * 4)."""
    return max(4, -(-int(row_lengths(plan).max()) // 4) * 4)


def polygon_plan(n_target: int, n_time: int, *, seed: int, sizes=(2, 3), n_groups: int = 0, **kw) -> SyntheticPlan:
    """A merged make_plan plan with exactly n_target real cells: the unmerged plan is sized (n_exact) so that n_groups
    groups of `sizes` (default about one group per ten cells) bring it to n_target."""
    n_groups = n_groups or max(4, n_target // 10)
    drop = int((group_sizes(sizes, n_groups) - 1).sum())
    n0 = n_target + drop
    nq = int(np.ceil(n0 / 1.15))
    ny = max(4, int(round(np.sqrt(nq / 1.5))))
    nx = -(-nq // ny)
    kw.setdefault("dry_fraction", 0.02)
    plan = make_plan(nx, ny, n_time, seed=seed, n_exact=n0, **kw)
    out = merge_cells(plan, sizes, n_groups, seed=seed)
    assert out.n_real == n_target
    return out
