"""The polygon-mesh generator of tests/polygon_mesh.py (no device needed): merged plans keep make_plan's conventions,
conserve volume, area and continuity, reach the ELL widths 8 and 12 the GPU tests are written for, and keep a uniform
concentration uniform on steady flow through the oracle."""
import numpy as np
import pytest

from clearwater_riverine_b200 import synthetic
from oracle import reference_step as ref
from tests.polygon_mesh import ell_width, merge_cells, merged_count, row_lengths


def _base():
    return synthetic.make_plan(40, 30, 6, tri_fraction=0.15, dry_fraction=0.02, seed=12)


MERGES = {"w8": dict(sizes=(2, 3), n_groups=110, seed=1), "w12": dict(sizes=(2, 4), n_groups=90, seed=2),
          "w8_interior": dict(sizes=(2, 3), n_groups=90, seed=3, interior_only=True)}


def _continuity(plan):
    """Per cell and step: |V[t+1] - V[t] + dt * net outflow[t]| / V[t+1] over the wet real cells."""
    n = plan.n_real
    internal = plan.f2 < n
    dt = np.diff(plan.time_seconds)
    worst = 0.0
    for t in range(plan.n_time - 1):
        q = plan.face_flow[t].astype(np.float64)
        out = np.bincount(plan.f1, q, n) - np.bincount(plan.f2[internal], q[internal], n)
        v0, v1 = plan.volume[t, :n].astype(np.float64), plan.volume[t + 1, :n].astype(np.float64)
        wet = v1 > 0
        worst = max(worst, float(np.max(np.abs(v1 - v0 + dt[t] * out)[wet] / v1[wet])))
    return worst


@pytest.mark.parametrize("name", list(MERGES))
def test_merged_plan_keeps_the_generators_conventions(name):
    plan = _base()
    kw = MERGES[name]
    m = merge_cells(plan, **kw)
    n, nn, F = plan.n_real, m.n_real, plan.n_face
    assert nn == merged_count(plan, kw["sizes"], kw["n_groups"])
    assert m.n_face == nn + (F - n) and m.n_time == plan.n_time
    # f1 real, max(f1) == n - 1, ghosts n..F-1 one per ghost edge in their old order, ghost centres unchanged
    assert m.f1.max() == nn - 1 and m.f1.min() >= 0
    g_old, g_new = plan.f2 >= n, m.f2 >= nn
    assert np.array_equal(m.f2[g_new], np.arange(nn, m.n_face))
    assert g_new.sum() == g_old.sum()
    assert np.array_equal(m.face_x[nn:], plan.face_x[n:]) and np.array_equal(m.face_y[nn:], plan.face_y[n:])
    assert np.array_equal(m.volume[:, nn:], plan.volume[:, n:])
    # the old cell -> new cell map, read off the kept ghost edges and the edges that survived
    old_of_ghost = plan.f1[g_old]
    new_of_ghost = m.f1[g_new]
    assert np.array_equal(m.face_flow[:, g_new], plan.face_flow[:, g_old])      # flow > 0 still leaves f1 on ghost edges
    # internal edges: kept ones carry their flow and velocity (one may be flipped with both signs negated)
    a, b = m.f1[~g_new], m.f2[~g_new]
    assert np.all(a != b), "an edge inside a group survived"
    assert np.all(b < nn)
    # every kept internal edge appears in the old plan with the same |flow| series
    assert np.abs(m.face_flow[:, ~g_new]).sum() <= np.abs(plan.face_flow[:, ~g_old]).sum()
    assert np.all((m.face_flow == 0) | (np.sign(m.face_flow) == np.sign(m.edge_velocity)))
    # dry cells are never merged: they keep a zero volume and their count
    assert len(m.dry_cells) == len(plan.dry_cells)
    assert np.all(m.volume[:, m.dry_cells] == 0)
    assert np.sum(np.all(m.volume[:, :nn] == 0, axis=0)) == len(plan.dry_cells)
    # volume and plan area conserved
    v_old, v_new = plan.volume[:, :n].astype(np.float64).sum(1), m.volume[:, :nn].astype(np.float64).sum(1)
    assert np.all(np.abs(v_new - v_old) <= 1e-6 * v_old)
    assert abs(m.cell_area[:nn].sum() - plan.cell_area[:n].sum()) <= 1e-12 * plan.cell_area[:n].sum()
    assert np.all((m.face_x[:nn] >= plan.face_x[:n].min()) & (m.face_x[:nn] <= plan.face_x[:n].max()))
    # per-cell continuity as good as the unmerged plan's (f32 rounding of the summed volumes)
    assert _continuity(m) <= max(2.0 * _continuity(plan), 2e-7), (_continuity(m), _continuity(plan))
    # boundary lines: the same ghost edges, renumbered
    for key, faces in plan.boundary_faces.items():
        got = m.boundary_faces[key]
        assert len(got) == len(faces) and np.all(m.f2[got] >= nn)
        assert np.array_equal(m.f2[got] - nn, plan.f2[faces] - n)
        assert np.array_equal(m.face_flow[:, got], plan.face_flow[:, faces])
    # groups of merged cells: a merged cell is the union of the old cells on its ghost edges (where it has any)
    pairs = set(zip(old_of_ghost.tolist(), new_of_ghost.tolist()))
    assert len({o for o, _ in pairs}) == len(pairs), "an old cell split over two new cells"
    # no two faces between the same pair of cells
    lo, hi = np.minimum(a, b), np.maximum(a, b)
    assert len(np.unique(lo.astype(np.int64) * nn + hi)) == len(lo)
    # the degree the merge is for
    deg = row_lengths(m)
    if name == "w12":
        assert deg.max() == 10 and ell_width(m) == 12
    else:
        assert deg.max() == 8 and ell_width(m) == 8
    if kw.get("interior_only"):
        # a cell with a ghost edge kept its own volume: it was merged with nothing
        assert np.array_equal(m.volume[:, new_of_ghost], plan.volume[:, old_of_ghost]), "a cell with a ghost edge was merged"
        assert np.array_equal(m.cell_area[new_of_ghost], plan.cell_area[old_of_ghost])


def test_parallel_faces_only_when_asked():
    """Two pairs side by side share two faces: refused by default, kept with allow_parallel."""
    plan = _base()
    counts = {}
    for allow in (False, True):
        m = merge_cells(plan, 2, 300, seed=5, allow_parallel=allow)
        internal = m.f2 < m.n_real
        a, b = m.f1[internal].astype(np.int64), m.f2[internal].astype(np.int64)
        key = np.minimum(a, b) * m.n_real + np.maximum(a, b)
        counts[allow] = len(key) - len(np.unique(key))
    assert counts[False] == 0 and counts[True] > 0, counts


def test_merge_is_seeded_and_refuses_what_does_not_fit():
    plan = _base()
    m1, m2 = merge_cells(plan, (2, 3), 80, seed=9), merge_cells(plan, (2, 3), 80, seed=9)
    assert np.array_equal(m1.f1, m2.f1) and np.array_equal(m1.volume, m2.volume)
    with pytest.raises(ValueError):
        merge_cells(plan, 4, plan.n_real // 3, seed=9)


def test_uniform_concentration_is_preserved_on_interior_merges():
    """IC == BC == 100 on steady flow: the oracle keeps c == 100 on the merged plan (groups away from the boundary) as
    closely as on the plan it was merged from -- the merged volumes keep continuity to f32 rounding."""
    plan = synthetic.make_plan(40, 30, 8, tri_fraction=0.15, seed=9, unsteady=0.0, tidal=0.0)
    dev = {}
    for name, p in (("plain", plan), ("merged", merge_cells(plan, (2, 3), 150, seed=4, interior_only=True))):
        assert name == "plain" or ell_width(p) == 8
        adv, _, _, cdiff, dt = ref.derive_coefficients(p.face_flow, p.edge_velocity, p.face_x, p.face_y, p.f1, p.f2, 0.1,
                                                       p.time_seconds)
        mesh = ref.HydroMesh(p.f1, p.f2, p.n_face, adv, cdiff, p.edge_velocity, p.volume, dt, 0.1)
        n = p.n_real
        inp = np.zeros((p.n_time, p.n_face)); inp[0, :n] = 100.0; inp[:, n:] = 100.0
        oracle = ref.OracleRiverine(mesh, {"c": inp})
        for _ in range(p.n_time - 1):
            oracle.update()
        dev[name] = float(np.abs(oracle.constituent_dict["c"].concentration[-1][:n] - 100.0).max())
    assert dev["merged"] <= max(2.0 * dev["plain"], 1e-5), dev
