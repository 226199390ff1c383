"""Host-side cell ordering (no device needed): reverse Cuthill-McKee + the flow-aligned multicolouring of the
Gauss-Seidel sweeps (csrc/cwr_topology.cpp through cwr_order_cells)."""
import numpy as np
import pytest

from clearwater_riverine_b200 import synthetic
from clearwater_riverine_b200.backend import order_cells
from tests.polygon_mesh import merge_cells, row_lengths


def colours_of(new_of_old, color_ptr):
    return np.searchsorted(color_ptr, new_of_old, side="right") - 1


def _quads():
    return synthetic.make_plan(37, 23, 6, tri_fraction=0.2, dry_fraction=0.02, seed=3)


def _polygons(sizes, n_groups):
    """The quad plan with groups of cells merged into polygons: rows of up to 8 (sizes 2, 3) or 10 (with 4) neighbours."""
    return lambda: merge_cells(_quads(), sizes, n_groups, seed=3)


_ORDER_CASES = [(_quads, nc, h) for nc, h in [(0, False), (5, False), (8, True), (16, True), (64, True)]]
_ORDER_IDS = [f"{nc}-{h}" for _, nc, h in _ORDER_CASES]
for _name, _factory in (("w8", _polygons((2, 3), 80)), ("w12", _polygons((2, 4), 70))):
    for _nc, _h in [(0, False), (5, False), (8, True), (16, True)]:
        _ORDER_CASES.append((_factory, _nc, _h))
        _ORDER_IDS.append(f"{_name}-{_nc}-{_h}")


@pytest.mark.parametrize("make_plan,n_colors,hinted", _ORDER_CASES, ids=_ORDER_IDS)
def test_order_is_a_permutation_and_colours_separate_neighbours(make_plan, n_colors, hinted):
    """Quad / triangle meshes and polygon meshes (ELL widths 8 and 12): a colour request below the largest degree + 1
    is raised to it."""
    plan = make_plan()
    n = plan.n_real
    hint = plan.face_flow.mean(0) if hinted else None
    p, cptr, n_levels = order_cells(plan.f1, plan.f2, plan.n_face, True, n_colors, hint)
    assert np.array_equal(np.sort(p), np.arange(n))
    assert cptr[0] == 0 and cptr[-1] == n and np.all(np.diff(cptr) >= 0)
    if n_colors == 0:
        assert len(cptr) == 2
        return
    assert len(cptr) - 1 >= max(min(n_colors, 64), int(row_lengths(plan).max()) + 1)
    col = colours_of(p, cptr)
    internal = plan.f2 < n
    assert np.all(col[plan.f1[internal]] != col[plan.f2[internal]]), "coupled rows share a colour"
    if hinted:
        assert n_levels > len(cptr) - 1


def test_hint_aligns_the_sweep_with_the_flow():
    """With the hint most of the flow crosses edges whose downstream cell comes later in the sweep order (edges
    that are weak next to their cells' strongest flow do not direct the colouring); without it about half does."""
    plan = synthetic.make_plan(60, 60, 6, tri_fraction=0.1, dry_fraction=0.02, seed=4, unsteady=0.0, tidal=0.0)
    n = plan.n_real
    q = plan.face_flow[2]
    internal = (plan.f2 < n) & (q != 0)
    a, b = plan.f1[internal], plan.f2[internal]
    up, down = np.where(q[internal] > 0, a, b), np.where(q[internal] > 0, b, a)
    frac = {}
    for hinted in (False, True):
        p, cptr, _ = order_cells(plan.f1, plan.f2, plan.n_face, True, 16, q if hinted else None)
        wq = np.abs(q[internal])
        frac[hinted] = float(np.sum(wq * (p[down] > p[up])) / np.sum(wq))       # flow-weighted
    assert 0.35 < frac[False] < 0.65
    assert frac[True] > 0.85, frac


def test_cyclic_flow_hint_terminates():
    """A hint with circulation (cycles in the flow graph) still yields a valid colouring."""
    plan = synthetic.make_plan(20, 20, 4, tri_fraction=0.3, seed=5)
    rng = np.random.default_rng(0)
    hint = rng.normal(size=plan.n_edge).astype(np.float32)          # random directions: cycles everywhere
    p, cptr, _ = order_cells(plan.f1, plan.f2, plan.n_face, True, 12, hint)
    col = colours_of(p, cptr)
    internal = plan.f2 < plan.n_real
    assert np.all(col[plan.f1[internal]] != col[plan.f2[internal]])


@pytest.mark.parametrize("n_parts", [2, 3, 8])
@pytest.mark.parametrize("n_colors", [0, 12])
def test_domain_decomposition_strips(n_parts, n_colors):
    """Rows are ordered (part, colour, ...): parts are equal contiguous row ranges, each part's colours tile
    its range, colours still separate coupled rows across parts, and only a thin layer of rows is read by
    other parts (strips across the flow / the RCM band)."""
    plan = synthetic.make_plan(64, 48, 6, tri_fraction=0.15, dry_fraction=0.02, seed=6)
    n = plan.n_real
    hint = plan.face_flow.mean(0)
    p, cptr, n_levels, part_ptr, n_send = order_cells(plan.f1, plan.f2, plan.n_face, True, n_colors, hint, n_parts)
    assert np.array_equal(np.sort(p), np.arange(n))
    assert part_ptr[0] == 0 and part_ptr[-1] == n
    sizes = np.diff(part_ptr)
    assert sizes.max() - sizes.min() <= 1
    part = np.searchsorted(part_ptr, p, side="right") - 1
    internal = plan.f2 < n
    a, b = plan.f1[internal], plan.f2[internal]
    cut = part[a] != part[b]
    # halo rows per part = rows with a neighbour in another part
    sent = np.zeros(n, bool); sent[a[cut]] = True; sent[b[cut]] = True
    assert np.array_equal(n_send, np.bincount(part[sent], minlength=n_parts))
    assert n_send.sum() < 0.35 * n            # thin strips boundaries (64 x 48 cells, up to 8 strips)
    if n_colors:
        assert cptr.shape == (n_parts, cptr.shape[1])
        for q in range(n_parts):
            assert cptr[q, 0] == part_ptr[q] and cptr[q, -1] == part_ptr[q + 1] and np.all(np.diff(cptr[q]) >= 0)
        colour = np.empty(n, np.int64)
        for q in range(n_parts):
            rows = np.arange(part_ptr[q], part_ptr[q + 1])
            colour_of_row = np.searchsorted(cptr[q], rows, side="right") - 1
            inv = np.empty(n, np.int64)
            colour[np.isin(p, rows)] = colour_of_row[p[np.isin(p, rows)] - part_ptr[q]]
        assert np.all(colour[a] != colour[b]), "coupled rows share a colour"


def test_topology_does_not_depend_on_the_host_thread_count(monkeypatch):
    """build_topology runs its order-independent loops on host threads (meshes of >= 2^18 cells): rows, colours, strips and
    strip neighbours are identical with 1, 3 and 5 threads."""
    from clearwater_riverine_b200 import synthetic
    from clearwater_riverine_b200.backend import strip_layout
    plan = synthetic.make_plan(530, 520, 3, tri_fraction=0.1, dry_fraction=0.02, seed=4)
    assert plan.n_real >= 1 << 18
    hint = plan.face_flow.mean(0)
    outs = []
    for threads in ("1", "3", "5"):
        monkeypatch.setenv("CWR_TOPO_THREADS", threads)
        outs.append(strip_layout(plan.f1, plan.f2, plan.n_face, 12, hint, 37, 2, strip_cap=256))
    for other in outs[1:]:
        assert set(other) == set(outs[0])
        for key, val in outs[0].items():
            assert np.array_equal(np.asarray(val), np.asarray(other[key])), key
