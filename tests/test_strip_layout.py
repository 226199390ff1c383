"""Host-side layout of the neighbour-synchronised Gauss-Seidel sweep kernel (precond_sync = 2; no device needed):
rows ordered (part, strip, colour, RCM position), one strip per CTA, and a numpy emulation of the kernel's
synchronisation rule -- "a strip starts step k once every strip it is coupled to has finished step k - 1" -- under
random legal interleavings, which must reproduce the sequential colour-by-colour sweep exactly."""
import numpy as np
import pytest
import scipy.sparse as sp

from clearwater_riverine_b200 import synthetic
from clearwater_riverine_b200.backend import strip_layout
from tests.polygon_mesh import merge_cells, row_lengths


def _plan(seed=3):
    return synthetic.make_plan(37, 29, 6, tri_fraction=0.2, dry_fraction=0.02, seed=seed)


def _polygons(sizes, n_groups):
    """_plan() with groups of cells merged into polygons: rows of up to 8 (sizes 2, 3) or 10 (with 4) neighbours."""
    return lambda: merge_cells(_plan(), sizes, n_groups, seed=4)


_STRIP_CASES = [(_plan, *c) for c in [(1, 1, 8), (1, 7, 8), (1, 24, 12), (2, 5, 9), (4, 3, 8)]]
_STRIP_IDS = ["-".join(map(str, c[1:])) for c in _STRIP_CASES]
for _name, _factory in (("w8", _polygons((2, 3), 90)), ("w12", _polygons((2, 4), 80))):
    for _c in [(1, 7, 8), (1, 24, 5), (2, 5, 9), (4, 3, 8)]:
        _STRIP_CASES.append((_factory, *_c))
        _STRIP_IDS.append(_name + "-" + "-".join(map(str, _c)))


@pytest.mark.parametrize("make_plan,n_parts,n_strips,n_colors", _STRIP_CASES, ids=_STRIP_IDS)
def test_strips_partition_the_rows_and_list_their_neighbours(make_plan, n_parts, n_strips, n_colors):
    """Quad / triangle meshes and polygon meshes (ELL widths 8 and 12; colour requests below the largest degree + 1 are
    raised to it)."""
    plan = make_plan()
    n = plan.n_real
    L = strip_layout(plan.f1, plan.f2, plan.n_face, n_colors, plan.face_flow.mean(0), n_strips, n_parts)
    p, cptr, nc = L["new_of_old"], L["strip_cptr"], L["n_colors"]
    NS = n_parts * n_strips
    assert nc >= max(n_colors, int(row_lengths(plan).max()) + 1)
    assert np.array_equal(np.sort(p), np.arange(n))
    # strips tile [0, n) contiguously, colours tile every strip, strips have equal sizes (+-1 per part)
    assert cptr[0, 0] == 0 and cptr[-1, -1] == n
    assert np.all(cptr[1:, 0] == cptr[:-1, -1]) and np.all(np.diff(cptr, axis=1) >= 0)
    sizes = cptr[:, -1] - cptr[:, 0]
    assert sizes.max() - sizes.min() <= 2
    # the colour of a row, from its position, equals color_of and separates coupled rows
    strip_of = np.searchsorted(cptr[:, 0], np.arange(n), side="right") - 1
    col_pos = np.array([np.searchsorted(cptr[strip_of[i]], i, side="right") - 1 for i in range(n)])
    assert np.array_equal(col_pos, L["color_of"])
    internal = plan.f2 < n
    a, b = p[plan.f1[internal]], p[plan.f2[internal]]
    assert np.all(col_pos[a] != col_pos[b])
    # neighbour lists: symmetric, global strip ids (strips of other parts included: the sweep kernel synchronises with
    # them through flag mirrors in peer memory), and complete for every internal edge
    nptr, nbr = L["strip_nptr"], L["strip_nbr"]
    pairs = {(s, int(q)) for s in range(NS) for q in nbr[nptr[s]:nptr[s + 1]]}
    assert all((q, s) in pairs for (s, q) in pairs)
    assert all(s != q for (s, q) in pairs)
    sa, sb = strip_of[a], strip_of[b]
    cross = sa != sb
    assert {(int(x), int(y)) for x, y in zip(sa[cross], sb[cross])} <= pairs
    if n_parts > 1:
        assert any(s // n_strips != q // n_strips for (s, q) in pairs), "the parts are coupled through their boundary strips"
    assert len(pairs) == 2 * len({(min(x, y), max(x, y)) for x, y in zip(sa[cross].tolist(), sb[cross].tolist())})


def test_neighbour_synchronised_schedule_equals_the_sequential_sweep():
    plan = _plan(seed=5)
    n = plan.n_real
    n_strips, n_sweeps = 9, 3
    L = strip_layout(plan.f1, plan.f2, plan.n_face, 8, plan.face_flow.mean(0), n_strips)
    p, cptr, nc, nptr, nbr = L["new_of_old"], L["strip_cptr"], L["n_colors"], L["strip_nptr"], L["strip_nbr"]
    rng = np.random.default_rng(0)
    internal = plan.f2 < n
    a, b = p[plan.f1[internal]], p[plan.f2[internal]]
    w = -rng.random(2 * len(a)) * 0.2
    Lo = sp.csr_matrix((w, (np.concatenate([a, b]), np.concatenate([b, a]))), shape=(n, n))     # off-diagonals of I + L
    u = rng.random(n)
    color_of = L["color_of"].astype(int)

    def relax(z, rows):
        z[rows] = u[rows] - Lo[rows] @ z

    # sequential reference: colour by colour over all strips
    zs = np.zeros(n)
    for s in range(n_sweeps):
        for c in range(nc):
            relax(zs, np.nonzero(color_of == c)[0])
    # random legal interleavings of the strips
    for trial in range(3):
        z = np.zeros(n)
        done = np.zeros(n_strips, int)               # steps finished per strip
        total = n_sweeps * nc
        while done.min() < total:
            ready = [s for s in range(n_strips) if done[s] < total and all(done[q] >= done[s] for q in nbr[nptr[s]:nptr[s + 1]])]
            assert ready, "deadlock"
            s = ready[rng.integers(len(ready))]
            c = done[s] % nc
            relax(z, np.arange(cptr[s, c], cptr[s, c + 1]))
            done[s] += 1
        assert np.array_equal(z, zs)


def test_strip_cap_moves_overflow_rows_to_legal_colours():
    """strip_cap: no (strip, colour) above the cap where a legal colour with room exists; colours still separate
    coupled rows; only rows of over-full colours move."""
    plan = synthetic.make_plan(120, 90, 6, tri_fraction=0.2, dry_fraction=0.02, seed=9)
    n = plan.n_real
    hint = plan.face_flow.mean(0)
    L0 = strip_layout(plan.f1, plan.f2, plan.n_face, 10, hint, 8)
    d0 = np.diff(L0["strip_cptr"], axis=1)
    cap = int(np.ceil(d0.sum(1).max() / 10 * 1.09))        # (a cap the strips cannot meet with 8 % to spare is relaxed)
    assert d0.max() > cap, "the case must have over-full colours"
    L = strip_layout(plan.f1, plan.f2, plan.n_face, 10, hint, 8, strip_cap=cap)
    d = np.diff(L["strip_cptr"], axis=1)
    assert d.max() <= cap and np.array_equal(d.sum(1), d0.sum(1))
    p, cptr = L["new_of_old"], L["strip_cptr"]
    assert np.array_equal(np.sort(p), np.arange(n))
    internal = plan.f2 < n
    col = L["color_of"].astype(int)
    a, b = p[plan.f1[internal]], p[plan.f2[internal]]
    assert np.all(col[a] != col[b])
    # rows that kept their colour: everything outside the over-full (strip, colour) pairs
    moved = (L["color_of"][p] != L0["color_of"][L0["new_of_old"]]).sum()
    assert 0 < moved <= np.maximum(d0 - cap, 0).sum()


@pytest.mark.parametrize("hinted", [False, True])
def test_whole_mesh_as_one_strip_balances_the_colours_for_the_on_chip_solver(hinted):
    """Without strips a cap makes the whole mesh the one strip (what create passes for meshes of <= 4096 cells): on the
    Ohio-shaped mesh every one of the 12 colours ends at <= 256 rows -- one pass of k_solve_chip's 256 threads -- with
    or without a flow hint (the unhinted greedy colouring starts at 1468 rows in its first colour); colours still
    separate coupled rows, and colour-major row ranges stay contiguous."""
    plan = synthetic.ohio_like(12, seed=2)
    n = plan.n_real
    hint = plan.face_flow.mean(0) if hinted else None
    L0 = strip_layout(plan.f1, plan.f2, plan.n_face, 12, hint, 0)
    L = strip_layout(plan.f1, plan.f2, plan.n_face, 12, hint, 0, strip_cap=256)
    assert L["n_colors"] == 12
    cnt0 = np.bincount(L0["color_of"], minlength=12)
    cnt = np.bincount(L["color_of"], minlength=12)
    assert cnt.sum() == n and cnt.max() <= 256
    if not hinted:
        assert cnt0.max() > 256, "the case must need balancing"
    p = L["new_of_old"]
    assert np.array_equal(np.sort(p), np.arange(n))
    internal = plan.f2 < n
    col = L["color_of"].astype(int)                  # by new id
    assert np.all(col[p[plan.f1[internal]]] != col[p[plan.f2[internal]]])
    assert np.all(np.diff(col) >= 0), "rows are colour-major"


def _chip_emulation(A, b, x0, col, n_sweeps, rtol=1e-13, f32=True, max_iter=50):
    """numpy restatement of k_solve_chip (cwr_small.cuh): right-preconditioned BiCGSTAB in fp64 on the row-scaled system,
    the preconditioner = n_sweeps multicolour Gauss-Seidel sweeps from zero -- in fp32 on fp32 copies of the values, applied to
    the input scaled by 2^-h (h = half the exponent of the squared norm handed over), the result widened and scaled back."""
    d = A.diagonal()
    As = sp.diags(1.0 / d) @ A
    L = (As - sp.identity(A.shape[0])).tocsr()              # unit diagonal implied
    bs = b / d
    L32 = L.astype(np.float32)
    rows_of = [np.nonzero(col == c)[0] for c in range(col.max() + 1)]

    def precondition(u, norm2):
        if not f32:
            z = np.zeros_like(u)
            for _ in range(n_sweeps):
                for rows in rows_of:
                    z[rows] = u[rows] - L[rows] @ z
            return z
        h = int(np.trunc((np.frexp(norm2)[1] - 1) / 2))    # exponent field - 1023, halved towards zero
        uf = (u * np.ldexp(1.0, -h)).astype(np.float32)
        z = np.zeros_like(uf)
        for _ in range(n_sweeps):
            for rows in rows_of:
                z[rows] = uf[rows] - L32[rows] @ z
        assert z.dtype == np.float32
        return z.astype(np.float64) * np.ldexp(1.0, h)

    x = x0.copy()
    r = bs - (x + L @ x)
    rhat, p = r.copy(), r.copy()
    bb, rr = bs @ bs, r @ r
    rho, its = rr, 0
    while rr > rtol * rtol * bb and its < max_iter:
        ph = precondition(p, rr)
        v = ph + L @ ph
        alpha = rho / (rhat @ v)
        s = r - alpha * v
        ss = s @ s
        if ss <= rtol * rtol * bb:
            x += alpha * ph
            its += 1
            rr = ss
            break
        sh = precondition(s, ss)
        t = sh + L @ sh
        omega = (t @ s) / (t @ t)
        rho_new = rhat @ s - omega * (rhat @ t)
        x += alpha * ph + omega * sh
        r = s - omega * t
        beta = (rho_new / rho) * (alpha / omega)
        p = r + beta * (p - omega * v)
        rho, rr = rho_new, r @ r
        its += 1
    return x, its, np.sqrt(rr / bb)


@pytest.mark.parametrize("units", [1.0, 1e-20, 1e+20])
def test_fp32_sweeps_inside_fp64_bicgstab_reach_the_fp64_answer_in_any_units(units):
    """What k_solve_chip does with precond_precision = 32, restated in numpy on the oracle's own system of the Ohio-shaped
    mesh: same iteration count as with fp64 sweeps, relative residual <= 1e-13, answer within 1e-9 of spsolve -- also when
    the concentrations are 1e-20 or 1e+20 (the power-of-two scaling keeps the fp32 sweeps in range)."""
    import scipy.sparse.linalg as spla
    from oracle import reference_step as ref
    plan = synthetic.ohio_like(4, seed=2)
    n = plan.n_real
    adv, _, _, cdiff, dt = ref.derive_coefficients(plan.face_flow, plan.edge_velocity, plan.face_x, plan.face_y,
                                                   plan.f1, plan.f2, 0.1, plan.time_seconds)
    mesh = ref.HydroMesh(plan.f1, plan.f2, plan.n_face, adv, cdiff, plan.edge_velocity, plan.volume, dt, 0.1)
    inputs = synthetic.make_inputs(plan, 1, seed=2)[0] * units
    lhs = ref.LHS(mesh); lhs.update_values(mesh, 1)
    A = lhs.to_csr(); A.sum_duplicates()
    rhs = ref.RHS(mesh, inputs)
    x0 = inputs[0][:n].copy()
    rhs.update_values(x0.copy(), mesh, 1)
    b = np.asarray(rhs.vals, dtype=np.float64)
    Lay = strip_layout(plan.f1, plan.f2, plan.n_face, 12, plan.face_flow.mean(0), 0, strip_cap=256)
    col = Lay["color_of"].astype(int)[Lay["new_of_old"]]                  # colour by original cell id
    want = spla.spsolve(A.tocsc(), b)
    x64, its64, rel64 = _chip_emulation(A, b, x0, col, 8, f32=False)
    x32, its32, rel32 = _chip_emulation(A, b, x0, col, 8, f32=True)
    assert its32 == its64 and its32 <= 3
    assert rel32 <= 1e-13 and rel64 <= 1e-13
    scale = np.abs(want).max()
    assert np.abs(x32 - want).max() <= 1e-9 * scale and np.abs(x64 - want).max() <= 1e-9 * scale
