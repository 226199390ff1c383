"""Seeded synthetic HEC-RAS-like 2D meshes + hydrodynamics for tests and benchmarks.

The reference ships only three tiny plan files here (50 and 2 real cells); the Ohio
River plan and all larger meshes are absent (SURVEY.md F4), so the benchmark
configurations of BASELINE.json run on meshes made by this generator.  It emits the
*raw* arrays a HEC-RAS plan holds -- cell-centre coordinates, `Faces Cell Indexes`
(f1, f2), `Face Flow`, `Face Velocity`, `Cell Volume` (all float32, as on disk,
reference io/hdf.py:255-305) and the time axis -- in the reference's conventions:

  * real cells are 0..n-1, one ghost cell per perimeter edge n..F-1;
  * f1 is always a real cell and max(f1) == n-1 (the reference *defines*
    nreal = max(edges_face1), io/hdf.py:268-269);
  * flow > 0 leaves f1.

Topology: an nx x ny block of jittered quads, a seeded fraction of which is split
into two triangles (quad-dominant unstructured mesh: row degree 3..4, plus diagonals).
Cells can be renumbered randomly to mimic HEC-RAS's arbitrary numbering (so that the
RCM reordering in the solver has something to do).

Hydrodynamics: flow = a(t) * curl(psi) + b(t) * grad(phi).  The stream-function part
is exactly divergence-free per cell; the potential part has zero-mean b(t) and is
integrated exactly into the volumes, so continuity V[t+1] = V[t] - dt * sum(out-flow[t])
holds to float32 rounding and a uniform concentration stays uniform (the property the
reference's tests/test_final_mass.py checks).  Dry cells (volume 0, all face flows 0)
sit on a sub-lattice so that they never share a node.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np


@dataclass
class SyntheticPlan:
    f1: np.ndarray              # (E,) int32
    f2: np.ndarray              # (E,) int32
    face_x: np.ndarray          # (F,) float64
    face_y: np.ndarray          # (F,) float64
    time_seconds: np.ndarray    # (T,) float64
    face_flow: np.ndarray       # (T,E) float32
    edge_velocity: np.ndarray   # (T,E) float32
    volume: np.ndarray          # (T,F) float32
    n_real: int                 # n  (number of real cells = matrix order)
    boundary_faces: Dict[str, np.ndarray]   # BC line name -> ghost-edge ids
    dry_cells: np.ndarray
    cell_area: Optional[np.ndarray] = None  # (F,) float64 plan areas (ghost cells: the full quad's)

    @property
    def n_face(self) -> int:
        return len(self.face_x)

    @property
    def n_edge(self) -> int:
        return len(self.f1)

    @property
    def n_time(self) -> int:
        return len(self.time_seconds)


def make_plan(nx: int, ny: int, n_time: int, *, dt: float = 30.0, dx: float = 10.0, depth: float = 2.0,
              tri_fraction: float = 0.1, dry_fraction: float = 0.0, courant: float = 1.5,
              tidal: float = 0.15, unsteady: float = 1.0, shuffle: bool = True, seed: int = 0,
              n_exact: Optional[int] = None) -> SyntheticPlan:
    """Build a plan with about nx*ny*(1+tri_fraction) real cells.

    n_exact: if given, the number of split quads is chosen so that n == n_exact
             (requires nx*ny <= n_exact <= 2*nx*ny).
    courant: target |Q| dt / V of the through-flow (eddies modulate it by about +-60 %).
    unsteady, tidal: amplitude of the time variation of the rotational / potential flow parts;
             with both 0 the flow is steady and a uniform concentration is preserved to rounding
             (unsteady flow is not: the reference evaluates the LHS at t and the boundary RHS at t+1).
    """
    rng = np.random.default_rng(seed)
    nq = nx * ny
    dy = dx
    # ---- nodes --------------------------------------------------------------------------
    NX, NY = nx + 1, ny + 1
    jx = (rng.random((NY, NX)) - 0.5) * 0.3 * dx
    jy = (rng.random((NY, NX)) - 0.5) * 0.3 * dy
    jx[:, 0] = jx[:, -1] = 0.0
    jy[0, :] = jy[-1, :] = 0.0
    node_x = (np.arange(NX)[None, :] * dx + jx)
    node_y = (np.arange(NY)[:, None] * dy + jy)

    # ---- which quads are split / dry ---------------------------------------------------------
    if n_exact is not None:
        n_split = int(n_exact) - nq
        if not 0 <= n_split <= nq:
            raise ValueError("n_exact out of range for this nx, ny")
    else:
        n_split = int(round(tri_fraction * nq))
    split = np.zeros(nq, dtype=bool)
    split[rng.choice(nq, size=n_split, replace=False)] = True
    split = split.reshape(ny, nx)
    # T2 (upper-left triangle) of split quad q gets a new id nq + rank(q)
    t2_id = np.full((ny, nx), -1, dtype=np.int64)
    t2_id[split] = nq + np.arange(n_split)
    n = nq + n_split
    base_id = np.arange(nq, dtype=np.int64).reshape(ny, nx)
    left_owner = np.where(split, t2_id, base_id)     # who owns the quad's left / top side
    top_owner = left_owner
    right_owner = base_id                            # T1 keeps bottom / right side
    bottom_owner = base_id

    # ---- edges: (P, N, node_start, node_end) with outward flux of P = psi[end] - psi[start] ----
    nid = (np.arange(NY)[:, None] * NX + np.arange(NX)[None, :]).astype(np.int64)
    P, N, A, B = [], [], [], []
    ghost = -1
    # vertical edges at column i between (i-1, j) [left] and (i, j) [right]
    L = right_owner[:, :-1]; R = left_owner[:, 1:]
    P.append(L.ravel()); N.append(R.ravel())
    A.append(nid[:-1, 1:-1].ravel()); B.append(nid[1:, 1:-1].ravel())
    # left boundary: P = left_owner of column 0, traversed downwards
    P.append(left_owner[:, 0]); N.append(np.full(ny, ghost))
    A.append(nid[1:, 0]); B.append(nid[:-1, 0])
    # right boundary: P = right_owner of last column, traversed upwards
    P.append(right_owner[:, -1]); N.append(np.full(ny, ghost))
    A.append(nid[:-1, -1]); B.append(nid[1:, -1])
    # horizontal edges at row j between (i, j-1) [below] and (i, j) [above]
    Bl = top_owner[:-1, :]; Ab = bottom_owner[1:, :]
    P.append(Bl.ravel()); N.append(Ab.ravel())
    A.append(nid[1:-1, 1:].ravel()); B.append(nid[1:-1, :-1].ravel())
    # bottom boundary: P = bottom_owner row 0, traversed left -> right
    P.append(bottom_owner[0, :]); N.append(np.full(nx, ghost))
    A.append(nid[0, :-1]); B.append(nid[0, 1:])
    # top boundary: P = top_owner last row, traversed right -> left
    P.append(top_owner[-1, :]); N.append(np.full(nx, ghost))
    A.append(nid[-1, 1:]); B.append(nid[-1, :-1])
    # diagonals of split quads: P = T1, N = T2, traversed (i+1,j+1) -> (i,j)
    sj, si = np.nonzero(split)
    P.append(base_id[sj, si]); N.append(t2_id[sj, si])
    A.append(nid[sj + 1, si + 1]); B.append(nid[sj, si])
    n_left, n_right, n_bottom, n_top = ny, ny, nx, nx
    P = np.concatenate(P); N = np.concatenate(N); A = np.concatenate(A); B = np.concatenate(B)
    E = len(P)
    is_ghost = N == ghost

    # ---- cell centres and plan areas --------------------------------------------------------
    nxf, nyf = node_x.ravel(), node_y.ravel()
    q_nodes = np.stack([nid[:-1, :-1], nid[:-1, 1:], nid[1:, 1:], nid[1:, :-1]], axis=-1).reshape(nq, 4)
    cx = np.empty(n); cy = np.empty(n); area = np.empty(n)
    cx[:nq] = nxf[q_nodes].mean(1); cy[:nq] = nyf[q_nodes].mean(1); area[:nq] = dx * dy
    sp = split.ravel()
    t1n = q_nodes[sp][:, [0, 1, 2]]; t2n = q_nodes[sp][:, [0, 2, 3]]
    cx[np.nonzero(sp)[0]] = nxf[t1n].mean(1); cy[np.nonzero(sp)[0]] = nyf[t1n].mean(1)
    cx[nq:] = nxf[t2n].mean(1); cy[nq:] = nyf[t2n].mean(1)
    area[np.nonzero(sp)[0]] = 0.5 * dx * dy; area[nq:] = 0.5 * dx * dy

    # ---- dry cells: unsplit quads on the even/even sub-lattice (no shared nodes) ---------------
    dry_quads = np.zeros((ny, nx), dtype=bool)
    if dry_fraction > 0:
        cand = np.zeros((ny, nx), dtype=bool)
        cand[1:-1:2, 1:-1:2] = True
        cand &= ~split
        idx = np.nonzero(cand.ravel())[0]
        k = min(len(idx), int(round(dry_fraction * n)))
        dry_quads.ravel()[rng.choice(idx, size=k, replace=False)] = True
    dry_cells = base_id[dry_quads]

    # ---- stream function psi (node) and potential phi (cell) -----------------------------------
    Lx, Ly = nx * dx, ny * dy
    U = courant * dx / dt                                   # through-flow speed for the target Courant number
    X, Y = node_x / Lx, node_y / Ly
    kx = max(1, int(round(nx / 40))); ky = max(1, int(round(ny / 40)))
    psi = U * depth * (node_y + 0.6 * Ly / (2 * np.pi * ky) * np.sin(2 * np.pi * kx * X) * np.sin(2 * np.pi * ky * Y)
                       * min(1.0, 4.0 * ky / max(kx, 1)))
    psi_b = 0.35 * U * depth * Ly / (2 * np.pi * max(ky, 1)) * np.cos(2 * np.pi * (kx + 1) * X) * np.sin(np.pi * Y)
    # walls: psi exactly constant along the south / north boundary rows -> exactly zero flow there
    psi[0, :] = 0.0; psi[-1, :] = U * depth * Ly
    psi_b[0, :] = 0.0; psi_b[-1, :] = 0.0
    for arr in (psi, psi_b):                                # dry quads: psi constant on their 4 nodes
        dj, di = np.nonzero(dry_quads)
        v = arr[dj, di]
        arr[dj, di + 1] = v; arr[dj + 1, di] = v; arr[dj + 1, di + 1] = v
    psi, psi_b = psi.ravel(), psi_b.ravel()
    q_psi = psi[B] - psi[A]                                 # steady part       (E,)
    q_psi_b = psi_b[B] - psi_b[A]                           # slowly modulated  (E,)
    # potential (tidal) part on internal edges only, zero across dry cells
    phi = np.cos(np.pi * cx / Lx) * (1.0 + 0.2 * np.cos(2 * np.pi * cy / Ly))
    elen = np.hypot(nxf[A] - nxf[B], nyf[A] - nyf[B])
    q_phi = np.zeros(E)
    ii = ~is_ghost
    dry_mask = np.zeros(n, dtype=bool); dry_mask[dry_cells] = True
    cdist = np.hypot(cx[P[ii]] - cx[N[ii]], cy[P[ii]] - cy[N[ii]])
    q_phi[ii] = depth * elen[ii] / cdist * (phi[P[ii]] - phi[N[ii]])
    q_phi[ii] *= ~(dry_mask[P[ii]] | dry_mask[N[ii]])
    div_phi = np.bincount(P[ii], q_phi[ii], n) - np.bincount(N[ii], q_phi[ii], n)
    # scale so that the volume oscillation amplitude is `tidal` * V0 at most
    V0 = area * depth
    V0[dry_cells] = 0.0

    # ---- time axis, a(t), b(t) -----------------------------------------------------------------
    t = np.arange(n_time) * float(dt)
    steps = np.arange(n_time)
    a_t = 1.0 + unsteady * 0.25 * np.sin(2 * np.pi * steps / 37.0)
    a2_t = unsteady * np.sin(2 * np.pi * steps / 23.0 + 0.7)
    b_raw = np.cos(2 * np.pi * (steps + 0.5) / 16.0)
    cum = np.concatenate([[0.0], np.cumsum(b_raw[:-1])]) * dt          # integral of b up to step t
    wet = V0 > 0
    amp = np.max(np.abs(cum)) * np.max(np.abs(div_phi[wet]) / V0[wet]) if wet.any() else 0.0
    s_phi = tidal / amp if amp > 0 else 0.0
    b_t = b_raw * s_phi

    flow = (a_t[:, None] * q_psi[None, :] + a2_t[:, None] * q_psi_b[None, :] + b_t[:, None] * q_phi[None, :])
    vol = V0[None, :] - (cum * s_phi)[:, None] * div_phi[None, :]
    vol[:, dry_cells] = 0.0
    face_area = depth * elen
    with np.errstate(invalid="ignore"):
        vel = flow / face_area[None, :]

    # ---- renumber cells (HEC-RAS-like arbitrary numbering), orient edges, append ghosts ----------
    perm = rng.permutation(n) if shuffle else np.arange(n)     # new id of old cell c = perm[c]
    Pn = perm[P]
    Nn = np.where(is_ghost, -1, perm[np.where(is_ghost, 0, N)])
    flip = (~is_ghost) & (rng.random(E) < 0.5)                 # internal edges in either order
    last = n - 1                                               # make sure max(f1) == n-1
    touch = np.nonzero(((Pn == last) | (Nn == last)))[0]
    if not np.any((Pn[touch] == last) & ~flip[touch] | (Nn[touch] == last) & flip[touch]):
        e0 = touch[0]
        flip[e0] = (Nn[e0] == last)
    f1 = np.where(flip, Nn, Pn)
    f2 = np.where(flip, Pn, Nn)
    sign = np.where(flip, -1.0, 1.0)
    eperm = rng.permutation(E) if shuffle else np.arange(E)    # edge order on "disk"
    f1, f2, sign, g_e = f1[eperm], f2[eperm], sign[eperm], is_ghost[eperm]
    n_ghost = int(g_e.sum())
    f2 = f2.copy()
    f2[g_e] = n + np.arange(n_ghost)
    F = n + n_ghost
    flow = (flow[:, eperm] * sign[None, :]).astype(np.float32)
    vel = (vel[:, eperm] * sign[None, :]).astype(np.float32)
    vel[flow == 0] = 0.0                                       # sign(vel) == sign(flow) everywhere
    inv = np.empty(n, dtype=np.int64); inv[perm] = np.arange(n)
    face_x = np.empty(F); face_y = np.empty(F)
    face_x[:n] = cx[inv]; face_y[:n] = cy[inv]
    # ghost cell centre = mirror of the real centre across the edge midpoint
    mx = 0.5 * (nxf[A] + nxf[B])[eperm][g_e]; my = 0.5 * (nyf[A] + nyf[B])[eperm][g_e]
    face_x[n:] = 2 * mx - face_x[f1[g_e]]; face_y[n:] = 2 * my - face_y[f1[g_e]]
    volume = np.zeros((n_time, F), dtype=np.float32)
    volume[:, :n] = vol[:, inv].astype(np.float32)
    volume[:, n:] = np.float32(dx * dy * depth)                # ghost-cell volumes are never read by the step
    cell_area = np.full(F, dx * dy)
    cell_area[:n] = area[inv]

    # boundary lines: which original side each ghost edge came from
    side = np.full(E, -1)
    o = (nx - 1) * ny
    side[o:o + n_left] = 0; o += n_left
    side[o:o + n_right] = 1; o += n_right
    o += nx * (ny - 1)
    side[o:o + n_bottom] = 2; o += n_bottom
    side[o:o + n_top] = 3
    side = side[eperm]
    bfaces = {"upstream": np.nonzero(side == 0)[0], "downstream": np.nonzero(side == 1)[0],
              "south": np.nonzero(side == 2)[0], "north": np.nonzero(side == 3)[0]}
    return SyntheticPlan(
        f1=f1.astype(np.int32), f2=f2.astype(np.int32), face_x=face_x, face_y=face_y, time_seconds=t,
        face_flow=flow, edge_velocity=vel, volume=volume, n_real=n, boundary_faces=bfaces,
        dry_cells=np.sort(perm[dry_cells]), cell_area=cell_area)


def make_inputs(plan: SyntheticPlan, n_constituents: int, *, seed: int = 0, ic_range=(0.0, 100.0),
                bc_scale: Optional[np.ndarray] = None) -> np.ndarray:
    """(K,T,F) float64 `input_array`s: independent random ICs; BC series on the upstream and
    downstream lines (a base level plus lognormal pulses, per constituent).  Zero means unset
    (reference constituents.py:32, linalg.py:199-200), so values are kept strictly positive."""
    rng = np.random.default_rng(seed + 7919)
    T, F, n = plan.n_time, plan.n_face, plan.n_real
    inp = np.zeros((n_constituents, T, F))
    lo, hi = ic_range
    for k in range(n_constituents):
        inp[k, 0, :n] = lo + (hi - lo) * rng.random(n) + 1e-3
        for name in ("upstream", "downstream"):
            faces = plan.boundary_faces[name]
            if len(faces) == 0:
                continue
            base = 20.0 + 60.0 * rng.random()
            pulses = np.exp(rng.normal(0.0, 0.5, size=T))
            series = base * (0.5 + 0.5 * pulses)
            if bc_scale is not None:
                series = series * bc_scale[k]
            inp[k][:, plan.f2[faces]] = series[:, None]
    return inp


# ------------------------------------------------------------------------------------------
# presets for the BASELINE.json configurations
# ------------------------------------------------------------------------------------------
def ohio_like(n_time: int = 913, seed: int = 2) -> SyntheticPlan:
    """Stand-in for the Ohio River plan (2943 real cells; HDF absent -- SURVEY.md F4): a
    490 x 6 river strip with 3 split quads -> n = 2943, hourly output (dt = 3600 s)."""
    return make_plan(490, 6, n_time, dt=3600.0, dx=400.0, depth=6.0, courant=2.5, tidal=0.05,
                     n_exact=2943, seed=seed)


def square_mesh(n_side: int, n_time: int, seed: int, **kw) -> SyntheticPlan:
    kw.setdefault("tri_fraction", 0.1)
    return make_plan(n_side, n_side, n_time, seed=seed, **kw)


def make_kinetics(inputs: np.ndarray, *, seed: int = 0, decay_range=(20.0, 200.0)):
    """A seeded first-order network over the K constituents of `inputs` ((K,T,F), make_inputs): every constituent
    decays (decay_range in 1/day, theta in 1.02..1.08) and constituent k yields to k + 1 with +0.8 for even k and -0.4 for
    odd k (a chain with negative yields).  K >= 4: the last constituent is the temperature instead (its values rescaled to
    10..30 deg C; it neither decays nor receives); K < 4: a constant 24 deg C (13 deg C for K = 1).
    Returns (inputs', dict of TransportBackend.set_kinetics arguments)."""
    rng = np.random.default_rng(seed + 104729)
    inputs = np.array(inputs, dtype=np.float64, copy=True)
    K = inputs.shape[0]
    temperature_k = K - 1 if K >= 4 else -1
    n_react = K - 1 if temperature_k >= 0 else K
    lo, hi = decay_range
    decay = np.zeros(K)
    decay[:n_react] = lo + (hi - lo) * rng.random(n_react)
    theta = np.ones(K)
    theta[:n_react] = 1.02 + 0.06 * rng.random(n_react)
    yields = np.zeros((K, K))
    for k in range(n_react - 1):
        yields[k + 1, k] = 0.8 if k % 2 == 0 else -0.4
    if temperature_k >= 0:
        a = inputs[temperature_k]
        inputs[temperature_k] = np.where(a != 0, 10.0 + 0.2 * a, 0.0)
    return inputs, dict(decay_per_day=decay, theta=theta, yields=yields, temperature_k=temperature_k,
                        temperature_c=13.0 if K == 1 else 24.0)


def make_kinetics_sources(kin: dict, *, seed: int = 0, rate_range=(20.0, 200.0)) -> dict:
    """Seeded zero-order sources and exchange for a network of make_kinetics (kin: its set_kinetics arguments), in the
    manner of a BOD-DO model: every reacting constituent k has a source of 5..50 x rate_range per day (a sink for odd k,
    like sediment oxygen demand) and, for even k, an exchange rate in rate_range (1/day) toward oxygen saturation
    (k = 2 mod 4, reaeration) or a constant 5..45 (k = 0 mod 4); thetas in 1.0..1.08.  The temperature constituent, if
    any, relaxes toward a constant 18 deg C with a small source (the equilibrium-temperature model).
    Returns a dict of TransportBackend.set_kinetics_sources arguments."""
    rng = np.random.default_rng(seed + 130363)
    K = len(kin["decay_per_day"])
    temperature_k = kin["temperature_k"]
    lo, hi = rate_range
    source, exchange = np.zeros(K), np.zeros(K)
    source_theta, exchange_theta = 1.0 + 0.08 * rng.random(K), 1.0 + 0.08 * rng.random(K)
    equilibrium, kind = np.zeros(K), np.zeros(K, np.int32)
    for k in range(K):
        if k == temperature_k:
            exchange[k] = lo + (hi - lo) * rng.random()
            equilibrium[k] = 18.0
            source[k] = 0.5 * lo * (rng.random() - 0.5)
            continue
        source[k] = (5.0 + 45.0 * rng.random()) * (lo + (hi - lo) * rng.random()) * (-1.0 if k % 2 else 1.0)
        if k % 2 == 0:
            exchange[k] = lo + (hi - lo) * rng.random()
            if k % 4 == 2 or K == 1:
                kind[k] = 1
            else:
                equilibrium[k] = 5.0 + 40.0 * rng.random()
    return dict(source_per_day=source, source_theta=source_theta, exchange_per_day=exchange, exchange_theta=exchange_theta,
                equilibrium=equilibrium, equilibrium_kind=kind)


def make_kinetics_limits(kin: dict, src: Optional[dict] = None, *, seed: int = 0) -> dict:
    """Seeded Monod factors for a network of make_kinetics (kin) and make_kinetics_sources (src, or None), in the manner
    of a BOD-DO-nitrogen model: every decay that consumes a constituent (a negative yield) is limited by it (K in
    0.05..0.5, so that the decay is capped where the consumed constituent runs out), every sink is limited by its own
    constituent (sediment-oxygen-demand-like, K in 0.5..2), the decay of every reacting k = 1 mod 3 is inhibited by
    constituent k + 1 (denitrification-like, K in 5..50) and the positive source of every k = 0 mod 4 by constituent
    k + 2, when they exist.  A network without a consuming decay or a sink (K = 1 with a positive source) gets no factor.
    Returns a dict of TransportBackend.set_kinetics_limits arguments."""
    rng = np.random.default_rng(seed + 160183)
    decay, yields = np.asarray(kin["decay_per_day"]), np.asarray(kin["yields"])
    K = len(decay)
    source = np.zeros(K) if src is None or src.get("source_per_day") is None else np.asarray(src["source_per_day"])
    rows = []                                   # (process, column, factor column, kind, half-saturation)
    for k in range(K):
        if decay[k] == 0.0:
            continue
        for j in np.nonzero(yields[:, k] < 0.0)[0]:
            rows.append((0, k, int(j), 0, 0.05 + 0.45 * rng.random()))
    for k in range(K):
        if source[k] < 0.0:
            rows.append((1, k, k, 0, 0.5 + 1.5 * rng.random()))
    for k in range(K):
        if decay[k] != 0.0 and k % 3 == 1 and k + 1 < K:
            rows.append((0, k, k + 1, 1, 5.0 + 45.0 * rng.random()))
        if source[k] > 0.0 and k % 4 == 0 and k + 2 < K:
            rows.append((1, k, k + 2, 1, 5.0 + 45.0 * rng.random()))
    cols = list(zip(*rows)) if rows else [()] * 5
    return dict(process=np.array(cols[0], np.int32), column=np.array(cols[1], np.int32),
                factor_column=np.array(cols[2], np.int32), factor_kind=np.array(cols[3], np.int32),
                half_saturation=np.array(cols[4], np.float64))


def make_kinetics_depth(kin: dict, src: Optional[dict] = None, *, seed: int = 0, depth: float = 2.0):
    """Seeded depth-scaled processes for a network of make_kinetics (kin) and make_kinetics_sources (src, or None), in the
    manner of a BOD-DO model: the decay of every reacting k = 0 mod 3 becomes a settling velocity, the source of every
    k = 1 mod 2 an areal flux (sediment-oxygen-demand-like sinks) and about half of the exchange rates transfer
    velocities, chosen with the seed.  Each flagged rate is multiplied by `depth` (mesh length units; make_plan's default
    depth), so that at that depth it is the rate it replaces.
    Returns (kin', src', dict of the flags of TransportBackend.set_kinetics_depth)."""
    rng = np.random.default_rng(seed + 179424673)
    decay = np.array(kin["decay_per_day"], np.float64, copy=True)
    K = len(decay)
    zero = np.zeros(K)
    source = np.array(zero if src is None or src.get("source_per_day") is None else src["source_per_day"], np.float64)
    exchange = np.array(zero if src is None or src.get("exchange_per_day") is None else src["exchange_per_day"], np.float64)
    k = np.arange(K)
    coin = rng.random(K) < 0.5
    flags = dict(decay_per_depth=((k % 3 == 0) & (decay != 0)).astype(np.int32),
                 source_per_depth=((k % 2 == 1) & (source != 0)).astype(np.int32),
                 exchange_per_depth=(coin & (exchange != 0)).astype(np.int32))
    decay[flags["decay_per_depth"] == 1] *= depth
    source[flags["source_per_depth"] == 1] *= depth
    exchange[flags["exchange_per_depth"] == 1] *= depth
    kin = dict(kin, decay_per_day=decay)
    if src is not None:
        src = dict(src, source_per_day=source, exchange_per_day=exchange)
    return kin, src, flags
