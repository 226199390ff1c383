/*
 * cwr.h -- C ABI of the B200-native ClearWater-Riverine transport step.
 *
 * The reference (EcohydrologyTeam/ClearWater-riverine, pure Python) has no FFI; the
 * seam this library drops into is the body of
 *     ClearwaterRiverine.update()            src/clearwater_riverine/transport.py:201-276
 * and the state it touches.  Each entry point below names the reference lines it
 * replaces.  All arrays are caller-owned, contiguous, row-major, in the REFERENCE's
 * cell / edge numbering (the library's internal RCM ordering never crosses the ABI);
 * every set_* call copies its input.  One handle = one device + one stream; a handle
 * is not thread-safe, distinct handles may be driven from distinct host threads.
 *
 * Return value: 0 (CWR_OK) or a negative cwr_status; cwr_last_error() gives the text.
 * No exceptions or C++ types cross this boundary.
 */
#ifndef CWR_H
#define CWR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cwr_handle cwr_handle;

typedef enum {
    CWR_OK = 0,
    CWR_EINVAL = -1,        /* bad argument / state not available */
    CWR_ECUDA = -2,         /* CUDA runtime error */
    CWR_ENOTCONVERGED = -3, /* the solver hit max_iter (results are still stored) */
    CWR_EBREAKDOWN = -4,    /* BiCGSTAB breakdown that restarts could not cure */
    CWR_ENAN = -5,          /* non-finite residual (NaN/Inf in the inputs, e.g. a NaN boundary value) */
    CWR_ESINGULAR = -6,     /* zero diagonal: the reference's spsolve would warn MatrixRankWarning */
    CWR_ENOMEM = -7
} cwr_status;

typedef struct {
    double rtol;            /* stop when ||r||_2 <= rtol * ||b||_2 (row-scaled system); default 1e-13 */
    int max_iter;           /* BiCGSTAB iterations / defect-correction cycles per solve; default 500 */
    int reorder;            /* 0 = keep cell order, 1 = reverse Cuthill-McKee (default) */
    int keep_history;       /* 1 = keep every c[t] on the device (default), 0 = only c[t], c[t+1] */
    int hydro_capacity;     /* time slices resident on the device; 0 = all n_time (default) */
    int mass_flux;          /* 1 = compute the three per-edge mass-flux arrays every step (default, as the
                               reference does, transport.py:267-273), 0 = skip */
    int solver_path;        /* 0 = auto, 1 = multi-CTA kernels, 2 = one CTA per constituent runs the whole solve (small meshes;
                               <= 4096 cells with Gauss-Seidel sweeps: entirely on chip -- cwr_get_options reports 3, or 4 where a
                               thread keeps one row of every colour: quad / triangle meshes with colours of <= 256 rows) */
    int solver;             /* large meshes (solver_path 1): 1 = right-preconditioned BiCGSTAB; 2 = defect correction with the
                               preconditioner sweeps themselves: x += M^-1 r, r -= A (M^-1 r) in fp64, no Krylov vectors -- with
                               flow-aligned Gauss-Seidel sweeps the sweeps ARE the solver (18-19 of them reach 1e-13 where
                               BiCGSTAB spends 25 plus its own vector traffic); the number of sweeps per cycle is planned on the
                               device from the measured error factor, and a solve whose sweeps stagnate or diverge (not an
                               M-matrix) falls back to BiCGSTAB by itself; 0 (default) = 2 with Gauss-Seidel sweeps, else 1 */
    int check_every;        /* large meshes: iterations launched per convergence poll once the launch-ahead burst is used up;
                               default 1 */
    int precond_steps;      /* m: the preconditioner applies m - 1 sweeps; 1 = diagonal (Jacobi) scaling only;
                               0 (default) = 6 with Gauss-Seidel sweeps on large meshes, 5 on chip (<= 4096 cells), 8 with
                               Jacobi steps.  Defect-correction solver: 0 = the sweeps of every cycle are planned on the device
                               from the measured error factor (2..10 in fp32), m > 0 = every cycle does exactly m - 1 */
    int precond_precision;  /* 32 (default): the sweeps and the preconditioned vectors are fp32 (half the bytes;
                               BiCGSTAB itself, its products A p^ / A s^ and its dots stay fp64, so the converged
                               answer is the fp64 one); 64: fp64 sweeps */
    int precond_sweep;      /* 1 (default) = multicolour Gauss-Seidel sweeps from z = 0, all sweeps of one application (or of
                               one defect-correction cycle) in one persistent kernel (see precond_sync); the rows are
                               regrouped by colour and the colours follow the flow (cwr_set_flow_hint, or the
                               first hydrodynamic slices uploaded -- upload hydro before inputs);
                               0 = Jacobi steps, z = (I + N + ... + N^(m-1)) u with N = I - D^-1 A */
    int precond_colors;     /* colours of the Gauss-Seidel sweeps (raised to max row degree + 1 if smaller);
                               0 (default) = chosen from the mesh size so that one colour moves ~20 MB */
    int dd_rank, dd_world;  /* domain decomposition: this handle is rank dd_rank of dd_world (<= 8) handles, one per
                               GPU/process, each given the WHOLE mesh and the same inputs; rows are cut into dd_world
                               strips and a handle computes its strip, exchanging boundary rows and dot products with
                               the others over NVLink peer memory (cwr_dd_export / cwr_dd_attach).  0 / 0 or 1: off */
    int dd_halo_per_colour; /* domain decomposition, Gauss-Seidel sweeps: 0 (default) = boundary rows cross NVLink once per sweep
                               (Gauss-Seidel inside a strip, one sweep of lag across strips; one halo barrier per sweep),
                               1 = after every colour (exact multi-rank Gauss-Seidel; a halo barrier per colour; precond_sync 1) */
    int precond_sync;       /* Gauss-Seidel sweep kernel: 1 = rows colour-major, a grid barrier between colours; 2 = rows cut into
                               one strip per CTA (colour-major inside), a CTA only waits for the strips its rows are coupled
                               to (per-strip flags: release/acquire between neighbours instead of a device-wide rendezvous);
                               3 = the same strips, software-pipelined across that wait: everything a colour reads except the
                               values of the colour swept just before it is fetched (cp.async into shared memory) BEFORE the
                               wait, so the dependent latency overlaps the streaming (16-byte packs: K a multiple of 4 with
                               fp32 sweeps; otherwise 2 is used);
                               4 = the schedule of 3 with the operands arriving the Blackwell way: the contiguous streams of a
                               colour step (column indices, matrix values, right-hand side) by cp.async.bulk + mbarrier into a
                               per-warp ring four steps deep (L2 evict-first), the neighbour gathers as predicated
                               ld.global.cg into registers (sector-exact where cp.async.cg fetches whole lines).  Written for
                               fp32 sweeps over 16 constituents, ELL width 4, one rank; otherwise 3 is used.
                               Same arithmetic in all four (bitwise equal results for the same colours);
                               0 (default) = 4 unless dd_halo_per_colour */
} cwr_options;

typedef struct {
    int iterations;         /* BiCGSTAB iterations (max over constituents) / defect-correction cycles */
    int restarts;
    int status;             /* cwr_status of the solve */
    double max_relres;      /* max over constituents of ||r|| / ||b|| at exit */
    int n_launches;         /* kernels this step launched */
    int sweeps;             /* Gauss-Seidel sweeps of the solve (defect-correction solver; 0 otherwise) */
} cwr_step_info;

typedef struct {
    double vol_start, mass_start, vol_end, mass_end;   /* postproc_util.py:36-59 */
} cwr_mass_totals;

/* defaults for every field of cwr_options */
int cwr_default_options(cwr_options* opt);

/* Replaces LHS.__init__ / RHS.__init__ (linalg.py:18-32, 159-175) and the per-step COO->CSR
 * rebuild (transport.py:215-218): builds the fixed CSR pattern, the slot->edge map and the
 * boundary-cell lists once.  n_real = nreal + 1 = max(f1) + 1 (io/hdf.py:268-269). */
int cwr_create(cwr_handle** h, int device, int n_real, int n_face, int n_edge, int n_time, int n_const,
               const int32_t* f1, const int32_t* f2, double diffusion_coefficient, const cwr_options* opt);
/* The same with the flow hint of cwr_set_flow_hint given up front ((E,) f32 or NULL): the ordering is built once
 * (it costs seconds on meshes of millions of cells). */
int cwr_create_with_hint(cwr_handle** h, int device, int n_real, int n_face, int n_edge, int n_time, int n_const,
                         const int32_t* f1, const int32_t* f2, double diffusion_coefficient, const cwr_options* opt,
                         const float* flow_hint);
void cwr_destroy(cwr_handle* h);
const char* cwr_last_error(const cwr_handle* h);   /* h may be NULL: error of the last failed cwr_create */

/* The mesh variables the step reads (linalg.py:61-66,89,225,372; produced by utilities.py:513-541):
 * slices [t0, t0+nt) of advection_coeff (nt,E) f32, coeff_to_diffusion (nt,E) f64,
 * edge_velocity (nt,E) f32, volume (nt,F) f32, dt (nt,) f64. */
int cwr_set_hydro(cwr_handle* h, int t0, int nt, const float* adv, const double* cdiff, const float* vel,
                  const float* vol, const double* dt);

/* "Next" row N1: the same, derived on the device from the raw HEC-RAS arrays as
 * WQVariableCalculator.calculate does (utilities.py:513-541).  cwr_set_geometry gives the cell
 * centres (face_x, face_y: (F,)) from which face_to_face_dist is computed (utilities.py:261-280). */
int cwr_set_geometry(cwr_handle* h, const double* face_x, const double* face_y);
int cwr_set_hydro_raw(cwr_handle* h, int t0, int nt, const float* face_flow, const float* edge_velocity,
                      const float* volume, const double* dt);

/* cwr_set_hydro_raw on a second stream: the copy and the derivation overlap whatever the handle's stream and the
 * caller do next (typically the device->host copy of the step just taken); the next call that reads the hydro
 * window waits for it on the device.  The host arrays must stay valid until then (page-locked for a truly
 * asynchronous copy). */
int cwr_prefetch_hydro_raw(cwr_handle* h, int t0, int nt, const float* face_flow, const float* edge_velocity,
                           const float* volume, const double* dt);

/* Optional, before any other set_* call: one representative signed face flow per edge ((E,) f32, e.g. the
 * time mean of `Face Flow`) for the flow-aligned colouring of the Gauss-Seidel sweeps (precond_sweep = 1).
 * Without it the first cwr_set_hydro* call's slices are used.  Affects speed only, never results beyond rtol. */
int cwr_set_flow_hint(cwr_handle* h, const float* face_flow);

/* Constituent.input_array (constituents.py:31,93,164): (T,F) f64, IC in row 0, BC values in
 * ghost-cell columns, 0 = "not set".  Also initialises c[0] as set_initial_conditions does. */
int cwr_set_inputs(cwr_handle* h, int k, const double* input_array);

/* update_concentration override (transport.py:233-236): overwrite c_k[t, 0:n]. */
int cwr_set_state(cwr_handle* h, int k, int t, const double* c);

/* One ClearwaterRiverine.update() (transport.py:201-276) for all constituents: LHS(t) assembly,
 * RHS per constituent, solve, store c[t+1] with BC re-imposition, mass flux.  info may be NULL. */
int cwr_step(cwr_handle* h, int t, cwr_step_info* info);

/* for (t = t_begin; t < t_end; ++t) cwr_step(h, t) without host round trips between steps
 * (the loop the reference's users write, examples/01_getting_started_riverine.ipynb cell 26). */
int cwr_run(cwr_handle* h, int t_begin, int t_end, cwr_step_info* worst);

/* mesh[name][t] (transport.py:252-264): (F,) f64 -- real cells, BC ghost values, NaN elsewhere. */
int cwr_get_state(cwr_handle* h, int k, int t, double* c_out);
/* All constituents at once, real cells only: (K, n) f64 (what a coupling loop reads each step). */
int cwr_get_state_all(cwr_handle* h, int t, double* c_out);
/* The same, every constituent straight into its own destination: rows[k] -> (n,) f64 (e.g. row t of the
 * caller's (T,F) output array of constituent k; NULL skips k).  One device->host copy per constituent with no
 * intermediate host buffer; at full PCIe rate when the destinations are page-locked (cwr_host_register). */
int cwr_get_state_rows(cwr_handle* h, int t, double* const* rows);
/* Asynchronous outputs of a step: c[t] (rows[k] -> (n,) f64, as cwr_get_state_rows) and, optionally, the three mass-flux
 * arrays of step t - 1 (adv/diff/tot_rows[k] -> (E,) f64, as cwr_get_mass_flux; any of the three arrays of pointers
 * may be NULL) are gathered into a staging slot on the handle's stream and copied to the host on a separate stream,
 * so the copies overlap the next cwr_step (two slots: the call only blocks if the copies of the fetch before the last
 * one are still running).  The destinations must be page-locked (cwr_host_register) for the overlap to be real and must
 * not be read before cwr_fetch_wait returns.  Replaces the per-step writes of transport.py:252-273. */
int cwr_fetch_async(cwr_handle* h, int t, double* const* state_rows, double* const* adv_rows, double* const* diff_rows,
                    double* const* tot_rows);
int cwr_fetch_wait(cwr_handle* h);
/* Page-lock / release a caller-owned host array (cudaHostRegister) so that the copies above run asynchronously
 * at full rate.  Optional; no handle needed (a CUDA device must be present). */
int cwr_host_register(void* p, size_t bytes);
int cwr_host_unregister(void* p);
/* All overrides at once: (K, n) f64; mask[k] != 0 selects the constituents to overwrite. */
int cwr_set_state_all(cwr_handle* h, int t, const double* c, const uint8_t* mask);

/* Constituent.{advection,diffusion,total}_mass_flux[t] (transport.py:406-429): (E,) f64 each; any
 * pointer may be NULL.  Only the most recent step's fluxes are held on the device. */
int cwr_get_mass_flux(cwr_handle* h, int k, int t, double* advection, double* diffusion, double* total);

/* "Next" row N2 (postproc_util.py:36-59): sum(V*c) over real cells at t_start and t_end. */
int cwr_mass_totals_at(cwr_handle* h, int k, int t_start, int t_end, cwr_mass_totals* out);
/* Per-edge running sums of total_mass_flux over the steps taken so far, split as the reference's
 * mass balance does (postproc_util.py:100-143): in = sum of entries <= 0, out = sum of entries >= 0.
 * (E,) f64 each, any may be NULL.  Enabled when options.mass_flux != 0. */
int cwr_get_flux_sums(cwr_handle* h, int k, double* total_sum, double* in_sum, double* out_sum);

/* The same for the water volume across the boundary faces (postproc_util.py:93-95, 112-134): per-edge running sums
 * of face_flow[t] * dt[t] over the steps taken so far, total / in (<= 0) / out (>= 0), NaN skipped; (E,) f64 each, zero on
 * internal edges.  (With cwr_set_hydro, which is not given the raw face flow, advection_coeff stands in for it.) */
int cwr_get_volume_sums(cwr_handle* h, double* total_sum, double* in_sum, double* out_sum);

/* --- first-order kinetics (decay with temperature correction, transformation chains) ---------------------------------
 * Step t first forms c~ as without kinetics: c[t], or the cwr_set_state override, with the non-zero real-cell entries of
 * input_array[t] merged in.  With kinetics set, every real cell i is then reacted before the load term V[t] c~ / dt is formed:
 *     T_i = temperature_c, or c~ of constituent temperature_k in cell i before any reaction of the step
 *     for k in topological order of the yield graph:
 *         r = decay_k * theta_k^(T_i - 20) / 86400          (decay in 1/day; theta^x = exp(x log theta))
 *         loss = c~_k * (-expm1(-r dt[t]));  c~_k -= loss;  c~_j += yields[j, k] * loss for every j
 *     then, with cwr_set_kinetics_sources, for every column k with a source or exchange term, in ascending k:
 *         s   = source_k * source_theta_k^(T_i - 20) / 86400        (concentration units per second; may be < 0)
 *         r   = exchange_k * exchange_theta_k^(T_i - 20) / 86400    (1/s, >= 0)
 *         ceq = equilibrium_k (kind 0) | O2sat(T_i) (kind 1, mg/L)
 *         phi = -expm1(-r dt[t]) / r, or dt[t] when r == 0
 *         c~_k += (s + r (ceq - c~_k)) * phi                        (exact solution of dc/dt = s + r (ceq - c) over dt)
 * and the rest of the step (ghost terms, warm start, solve, BC re-imposition, mass flux) takes the reacted c~'.  History
 * rows are not rewritten: c[t] stays what transport or the override produced; the reaction of step t shows in c[t+1].
 * Ghost cells and BC values are not reacted; without Monod factors nothing is clamped.  Rates are per column (a scenario
 * ensemble may sweep them).
 * With cwr_set_kinetics_limits, a process (the decay of column k, or the source of column k) carries Monod factors on
 * constituents j with half-saturations K > 0, c+ = max(c, 0):
 *         limitation f = c+_j / (K + c+_j),  inhibition f = K / (K + c+_j),  M = product of the process's factors in the
 *         order given, from 1.0
 *     c_j is read as the row holds it when the process is applied (decays in the topological order above -- factors add no
 *     edges to the yield graph --, then the source columns in ascending k); T is still the value before the reactions.
 *     decay:  r_eff = r M;  loss = c~_k * (-expm1(-r_eff dt[t]));  for every limitation on a j the decay consumes
 *             (yields[j, k] < 0): loss = min(loss, c+_j / -yields[j, k]), the quotient rounded toward -inf;  then c~_k
 *             and the yields as above
 *     source: a factor on another column: s M in place of s.  A limitation on the column itself (a sink, s < 0) is the
 *             first-order sink a = -s M' / (K + c+_k) (M': the other factors), frozen at the value before the term:
 *             c~_k += (r ceq - (r + a) c~_k) * phi, phi = -expm1(-(r + a) dt[t]) / (r + a), or dt[t] when r + a == 0
 *     So a constituent stays >= 0 at every step size when it starts >= 0, every process that consumes it is limited by
 *     it, its own sink is self-limited and its equilibrium is >= 0.  The cap holds exactly in floating point for any
 *     yield: the rounded-down quotient keeps -yields[j, k] * loss <= c+_j.  This covers the reaction; transport adds
 *     only solver-tolerance noise.  Processes without factors are computed exactly as without cwr_set_kinetics_limits.
 * With cwr_set_kinetics_depth, a process may be given per unit depth -- a settling velocity, an areal source such as
 * sediment oxygen demand, a surface transfer velocity -- and acts through the depth of cell i at step t:
 *         h_i = max(V_i[t] / A_i, min_depth)      (V[t]: the f32 volume of the load term and the reaction mass, in f64)
 *     with A_i the cell's plan area.  A flagged rate, its theta^(T_i - 20) included, is divided by h_i before use, as a
 *     product with the rounded reciprocal g_i = 1 / h_i (one division per cell):
 *         decay:    r = decay_k * theta_k^(T_i - 20) / 86400 * g_i          (decay_k: a velocity, length / day)
 *         source:   s = source_k * source_theta_k^(T_i - 20) / 86400 * g_i  (source_k: concentration x length / day)
 *         exchange: r = exchange_k * exchange_theta_k^(T_i - 20) / 86400 * g_i   (exchange_k: length / day)
 *     Everything else -- the yields, the Monod factors and the cap, the self-limited sink a = -s M' / (K + c+_k) with this
 *     s, the order of the chain, the exact per-step solutions -- is unchanged, so the non-negativity guarantee above holds
 *     at any depth, min_depth included.  Lengths are in the mesh's unit, volume unit / area unit: m for SI plans, ft for
 *     US-customary ones.  An areal flux in g/m2/day on a plan in ft is given as flux / 0.3048 (mg/L ft/day); a velocity in
 *     m/day as v / 0.3048.  A dry cell (V = 0) takes h = min_depth: its rates stay finite and its load term is 0.
 * O2sat is the APHA / Benson-Krause freshwater saturation at 1 atm, Ta = T + 273.15 K:
 *     ln O2sat = -139.34411 + 1.575701e5/Ta - 6.642308e7/Ta^2 + 1.243800e10/Ta^3 - 8.621949e11/Ta^4
 *
 * decay_per_day (K) or NULL = kinetics off; theta (K) or NULL = all 1; yields (K,K) row-major,
 * yields[j*K + k] = mass of j formed per mass of k decayed, or NULL = none; temperature_k = index of the
 * temperature constituent or -1 for the constant temperature_c.  Takes effect for steps queued after the call
 * (stream-ordered upload) and clears the sources, the limits and the depth flags.  CWR_EINVAL for a negative or non-finite decay, theta <= 0 or
 * non-finite, a non-finite yield or yields[k*K + k] != 0, a cycle in the yield graph, a temperature constituent that
 * decays or receives a yield, an index out of range.  Domain decomposition: every rank makes the same call. */
int cwr_set_kinetics(cwr_handle* h, const double* decay_per_day, const double* theta, const double* yields,
                     int temperature_k, double temperature_c);
/* Zero-order sources and relaxation toward an equilibrium (reaeration, equilibrium temperature), applied after the
 * first-order chain of the kinetics set last (see above); all arrays (K).  source_per_day (concentration units per day)
 * or NULL = none; exchange_per_day (1/day) or NULL = none; both NULL = sources off; a theta NULL = all 1; equilibrium
 * (the constant target of kind 0); equilibrium_kind 0 = constant, 1 = O2sat(T), or NULL = all 0.  Acts only while
 * kinetics is set (all-zero decay rates are allowed); cwr_set_kinetics clears it; it clears the limits and the depth flags.  Stream-ordered
 * upload.  CWR_EINVAL
 * when kinetics is not set, for a non-finite source, a theta <= 0 or non-finite, a negative or non-finite exchange, a kind
 * other than 0 or 1, exchange without equilibrium, a non-finite equilibrium of a kind-0 column with exchange > 0, or kind 1
 * on the temperature constituent.  The reaction mass includes these terms.  Domain decomposition: every rank makes the
 * same call. */
int cwr_set_kinetics_sources(cwr_handle* h, const double* source_per_day, const double* source_theta,
                             const double* exchange_per_day, const double* exchange_theta,
                             const double* equilibrium, const int* equilibrium_kind);
/* Monod limitation and inhibition of the kinetics and sources set last (see above); arrays (n): factor i scales process
 * process[i] (0 = the decay of column[i], 1 = its source) by a factor of kind factor_kind[i] (0 = limitation, 1 =
 * inhibition) on constituent factor_column[i] with half-saturation half_saturation[i].  n == 0 or a NULL array = limits
 * off.  Acts only while kinetics is set; cwr_set_kinetics and cwr_set_kinetics_sources clear it, so the order is kinetics,
 * sources, limits.  Stream-ordered upload.  CWR_EINVAL when kinetics is not set, for n < 0, a process or kind other than 0
 * or 1, a column index out of range, a half-saturation <= 0 or non-finite, a decay factor on a column whose decay is 0 or
 * a source factor on a column whose source is 0, a decay factor on its own column, a source factor on its own column that
 * is an inhibition or whose source is >= 0, or the same (process, column, factor column, kind) twice.  Domain
 * decomposition: every rank makes the same call. */
int cwr_set_kinetics_limits(cwr_handle* h, int n, const int* process, const int* column, const int* factor_column,
                            const int* factor_kind, const double* half_saturation);
/* Depth-scaled processes of the kinetics and sources set last (see above).  cell_area (F) in reference numbering, the plan
 * area of every cell (only the real cells are read); min_depth > 0 the floor of h; decay_per_depth, source_per_depth,
 * exchange_per_depth (K) each 0 / 1 or NULL = none: 1 divides that process's rate of column k by h.  All flags NULL or 0 =
 * depth off (cell_area may then be NULL).  Acts only while kinetics is set; cwr_set_kinetics and cwr_set_kinetics_sources
 * clear it; it and cwr_set_kinetics_limits do not clear each other, so the order is kinetics, sources, then limits and
 * depth in either order.  Stream-ordered upload, the areas permuted to the device order like the volumes.  CWR_EINVAL
 * when kinetics is not set, for a flag other than 0 or 1, a flag on a process whose rate is 0, a flag with cell_area NULL,
 * a real cell's area not finite and > 0, or min_depth not finite and > 0.  Domain decomposition: every rank makes the
 * same call. */
int cwr_set_kinetics_depth(cwr_handle* h, const double* cell_area, double min_depth, const int* decay_per_depth,
                           const int* source_per_depth, const int* exchange_per_depth);
/* Time-varying forcing of the kinetics and sources set last (see above): n series of n_time values each, values (n,
 * n_time) row-major, one per model time index; step t uses entry t (the index of vol[t] and dt[t]), held over the step.
 * Series i has target[i] and column[i]:
 *     CWR_FORCE_TEMPERATURE     column -1: replaces temperature_c (only while temperature_k == -1); O2sat(T) follows it
 *     CWR_FORCE_EQUILIBRIUM     replaces the constant equilibrium of column k (exchange > 0, equilibrium kind 0)
 *     CWR_FORCE_DECAY_SCALE     multiplies the decay rate of column k
 *     CWR_FORCE_SOURCE_SCALE    multiplies the source of column k
 *     CWR_FORCE_EXCHANGE_SCALE  multiplies the exchange rate of column k
 * A scale f multiplies the per-day rate (rate * f[t] in fp64) before anything else acts on it: the theta^(T - 20)
 * correction, the depth, the Monod factors and the cap, the exact per-step solutions.  A scale of 1, or a series equal to
 * the constant it replaces, gives the bits of the unforced step.  Scales are >= 0, so a sink stays a sink and the
 * non-negativity guarantee above holds; under an equilibrium series it holds where the series is >= 0 (not checked).
 * n == 0 = forcing off.  Acts only while kinetics is set; cwr_set_kinetics and cwr_set_kinetics_sources clear it; it,
 * cwr_set_kinetics_limits and cwr_set_kinetics_depth do not clear each other.  Stream-ordered upload.  CWR_EINVAL when
 * kinetics is not set, for n < 0, n_time other than the handle's, a NULL array with n > 0, an unknown target, a column
 * out of range or a temperature series with a column other than -1, the same (target, column) twice, a non-finite
 * value, a negative scale, a scale on a process whose rate is 0, a temperature series while a temperature constituent
 * is set, or an equilibrium series on a column without exchange or one that relaxes toward O2sat.  The reaction mass
 * includes the forced rates.  Domain decomposition: every rank makes the same call. */
enum {
    CWR_FORCE_TEMPERATURE = 0,
    CWR_FORCE_EQUILIBRIUM = 1,
    CWR_FORCE_DECAY_SCALE = 2,
    CWR_FORCE_SOURCE_SCALE = 3,
    CWR_FORCE_EXCHANGE_SCALE = 4
};
int cwr_set_kinetics_forcing(cwr_handle* h, int n, int n_time, const int* target, const int* column,
                             const double* values);
/* Reaction mass of constituent k, sum over the steps taken of sum_i V[t]_i (c~'_ik - c~_ik), reduced on the device in a fixed
 * order (the same bits every run): a running sum since cwr_create, 0 while kinetics was never set.  Domain decomposition:
 * the partial sum over the rows the rank owns (as cwr_mass_totals_at). */
int cwr_get_reaction_mass(cwr_handle* h, int k, double* total);

/* --- domain decomposition over NVLink (SURVEY.md 8e-ii; BASELINE configs[4]) ----------------------------
 * One process per GPU creates a handle with options.dd_rank / dd_world set, every rank with the SAME mesh,
 * hydrodynamics and inputs (the mesh is replicated, the rows are not: a rank assembles, solves and stores
 * only its strip).  cwr_dd_export gives the CUDA IPC handle of the rank's symmetric slab (CWR_IPC_HANDLE_BYTES
 * bytes); the host exchanges them (torch.distributed / MPI all-gather) and passes all dd_world of them, in
 * rank order, to cwr_dd_attach.  From then on the kernels store boundary rows straight into the peers that read
 * them and all-reduce the BiCGSTAB dot products through peer inboxes; every rank must make the same calls in
 * the same order.  Outputs of a rank are valid for the cells / edges it owns (cwr_dd_layout masks, reference
 * numbering) plus its halo; mass totals and flux sums are partial sums over the owned part. */
#define CWR_IPC_HANDLE_BYTES 64
typedef struct {
    int rank, world;
    int rows_owned;         /* cells of this rank's strip */
    int rows_sent;          /* of those, cells other ranks read (halo volume per exchange) */
    int neighbour_mask;     /* bit q: rank q exchanges rows with this one */
    int n_colors, n_levels;
} cwr_dd_info;
int cwr_dd_export(cwr_handle* h, void* ipc_handle);
int cwr_dd_attach(cwr_handle* h, const void* ipc_handles /* dd_world * CWR_IPC_HANDLE_BYTES */);
int cwr_dd_layout(cwr_handle* h, cwr_dd_info* info, uint8_t* owned_cells /* (n_real,) or NULL */,
                  uint8_t* owned_edges /* (E,) or NULL */);

/* --- introspection used by the parity tests -------------------------------------------------- */
/* CSR of A(t) as last assembled, reference numbering, diagonal included, columns sorted:
 * call with NULL arrays to get nnz. */
int cwr_get_lhs(cwr_handle* h, int64_t* nnz, int32_t* indptr, int32_t* indices, double* data);
int cwr_get_rhs(cwr_handle* h, int k, double* b);           /* (n,) f64, unscaled */
int cwr_get_permutation(cwr_handle* h, int32_t* new_of_old); /* (n,) */
int cwr_get_options(const cwr_handle* h, cwr_options* resolved); /* the options in force (autos resolved) */
int cwr_stream(cwr_handle* h, void** cuda_stream);           /* the handle's cudaStream_t */
int cwr_counters(cwr_handle* h, int64_t* kernel_launches, int64_t* solver_iterations);
/* Defect-correction solver: Gauss-Seidel sweeps done so far, solves that fell back to BiCGSTAB; the strips of the
 * neighbour-synchronised sweep kernel (0 when it is not in use) and the most strips any strip waits for.  Any may be NULL. */
int cwr_solver_stats(cwr_handle* h, int64_t* sweeps, int64_t* fallbacks, int* n_strips, int* max_strip_neighbours);
/* Host only (no device needed): the cell ordering cwr_create / the first cwr_set_hydro* would build --
 * reverse Cuthill-McKee, then (n_colors > 0) the flow-aligned multicolouring of the Gauss-Seidel sweeps, then
 * (n_parts > 1) the strips of the domain decomposition; rows end up ordered (part, colour, level, RCM).
 * flow_hint: (E,) signed face flow (> 0 leaves f1) or NULL; new_of_old: (n_real,); color_ptr: (n_parts, n_colors_out+1)
 * absolute row ranges of each part's colours (room for 8 * 65 entries), may be NULL; part_ptr: (n_parts+1) rows owned
 * by each part, may be NULL; n_send: (n_parts) rows of a part that other parts read (halo volume), may be NULL. */
int cwr_order_cells(int n_real, int n_face, int n_edge, const int32_t* f1, const int32_t* f2, int reorder, int n_colors,
                    const float* flow_hint, int n_parts, int32_t* new_of_old, int32_t* color_ptr, int* n_colors_out,
                    int* n_levels, int32_t* part_ptr, int32_t* n_send);

/* Host only: the strips of the neighbour-synchronised sweep kernel (precond_sync = 2) build_topology makes -- every part
 * cut into n_strips equal chunks of the RCM order, rows ordered (part, strip, colour, RCM position).  Call once with the
 * array pointers NULL for the sizes (n_colors_out, nbr_total), then with arrays: new_of_old (n_real), strip_cptr
 * (n_parts * n_strips, n_colors + 1: absolute row ranges of a strip's colours), strip_nptr (n_parts * n_strips + 1) and
 * strip_nbr (nbr_total): the strips (global ids, other parts included) a strip shares an edge with, color_of (n_real, new numbering).
 * strip_cap > 0: the rows a (strip, colour) would hold beyond strip_cap (one pass of the sweep kernel's CTA: 256 at
 * K = 16) are moved to the nearest later colour that no neighbour has and that has room; 0 = colours as levelled. */
int cwr_strip_layout(int n_real, int n_face, int n_edge, const int32_t* f1, const int32_t* f2, int n_colors, const float* flow_hint,
                     int n_parts, int n_strips, int* n_colors_out, int* nbr_total, int32_t* new_of_old, int32_t* strip_cptr,
                     int32_t* strip_nptr, int32_t* strip_nbr, uint8_t* color_of, int strip_cap);

/* --- device timing of the dominant kernel (bench.py roofline) -------------------------------- */
/* Per-kernel-family device time inside cwr_step, measured with CUDA events recorded on the handle's
 * stream between the launches.  cwr_profile(h, 1, NULL, NULL) switches it on (and zeroes the sums),
 * (h, 0, ...) off, (h, -1, ms, counts) only reads: accumulated milliseconds and launch counts. */
enum {
    CWR_FAM_ASSEMBLE = 0,   /* k_boundary_diag + k_assemble */
    CWR_FAM_RHS,            /* k_rhs + k_boundary_rhs */
    CWR_FAM_SPMM_INIT,      /* r = b - A x0 */
    CWR_FAM_SPMM_V,         /* v = A p  with (rhat, v) */
    CWR_FAM_UPDATE_S,       /* s = r - alpha v with (s, s): the half-step convergence test */
    CWR_FAM_SPMM_T,         /* t = A s  with the four dots */
    CWR_FAM_UPDATE_XRP,     /* x, r, p updates with (r, r) */
    CWR_FAM_MASS_FLUX,
    CWR_FAM_PRECOND,        /* the preconditioner: one k_precond_gs launch = all Gauss-Seidel sweeps of one application
                               (precond_sweep = 1), or one Jacobi step out = u + N z per launch (precond_sweep = 0) */
    CWR_FAM_SOLVE_SMALL,    /* small meshes: the whole solve of every column, one CTA each (k_solve_tiny / k_solve_small) */
    CWR_FAM_DC_UPDATE,      /* defect-correction solver: r -= A z, x += z with (r, r) and the plan of the next cycle */
    CWR_PROFILE_FAMILIES
};
int cwr_profile(cwr_handle* h, int enable, double* ms, int64_t* counts);

/* Time `reps` launches of the SpMM/SpMV kernel (y = A x over all K columns) with CUDA events on
 * the handle's stream; returns average milliseconds per launch and the algorithmic bytes of one
 * launch (12*nnz_off + 4*(n+1) + 16*n*K, SURVEY.md 8d). */
int cwr_time_spmm(cwr_handle* h, int reps, double* ms_per_launch, double* algorithmic_bytes);

#ifdef __cplusplus
}
#endif
#endif /* CWR_H */
