// sm_100a kernels of the transport step.  Results, BiCGSTAB recurrences, products and dot products are fp64; only
// the preconditioner sweeps and the preconditioned vectors are fp32.  HBM-bound gather/stream work, so the
// design rules are: coalescing (constituents interleaved, x[row*K + k]: one 128 B line per row at
// K = 16, moved as 128-bit packs per lane), a fixed-width row-major ELL matrix (one int4 + two
// double2 broadcast loads per row, no rowptr dependency in front of the gathers), persistent grids
// sized from the SM count, fused dot products with a deterministic two-level reduction (no
// floating-point atomics anywhere), per-step parameters read from a device-resident struct so
// that a step is the same launch sequence every time, and -- across GPUs -- boundary rows and dot products
// exchanged through peer-mapped memory from inside the kernels (see the domain-decomposition section).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "cwr_topology.h"   // kColMask: ell_col bit 31 marks a neighbour visited later in a Gauss-Seidel sweep

namespace cwr {

constexpr int kThreads = 256;
constexpr int kMaxK = 128;      // constituents per handle
constexpr int kMaxDots = 4;
#ifndef CWR_SPMM_MIN_BLOCKS
#define CWR_SPMM_MIN_BLOCKS 4   // resident CTAs per SM the SpMM kernels are compiled for (register cap 64)
#endif
#ifndef CWR_AT_MIN_BLOCKS
#define CWR_AT_MIN_BLOCKS 3     // the four-dot product t = A s^ (MODE_AT): 80 registers, no spills (157 -> 118 us; 2: 137 us)
#endif

// Per-step pointers/values; written by k_set_step and read by every kernel of the step.
struct StepParams {
    const float* adv_t;      // (E)  advection_coeff[t]       device edge order
    const double* cdiff_t;   // (E)  coeff_to_diffusion[t]
    const float* vol_t;      // (n)  volume[t]   real cells, device cell order
    const float* vol_t1;     // (n)  volume[t+1]
    const float* adv_t1;     // (E)  advection_coeff[t+1]
    const double* cdiff_t1;  // (E)  coeff_to_diffusion[t+1]
    const float* velg_t1;    // (E_g) edge_velocity[t+1] of ghost edges
    const float* flowg_t;    // (E_g) face_flow[t] of ghost edges (boundary volume sums, postproc_util.py:93-95)
    const double* bc_t1;     // (G,K) input_array[t+1][ghost cells]
    const double* state_t;   // (n,K) c[t]
    double* state_t1;        // (n,K) c[t+1]  (the solver iterates in place on it)
    double dt;               // dt[t]
    int t;
    int apply_ic;            // t == 0: input_array[0] overrides c~ where non-zero (linalg.py:199-200)
};

enum ScalarRow { SC_RHO = 0, SC_ALPHA, SC_OMEGA, SC_BETA, SC_BNORM2, SC_RNORM2, SC_RHATV, SC_ROWS };
enum ColFlag { FL_CONVERGED = 1, FL_BREAKDOWN = 2, FL_NAN = 4, FL_ZERO_RHS = 8, FL_PENDING = 16, FL_HALF = 32 };

struct SolverCtl {
    int all_done;       // every column converged / failed / fixed
    int iter;           // BiCGSTAB iterations done in this solve
    int flags_or;       // OR of column flags that matter to the host (breakdown, nan)
    int singular;       // a zero diagonal was met during assembly
    int hit_max_iter;
    int barrier_timeout; // a grid barrier of the persistent sweep kernel gave up (never expected)
    int pad[2];
    unsigned ticket[4]; // last-block tickets (one per kernel family)
    unsigned ticket_halo; // k_halo_push
    unsigned ticket_s;    // k_update_s
    int finish_half;      // every active column converged at the half step: skip the sweeps on s and t = A s^
    unsigned gs_bar[2]; // k_precond_gs: grid barrier arrivals, exits
    // defect-correction solver (solver = 2): x += GS^S(r), r -= A z, with S planned on the device after every cycle
    unsigned long long strip_base;   // k_gs_strip: warp arrivals every strip's flag has counted in the launches so far
    int dc_sweeps;        // sweeps of the next cycle
    int dc_fail;          // the sweeps stagnate or diverge (not an M-matrix?): the host falls back to BiCGSTAB
    int dc_slow;          // consecutive cycles that reduced the residual by less than 0.7
    int sweeps_done;      // Gauss-Seidel sweeps of this solve
    double dc_rate;       // error factor per sweep measured over the last cycle (kept across steps)
    double dc_worst;      // max over columns of (||r|| / ||b||) / rtol after the last cycle
};

constexpr int kMaxRanks = 8;

// Control block of the domain-decomposed path, at the start of every rank's symmetric slab: peers write
// their announcements straight into it over NVLink (peer-mapped stores).
struct DdCtl {
    unsigned long long bar_flag[kMaxRanks];   // [q]: last halo/barrier epoch rank q announced   (written by rank q)
    unsigned long long dot_flag[kMaxRanks];   // [q]: last dot-product epoch rank q announced     (written by rank q)
    unsigned long long bar_epoch, dot_epoch;  // this rank's own counters (local use only)
    int timeout;                              // a bounded wait on a peer gave up (never expected)
    int pad[27];
    double dot_inbox[2][kMaxRanks][kMaxDots * kMaxK];   // [epoch parity][from rank][dot * K + k]
};
constexpr int kFlagStride = 16;                // strip flags: one per 128-byte line
constexpr size_t kDdCtlBytes = 1 << 20;       // room reserved at the head of the slab: DdCtl, and from kDdFlagOffset the strip flags
constexpr size_t kDdFlagOffset = 512 << 10;   // (several ranks: a strip's flag is mirrored into the ranks that read its rows)

struct DeviceModel {
    int n, K, E, E_int, E_g, G, nb, W;     // W = ELL width (multiple of 4)
    // rows / edges / boundary cells this rank owns (everything when world == 1)
    int row_lo, row_hi, ie_lo, ie_hi, ge_lo, ge_hi, b_lo, b_hi;
    int rank, world;
    unsigned nbr_mask;            // ranks this one exchanges halo rows with
    const uint8_t* send_mask;     // (n) bit q: rank q reads this row (0 for interior rows)
    const int32_t* send_rows; int n_send;   // this rank's rows with a non-zero send_mask
    int halo_per_sweep;           // Gauss-Seidel kernel: halo rows cross once per sweep (1) or after every colour (0)
    char* peer_base[kMaxRanks];   // every rank's symmetric slab (own included): DdCtl, p^, s^, tmp, state slots
    char* sym_base;               // == peer_base[rank]
    DdCtl* dd;
    const int32_t* ell_col;   // (n,W) neighbour row (& kColMask), padded with the row itself
    const int32_t* ell_code;  // (n,W) (e' << 1) | side, -1 = padding
    const int32_t* f1p; const int32_t* f2p;
    const int32_t* bcell; const int32_t* bptr; const int32_t* bedge;
    const int32_t* color_ptr; int n_colors;   // (n_colors+1) row ranges of the Gauss-Seidel colours
    // strips of the neighbour-synchronised Gauss-Seidel kernel (cwr_topology.h): CTA b owns strip strip0 + b
    const int32_t* strip_cptr; const int32_t* strip_nptr; const int32_t* strip_nbr;
    const uint8_t* strip_peers;       // (all strips, global ids) bit q: rank q reads rows of the strip
    unsigned long long* strip_flag;   // (all strips, global ids; x kFlagStride: one 128-byte line per strip -- the polls of 48 warps per flag would
                                      // otherwise queue at the one L2 slice that owns 16 flags) progress of a strip, see the sweep kernels
    int n_strips, strip0;
    int us_from_producer;             // the kernels that produce the residual also write it in the sweep type to M.us (k_gs_strip)
    int sweep_f32;                    // sweep type is float
    int dc_smin, dc_smax;             // sweeps per defect-correction cycle: bounds of the device-side plan
    double dc_floor;                  // largest residual reduction one cycle can deliver in the sweep precision
    double* val;        // (n,W) off-diagonals of D^-1 A
    float* valf;        // (n,W) the same in fp32 (fp32 preconditioner sweeps), or nullptr
    double* diag;       // (n)   D
    double* gdiag;      // (n)   ghost-edge diagonal terms (boundary cells only, 0 elsewhere)
    const double* ic;   // (n,K) input_array[0][0:n]
    double *b, *r, *rhat, *p, *v, *tt, *xc;   // (n,K) work vectors (b is the row-scaled RHS)
    // preconditioned vectors p^ and s^, the sweep ping-pong partner and the sweep-precision copy of the
    // preconditioner's input: (n,K) of the SWEEP type (float by default, double with precond_precision = 64;
    // the small-mesh path uses them as double).  Allocated 8 bytes per entry either way.
    void *ph, *sh, *tmp, *us;
    double* partials;   // (kMaxDots * K, grid): per-CTA partial dot products, block index fastest
    double* sc;         // (SC_ROWS, K) per-column scalars
    int* colflags;      // (K)
    int* coliters;      // (K)
    SolverCtl* ctl;
    const StepParams* sp;
    double* flux;       // (3, E, K) advection / diffusion / total mass flux of the last step
    double* bsum;       // (3, E_g, K) running total / in / out sums of the total mass flux on ghost edges
    double* vsum;       // (3, E_g) running total / in / out sums of face_flow * dt on ghost edges
    double tol2;        // rtol^2
    double diffusion_coefficient;
    int max_iter;
    int want_flux;
};

// Programmatic dependent launch (small-mesh path: a step is a chain of 6 - 8 launches of a few microseconds each, so the
// gaps between them count).  The host launches these kernels with programmaticStreamSerialization; each lets its successor
// be scheduled at once and waits for its predecessor's memory before it touches anything.  Launched without the attribute
// (the large path) both instructions do nothing.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_enter() {
    pdl_launch_dependents();
    pdl_wait();
}

__global__ void k_set_step(StepParams p, StepParams* dst, SolverCtl* ctl, DdCtl* dd) {
    pdl_enter();
    *dst = p;
    if (dd) dd->timeout = 0;            // (a peer that was slow in an earlier step is waited for again)
    ctl->all_done = 0; ctl->iter = 0; ctl->flags_or = 0; ctl->hit_max_iter = 0; ctl->finish_half = 0;
    ctl->singular = 0; ctl->dc_fail = 0; ctl->dc_slow = 0; ctl->sweeps_done = 0;
}

// The solver's control block and per-column scalars, written into page-locked host memory that the device maps
// (zero-copy): the host polls convergence by synchronising the stream and reading its own memory.  A cudaMemcpy
// would queue behind the bulk device->host copies of the asynchronous output path on the same copy engine.
struct HostMirror {
    SolverCtl ctl;
    double sc[SC_ROWS * kMaxK];
    int flags[kMaxK];
};
__global__ void k_mirror(const SolverCtl* __restrict__ ctl, const double* __restrict__ sc, const int* __restrict__ flags, int K,
                         HostMirror* __restrict__ dst, int with_columns) {
    if (with_columns) {
        for (int q = threadIdx.x; q < SC_ROWS * K; q += blockDim.x) dst->sc[q] = sc[q];
        for (int q = threadIdx.x; q < K; q += blockDim.x) dst->flags[q] = flags[q];
    }
    const int words = (int)(sizeof(SolverCtl) / sizeof(int));
    for (int q = threadIdx.x; q < words; q += blockDim.x) reinterpret_cast<int*>(&dst->ctl)[q] = reinterpret_cast<const int*>(ctl)[q];
    __threadfence_system();
}

// ---------------------------------------------------------------------------------------------
// upload helpers: reference order -> device order
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_gather(T* __restrict__ dst, const T* __restrict__ src, const int32_t* __restrict__ idx, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[idx[i]];
}

__global__ void k_scatter_column(double* __restrict__ dst, const double* __restrict__ src,
                                 const int32_t* __restrict__ old_of_new, int n, int K, int k) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        dst[(size_t)i * K + k] = src[old_of_new[i]];
}

// bc[(t*G + g)*K + k] = input[t*F + n + g]
__global__ void k_scatter_bc(double* __restrict__ bc, const double* __restrict__ input, int T, int F, int n, int G, int K, int k) {
    size_t total = (size_t)T * G;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        size_t t = i / G, g = i % G;
        bc[i * K + k] = input[t * F + n + g];
    }
}

__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000LL); }

// out[F]: real cells from the interleaved state (reference order), ghost cells: BC value or NaN
__global__ void k_extract_state(double* __restrict__ out, const double* __restrict__ state, const double* __restrict__ bc_t,
                                const int32_t* __restrict__ new_of_old, int n, int F, int K, int k) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < F; j += gridDim.x * blockDim.x) {
        double v;
        if (j < n) v = state[(size_t)new_of_old[j] * K + k];
        else {
            v = bc_t ? bc_t[(size_t)(j - n) * K + k] : 0.0;
            if (v == 0.0) v = qnan();   // transport.py:258-264: unset ghost cells stay NaN
        }
        out[j] = v;
    }
}

// out[(k, j)] for all constituents, reference order: rows of the interleaved (rows, K) array `src` gathered through
// `perm` (reference index j -> device row) and transposed through shared memory, so that both the reads (K values of
// one row: one 8K-byte segment) and the writes (32 consecutive j of one column) are coalesced.  Used for c[t+1]
// (perm = new_of_old over the n real cells) and for the three mass-flux arrays (perm = einv over the E edges).
constexpr int kXposeRows = 32;
__global__ void __launch_bounds__(kThreads) k_extract_all(double* __restrict__ out, const double* __restrict__ src,
                                                          const int32_t* __restrict__ perm, int n, int K, size_t out_stride_k) {
    extern __shared__ double xt[];                     // [kXposeRows][K + 1]
    const int ld = K + 1;
    for (int j0 = blockIdx.x * kXposeRows; j0 < n; j0 += gridDim.x * kXposeRows) {
        const int rows = min(kXposeRows, n - j0);
        for (int q = threadIdx.x; q < rows * K; q += blockDim.x) {
            const int r = q / K, k = q % K;
            xt[r * ld + k] = src[(size_t)perm[j0 + r] * K + k];
        }
        __syncthreads();
        for (int q = threadIdx.x; q < rows * K; q += blockDim.x) {
            const int k = q / rows, r = q % rows;
            out[(size_t)k * out_stride_k + j0 + r] = xt[r * ld + k];
        }
        __syncthreads();
    }
}

__global__ void k_scatter_all(double* __restrict__ state, const double* __restrict__ src, const uint8_t* __restrict__ mask,
                              const int32_t* __restrict__ new_of_old, int n, int K) {
    size_t total = (size_t)n * K;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        int k = (int)(i / n), j = (int)(i % n);
        if (mask == nullptr || mask[k]) state[(size_t)new_of_old[j] * K + k] = src[i];
    }
}

// out[e] (reference edge order) = flux[which][e'][k]
__global__ void k_extract_flux(double* __restrict__ out, const double* __restrict__ flux, const int32_t* __restrict__ einv,
                               int E, int K, int k) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < E; e += gridDim.x * blockDim.x)
        out[e] = flux[(size_t)einv[e] * K + k];
}

// ---------------------------------------------------------------------------------------------
// "next" row N1: derive adv / cdiff from the raw HEC-RAS arrays (reference utilities.py:513-541)
//   adv = face_flow * sign(|vel|)  (f32);  area = adv / vel, NaN -> 0 (f32);
//   cdiff = f64(f32(area * D)) / dist
// input in reference edge order, output in device edge order.
// ---------------------------------------------------------------------------------------------
__global__ void k_derive(float* __restrict__ adv, double* __restrict__ cdiff, float* __restrict__ velg, float* __restrict__ flowg,
                         const float* __restrict__ flow, const float* __restrict__ vel, const double* __restrict__ dist,
                         const int32_t* __restrict__ eperm, int E, int E_int, float Df) {
    for (int ep = blockIdx.x * blockDim.x + threadIdx.x; ep < E; ep += gridDim.x * blockDim.x) {
        int e = eperm[ep];
        float q = flow[e], u = vel[e];
        float au = fabsf(u);
        float sg = (au > 0.f) ? 1.f : ((au == 0.f) ? 0.f : au);     // sign(|u|); NaN stays NaN
        float a = __fmul_rn(q, sg);
        float area = __fdiv_rn(a, u);
        if (area != area) area = 0.f;                                // fillna(0)
        float ad = __fmul_rn(area, Df);
        adv[ep] = a;
        cdiff[ep] = (double)ad / dist[e];
        if (ep >= E_int) { velg[ep - E_int] = u; flowg[ep - E_int] = q; }
    }
}

__global__ void k_dist(double* __restrict__ dist, const double* __restrict__ fx, const double* __restrict__ fy,
                       const int32_t* __restrict__ f1, const int32_t* __restrict__ f2, int E) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < E; e += gridDim.x * blockDim.x) {
        double dx = fx[f1[e]] - fx[f2[e]], dy = fy[f1[e]] - fy[f2[e]];
        dist[e] = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));   // no fma contraction: matches numpy
    }
}

// ---------------------------------------------------------------------------------------------
// LHS assembly  (reference linalg.py:34-156 + transport.py:215-218)
// ---------------------------------------------------------------------------------------------
// ghost-edge diagonal terms: sum over a boundary cell's ghost edges of cdiff + max(adv, 0)
// (linalg.py:92-97 and 113-115 applied to ghost edges).
__global__ void k_boundary_diag(DeviceModel M) {
    pdl_enter();
    const StepParams& sp = *M.sp;
    for (int b = M.b_lo + blockIdx.x * blockDim.x + threadIdx.x; b < M.b_hi; b += gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int j = M.bptr[b]; j < M.bptr[b + 1]; ++j) {
            int e = M.bedge[j];
            s += sp.cdiff_t[e] + fmax((double)sp.adv_t[e], 0.0);
        }
        M.gdiag[M.bcell[b]] = s;
    }
}

// One thread per row: diagonal D_i and the row's off-diagonals, written once into their fixed
// slots, already divided by D_i (row-scaled system D^-1 A, unit diagonal implied).
//   internal edge e = (P = f1, N = f2), a = adv[t,e], d = cdiff[t,e]:
//     A[P,N] = -d + min(a,0)   A[N,P] = -d - max(a,0)
//     A[P,P] += d + max(a,0)   A[N,N] += d - min(a,0)
//   A[i,i] += vol[t+1,i]/dt[t]  (+1 if vol[t+1,i] == 0, linalg.py:66,77-81)
__global__ void __launch_bounds__(kThreads) k_assemble(DeviceModel M) {
    pdl_enter();
    const StepParams& sp = *M.sp;
    const double dt = sp.dt;
    const int W = M.W;
    for (int i = M.row_lo + blockIdx.x * blockDim.x + threadIdx.x; i < M.row_hi; i += gridDim.x * blockDim.x) {
        const float vol = sp.vol_t1[i];
        double diag = (vol == 0.f ? 1.0 : 0.0) + (double)vol / dt + M.gdiag[i];
        const int32_t* code = M.ell_code + (size_t)i * W;
        double* val = M.val + (size_t)i * W;
        if (W == 4) {      // the common width: everything stays in registers, every value is written once
            const int4 c4 = *reinterpret_cast<const int4*>(code);
            const int cs[4] = {c4.x, c4.y, c4.z, c4.w};
            double a[4], d[4], off[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {       // all eight gathers in flight together
                a[u] = cs[u] >= 0 ? (double)sp.adv_t[cs[u] >> 1] : 0.0;
                d[u] = cs[u] >= 0 ? sp.cdiff_t[cs[u] >> 1] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                off[u] = 0.0;
                if (cs[u] >= 0) {
                    if (cs[u] & 1) { off[u] = -d[u] - fmax(a[u], 0.0); diag += d[u] - fmin(a[u], 0.0); }
                    else           { off[u] = -d[u] + fmin(a[u], 0.0); diag += d[u] + fmax(a[u], 0.0); }
                }
            }
            const double inv = 1.0 / diag;
#pragma unroll
            for (int u = 0; u < 4; ++u) off[u] *= inv;
            *reinterpret_cast<double2*>(val) = make_double2(off[0], off[1]);
            *reinterpret_cast<double2*>(val + 2) = make_double2(off[2], off[3]);
            if (M.valf) *reinterpret_cast<float4*>(M.valf + (size_t)i * 4) = make_float4((float)off[0], (float)off[1], (float)off[2], (float)off[3]);
            M.diag[i] = diag;
            if (diag == 0.0) M.ctl->singular = 1;
            continue;
        }
        for (int w = 0; w < W; w += 4) {
            const int4 c4 = *reinterpret_cast<const int4*>(code + w);
            const int cs[4] = {c4.x, c4.y, c4.z, c4.w};
            double off[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                off[u] = 0.0;
                if (cs[u] >= 0) {
                    const double a = (double)sp.adv_t[cs[u] >> 1];
                    const double d = sp.cdiff_t[cs[u] >> 1];
                    if (cs[u] & 1) { off[u] = -d - fmax(a, 0.0); diag += d - fmin(a, 0.0); }
                    else           { off[u] = -d + fmin(a, 0.0); diag += d + fmax(a, 0.0); }
                }
            }
            *reinterpret_cast<double2*>(val + w) = make_double2(off[0], off[1]);
            *reinterpret_cast<double2*>(val + w + 2) = make_double2(off[2], off[3]);
        }
        const double inv = 1.0 / diag;
        for (int w = 0; w < W; w += 2) {
            double2 o = *reinterpret_cast<double2*>(val + w);
            o.x *= inv; o.y *= inv;
            *reinterpret_cast<double2*>(val + w) = o;
            if (M.valf) *reinterpret_cast<float2*>(M.valf + (size_t)i * W + w) = make_float2((float)o.x, (float)o.y);
        }
        M.diag[i] = diag;
        if (diag == 0.0) M.ctl->singular = 1;
    }
}

// ---------------------------------------------------------------------------------------------
// (row, column) thread mapping shared by all vector kernels: KC lanes per row, each lane owns VEC
// adjacent columns (VEC = 2: 128-bit accesses); rows are dealt to lane groups grid-stride.
// ---------------------------------------------------------------------------------------------
template <int VEC> struct Vd { double a[VEC]; };

template <int VEC>
__device__ __forceinline__ Vd<VEC> ldv(const double* p) {
    Vd<VEC> r;
    if (VEC == 2) { const double2 t = *reinterpret_cast<const double2*>(p); r.a[0] = t.x; r.a[VEC - 1] = t.y; }
    else r.a[0] = *p;
    return r;
}
template <int VEC>
__device__ __forceinline__ void stv(double* p, const Vd<VEC>& v) {
    if (VEC == 2) *reinterpret_cast<double2*>(p) = make_double2(v.a[0], v.a[VEC - 1]);
    else *p = v.a[0];
}

// RHS  (reference linalg.py:177-275), K constituents at once, row-scaled by 1/D; warm start x0 = c~
template <int KC, int VEC>
__global__ void __launch_bounds__(kThreads) k_rhs(DeviceModel M) {
    pdl_enter();
    const StepParams& sp = *M.sp;
    const int K = M.K, lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kThreads / KC;
    const double dt = sp.dt;
    for (int c = lane * VEC; c < K; c += KC * VEC)
        for (int i = M.row_lo + blockIdx.x * GPB + group; i < M.row_hi; i += gridDim.x * GPB) {
            const size_t idx = (size_t)i * K + c;
            Vd<VEC> conc = ldv<VEC>(sp.state_t + idx);
            if (sp.apply_ic) {
                const Vd<VEC> ic = ldv<VEC>(M.ic + idx);
#pragma unroll
                for (int q = 0; q < VEC; ++q) if (ic.a[q] != 0.0) conc.a[q] = ic.a[q];
            }
            const double vol = (double)sp.vol_t[i], dg = M.diag[i];
            Vd<VEC> bb;
#pragma unroll
            for (int q = 0; q < VEC; ++q) bb.a[q] = (vol * conc.a[q] / dt) / dg;      // linalg.py:239
            stv<VEC>(M.b + idx, bb);
            stv<VEC>(sp.state_t1 + idx, conc);
        }
}

// Sparse real-cell entries of input_array at t >= 1 (rare): before the solve they replace c~ where non-zero
// (linalg.py:199-200: state and load term recomputed; k_boundary_rhs, which runs afterwards, adds the ghost terms),
// after it they are re-imposed on the stored row (transport.py:258-264).  idx = row * K + column, device order.
__global__ void k_patch_rows(DeviceModel M, const long long* __restrict__ idx, const double* __restrict__ val, int count, int before_solve) {
    pdl_enter();
    const StepParams& sp = *M.sp;
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < count; q += gridDim.x * blockDim.x) {
        const long long i = idx[q];
        const int row = (int)(i / M.K);
        sp.state_t1[i] = val[q];
        if (before_solve) M.b[i] = ((double)sp.vol_t[row] * val[q] / sp.dt) / M.diag[row];
    }
}

// Boundary cells: b_i = load + ghost_in + ghost_out with the reference's selection and
// last-edge-wins assignment (linalg.py:349-351, 372-378, 390).  One lane per (cell, column).
__global__ void __launch_bounds__(kThreads) k_boundary_rhs(DeviceModel M) {
    pdl_enter();
    const StepParams& sp = *M.sp;
    const int K = M.K;
    const double dt = sp.dt;
    const bool has_diffusion = M.diffusion_coefficient != 0.0;
    const size_t total = (size_t)(M.b_hi - M.b_lo) * K;
    for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int b = M.b_lo + (int)(q / K), c = (int)(q % K);
        const int i = M.bcell[b];
        double m_in = 0.0, ca_in = 0.0, cd_in = 0.0, m_out = 0.0, cd_out = 0.0;
        for (int j = M.bptr[b]; j < M.bptr[b + 1]; ++j) {
            const int e = M.bedge[j];
            const float u = sp.velg_t1[e - M.E_int];
            const double bc = sp.bc_t1[(size_t)(M.f2p[e] - M.n) * K + c];
            const double cd = has_diffusion ? fabs(sp.cdiff_t1[e]) : 0.0;
            if (u < 0.f) { m_in = bc; ca_in = fabs((double)sp.adv_t1[e]); cd_in = cd; }
            if (u > 0.f) { m_out = bc; cd_out = cd; }
        }
        const size_t idx = (size_t)i * K + c;
        const double conc = sp.state_t1[idx];                    // c~ written by k_rhs
        const double load = (double)sp.vol_t[i] * conc / dt;
        const double rhs = load + (ca_in + cd_in) * m_in + cd_out * m_out;
        M.b[idx] = rhs / M.diag[i];
    }
}

// ---------------------------------------------------------------------------------------------
// deterministic block / grid reduction of per-column dot products
// ---------------------------------------------------------------------------------------------
// acc[d*VEC + q]: dot d of column (chunk*KC + lane)*VEC + q.  partials layout: [(d*K + k)][block] with
// the block index fastest, so that the final reduction reads them coalesced.
template <int ND, int KC, int VEC>
__device__ __forceinline__ void block_dots(double (&acc)[ND * VEC], double* smem, double* partials, int K, int chunk) {
    constexpr int NA = ND * VEC;
#pragma unroll
    for (int off = KC; off < 32; off <<= 1)
#pragma unroll
        for (int d = 0; d < NA; ++d) acc[d] += __shfl_xor_sync(0xffffffffu, acc[d], off);
    const int wl = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NW = kThreads / 32;
    if (wl < KC)
#pragma unroll
        for (int d = 0; d < NA; ++d) smem[(warp * NA + d) * KC + wl] = acc[d];
    __syncthreads();
    if (threadIdx.x < NA * KC) {
        const int a = threadIdx.x / KC, l = threadIdx.x % KC;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) s += smem[(w * NA + a) * KC + l];
        const int d = a / VEC, q = a % VEC;
        const int c = (chunk * KC + l) * VEC + q;
        if (c < K) partials[(size_t)(d * K + c) * gridDim.x + blockIdx.x] = s;
    }
    __syncthreads();
}

// true in exactly one block: the last one to arrive.  All of the grid's partials are visible to it.
__device__ __forceinline__ bool last_block_arrives(unsigned* ticket) {
    __shared__ int is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(ticket, 1u);
        is_last = (t == gridDim.x - 1);
        if (is_last) *ticket = 0;
    }
    __syncthreads();
    if (is_last) __threadfence();
    return is_last != 0;
}

// Sum the grid's partials -> tot[d*K + k] (shared memory), by the last CTA.  One warp per (dot, column)
// pair: lanes read consecutive blocks (coalesced), accumulate in a fixed order, then a fixed shuffle
// tree combines the lanes -> bitwise deterministic for a given grid size.
template <int ND>
__device__ __forceinline__ void grid_totals(const double* partials, double* tot, int K) {
    const int pairs = ND * K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned G = gridDim.x;
    for (int pair = warp; pair < pairs; pair += kThreads / 32) {
        const double* src = partials + (size_t)pair * G;
        double s0 = 0.0, s1 = 0.0;
        unsigned b = lane;
        for (; b + 32 < G; b += 64) { s0 += __ldcg(src + b); s1 += __ldcg(src + b + 32); }
        if (b < G) s0 += __ldcg(src + b);
        double s = s0 + s1;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        if (lane == 0) tot[pair] = s;
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// First-order kinetics (cwr_set_kinetics): after c~ is formed (k_rhs, k_patch_rows), every owned real row is reacted
//   for the reacting constituents k in topological order of the yield graph:
//     r = decay_k * theta_k^(T - 20) / 86400,  loss = c~_k * (-expm1(-r dt)),  c~_k -= loss,  c~_j += yield[j,k] * loss
// and the load term b = (vol c~' / dt) / D is rewritten with k_rhs's expression (k_boundary_rhs, which runs afterwards,
// reads the reacted c~'), so a zero rate leaves every bit as it was.  The step's reaction mass sum_i vol_i (c~'_ik - c~_ik)
// is reduced per column without atomics: per-thread sums over a fixed set of rows, per-CTA partials, and the last CTA adds
// them in block order (grid_totals).
// Sources and exchange (cwr_set_kinetics_sources) follow the chain in the same row, for the listed columns in ascending k:
//     s = source_k theta_s^(T - 20) / 86400,  r = exchange_k theta_e^(T - 20) / 86400,  ceq = equilibrium_k | O2sat(T)
//     phi = -expm1(-r dt) / r (dt when r == 0),  c~_k += (s + r ceq - r c~_k) phi
// the exact solution of dc/dt = s + r (ceq - c) over dt.  T is the value before any of the step's reactions.
// Monod factors (cwr_set_kinetics_limits) scale a process -- the decay of step p or the source of source column p -- by
// M = prod f in the order given, f = c+_j / (K + c+_j) (limitation) or K / (K + c+_j) (inhibition), c+ = max(c, 0), with
// c_j as the row holds it when the process is applied:
//     decay:   loss = c~_k * (-expm1(-r M dt)), then loss = min(loss, c+_j / -yield[j,k]) for every limitation on a j the
//              process consumes (KinFac.use > 0), the quotient rounded toward -inf so that c~_j + yield[j,k] * loss >= 0
//              holds in floating point for any yield; c~_k and the yields as above
//     source:  s M in place of s; a limitation on the column itself (a sink only) is the first-order sink
//              a = -s M' / (K + c+_k) (M': the other factors), c~_k += (r ceq - (r + a) c~_k) phi(r + a)
// Process q's factors are fl[fptr[q], fptr[q + 1]), q = p for step p and n_steps + p for source column p.  A process with
// factors is evaluated per row (at a constant temperature too); the others take exactly the unfactored code.  Only
// k_react<true> (launched while factors are set) has the factored code: k_react<false> keeps the registers, hence the
// occupancy and the grid (kin_grid_max), that it has without it, and both take that grid, so the column sums of the
// reaction mass are added in the same order with or without factors.
// Depth-scaled processes (cwr_set_kinetics_depth) multiply a flagged rate -- the decay of step p, or the source or the
// exchange of source column p -- by 1 / h, h = max(vol / area, min_depth) the row's depth: vol[t] from the tile (svol),
// area read by the row's thread (coalesced).  One division per row, none per process: a division in the chain is a call
// whose saved registers spill.  dfl[q] holds the flags of process q (numbered as fptr): bit 0 the decay or the source,
// bit 1 the exchange.  A flagged process is evaluated per row by the factored code (at a constant temperature too); the
// others keep their per-CTA coefficients.  Only k_react<true, true> (launched while depth flags are set, with an
// all-empty fptr when there are no factors) has the depth code; it takes the same tile and grid as the others.
// ---------------------------------------------------------------------------------------------
struct KinStep { int col, y_begin, y_end, pad; double decay, log_theta; };   // a reacting constituent; its yields
struct KinYield { int col, pad; double y; };                                 // [y_begin, y_end)
struct KinState { unsigned ticket; int pad; double mass[kMaxK]; };           // last-CTA ticket, running reaction mass
// a column with a source or exchange term; kind 1: ceq = O2sat(T) (listed only with exchange > 0), kind 0: ceq = equilibrium
struct KinSrc { int col, kind; double source, log_source_theta, exchange, log_exchange_theta, equilibrium; };
// a Monod factor on column col: kind 0 limitation, 1 inhibition; half: K > 0; use: -yield[col, k] of a decay process that
// consumes col and is limited by it (the cap), else 0
struct KinFac { int col, kind; double half, use; };

// c+_j / (K + c+_j) or K / (K + c+_j)
__device__ __forceinline__ double monod(const KinFac& a, double cj) {
    const double cp = fmax(cj, 0.0);
    return (a.kind ? a.half : cp) / (a.half + cp);
}

// Dissolved-oxygen saturation (mg/L) of fresh water at 1 atm, T in deg C (APHA / Benson-Krause), as written: no clamp
__device__ __forceinline__ double o2_saturation(double T) {
    const double x = 1.0 / (T + 273.15);
    return exp(-139.34411 + x * (1.575701e5 + x * (-6.642308e7 + x * (1.243800e10 + x * -8.621949e11))));
}

// s + r ceq, r and phi of one source column at temperature T (o2 = O2sat(T), read only for kind 1)
__device__ __forceinline__ void kin_src_coef(const KinSrc& s, double T, double o2, double dt, double& sr, double& r, double& phi) {
    const double dT = T - 20.0;
    r = s.exchange * exp(dT * s.log_exchange_theta) / 86400.0;
    sr = s.source * exp(dT * s.log_source_theta) / 86400.0 + r * (s.kind ? o2 : s.equilibrium);
    phi = r > 0.0 ? -expm1(-r * dt) / r : dt;
}

// The loss of decay step s with its nf factors a[] (the row c as it is now); kDepth: df = 1 scales the rate by hinv = 1 / h
template <bool kDepth = false>
__device__ __forceinline__ double kin_decay_limited(const double* c, const KinStep& s, const KinFac* __restrict__ a, int nf,
                                                 double T, double dt, double hinv = 1.0, int df = 0) {
    double r = s.decay * exp((T - 20.0) * s.log_theta) / 86400.0;
    if (kDepth && df) r = r * hinv;
    double m = 1.0;
    for (int q = 0; q < nf; ++q) {
        const KinFac f = a[q];
        m *= monod(f, c[f.col]);
    }
    double loss = c[s.col] * (-expm1(-(r * m) * dt));
    for (int q = 0; q < nf; ++q) {
        const KinFac f = a[q];
        if (f.use > 0.0) loss = fmin(loss, __ddiv_rd(fmax(c[f.col], 0.0), f.use));   // rounded down: use * cap <= c+_j
    }
    return loss;
}

// Source column *sp with its nf factors a[] applied to the row c (o2 = O2sat(T), read only for kind 1); kDepth: bit 0
// of df scales the source by hinv = 1 / h, bit 1 the exchange rate
template <bool kDepth = false>
__device__ __forceinline__ void kin_src_limited(double* c, const KinSrc* __restrict__ sp, const KinFac* __restrict__ a, int nf,
                                             double T, double o2, double dt, double hinv = 1.0, int df = 0) {
    const KinSrc s = *sp;
    const double dT = T - 20.0;
    double r = s.exchange * exp(dT * s.log_exchange_theta) / 86400.0;
    double src = s.source * exp(dT * s.log_source_theta) / 86400.0;
    if (kDepth && (df & 2)) r = r * hinv;
    if (kDepth && (df & 1)) src = src * hinv;
    const double req = r * (s.kind ? o2 : s.equilibrium);
    double m = 1.0, self_half = 0.0;
    for (int q = 0; q < nf; ++q) {
        const KinFac f = a[q];
        if (f.col == s.col) self_half = f.half;   // the self-limitation of a sink (K > 0)
        else m *= monod(f, c[f.col]);
    }
    double& v = c[s.col];
    if (self_half > 0.0) {
        const double rr = r + -src * m / (self_half + fmax(v, 0.0));
        const double phi = rr > 0.0 ? -expm1(-rr * dt) / rr : dt;
        v += (req - rr * v) * phi;
    } else {
        const double phi = r > 0.0 ? -expm1(-r * dt) / r : dt;
        v += (src * m + req - r * v) * phi;
    }
}

// Shared memory of k_react: st[kMaxK] and last_block_arrives' flag (static, kReactStaticSmem bounds them), then the dynamic
// part: a tile of R rows x (K + 1) doubles (odd stride: the one-row-per-thread chain is free of bank conflicts), vol and D
// of its rows, fac[kMaxK] and red[kThreads].  R is the largest multiple of 32 (at most kThreads) that keeps the whole within
// the 48 KB a kernel may use without opting in, for every K <= kMaxK.  With source columns at a constant temperature, their
// coefficients follow (react_src_smem_bytes, opted in); the tile does not shrink for them, so R is the same with or without.
constexpr size_t kReactSmemLimit = 48 * 1024;
constexpr size_t kReactStaticSmem = sizeof(KinStep) * kMaxK + 64;
__host__ __device__ constexpr int react_tile_rows(int K) {
    return (int)((kReactSmemLimit - kReactStaticSmem - (kMaxK + kThreads) * sizeof(double)) / ((K + 3) * sizeof(double))) >= kThreads
               ? kThreads
               : (int)((kReactSmemLimit - kReactStaticSmem - (kMaxK + kThreads) * sizeof(double)) / ((K + 3) * sizeof(double))) / 32 * 32;
}
__host__ __device__ constexpr size_t react_smem_bytes(int K) {
    return (size_t)react_tile_rows(K) * (K + 1 + 2) * sizeof(double) + (size_t)(kMaxK + kThreads) * sizeof(double);
}
constexpr bool react_smem_fits_every_k() {
    for (int K = 1; K <= kMaxK; ++K)
        if (react_tile_rows(K) < 32 || react_smem_bytes(K) + kReactStaticSmem > kReactSmemLimit) return false;
    return true;
}
static_assert(react_smem_fits_every_k(), "k_react's shared memory must fit in 48 KB for every K <= kMaxK");
// [3 n_src] s + r ceq, r, phi per source column; only at a constant temperature (a temperature constituent: per row)
__host__ __device__ constexpr size_t react_src_smem_bytes(int n_src, int temp_k) {
    return temp_k < 0 ? (size_t)3 * n_src * sizeof(double) : 0;
}

// f(e) for the elements [0, cnt) of a tile of the interleaved state that starts at `base`: each thread takes pairs that
// are 16-byte aligned there, the unpaired element at either end is taken by one thread.  (A state slot starts at an odd
// element when n K is odd.)
template <typename F>
__device__ __forceinline__ void react_pairs(const double* base, int cnt, F f) {
    const int head = (int)((reinterpret_cast<uintptr_t>(base) >> 3) & 1);
    const int pairs = (cnt - head) >> 1;
    for (int q = threadIdx.x; q < pairs; q += blockDim.x) f(head + 2 * q, true);
    if (threadIdx.x == 0) {
        if (head && cnt > 0) f(0, false);
        if (cnt > head && ((cnt - head) & 1)) f(cnt - 1, false);
    }
}

template <bool kLimited, bool kDepth = false>
__global__ void __launch_bounds__(kThreads) k_react(DeviceModel M, const KinStep* __restrict__ steps, int n_steps,
                                                    const KinYield* __restrict__ yl, int temp_k, double temp_c,
                                                    const KinSrc* __restrict__ srcs, int n_src, int src_o2,
                                                    const KinFac* __restrict__ fl, const int* __restrict__ fptr,
                                                    double* __restrict__ partials, KinState* __restrict__ ks, int accumulate,
                                                    const double* __restrict__ area, const int* __restrict__ dfl,
                                                    double min_depth) {
    static_assert(kLimited || !kDepth, "the depth code is in the factored instantiation");
    extern __shared__ double rs[];
    __shared__ KinStep st[kMaxK];
    pdl_enter();
    const StepParams& sp = *M.sp;
    const int K = M.K, ld = K + 1, R = react_tile_rows(K);
    double* tile = rs;                        // [R][K + 1]: c~, then c~', then vol * (c~' - c~)
    double* svol = tile + (size_t)R * ld;     // [R] vol[t] of the tile's rows
    double* sdg = svol + R;                   // [R] D
    double* fac = sdg + R;                    // [kMaxK] constant temperature: 1 - exp(-r dt) of every step
    double* red = fac + kMaxK;                // [kThreads] column sums
    double* sco = red + kThreads;             // [3 n_src] constant temperature: s + r ceq, r, phi (react_src_smem_bytes)
    const double dt = sp.dt;
    for (int p = threadIdx.x; p < n_steps; p += blockDim.x) {
        const KinStep s = steps[p];
        st[p] = s;
        if (temp_k < 0) fac[p] = -expm1(-(s.decay * exp((temp_c - 20.0) * s.log_theta) / 86400.0) * dt);
    }
    if (temp_k < 0)
        for (int p = threadIdx.x; p < n_src; p += blockDim.x) {
            const KinSrc s = srcs[p];
            kin_src_coef(s, temp_c, s.kind ? o2_saturation(temp_c) : 0.0, dt, sco[3 * p], sco[3 * p + 1], sco[3 * p + 2]);
        }
    __syncthreads();
    // column sums: thread (g, k) adds rows g, g + G, ... of every tile the CTA takes, in that order
    const int G = kThreads / K, kc = threadIdx.x % K, g = threadIdx.x / K;
    double acc = 0.0;
    const int nrows = M.row_hi - M.row_lo;
    double* __restrict__ x = sp.state_t1;
    for (int r0 = blockIdx.x * R; r0 < nrows; r0 += gridDim.x * R) {
        const int rows = min(R, nrows - r0), row0 = M.row_lo + r0, cnt = rows * K;
        const size_t g0 = (size_t)row0 * K;
        const bool b_aligned = ((reinterpret_cast<uintptr_t>(M.b + g0) ^ reinterpret_cast<uintptr_t>(x + g0)) & 15) == 0;
        react_pairs(x + g0, cnt, [&](int e, bool pair) {
            const int r = e / K, k = e - r * K;
            if (pair) {
                const double2 v = *reinterpret_cast<const double2*>(x + g0 + e);
                tile[r * ld + k] = v.x;
                const int r1 = (e + 1) / K, k1 = e + 1 - r1 * K;
                tile[r1 * ld + k1] = v.y;
            } else tile[r * ld + k] = x[g0 + e];
        });
        for (int r = threadIdx.x; r < rows; r += blockDim.x) { svol[r] = (double)sp.vol_t[row0 + r]; sdg[r] = M.diag[row0 + r]; }
        __syncthreads();
        if (threadIdx.x < rows) {             // one row's chain per thread
            double* c = tile + threadIdx.x * ld;
            const double T = temp_k < 0 ? temp_c : c[temp_k];
            const double hinv = kDepth ? 1.0 / fmax(svol[threadIdx.x] / area[row0 + threadIdx.x], min_depth) : 1.0;
            for (int p = 0; p < n_steps; ++p) {
                const KinStep& s = st[p];
                const int fb = kLimited ? fptr[p] : 0, fe = kLimited ? fptr[p + 1] : 0;
                const int df = kDepth ? dfl[p] : 0;
                double loss;
                if (fb == fe && !df) {
                    const double f = temp_k < 0 ? fac[p] : -expm1(-(s.decay * exp((T - 20.0) * s.log_theta) / 86400.0) * dt);
                    loss = c[s.col] * f;
                } else loss = kin_decay_limited<kDepth>(c, s, fl + fb, fe - fb, T, dt, hinv, df);
                c[s.col] -= loss;
                for (int q = s.y_begin; q < s.y_end; ++q) {
                    const KinYield y = yl[q];
                    c[y.col] += y.y * loss;
                }
            }
            if (kLimited) {                   // factored source columns per row; the others as below
                const double o2 = src_o2 ? o2_saturation(T) : 0.0;
                for (int p = 0; p < n_src; ++p) {
                    const int fb = fptr[n_steps + p], fe = fptr[n_steps + p + 1];
                    const int df = kDepth ? dfl[n_steps + p] : 0;
                    if (fb != fe || df) {
                        kin_src_limited<kDepth>(c, srcs + p, fl + fb, fe - fb, T, o2, dt, hinv, df);
                    } else if (temp_k < 0) {
                        const double* q = sco + 3 * p;
                        double& v = c[srcs[p].col];
                        v += (q[0] - q[1] * v) * q[2];
                    } else {
                        double sr, r, phi;
                        kin_src_coef(srcs[p], T, o2, dt, sr, r, phi);
                        double& v = c[srcs[p].col];
                        v += (sr - r * v) * phi;
                    }
                }
            } else if (temp_k < 0) {
                for (int p = 0; p < n_src; ++p) {
                    const double* q = sco + 3 * p;
                    double& v = c[srcs[p].col];
                    v += (q[0] - q[1] * v) * q[2];
                }
            } else if (n_src > 0) {
                const double o2 = src_o2 ? o2_saturation(T) : 0.0;
                for (int p = 0; p < n_src; ++p) {
                    const KinSrc s = srcs[p];
                    double sr, r, phi;
                    kin_src_coef(s, T, o2, dt, sr, r, phi);
                    double& v = c[s.col];
                    v += (sr - r * v) * phi;
                }
            }
        }
        __syncthreads();
        // c~' and b = (vol c~' / dt) / D out (k_rhs's expression); the tile keeps vol * (c~' - c~) (c~ re-read from L2)
        react_pairs(x + g0, cnt, [&](int e, bool pair) {
            double nv[2], bb[2];
            const int m = pair ? 2 : 1;
            for (int u = 0; u < m; ++u) {
                const int r = (e + u) / K, k = e + u - r * K;
                const double v = tile[r * ld + k], vol = svol[r];
                nv[u] = v;
                bb[u] = (vol * v / dt) / sdg[r];
                tile[r * ld + k] = vol * (v - x[g0 + e + u]);
            }
            if (pair) *reinterpret_cast<double2*>(x + g0 + e) = make_double2(nv[0], nv[1]);
            else x[g0 + e] = nv[0];
            if (pair && b_aligned) *reinterpret_cast<double2*>(M.b + g0 + e) = make_double2(bb[0], bb[1]);
            else for (int u = 0; u < m; ++u) M.b[g0 + e + u] = bb[u];
        });
        __syncthreads();
        if (g < G)
            for (int r = g; r < rows; r += G) acc += tile[r * ld + kc];
        __syncthreads();
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < K) {
        double s = 0.0;
        for (int q = 0; q < G; ++q) s += red[q * K + threadIdx.x];
        partials[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = s;
    }
    if (!last_block_arrives(&ks->ticket)) return;
    grid_totals<1>(partials, red, K);
    if (accumulate && threadIdx.x < K) ks->mass[threadIdx.x] += red[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------
// Domain decomposition over NVLink: one process per GPU, every rank holds the whole mesh's index space
// (global row numbers everywhere) but computes only its rows [row_lo, row_hi).  The vectors other
// ranks gather from (p^, s^, x) live in a symmetric slab that every rank maps from every peer (CUDA
// IPC), so a producer kernel stores a boundary row straight into the peers that read it, and one
// 8-byte flag store per peer announces "everything up to epoch e has been written".  Dot products are
// all-reduced the same way: every rank writes its partial totals into every rank's inbox and adds the
// inbox in rank order -- identical bits on every rank, so all ranks take identical decisions.
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T* peer_ptr(const DeviceModel& M, int q, T* local) {
    return reinterpret_cast<T*>(M.peer_base[q] + (reinterpret_cast<char*>(local) - M.sym_base));
}
__device__ __forceinline__ void st_flag(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_flag(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// one thread: announce epoch e to the ranks in `mask` / wait for theirs (bounded)
__device__ __forceinline__ void dd_signal(const DeviceModel& M, bool dots, unsigned long long e, unsigned mask) {
    for (int q = 0; q < M.world; ++q)
        if (q != M.rank && ((mask >> q) & 1u)) {
            DdCtl* pd = peer_ptr(M, q, M.dd);
            st_flag(dots ? &pd->dot_flag[M.rank] : &pd->bar_flag[M.rank], e);
        }
}
__device__ __forceinline__ bool dd_arrived(const DeviceModel& M, bool dots, unsigned long long e, unsigned mask) {
    for (int q = 0; q < M.world; ++q)
        if (q != M.rank && ((mask >> q) & 1u))
            if (ld_flag(dots ? &M.dd->dot_flag[q] : &M.dd->bar_flag[q]) < e) return false;
    return true;
}
__device__ __forceinline__ void dd_wait(const DeviceModel& M, bool dots, unsigned long long e, unsigned mask) {
    unsigned spins = 0;
    if (*reinterpret_cast<volatile int*>(&M.dd->timeout)) return;     // a peer already went missing in this step: fail fast
    // never hang the device, but ordinary rank skew (a host stall, a slow first step on one rank) must not fail the
    // handle: the bound is wall time (30 s on %globaltimer, looked at every 4096 polls), and cwr_step re-arms it
    unsigned long long t0 = 0;
    while (!dd_arrived(M, dots, e, mask)) {
        if ((++spins & 4095u) != 0) continue;
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > 30000000000ull) { M.dd->timeout = 1; break; }
    }
    // The rows / totals the peer announced were performed at system scope before its flag store (its
    // fence.sys), they live in THIS device's memory and are read through L2 (ld.cg / cp.async.cg / the next
    // kernel): a device-scope fence orders those reads after the flag read.  (fence.sys costs 1.75 us on
    // B200, fence.gpu 0.4 us -- tools/microbench/peer_latency.cu.)
    __threadfence();
}

// tot[0 .. pairs) (shared memory, this rank's totals, complete) -> sums over all ranks, by the whole CTA
__device__ __forceinline__ void dd_allreduce(const DeviceModel& M, double* tot, int pairs) {
    if (M.world == 1) return;
    __shared__ unsigned long long e_sh;
    if (threadIdx.x == 0) e_sh = ++M.dd->dot_epoch;
    __syncthreads();
    const unsigned long long e = e_sh;
    const int buf = (int)(e & 1ull);
    for (int pair = threadIdx.x; pair < pairs; pair += blockDim.x) {
        const double v = tot[pair];
        for (int q = 0; q < M.world; ++q) peer_ptr(M, q, M.dd)->dot_inbox[buf][M.rank][pair] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned all = (1u << M.world) - 1u;
        __threadfence_system();               // the CTA's inbox stores (ordered before it by the barrier), then the flags
        dd_signal(M, true, e, all);
        dd_wait(M, true, e, all);
    }
    __syncthreads();
    for (int pair = threadIdx.x; pair < pairs; pair += blockDim.x) {
        double s = 0.0;
        for (int q = 0; q < M.world; ++q) s += __ldcg(&M.dd->dot_inbox[buf][q][pair]);
        tot[pair] = s;
    }
    __syncthreads();
}

// boundary rows of a slab vector -> the peers that read them, then the halo barrier: when the kernel
// has finished, every neighbour's rows have landed here as well.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_halo_push(DeviceModel M, T* vec, const int32_t* __restrict__ send_rows, int n_send) {
    const int K = M.K;
    const size_t total = (size_t)n_send * K;
    for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int row = send_rows[q / K], k = (int)(q % K);
        const T v = vec[(size_t)row * K + k];
        unsigned m = M.send_mask[row];
        while (m) {
            const int r = __ffs(m) - 1;
            m &= m - 1;
            peer_ptr(M, r, vec)[(size_t)row * K + k] = v;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) __threadfence_system();        // this CTA's peer stores, before its arrival below
    if (!last_block_arrives(&M.ctl->ticket_halo)) return;
    if (threadIdx.x == 0) {
        const unsigned long long e = ++M.dd->bar_epoch;
        dd_signal(M, false, e, M.nbr_mask);
        dd_wait(M, false, e, M.nbr_mask);
    }
}

__device__ __forceinline__ void publish_done(DeviceModel& M, int K) {
    int done = 1, flags = 0;
    for (int k = 0; k < K; ++k) {
        const int f = M.colflags[k];
        flags |= f;
        if (!(f & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN)) || (f & FL_PENDING)) done = 0;
    }
    M.ctl->flags_or = flags;
    if (M.ctl->iter >= M.max_iter && !done) { M.ctl->hit_max_iter = 1; done = 1; }
    M.ctl->all_done = done;
}

// ---------------------------------------------------------------------------------------------
// packs of V adjacent columns of type T moved with one (<= 128-bit) access
// ---------------------------------------------------------------------------------------------
template <typename T, int V> struct alignas(sizeof(T) * V > 16 ? 16 : sizeof(T) * V) Pk { T a[V]; };
template <typename T, int V>
__device__ __forceinline__ Pk<T, V> ldk(const T* p) { return *reinterpret_cast<const Pk<T, V>*>(p); }
template <typename T, int V>
__device__ __forceinline__ void stk(T* p, const Pk<T, V>& v) { *reinterpret_cast<Pk<T, V>*>(p) = v; }
// VEC columns of a ZT vector, widened (exactly) to double
template <typename ZT, int VEC>
__device__ __forceinline__ Vd<VEC> ldz(const ZT* p) {
    const Pk<ZT, VEC> t = ldk<ZT, VEC>(p);
    Vd<VEC> r;
#pragma unroll
    for (int q = 0; q < VEC; ++q) r.a[q] = (double)t.a[q];
    return r;
}

// ---------------------------------------------------------------------------------------------
// Preconditioner sweeps over the row-scaled matrix  A = I + L  (L = off-diagonals in ELL; N := -L is
// the Jacobi iteration matrix):   out_i = u_i - (L z)_i   for rows [row_begin, row_end).
//   * Jacobi step: z != out, whole row range; m - 1 of them give z = (I + N + ... + N^(m-1)) u.
//   * one colour of a multicolour Gauss-Seidel sweep: z == out (in place), [row_begin, row_end) = the
//     rows of ONE colour -- rows of a colour are not coupled, so the range is updated in parallel.
// ST is the sweep precision: float by default.  The preconditioner only has to be a fixed linear
// operator close to A^-1; BiCGSTAB's own vectors, products A p^ / A s^ and dot products stay fp64 (p^,
// s^ are widened exactly), so the converged answer is the fp64 one and the sweeps move half the bytes.
// FIRST: z = u is the solver's fp64 vector (gathered as double); the step also leaves the ST copy of
// u in M.us for the following sweeps.
// ---------------------------------------------------------------------------------------------
template <typename ST, int KC, int VEC, bool FIRST>
__global__ void __launch_bounds__(kThreads, CWR_SPMM_MIN_BLOCKS) k_sweep(DeviceModel M, const double* __restrict__ u64,
                                                                         const ST* z, ST* out, int row_begin, int row_end) {
    if (M.ctl->all_done || M.ctl->finish_half) return;
    const int K = M.K, W = M.W;
    const int lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kThreads / KC;
    const int32_t* __restrict__ ecol = M.ell_col;
    const ST* __restrict__ eval = sizeof(ST) == 4 ? reinterpret_cast<const ST*>(M.valf) : reinterpret_cast<const ST*>(M.val);
    ST* us = reinterpret_cast<ST*>(M.us);
    const int stride = gridDim.x * GPB;
    for (int c = lane * VEC; c < K; c += KC * VEC) {
        // software pipeline: the next row's indices / values are fetched under this row's gathers
        int i = row_begin + blockIdx.x * GPB + group;
        int4 c4n = make_int4(0, 0, 0, 0);
        Pk<ST, 4> vn = {};
        if (i < row_end) {
            c4n = *reinterpret_cast<const int4*>(ecol + (size_t)i * W);
            vn = ldk<ST, 4>(eval + (size_t)i * W);
        }
        for (; i < row_end; i += stride) {
            const size_t idx = (size_t)i * K + c;
            const int4 c4 = make_int4(c4n.x & kColMask, c4n.y & kColMask, c4n.z & kColMask, c4n.w & kColMask);
            const Pk<ST, 4> v = vn;
            Pk<ST, VEC> x0, x1, x2, x3, own;
            if (FIRST) {
                // u is one of the solver's own vectors: under domain decomposition only this rank's rows of it exist,
                // the other ranks' rows count as 0 in this first step (their z arrives with the halo push that follows)
                const bool dd = M.world > 1;
                const int lo = M.row_lo, hi = M.row_hi;
                const Pk<double, VEC> dz = {};
                const Pk<double, VEC> d0 = dd && (c4.x < lo || c4.x >= hi) ? dz : ldk<double, VEC>(u64 + (size_t)c4.x * K + c);
                const Pk<double, VEC> d1 = dd && (c4.y < lo || c4.y >= hi) ? dz : ldk<double, VEC>(u64 + (size_t)c4.y * K + c);
                const Pk<double, VEC> d2 = dd && (c4.z < lo || c4.z >= hi) ? dz : ldk<double, VEC>(u64 + (size_t)c4.z * K + c);
                const Pk<double, VEC> d3 = dd && (c4.w < lo || c4.w >= hi) ? dz : ldk<double, VEC>(u64 + (size_t)c4.w * K + c);
                const Pk<double, VEC> dn = ldk<double, VEC>(u64 + idx);
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    x0.a[q] = (ST)d0.a[q]; x1.a[q] = (ST)d1.a[q]; x2.a[q] = (ST)d2.a[q]; x3.a[q] = (ST)d3.a[q]; own.a[q] = (ST)dn.a[q];
                }
            } else {
                x0 = ldk<ST, VEC>(z + (size_t)c4.x * K + c); x1 = ldk<ST, VEC>(z + (size_t)c4.y * K + c);
                x2 = ldk<ST, VEC>(z + (size_t)c4.z * K + c); x3 = ldk<ST, VEC>(z + (size_t)c4.w * K + c);
                own = ldk<ST, VEC>(us + idx);
            }
            const int inext = i + stride;
            if (inext < row_end) {
                c4n = *reinterpret_cast<const int4*>(ecol + (size_t)inext * W);
                vn = ldk<ST, 4>(eval + (size_t)inext * W);
            }
            Pk<ST, VEC> o;
#pragma unroll
            for (int q = 0; q < VEC; ++q)
                o.a[q] = v.a[3] * x3.a[q] + (v.a[2] * x2.a[q] + (v.a[1] * x1.a[q] + v.a[0] * x0.a[q]));
            for (int w = 4; w < W; w += 4) {      // rows wider than 4 (not pipelined)
                const int4 d4 = *reinterpret_cast<const int4*>(ecol + (size_t)i * W + w);
                const Pk<ST, 4> wv = ldk<ST, 4>(eval + (size_t)i * W + w);
                const int cs[4] = {d4.x & kColMask, d4.y & kColMask, d4.z & kColMask, d4.w & kColMask};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    Pk<ST, VEC> y;
                    if (FIRST) {
                        Pk<double, VEC> d = {};
                        if (!(M.world > 1 && (cs[u] < M.row_lo || cs[u] >= M.row_hi))) d = ldk<double, VEC>(u64 + (size_t)cs[u] * K + c);
#pragma unroll
                        for (int q = 0; q < VEC; ++q) y.a[q] = (ST)d.a[q];
                    } else y = ldk<ST, VEC>(z + (size_t)cs[u] * K + c);
#pragma unroll
                    for (int q = 0; q < VEC; ++q) o.a[q] += wv.a[u] * y.a[q];
                }
            }
#pragma unroll
            for (int q = 0; q < VEC; ++q) o.a[q] = own.a[q] - o.a[q];
            stk<ST, VEC>(out + idx, o);
            if (FIRST) stk<ST, VEC>(us + idx, own);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Multicolour Gauss-Seidel preconditioner, all sweeps of one application in ONE persistent kernel:
//   z = 0;  repeat n_sweeps times:  for colour = 0 .. n_colors-1:  z_i = u_i - (L z)_i  for the rows of
//   that colour (in place),
// with a grid-wide barrier between colours (cooperative launch: every CTA is resident).  The colours
// follow the flow (cwr_topology.cpp), so one sweep carries information ~n_colors cells downstream, at
// the memory traffic of ONE Jacobi step -- the colours only cut that step into slices.  During the first
// sweep neighbours of a later colour have not been visited yet (z = 0 there: index >= the colour's first
// row) and u arrives as the solver's fp64 vector; its ST copy is kept in M.us for the later sweeps.
// Gathers bypass L1 (ld.cg): the values were written by other SMs a barrier ago.
// ---------------------------------------------------------------------------------------------
template <typename T, int V>
__device__ __forceinline__ Pk<T, V> ldk_cg(const T* p) {
    Pk<T, V> r;
    if constexpr (sizeof(T) * V == 16) { const int4 t = __ldcg(reinterpret_cast<const int4*>(p)); r = *reinterpret_cast<const Pk<T, V>*>(&t); }
    else if constexpr (sizeof(T) * V == 8) { const int2 t = __ldcg(reinterpret_cast<const int2*>(p)); r = *reinterpret_cast<const Pk<T, V>*>(&t); }
    else if constexpr (sizeof(T) * V == 4) { const int t = __ldcg(reinterpret_cast<const int*>(p)); r = *reinterpret_cast<const Pk<T, V>*>(&t); }
    else {
#pragma unroll
        for (int q = 0; q < V; ++q) r.a[q] = __ldcg(p + q);
    }
    return r;
}

// Grid barrier of the persistent sweep kernel.  With several ranks it is also the halo barrier: the last
// CTA of this rank to arrive (every CTA's stores, peer stores included, are fenced before its arrival)
// announces epoch `e` to the neighbour ranks, and every CTA also waits for the neighbours' announcements.
// cross: this barrier is also a halo barrier (epoch e) -- else it only synchronises this device's CTAs.
__device__ __forceinline__ void grid_barrier(const DeviceModel& M, unsigned target, unsigned long long e, bool pushed, bool cross) {
    SolverCtl* ctl = M.ctl;
    // system-scope fence only in the CTAs that stored rows into a peer since the last barrier
    const int any_pushed = cross ? __syncthreads_or(pushed) : (__syncthreads(), 0);
    if (threadIdx.x == 0) {
        if (any_pushed) __threadfence_system(); else asm volatile("fence.acq_rel.gpu;" ::: "memory");
        const unsigned t = atomicAdd(&ctl->gs_bar[0], 1u);
        // every CTA that stored into a peer fenced at system scope BEFORE its arrival; seeing all arrivals
        // (device-scope fence) therefore orders all of this rank's peer stores before the announcement
        if (cross && t == target - 1) { __threadfence(); dd_signal(M, false, e, M.nbr_mask); }
        unsigned spins = 0;
        // never hang the device: a barrier that gave up once (never expected) makes the later ones fall through
        const unsigned limit = *reinterpret_cast<volatile int*>(&ctl->barrier_timeout) ? 0u : (1u << 27);
        while (*reinterpret_cast<volatile unsigned*>(&ctl->gs_bar[0]) < target)
            if (++spins > limit) { ctl->barrier_timeout = 1; break; }
        if (cross) dd_wait(M, false, e, M.nbr_mask); else asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
    __syncthreads();
}

// Two CTAs of 512 threads per SM.  Every lane group owns up to kGsRows rows of a colour at a time.  The
// loads that do not depend on other CTAs -- the rows' column indices and matrix values -- are issued
// BEFORE the barrier in front of the colour; after it all gathers of those rows go out together as
// 16-byte cp.async.cg copies into per-thread shared-memory slots (no destination registers held while in
// flight, L1 bypassed), so a colour costs one barrier plus one gather latency.  Packs narrower than 16
// bytes gather into registers.  (Measured and rejected, profiles/r01_notes.md: splitting the columns into
// two independently synchronised halves to overlap one half's barrier with the other half's work; three
// pipelined rows, which spill.)
constexpr int kGsThreads = 512;
constexpr int kGsRows = 2;
constexpr int kGsSmemBytes = kGsRows * 4 * 16 * kGsThreads;

__device__ __forceinline__ void cp_async_cg16(void* smem_dst, const void* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
// predicated copy: nothing when !pred; `bytes` = 16 copies, 0 fills the slot with zeros without reading the source
__device__ __forceinline__ void cp_async_cg16_if(void* smem_dst, const void* gsrc, bool pred, int bytes) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %3, 0;\n @p cp.async.cg.shared.global [%0], [%1], 16, %2;\n}"
                 ::"r"(d), "l"(gsrc), "r"(bytes), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

// STRIP = false: rows colour-major (color_ptr), lane groups dealt grid-wide, a GRID barrier between colours.
// STRIP = true (precond_sync = 2): rows strip-major -- CTA b owns the contiguous strip strip0 + b, colour-major
// inside (strip_cptr) -- and a colour only waits for the strips this strip's rows are coupled to (strip_nbr; two
// or three of them when the strips are cut from the RCM order): every CTA publishes (launch sequence, step)
// in strip_flag after a step and polls its neighbours' flags before the next one.  A CTA is then never more
// than one step ahead of a strip it exchanges values with, which orders exactly the reads and writes the grid
// barrier ordered -- the results are bit-identical to the grid-barrier sweep over the same colours -- but a
// step costs one release/acquire between neighbours instead of a device-wide rendezvous, and slow CTAs only
// hold up their neighbours.  n_sweeps <= 0: the count is read from ctl->dc_sweeps (planned on the device by the
// defect-correction solver).
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

constexpr int kMaxColors = 64;

template <typename ST, int KC, int VEC, bool STRIP>
__global__ void __launch_bounds__(kGsThreads, 2) k_precond_gs(DeviceModel M, const double* __restrict__ u64, ST* z, int n_sweeps_arg,
                                                              unsigned long long seq) {
    constexpr bool SMEM = sizeof(ST) * VEC == 16;
    constexpr int NR = kGsRows;
    extern __shared__ int4 gs_land[];          // [NR rows][4 neighbours][kGsThreads] landing slots (SMEM path)
    __shared__ int s_cp[kMaxColors + 1];       // row ranges of the colours this CTA sweeps
    if (M.ctl->all_done || M.ctl->finish_half) return;
    const int n_sweeps = n_sweeps_arg > 0 ? n_sweeps_arg : M.ctl->dc_sweeps;
    const int K = M.K, W = M.W, nc = M.n_colors;
    const int vb = blockIdx.x, nvb = gridDim.x, c_end = K;
    const int lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kGsThreads / KC;
    const int32_t* __restrict__ ecol = M.ell_col;
    const ST* __restrict__ eval = sizeof(ST) == 4 ? reinterpret_cast<const ST*>(M.valf) : reinterpret_cast<const ST*>(M.val);
    ST* us = reinterpret_cast<ST*>(M.us);
    // lane groups that share a colour's rows, and this group's position among them
    const int TG = STRIP ? GPB : nvb * GPB, gid = STRIP ? group : vb * GPB + group;
    const int sid = M.strip0 + vb;                                          // STRIP: the strip this CTA owns
    const int32_t* __restrict__ cp_src = STRIP ? M.strip_cptr + (size_t)sid * (nc + 1) : M.color_ptr;
    for (int q = threadIdx.x; q <= nc; q += kGsThreads) s_cp[q] = cp_src[q];
    const int nb0 = STRIP ? M.strip_nptr[sid] : 0, n_nbr = STRIP ? M.strip_nptr[sid + 1] - nb0 : 0;
    __syncthreads();
    const int c = lane * VEC;
    const bool lane_on = c < c_end;
    const int n_steps = n_sweeps * nc;
    unsigned epoch = 0;
    const bool multi = M.world > 1;
    // Several ranks: either every finished boundary row goes to its readers at once and every colour's barrier is
    // a halo barrier (exact multi-rank Gauss-Seidel; grid-barrier kernel only), or (halo_per_sweep, default) the
    // boundary rows cross once at the end of each sweep: within a sweep the neighbours' rows are one sweep old (zero
    // in the first sweep) -- Gauss-Seidel inside a rank's rows, Jacobi across ranks -- and only one barrier per sweep
    // waits for NVLink.
    // STRIP with several ranks (xs): EXACT Gauss-Seidel across the cut -- a finished row that another rank reads goes
    // there at once (peer store), the strip's flag is mirrored into those ranks after a system-scope fence, and a
    // boundary strip waits for the strips of the neighbouring rank exactly as for its local neighbours: no halo barrier,
    // no sweep of lag (the sweep-lagged halo cost 25 sweeps against 13 on the 16M-cell mesh).
    const bool xs = multi && STRIP;
    const bool per_sweep = multi && !STRIP && M.halo_per_sweep, per_colour = multi && !STRIP && !per_sweep;
    const unsigned my_peers = xs ? (unsigned)M.strip_peers[sid] & ~(1u << M.rank) : 0u;
    const int row_lo = M.row_lo, row_hi = M.row_hi;
    const unsigned long long e0 = multi ? M.dd->bar_epoch : 0ull;     // halo epochs continue where the last kernel stopped
    unsigned long long xe = 0;                                         // halo barriers of this launch
    // a finished row also goes to the ranks that read it (NVLink peer stores)
    bool pushed = false;
    auto push = [&](int i, int cc, const Pk<ST, VEC>& o) {
        if (!(per_colour || xs)) return;
        unsigned m = M.send_mask[i];
        pushed |= m != 0;
        while (m) {
            const int q = __ffs(m) - 1;
            m &= m - 1;
            stk<ST, VEC>(peer_ptr(M, q, z) + (size_t)i * K + cc, o);
        }
    };
    auto load_own = [&](int i, int cc, bool first_sweep) {
        Pk<ST, VEC> own;
        if (first_sweep) {
            const Pk<double, VEC> d = ldk<double, VEC>(u64 + (size_t)i * K + cc);
#pragma unroll
            for (int q = 0; q < VEC; ++q) own.a[q] = (ST)d.a[q];
        } else own = ldk<ST, VEC>(us + (size_t)i * K + cc);      // written by this very thread in sweep 0
        return own;
    };
    // pipeline registers: indices / values of the first NR rows of the coming colour
    int4 pc[NR]; Pk<ST, 4> pv[NR];
    auto prefetch = [&](int step) {
        const int col = step % nc;
        const int rb = s_cp[col], re = s_cp[col + 1];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int i = rb + gid + r * TG;
            if (i < re) {
                pc[r] = *reinterpret_cast<const int4*>(ecol + (size_t)i * W);
                pv[r] = ldk<ST, 4>(eval + (size_t)i * W);
            }
        }
    };
    // STRIP: this strip has finished `step` (all of the CTA's stores, then the flag) / wait until the
    // neighbouring strips have
    auto publish = [&](int step) {
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned long long v = (seq << 20) | (unsigned long long)(step + 1);
            if (my_peers) {              // rows of this strip went into other ranks: their mirrors of the flag, after a system-scope fence
                __threadfence_system();
                for (unsigned m = my_peers; m; m &= m - 1)
                    st_flag(peer_ptr(M, __ffs(m) - 1, M.strip_flag) + (size_t)sid * kFlagStride, v);
            } else __threadfence();
            st_flag(M.strip_flag + (size_t)sid * kFlagStride, v);
        }
    };
    auto wait_nbrs = [&](int step) {
        const unsigned long long target = (seq << 20) | (unsigned long long)(step + 1);
        for (int j = threadIdx.x; j < n_nbr; j += kGsThreads) {
            const unsigned long long* f = M.strip_flag + (size_t)M.strip_nbr[nb0 + j] * kFlagStride;
            unsigned spins = 0;
            const unsigned limit = *reinterpret_cast<volatile int*>(&M.ctl->barrier_timeout) ? 0u : (1u << 26);
            while (ld_acquire_u64(f) < target)
                if (++spins > limit) { M.ctl->barrier_timeout = 1; break; }      // never hang the device
        }
        __syncthreads();
    };
    // one row, columns [cc, cc + VEC): remaining ELL blocks through registers, then the update and the store
    auto relax_tail = [&](int i, int cc, int w0, Pk<ST, VEC> acc, const Pk<ST, VEC>& own, bool first_sweep) {
        for (int w = w0; w < W; w += 4) {
            const int4 d4 = *reinterpret_cast<const int4*>(ecol + (size_t)i * W + w);
            const Pk<ST, 4> wv = ldk<ST, 4>(eval + (size_t)i * W + w);
            const int ds[4] = {d4.x, d4.y, d4.z, d4.w};
            Pk<ST, VEC> y[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int dj = ds[u] & kColMask;
                if (first_sweep && (ds[u] < 0 || (per_sweep && (dj < row_lo || dj >= row_hi)))) {   // not visited yet: still 0
#pragma unroll
                    for (int q = 0; q < VEC; ++q) y[u].a[q] = (ST)0;
                } else y[u] = ldk_cg<ST, VEC>(z + (size_t)(ds[u] & kColMask) * K + cc);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int q = 0; q < VEC; ++q) acc.a[q] += wv.a[u] * y[u].a[q];
        }
#pragma unroll
        for (int q = 0; q < VEC; ++q) acc.a[q] = own.a[q] - acc.a[q];
        stk<ST, VEC>(z + (size_t)i * K + cc, acc);
        if (first_sweep) stk<ST, VEC>(us + (size_t)i * K + cc, own);
        push(i, cc, acc);
    };
    Pk<ST, VEC> zero;
#pragma unroll
    for (int q = 0; q < VEC; ++q) zero.a[q] = (ST)0;

    prefetch(0);
    for (int step = 0; step < n_steps; ++step) {
        const int col = step % nc;
        const bool first_sweep = step < nc;
        const int rb = s_cp[col], re = s_cp[col + 1];
        bool on[NR]; int row[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) { row[r] = rb + gid + r * TG; on[r] = row[r] < re && lane_on; }
        // ---- all gathers of the pipelined rows go out together ------------------------------------------------
        Pk<ST, VEC> xr[SMEM ? 1 : NR][SMEM ? 1 : 4], own[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            if (!on[r]) continue;
            const int cs[4] = {pc[r].x, pc[r].y, pc[r].z, pc[r].w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int cj = cs[u] & kColMask;                     // bit 31: visited later in the sweep from z = 0
                const bool skip = first_sweep && (cs[u] < 0 || (per_sweep && (cj < row_lo || cj >= row_hi)));
                if constexpr (SMEM) {
                    int4* slot = gs_land + (r * 4 + u) * kGsThreads + threadIdx.x;
                    if (skip) *slot = make_int4(0, 0, 0, 0);
                    else cp_async_cg16(slot, z + (size_t)(cs[u] & kColMask) * K + c);
                } else {
                    xr[r][u] = skip ? zero : ldk_cg<ST, VEC>(z + (size_t)(cs[u] & kColMask) * K + c);
                }
            }
            own[r] = load_own(row[r], c, first_sweep);
        }
        if constexpr (SMEM) cp_async_wait_all();
        // ---- update, store ------------------------------------------------------------------------------------
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            if (!on[r]) continue;
            Pk<ST, VEC> o = zero;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                Pk<ST, VEC> x;
                if constexpr (SMEM) x = *reinterpret_cast<const Pk<ST, VEC>*>(gs_land + (r * 4 + u) * kGsThreads + threadIdx.x);
                else x = xr[r][u];
#pragma unroll
                for (int q = 0; q < VEC; ++q) o.a[q] += pv[r].a[u] * x.a[q];
            }
            relax_tail(row[r], c, 4, o, own[r], first_sweep);
        }
        // further column chunks of those rows (more columns than lanes x VEC), and colours with more rows per lane group
#pragma unroll 1
        for (int r = 0; r < NR; ++r)
            if (row[r] < re)
                for (int cc = c + KC * VEC; cc < c_end; cc += KC * VEC)
                    relax_tail(row[r], cc, 0, zero, load_own(row[r], cc, first_sweep), first_sweep);
#pragma unroll 1
        for (int i = rb + gid + NR * TG; i < re; i += TG)
            for (int cc = c; cc < c_end; cc += KC * VEC)
                relax_tail(i, cc, 0, zero, load_own(i, cc, first_sweep), first_sweep);
        const bool last_step = step + 1 == n_steps;
        if (STRIP && (!last_step || xs)) publish(step);
        if (per_sweep && col == nc - 1) {
            // end of a sweep: once the last colour is complete on this device, the rank's boundary rows go to
            // the ranks that read them, and the next barrier also waits for theirs
            ++epoch;
            grid_barrier(M, epoch * nvb, 0, false, false);
            const int packs = (K + VEC - 1) / VEC;
            for (int q = blockIdx.x * kGsThreads + threadIdx.x; q < M.n_send * packs; q += gridDim.x * kGsThreads) {
                const int i = M.send_rows[q / packs], cc = (q % packs) * VEC;
                if (cc + VEC > K) continue;
                const Pk<ST, VEC> o = ldk_cg<ST, VEC>(z + (size_t)i * K + cc);
                unsigned m = M.send_mask[i];
                pushed |= m != 0;
                while (m) {
                    const int r = __ffs(m) - 1;
                    m &= m - 1;
                    stk<ST, VEC>(peer_ptr(M, r, z) + (size_t)i * K + cc, o);
                }
            }
            if (!last_step) prefetch(step + 1);
            ++epoch; ++xe;
            grid_barrier(M, epoch * nvb, e0 + xe, pushed, true);
            pushed = false;
        } else if (STRIP) {
            if (!last_step) { prefetch(step + 1); wait_nbrs(step); }
            else if (xs) wait_nbrs(step);      // the products that follow gather the neighbouring ranks' last colour too
        } else if (!last_step) {
            prefetch(step + 1);
            ++epoch;
            if (per_colour) ++xe;
            grid_barrier(M, epoch * nvb, e0 + xe, pushed, per_colour);
            pushed = false;
        } else if (per_colour) {       // the products that follow gather the neighbours' last colour too
            ++epoch; ++xe;
            grid_barrier(M, epoch * nvb, e0 + xe, pushed, true);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) M.ctl->sweeps_done += n_sweeps;
    if (STRIP) return;                     // no grid barrier was used: nothing to re-arm
    // the last CTA to leave re-arms the barrier for the next launch
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(&M.ctl->gs_bar[1], 1u);
        if (t == (unsigned)nvb - 1) {
            M.ctl->gs_bar[0] = 0; M.ctl->gs_bar[1] = 0;
            if (multi) M.dd->bar_epoch = e0 + xe;
            __threadfence();
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Strip sweep kernel, software-pipelined across the synchronisation (precond_sync = 3; 16-byte packs only).
// Same rows, colours, flags and arithmetic as k_precond_gs<STRIP = true>; what changes is WHEN the loads go out.
// Measured on the 1M x 16 benchmark, a colour step of that kernel costs ~3.5 us of dependent latency (fence,
// flag, poll, gathers: three round trips through a saturated memory system) on top of its ~2.5 us of bandwidth,
// with or without the grid barrier.  But of everything step k reads, only the neighbours of the colour swept
// in step k - 1 (kPrevBit) can still be missing when step k - 1 has finished here: a strip is never more than
// one step ahead of the strips it is coupled to, so every other neighbour already holds exactly the version step
// k must see, and cannot be overwritten before this strip has published step k.  So after its own step k - 1 a
// CTA issues, as cp.async copies into per-thread shared-memory slots, the matrix values, the right-hand side u
// and all EARLY gathers of step k, publishes step k - 1, waits for its neighbours, issues the few LATE gathers
// (L2 hits: written a moment ago), and computes: the dependent chain overlaps the streaming instead of
// alternating with it.  u arrives in the sweep type (M.us, written by the kernel that produced the residual), so
// a row is 16 B indices (registers, prefetched one step ahead) + 6 slots of 16 B.
// ---------------------------------------------------------------------------------------------
template <typename ST> struct GsSlots { static constexpr int val = sizeof(ST) * 4 / 16, total = 5 + val; };
template <typename ST> constexpr int gs3_smem_bytes() { return kGsRows * GsSlots<ST>::total * 16 * kGsThreads; }

template <typename ST, int KC, int VEC>
__global__ void __launch_bounds__(kGsThreads, 2) k_gs_strip(DeviceModel M, ST* z, int n_sweeps_arg, unsigned long long seq) {
    static_assert(sizeof(ST) * VEC == 16, "k_gs_strip moves 16-byte packs");
    constexpr int NR = kGsRows, VS = GsSlots<ST>::val, NS = GsSlots<ST>::total;
    extern __shared__ int4 gs_land[];          // [NR rows][4 gathers | u | values][kGsThreads]
    __shared__ int s_cp[kMaxColors + 1];
    if (M.ctl->all_done || M.ctl->finish_half) return;
    const int n_sweeps = n_sweeps_arg > 0 ? n_sweeps_arg : M.ctl->dc_sweeps;
    const int K = M.K, W = M.W, nc = M.n_colors;
    const int vb = blockIdx.x, nvb = gridDim.x;
    const int lane = threadIdx.x % KC, group = threadIdx.x / KC;
    constexpr int GPB = kGsThreads / KC;
    const int32_t* __restrict__ ecol = M.ell_col;
    const ST* __restrict__ eval = sizeof(ST) == 4 ? reinterpret_cast<const ST*>(M.valf) : reinterpret_cast<const ST*>(M.val);
    const ST* __restrict__ us = reinterpret_cast<const ST*>(M.us);
    const int sid = vb;                        // (one rank: several ranks run k_precond_gs<STRIP>)
    const int32_t* __restrict__ cp_src = M.strip_cptr + (size_t)sid * (nc + 1);
    for (int q = threadIdx.x; q <= nc; q += kGsThreads) s_cp[q] = cp_src[q];
    const int nb0 = M.strip_nptr[sid], n_nbr = M.strip_nptr[sid + 1] - nb0;
    __syncthreads();
    const int c = lane * VEC;
    const bool lane_on = c < K;
    const int n_steps = n_sweeps * nc;
    auto slot = [&](int r, int s) { return gs_land + (r * NS + s) * kGsThreads + threadIdx.x; };
    auto skipped = [&](int cj, bool first_sweep) { return first_sweep && cj < 0; };     // first sweep from z = 0: not visited yet
    int4 pc[NR], pcn[NR];
    auto load_idx = [&](int4 (&dst)[NR], int step) {
        const int col = step % nc;
        const int rb = s_cp[col], re = s_cp[col + 1];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int i = rb + group + r * GPB;
            if (i < re) dst[r] = *reinterpret_cast<const int4*>(ecol + (size_t)i * W);
        }
    };
    // everything of `step` that does not depend on the step before it.  Branch-free: every copy is predicated, and a
    // neighbour that counts as 0 (first sweep: not visited yet / another rank's row) is a zero-filling copy
    const ST* __restrict__ zc = z + c;
    const ST* __restrict__ usc = us + c;
    auto issue_early = [&](int step) {
        const int col = step % nc;
        const bool first_sweep = step < nc;
        const int rb = s_cp[col], re = s_cp[col + 1];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int i = rb + group + r * GPB;
            const bool act = i < re && lane_on;
            const int cs[4] = {pc[r].x, pc[r].y, pc[r].z, pc[r].w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool skip = skipped(cs[u], first_sweep);
                cp_async_cg16_if(slot(r, u), zc + (size_t)(cs[u] & kColMask) * K, act && (skip || !(cs[u] & kPrevBit)), skip ? 0 : 16);
            }
            cp_async_cg16_if(slot(r, 4), usc + (size_t)i * K, act, 16);
#pragma unroll
            for (int v = 0; v < VS; ++v) cp_async_cg16_if(slot(r, 5 + v), reinterpret_cast<const char*>(eval + (size_t)i * W) + 16 * v, act, 16);
        }
    };
    auto issue_late = [&](int step) {
        const int col = step % nc;
        const bool first_sweep = step < nc;
        const int rb = s_cp[col], re = s_cp[col + 1];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int i = rb + group + r * GPB;
            const bool act = i < re && lane_on;
            const int cs[4] = {pc[r].x, pc[r].y, pc[r].z, pc[r].w};
#pragma unroll
            for (int u = 0; u < 4; ++u)
                cp_async_cg16_if(slot(r, u), zc + (size_t)(cs[u] & kColMask) * K, act && (cs[u] & kPrevBit) && !skipped(cs[u], first_sweep), 16);
        }
    };
    // Synchronisation is per WARP, not per CTA: strip_flag[s] counts the warp arrivals of strip s (every warp of a
    // strip arrives once per step, after its own stores and a fence), and a warp starts step k + 1 when its own strip
    // and the neighbouring strips show all their warps' arrivals for step k.  No __syncthreads() in the sweep loop:
    // the warps of a CTA drift apart by up to a step, a slow warp holds up only the warps that read its rows.
    constexpr unsigned kWarps = kGsThreads / 32;
    const unsigned long long base = M.ctl->strip_base;
    const int wl = threadIdx.x & 31;
    auto publish = [&](int step) {
        (void)step;
        __syncwarp();
        if (wl == 0) {
            __threadfence();
            atomicAdd(M.strip_flag + (size_t)vb * kFlagStride, 1ull);
        }
    };
    auto wait_nbrs = [&](int step) {
        const unsigned long long target = base + (unsigned long long)kWarps * (unsigned long long)(step + 1);
        // lane 0: this strip; lanes 1..: the neighbouring strips (a strip of an RCM band has two or three)
        for (int j = wl; j <= n_nbr; j += 32) {
            const unsigned long long* f = M.strip_flag + (size_t)(j == 0 ? vb : M.strip_nbr[nb0 + j - 1]) * kFlagStride;
            unsigned spins = 0;
            const unsigned limit = *reinterpret_cast<volatile int*>(&M.ctl->barrier_timeout) ? 0u : (1u << 26);
            while (ld_acquire_u64(f) < target)
                if (++spins > limit) { M.ctl->barrier_timeout = 1; break; }      // never hang the device
        }
        __syncwarp();
    };
    // a row through registers (rows beyond the pipelined ones, ELL blocks beyond the first, further column chunks)
    auto relax_slow = [&](int i, int cc, int w0, Pk<ST, VEC> acc, bool first_sweep) {
        for (int w = w0; w < W; w += 4) {
            const int4 d4 = *reinterpret_cast<const int4*>(ecol + (size_t)i * W + w);
            const Pk<ST, 4> wv = ldk<ST, 4>(eval + (size_t)i * W + w);
            const int ds[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (skipped(ds[u], first_sweep)) continue;
                const Pk<ST, VEC> y = ldk_cg<ST, VEC>(z + (size_t)(ds[u] & kColMask) * K + cc);
#pragma unroll
                for (int q = 0; q < VEC; ++q) acc.a[q] += wv.a[u] * y.a[q];
            }
        }
        const Pk<ST, VEC> own = ldk_cg<ST, VEC>(us + (size_t)i * K + cc);
#pragma unroll
        for (int q = 0; q < VEC; ++q) acc.a[q] = own.a[q] - acc.a[q];
        stk<ST, VEC>(z + (size_t)i * K + cc, acc);
    };
    Pk<ST, VEC> zero;
#pragma unroll
    for (int q = 0; q < VEC; ++q) zero.a[q] = (ST)0;

    load_idx(pc, 0);
    issue_early(0);
    for (int step = 0; step < n_steps; ++step) {
        const int col = step % nc;
        const bool first_sweep = step < nc, last_step = step + 1 == n_steps;
        const int rb = s_cp[col], re = s_cp[col + 1];
        if (!last_step) load_idx(pcn, step + 1);                 // indices of the next step, in flight across this one
        if (step > 0) wait_nbrs(step - 1);
        issue_late(step);
        cp_async_wait_all();
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int i = rb + group + r * GPB;
            if (i >= re || !lane_on) continue;
            ST vals[4];
#pragma unroll
            for (int v = 0; v < VS; ++v) *reinterpret_cast<int4*>(reinterpret_cast<char*>(vals) + 16 * v) = *slot(r, 5 + v);
            Pk<ST, VEC> o = zero;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const Pk<ST, VEC> x = *reinterpret_cast<const Pk<ST, VEC>*>(slot(r, u));
#pragma unroll
                for (int q = 0; q < VEC; ++q) o.a[q] += vals[u] * x.a[q];
            }
            if (W > 4) {
                // wider rows: the remaining ELL blocks through registers, then the update from the accumulated sum
                for (int w = 4; w < W; w += 4) {
                    const int4 d4 = *reinterpret_cast<const int4*>(ecol + (size_t)i * W + w);
                    const Pk<ST, 4> wv = ldk<ST, 4>(eval + (size_t)i * W + w);
                    const int ds[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (skipped(ds[u], first_sweep)) continue;
                        const Pk<ST, VEC> y = ldk_cg<ST, VEC>(z + (size_t)(ds[u] & kColMask) * K + c);
#pragma unroll
                        for (int q = 0; q < VEC; ++q) o.a[q] += wv.a[u] * y.a[q];
                    }
                }
            }
            const Pk<ST, VEC> own = *reinterpret_cast<const Pk<ST, VEC>*>(slot(r, 4));
#pragma unroll
            for (int q = 0; q < VEC; ++q) o.a[q] = own.a[q] - o.a[q];
            stk<ST, VEC>(z + (size_t)i * K + c, o);
        }
        // further column chunks of those rows (more columns than lanes x VEC), colours with more rows per lane group
#pragma unroll 1
        for (int r = 0; r < NR; ++r) {
            const int i = rb + group + r * GPB;
            if (i < re)
                for (int cc = c + KC * VEC; cc < K; cc += KC * VEC) relax_slow(i, cc, 0, zero, first_sweep);
        }
#pragma unroll 1
        for (int i = rb + group + NR * GPB; i < re; i += GPB)
            for (int cc = c; cc < K; cc += KC * VEC) relax_slow(i, cc, 0, zero, first_sweep);
        if (last_step) break;
        publish(step);
#pragma unroll
        for (int r = 0; r < NR; ++r) pc[r] = pcn[r];
        issue_early(step + 1);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) M.ctl->sweeps_done += n_sweeps;
    __syncthreads();
    if (threadIdx.x == 0) {        // the last CTA to leave: arrivals every strip has counted, the grid barrier re-armed
        const unsigned t = atomicAdd(&M.ctl->gs_bar[1], 1u);
        if (t == (unsigned)nvb - 1) {
            M.ctl->gs_bar[0] = 0; M.ctl->gs_bar[1] = 0;
            M.ctl->strip_base = base + (unsigned long long)kWarps * (unsigned long long)(n_steps - 1);
            __threadfence();
        }
    }
}

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_add1(unsigned long long* p) {
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(p) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Strip sweep kernel with a TMA-fed operand ring (precond_sync = 4: fp32 sweeps, K = 16 -- 4 lanes x 16 bytes per row --,
// ELL width 4, one rank; same schedule, flags and arithmetic -- bitwise the same results).
// What the ncu counters of k_gs_strip and of a leaner cp.async form of it said (profiles/r02_notes.md): the pace is set by (a) two DRAM latencies in
// series per colour step -- the column indices of step k + 1 are loaded during step k, and only then can the copies
// of step k + 1 go out, one step ahead of their use -- and (b) L2 -> SM traffic: cp.async.cg (LDGSTS.BYPASS) moves
// whole 128-byte lines per quarter warp, so a 64-byte row gather, and above all the 16-byte-per-row value and index
// streams, fetch 1.5 - 4 x the sectors they use (127 M sectors per 6 sweeps against 66 M useful), where ld.global.cg
// is sector-exact.  Here:
//  * the three STREAMS of a step (column indices, matrix values, right-hand side u: contiguous per warp, 8 rows per
//    pass) arrive by cp.async.bulk -- one elected lane, three bulk copies per pass, completion on an mbarrier -- into
//    a per-warp ring kTmaStages steps deep: no registers, no per-lane address arithmetic, sector-exact, an L2
//    evict-first policy (they are read once per sweep; z, which every row gathers four times, keeps the L2), and
//    their DRAM latency is off the step's dependent chain;
//  * the GATHERS are predicated ld.global.cg into registers: the early ones (every neighbour but those of the
//    colour swept just before) go out after the step before, the late ones after the neighbour wait.
// ---------------------------------------------------------------------------------------------
constexpr int kTmaStages = 4;
constexpr int kTmaStageBytes = kGsRows * 8 * (16 + 16 + 64);              // per warp and stage: indices | values | u
constexpr int kTmaSmemBytes = (kGsThreads / 32) * kTmaStages * kTmaStageBytes;

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile("{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @!p bra WAIT_%=;\n}"
                 ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned sdst, const void* gsrc, unsigned bytes, unsigned bar, unsigned long long policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(sdst), "l"(gsrc), "r"(bytes), "r"(bar), "l"(policy) : "memory");
}

template <bool DBG>
__global__ void __launch_bounds__(kGsThreads, 2) k_gs_tma(DeviceModel M, float* __restrict__ z, int n_sweeps_arg) {
    constexpr int NR = kGsRows, GPB = kGsThreads / 4, ST = kTmaStages, kWarps = kGsThreads / 32;
    // DBG (development, CWR_GS_DEBUG = bits): timing experiments, some of which break the sweep's semantics -- 1: no neighbour
    // wait, 2: no publish (no release fence), 8: no __nanosleep between polls, 16: streams without the evict-first policy
    const int dbg = DBG ? n_sweeps_arg >> 16 : 0;
    n_sweeps_arg &= 0xffff;
    static_assert(NR == 2, "two rows per lane group");
    extern __shared__ int4 gs_land[];                    // [warp][stage][ idx[NR][8] | val[NR][8] | u[NR][8][4] ] (16-byte units)
    __shared__ int s_cp[kMaxColors + 1];
    __shared__ __align__(8) unsigned long long s_bar[kWarps * ST];
    if (M.ctl->all_done || M.ctl->finish_half) return;
    const int n_sweeps = n_sweeps_arg > 0 ? n_sweeps_arg : M.ctl->dc_sweeps;
    const int nc = M.n_colors, vb = blockIdx.x, nvb = gridDim.x;
    const int lane = threadIdx.x & 3, group = threadIdx.x >> 2, wl = threadIdx.x & 31, warp = threadIdx.x >> 5, gl = group & 7;
    const int32_t* __restrict__ cp_src = M.strip_cptr + (size_t)vb * (nc + 1);
    for (int q = threadIdx.x; q <= nc; q += kGsThreads) s_cp[q] = cp_src[q];
    const int nb0 = M.strip_nptr[vb], n_nbr = M.strip_nptr[vb + 1] - nb0;
    unsigned long long* const own_flag = M.strip_flag + (size_t)vb * kFlagStride;
    const unsigned long long* const my_flag = wl == 0 ? own_flag : (wl <= n_nbr ? M.strip_flag + (size_t)M.strip_nbr[nb0 + wl - 1] * kFlagStride : nullptr);
    unsigned long long target = M.ctl->strip_base;
    const unsigned long long base = target;
    const unsigned spin_limit = M.ctl->barrier_timeout ? 0u : (1u << 26);
    const unsigned bar0 = (unsigned)__cvta_generic_to_shared(s_bar + warp * ST);
    if (wl == 0) {
#pragma unroll
        for (int s = 0; s < ST; ++s) mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int n_steps = n_sweeps * nc;
    int4* const ring = gs_land + warp * (ST * kTmaStageBytes / 16);            // this warp's ring
    const unsigned ring_s = (unsigned)__cvta_generic_to_shared(ring);
    const int4* __restrict__ ecol4 = reinterpret_cast<const int4*>(M.ell_col);
    const int4* __restrict__ val4 = reinterpret_cast<const int4*>(M.valf);
    int4* const zq = reinterpret_cast<int4*>(z);                               // pack 4 * row + lane
    const int4* __restrict__ usq = reinterpret_cast<const int4*>(M.us);
    unsigned long long policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
    if (DBG && (dbg & 16)) asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(policy));
    auto nbr_ptr = [&](int cs) { return zq + (((unsigned)cs << 2) + (unsigned)lane); };
    auto row_pack = [&](int i) { return ((unsigned)i << 2) + (unsigned)lane; };
    // the streams of `step` into its stage (one elected lane): rows rb + 128 r + 8 warp + [0, 8) of the step's colour
    auto fill = [&](int step, int col) {
        const int stage = step % ST;
        const int b = s_cp[col], e = s_cp[col + 1];
        const unsigned sbase = ring_s + stage * kTmaStageBytes, bar = bar0 + 8 * stage;
        int cnt[NR];
#pragma unroll
        for (int r = 0; r < NR; ++r) cnt[r] = max(0, min(8, e - (b + r * GPB + 8 * warp)));
        mbar_expect_tx(bar, 96u * (unsigned)(cnt[0] + cnt[1]));
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            if (cnt[r] <= 0) continue;
            const int row0 = b + r * GPB + 8 * warp;
            bulk_g2s(sbase + r * 128, ecol4 + row0, 16u * cnt[r], bar, policy);
            bulk_g2s(sbase + NR * 128 + r * 128, val4 + row0, 16u * cnt[r], bar, policy);
            bulk_g2s(sbase + 2 * NR * 128 + r * 512, usq + (size_t)row0 * 4, 64u * cnt[r], bar, policy);
        }
    };
    float4 x[NR][4];
    int act[NR];
    // early gathers of `step` (its indices have landed): everything but the neighbours of the colour swept just before
    auto gather_early = [&](int step, int b, int e) {
        const int4* st = ring + (step % ST) * (kTmaStageBytes / 16);
        const int emask = step < nc ? (int)(kLaterBit | kPrevBit) : (int)kPrevBit;
        const int zmask = step < nc ? (int)kLaterBit : 0;
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            act[r] = b + group + r * GPB < e;
            const int4 c4 = st[r * 8 + gl];
            const int cs[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                x[r][u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (act[r] && (cs[u] & emask) != kPrevBit && !(cs[u] & zmask)) x[r][u] = __ldcg(reinterpret_cast<const float4*>(nbr_ptr(cs[u])));
            }
        }
    };
    auto gather_late = [&](int step) {
        const int4* st = ring + (step % ST) * (kTmaStageBytes / 16);
        const int emask = step < nc ? (int)(kLaterBit | kPrevBit) : (int)kPrevBit;
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int4 c4 = st[r * 8 + gl];
            const int cs[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (act[r] && (cs[u] & emask) == kPrevBit) x[r][u] = __ldcg(reinterpret_cast<const float4*>(nbr_ptr(cs[u])));
        }
    };

    // prologue: the streams of the first ST steps, the early gathers of step 0
    if (wl == 0)
        for (int s = 0, c = 0; s < ST && s < n_steps; ++s) { fill(s, c); c = c + 1 == nc ? 0 : c + 1; }
    int rb = s_cp[0], re = s_cp[1];
    int col = 0, col_fill = ST % nc;              // colour of the step the next refill is for (step + ST - 1 at the top of `step`)
    mbar_wait(bar0, 0);
    gather_early(0, rb, re);
    for (int step = 0; step < n_steps; ++step) {
        const bool last_step = step + 1 == n_steps;
        const int stage = step % ST;
        const int coln = col + 1 == nc ? 0 : col + 1;
        const int rbn = s_cp[coln], ren = s_cp[coln + 1];
        if (step > 0) {
            // the stage of step - 1 is free (every lane has used it): the streams of step - 1 + ST go there
            __syncwarp();
            if (wl == 0 && step - 1 + ST < n_steps) fill(step - 1 + ST, col_fill);
            col_fill = col_fill + 1 == nc ? 0 : col_fill + 1;
            // every warp of this strip and of the neighbouring strips has finished step - 1
            if (my_flag && !(dbg & 1)) {
                unsigned spins = 0;
                while (ld_relaxed_u64(my_flag) < target) {
                    if (++spins > spin_limit) { M.ctl->barrier_timeout = 1; break; }      // never hang the device
                    if (!(dbg & 8)) __nanosleep(DBG && (dbg & 32) ? 20 : 64);
                }
            }
            __syncwarp();
        }
        gather_late(step);
        const int4* st = ring + stage * (kTmaStageBytes / 16);
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const float4 v = *reinterpret_cast<const float4*>(st + NR * 8 + r * 8 + gl);
            const float4 own = *reinterpret_cast<const float4*>(st + 2 * NR * 8 + r * 32 + gl * 4 + lane);
            const float4 x0 = x[r][0], x1 = x[r][1], x2 = x[r][2], x3 = x[r][3];
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
            o.x += v.x * x0.x; o.y += v.x * x0.y; o.z += v.x * x0.z; o.w += v.x * x0.w;
            o.x += v.y * x1.x; o.y += v.y * x1.y; o.z += v.y * x1.z; o.w += v.y * x1.w;
            o.x += v.z * x2.x; o.y += v.z * x2.y; o.z += v.z * x2.z; o.w += v.z * x2.w;
            o.x += v.w * x3.x; o.y += v.w * x3.y; o.z += v.w * x3.z; o.w += v.w * x3.w;
            o.x = own.x - o.x; o.y = own.y - o.y; o.z = own.z - o.z; o.w = own.w - o.w;
            const int i = rb + group + r * GPB;
            if (act[r]) *reinterpret_cast<float4*>(zq + row_pack(i)) = o;
        }
        // rows beyond one pass of the CTA (rare: strip_cap): through registers, all gathers after the wait
#pragma unroll 1
        for (int i = rb + group + NR * GPB; i < re; i += GPB) {
            const int4 d4 = __ldg(ecol4 + i);
            const float4 wv = __ldg(reinterpret_cast<const float4*>(val4) + i);
            const int ds[4] = {d4.x, d4.y, d4.z, d4.w};
            const float ws[4] = {wv.x, wv.y, wv.z, wv.w};
            float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (step < nc && ds[u] < 0) continue;
                const float4 y = __ldcg(reinterpret_cast<const float4*>(nbr_ptr(ds[u])));
                o.x += ws[u] * y.x; o.y += ws[u] * y.y; o.z += ws[u] * y.z; o.w += ws[u] * y.w;
            }
            const float4 own = __ldcg(reinterpret_cast<const float4*>(usq + row_pack(i)));
            o.x = own.x - o.x; o.y = own.y - o.y; o.z = own.z - o.z; o.w = own.w - o.w;
            *reinterpret_cast<float4*>(zq + row_pack(i)) = o;
        }
        if (last_step) break;
        // The early gathers of the next step go out BEFORE this step is published: the release fence waits for the
        // warp's outstanding stores (~1 us: ncu, 90 of 373 us per 6 sweeps), and gathers issued behind it would
        // start a store latency late in every step.  They are safe here: the neighbouring strips have finished
        // step - 1 and cannot start step + 1 before this strip publishes, so all they may be writing is this
        // step's colour -- which is exactly what a step's early gathers leave out.
        rb = rbn; re = ren; col = coln;
        mbar_wait(bar0 + 8 * ((step + 1) % ST), ((step + 1) / ST) & 1);
        gather_early(step + 1, rb, re);
        // publish this warp's step: its lanes' stores, then one release per warp
        __syncwarp();
        if (wl == 0 && !(dbg & 2)) red_release_add1(own_flag);
        target += kWarps;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) M.ctl->sweeps_done += n_sweeps;
    __syncthreads();
    if (threadIdx.x == 0) {        // the last CTA to leave: arrivals every strip has counted
        const unsigned t = atomicAdd(&M.ctl->gs_bar[1], 1u);
        if (t == (unsigned)nvb - 1) {
            M.ctl->gs_bar[0] = 0; M.ctl->gs_bar[1] = 0;
            M.ctl->strip_base = DBG && (dbg & 2) ? base : base + (unsigned long long)kWarps * (unsigned long long)(n_steps - 1);
            __threadfence();
        }
    }
}

// u (fp64) -> the sweep type, own rows (the BiCGSTAB path in front of k_gs_strip: its vectors are fp64)
template <typename ST>
__global__ void __launch_bounds__(kThreads) k_to_sweep_type(DeviceModel M, const double* __restrict__ u, ST* __restrict__ out) {
    const size_t lo = (size_t)M.row_lo * M.K, hi = (size_t)M.row_hi * M.K;
    if (M.ctl->all_done || M.ctl->finish_half) return;
    for (size_t q = lo + blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < hi; q += (size_t)gridDim.x * blockDim.x) out[q] = (ST)u[q];
}

// ---------------------------------------------------------------------------------------------
// SpMM over the row-scaled matrix, fused with the BiCGSTAB step that consumes it.  z (type ZT: the
// solver's own fp64 vector, or a preconditioned vector in the sweep precision) is gathered and widened.
//   INIT : r = b - (x + L x)          ; rhat = p = r ; dots (r,r), (b,b)
//   AV   : v = z + L z                ; dot (rhat, v)                      -> alpha
//   AT   : t = z + L z                ; dots (t,s),(t,t),(rhat,t),(rhat,s) -> omega, rho', beta
//   PLAIN: y = z + L z                (timing / tests)
// Defect-correction solver (solver = 2; no Krylov vectors at all):
//   INIT_DC: r = b - (x + L x)        ; dots (r,r), (b,b); plans the first cycle's sweeps
//   DC     : r -= z + L z ; x += z    ; dot (r,r); convergence, stagnation test, plan of the next cycle
// ---------------------------------------------------------------------------------------------
enum SpmmMode { MODE_INIT = 0, MODE_AV = 1, MODE_AT = 2, MODE_PLAIN = 4, MODE_INIT_DC = 5, MODE_DC = 6 };

// Sweeps of the next defect-correction cycle: `worst` = how far the worst column is from the tolerance
// ((||r||/||b||)/rtol > 1), `rate` = measured error factor per sweep.  A cycle in the sweep precision cannot
// reduce the residual by more than ~1/floor_gain (fp32: ~1e-7), so longer cycles would be wasted; the last
// cycle gets one sweep of margin (another cycle costs about four sweeps of memory traffic).
__device__ __forceinline__ int dc_plan(double worst, double rate, int smin, int smax, double floor_gain) {
    rate = fmin(fmax(rate, 0.02), 0.97);
    const double l = -log(rate);
    int cap = (int)floor(log(floor_gain) / l);
    cap = max(smin, min(cap, smax));
    int s = (int)ceil(log(fmax(worst, 1.0)) / l + 1.0);
    if (s > cap) {
        const int cycles = (s + cap - 1) / cap;
        s = (s + cycles - 1) / cycles;
    }
    return max(smin, min(s, cap));
}

template <int KC, int VEC, int MODE, typename ZT>
__global__ void __launch_bounds__(kThreads, MODE == 2 ? CWR_AT_MIN_BLOCKS : CWR_SPMM_MIN_BLOCKS) k_spmm(DeviceModel M, const ZT* __restrict__ zin,
                                                                        double* __restrict__ out) {
    constexpr bool IS_INIT = MODE == MODE_INIT || MODE == MODE_INIT_DC;
    constexpr int ND = IS_INIT ? 2 : MODE == MODE_AV ? 1 : MODE == MODE_AT ? 4 : 1;
    constexpr bool HAS_DOTS = IS_INIT || MODE == MODE_AV || MODE == MODE_AT || MODE == MODE_DC;
    __shared__ double smem[HAS_DOTS ? (kThreads / 32) * kMaxDots * 2 * 32 : 1];
    __shared__ double tot[HAS_DOTS ? kMaxDots * kMaxK : 1];
    if (MODE == MODE_AV || MODE == MODE_AT || MODE == MODE_DC) { if (M.ctl->all_done) return; }
    if (MODE == MODE_AT) { if (M.ctl->finish_half) return; }
    const int K = M.K, n = M.row_hi, W = M.W;
    const int lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kThreads / KC;
    const int32_t* __restrict__ ecol = M.ell_col;
    const double* __restrict__ eval = M.val;
    if (IS_INIT) zin = reinterpret_cast<const ZT*>(M.sp->state_t1);     // ZT = double
    double* __restrict__ xs = M.sp->state_t1;
    const int nchunk = (K + KC * VEC - 1) / (KC * VEC);
    for (int chunk = 0; chunk < nchunk; ++chunk) {
        const int c = (chunk * KC + lane) * VEC;
        const bool active = c < K;
        double acc[ND * VEC];
#pragma unroll
        for (int d = 0; d < ND * VEC; ++d) acc[d] = 0.0;
        if (active) {
            // Software pipeline: the next row's column indices and values (the loads the gathers depend
            // on) are fetched while this row's gathers are in flight, so a row costs one memory latency,
            // not two.
            const int stride = gridDim.x * GPB;
            int i = M.row_lo + blockIdx.x * GPB + group;
            int4 c4n = make_int4(0, 0, 0, 0);
            double2 v01n = make_double2(0.0, 0.0), v23n = v01n;
            if (i < n) {
                c4n = *reinterpret_cast<const int4*>(ecol + (size_t)i * W);
                v01n = *reinterpret_cast<const double2*>(eval + (size_t)i * W);
                v23n = *reinterpret_cast<const double2*>(eval + (size_t)i * W + 2);
            }
            for (; i < n; i += stride) {
                const size_t idx = (size_t)i * K + c;
                const int4 c4 = make_int4(c4n.x & kColMask, c4n.y & kColMask, c4n.z & kColMask, c4n.w & kColMask);
                const double2 v01 = v01n, v23 = v23n;
                const Vd<VEC> x0 = ldz<ZT, VEC>(zin + (size_t)c4.x * K + c);
                const Vd<VEC> x1 = ldz<ZT, VEC>(zin + (size_t)c4.y * K + c);
                const Vd<VEC> x2 = ldz<ZT, VEC>(zin + (size_t)c4.z * K + c);
                const Vd<VEC> x3 = ldz<ZT, VEC>(zin + (size_t)c4.w * K + c);
                // the row's own operands are issued now as well, so nothing waits behind the gathers
                const Vd<VEC> own = ldz<ZT, VEC>(zin + idx);
                Vd<VEC> aux1 = own, aux2 = own;
                if (IS_INIT) aux1 = ldv<VEC>(M.b + idx);
                if (MODE == MODE_AV || MODE == MODE_AT) aux1 = ldv<VEC>(M.rhat + idx);
                if (MODE == MODE_DC) { aux1 = ldv<VEC>(M.r + idx); aux2 = ldv<VEC>(xs + idx); }
                if (MODE == MODE_AT) aux2 = ldv<VEC>(M.r + idx);          // s lives in the r buffer
                const int inext = i + stride;
                if (inext < n) {
                    c4n = *reinterpret_cast<const int4*>(ecol + (size_t)inext * W);
                    v01n = *reinterpret_cast<const double2*>(eval + (size_t)inext * W);
                    v23n = *reinterpret_cast<const double2*>(eval + (size_t)inext * W + 2);
                }
                Vd<VEC> s;
#pragma unroll
                for (int q = 0; q < VEC; ++q)
                    s.a[q] = fma(v23.y, x3.a[q], fma(v23.x, x2.a[q], fma(v01.y, x1.a[q], v01.x * x0.a[q])));
                for (int w = 4; w < W; w += 4) {      // rows wider than 4 (not pipelined)
                    int4 d4 = *reinterpret_cast<const int4*>(ecol + (size_t)i * W + w);
                    d4.x &= kColMask; d4.y &= kColMask; d4.z &= kColMask; d4.w &= kColMask;
                    const double2 w01 = *reinterpret_cast<const double2*>(eval + (size_t)i * W + w);
                    const double2 w23 = *reinterpret_cast<const double2*>(eval + (size_t)i * W + w + 2);
                    const Vd<VEC> y0 = ldz<ZT, VEC>(zin + (size_t)d4.x * K + c);
                    const Vd<VEC> y1 = ldz<ZT, VEC>(zin + (size_t)d4.y * K + c);
                    const Vd<VEC> y2 = ldz<ZT, VEC>(zin + (size_t)d4.z * K + c);
                    const Vd<VEC> y3 = ldz<ZT, VEC>(zin + (size_t)d4.w * K + c);
#pragma unroll
                    for (int q = 0; q < VEC; ++q)
                        s.a[q] = fma(w23.y, y3.a[q], fma(w23.x, y2.a[q], fma(w01.y, y1.a[q], fma(w01.x, y0.a[q], s.a[q]))));
                }
                Vd<VEC> y;
#pragma unroll
                for (int q = 0; q < VEC; ++q) y.a[q] = own.a[q] + s.a[q];
                if (IS_INIT) {
                    const Vd<VEC> bi = aux1;
                    Vd<VEC> r;
#pragma unroll
                    for (int q = 0; q < VEC; ++q) {
                        r.a[q] = bi.a[q] - y.a[q];
                        acc[0 * VEC + q] = fma(r.a[q], r.a[q], acc[0 * VEC + q]);
                        acc[1 * VEC + q] = fma(bi.a[q], bi.a[q], acc[1 * VEC + q]);
                    }
                    stv<VEC>(M.r + idx, r);
                    if (MODE == MODE_INIT) { stv<VEC>(M.rhat + idx, r); stv<VEC>(M.p + idx, r); }
                    if (MODE == MODE_INIT_DC && M.us_from_producer) {
                        if (M.sweep_f32) {
                            Pk<float, VEC> rs;
#pragma unroll
                            for (int q = 0; q < VEC; ++q) rs.a[q] = (float)r.a[q];
                            stk<float, VEC>(reinterpret_cast<float*>(M.us) + idx, rs);
                        } else stv<VEC>(reinterpret_cast<double*>(M.us) + idx, r);
                    }
                } else if (MODE == MODE_DC) {
                    Vd<VEC> r = aux1, xv = aux2;
#pragma unroll
                    for (int q = 0; q < VEC; ++q) {
                        r.a[q] -= y.a[q];
                        xv.a[q] += own.a[q];
                        acc[q] = fma(r.a[q], r.a[q], acc[q]);
                    }
                    stv<VEC>(M.r + idx, r); stv<VEC>(xs + idx, xv);
                    if (M.us_from_producer) {
                        Pk<ZT, VEC> rs;
#pragma unroll
                        for (int q = 0; q < VEC; ++q) rs.a[q] = (ZT)r.a[q];
                        stk<ZT, VEC>(reinterpret_cast<ZT*>(M.us) + idx, rs);
                    }
                } else if (MODE == MODE_AV) {
                    const Vd<VEC> rh = aux1;
                    stv<VEC>(M.v + idx, y);
#pragma unroll
                    for (int q = 0; q < VEC; ++q) acc[q] = fma(rh.a[q], y.a[q], acc[q]);
                } else if (MODE == MODE_AT) {
                    const Vd<VEC> rh = aux1, sv = aux2;
                    stv<VEC>(M.tt + idx, y);
#pragma unroll
                    for (int q = 0; q < VEC; ++q) {
                        acc[0 * VEC + q] = fma(y.a[q], sv.a[q], acc[0 * VEC + q]);
                        acc[1 * VEC + q] = fma(y.a[q], y.a[q], acc[1 * VEC + q]);
                        acc[2 * VEC + q] = fma(rh.a[q], y.a[q], acc[2 * VEC + q]);
                        acc[3 * VEC + q] = fma(rh.a[q], sv.a[q], acc[3 * VEC + q]);
                    }
                } else {
                    stv<VEC>(out + idx, y);
                }
            }
        }
        if (HAS_DOTS) block_dots<ND, KC, VEC>(acc, smem, M.partials, K, chunk);
    }
    if (!HAS_DOTS) return;
    if (!last_block_arrives(&M.ctl->ticket[MODE == MODE_INIT_DC ? 0 : MODE == MODE_DC ? 1 : MODE])) return;
    grid_totals<ND>(M.partials, tot, K);
    dd_allreduce(M, tot, ND * K);
    double* sc = M.sc;
    if constexpr (MODE == MODE_INIT_DC || MODE == MODE_DC) {
        // defect correction: convergence per column, the worst distance from the tolerance, the plan of the next cycle
        __shared__ unsigned long long worst_bits;
        __shared__ int not_done, failed, any_flags;
        if (threadIdx.x == 0) { worst_bits = 0ull; not_done = 0; failed = 0; any_flags = 0; }
        __syncthreads();
        const int iter_now = M.ctl->iter + (MODE == MODE_DC ? 1 : 0);
        for (int k = threadIdx.x; k < K; k += blockDim.x) {
            int f = M.colflags[k];
            if (MODE == MODE_INIT_DC) {
                const double rr = tot[0 * K + k], bb = tot[1 * K + k];
                sc[SC_BNORM2 * K + k] = bb; sc[SC_RNORM2 * K + k] = rr;
                f &= ~(FL_CONVERGED | FL_BREAKDOWN | FL_PENDING | FL_ZERO_RHS | FL_NAN | FL_HALF);
                if (!(rr == rr) || !(bb == bb) || isinf(rr) || isinf(bb)) f |= FL_NAN | FL_PENDING;
                else if (bb == 0.0 && rr != 0.0) f |= FL_ZERO_RHS | FL_PENDING;     // b == 0  =>  x = 0
            }
            if (!(f & FL_PENDING)) {
                const double rr = tot[k], bb = sc[SC_BNORM2 * K + k];
                if (MODE == MODE_DC) sc[SC_RNORM2 * K + k] = rr;
                if (!(rr == rr) || isinf(rr)) atomicOr(&failed, 1);                 // finite at the start, not any more
                else if (rr <= M.tol2 * bb) { if (!(f & FL_CONVERGED)) { f |= FL_CONVERGED; M.coliters[k] = iter_now; } }
                else {
                    f &= ~FL_CONVERGED;
                    atomicOr(&not_done, 1);
                    atomicMax(&worst_bits, (unsigned long long)__double_as_longlong(rr / (M.tol2 * bb)));
                }
            }
            atomicOr(&any_flags, f);
            M.colflags[k] = f;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            SolverCtl* ctl = M.ctl;
            ctl->iter = iter_now;
            ctl->flags_or = any_flags;
            int done = !not_done, fail = failed;
            if (!done && !fail) {
                const double worst = sqrt(__longlong_as_double((long long)worst_bits));
                double rate = ctl->dc_rate;
                if (!(rate > 0.0)) rate = 0.3;
                if (MODE == MODE_DC) {
                    const double prev = ctl->dc_worst;
                    const int S = max(1, ctl->dc_sweeps);
                    if (prev > 0.0 && worst < prev) rate = pow(worst / prev, 1.0 / S); else rate = 0.97;
                    if (worst > 0.7 * prev) ctl->dc_slow += 1; else ctl->dc_slow = 0;
                    if (ctl->dc_slow >= 2) fail = 1;
                } else ctl->dc_slow = 0;
                ctl->dc_rate = rate;
                ctl->dc_worst = worst;
                ctl->dc_sweeps = dc_plan(worst, rate, M.dc_smin, M.dc_smax, M.dc_floor);
            }
            if (!done && !fail && iter_now >= M.max_iter) { ctl->hit_max_iter = 1; done = 1; }
            if (fail) { ctl->dc_fail = 1; done = 1; }
            ctl->all_done = done;
        }
    } else {
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        int f = M.colflags[k];
        if (MODE == MODE_INIT) {
            const double rr = tot[0 * K + k], bb = tot[1 * K + k];
            sc[SC_RHO * K + k] = rr; sc[SC_BNORM2 * K + k] = bb; sc[SC_RNORM2 * K + k] = rr;
            sc[SC_ALPHA * K + k] = 0.0; sc[SC_OMEGA * K + k] = 0.0; sc[SC_BETA * K + k] = 0.0;
            f &= ~(FL_CONVERGED | FL_BREAKDOWN | FL_PENDING | FL_ZERO_RHS | FL_NAN | FL_HALF);
            if (!(rr == rr) || !(bb == bb) || isinf(rr) || isinf(bb)) f |= FL_NAN | FL_PENDING;
            else if (bb == 0.0 && rr != 0.0) f |= FL_ZERO_RHS | FL_PENDING;     // b == 0  =>  x = 0
            else if (rr <= M.tol2 * bb) { f |= FL_CONVERGED; M.coliters[k] = M.ctl->iter; }
        } else if (MODE == MODE_AV) {
            const double rv = tot[k];
            sc[SC_RHATV * K + k] = rv;
            double alpha = 0.0;
            if (!(f & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN | FL_PENDING))) {
                if (rv == 0.0 || !(rv == rv)) f |= FL_BREAKDOWN;
                else alpha = sc[SC_RHO * K + k] / rv;
            }
            sc[SC_ALPHA * K + k] = alpha;
        } else {
            const double ts = tot[0 * K + k], t2 = tot[1 * K + k], rt = tot[2 * K + k], rs = tot[3 * K + k];
            double omega = 0.0, beta = 0.0;
            if (!(f & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN | FL_PENDING | FL_HALF))) {
                const double rho = sc[SC_RHO * K + k], alpha = sc[SC_ALPHA * K + k];
                omega = t2 > 0.0 ? ts / t2 : 0.0;
                const double rho_new = rs - omega * rt;          // (rhat, s - omega t)
                if (omega != 0.0 && rho != 0.0) beta = (rho_new / rho) * (alpha / omega);
                else if (t2 > 0.0) f |= FL_BREAKDOWN;            // omega == 0 with s != 0: stagnation
                if (!(beta == beta) || isinf(beta)) { beta = 0.0; f |= FL_BREAKDOWN; }
                sc[SC_RHO * K + k] = rho_new;
            }
            sc[SC_OMEGA * K + k] = omega; sc[SC_BETA * K + k] = beta;
        }
        M.colflags[k] = f;
    }
    __syncthreads();
    if (MODE == MODE_INIT && threadIdx.x == 0) publish_done(M, K);
    }
}

// Defect-correction solver, after the last cycle: columns that cannot be iterated -- a non-finite right-hand side
// fills the column with NaN as spsolve does, b == 0 gives x = 0 (the BiCGSTAB path does this in k_update_xrp).
__global__ void __launch_bounds__(kThreads) k_fix_columns(DeviceModel M) {
    const int K = M.K;
    double* __restrict__ x = M.sp->state_t1;
    const size_t total = (size_t)(M.row_hi - M.row_lo) * K;
    for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int k = (int)(q % K);
        const int f = M.colflags[k];
        if (f & FL_PENDING) x[(size_t)M.row_lo * K + q] = (f & FL_NAN) ? qnan() : 0.0;
    }
}
__global__ void k_fix_flags(DeviceModel M) {
    for (int k = threadIdx.x; k < M.K; k += blockDim.x) {
        int f = M.colflags[k];
        if (f & FL_PENDING) {
            f &= ~FL_PENDING;
            if (f & FL_ZERO_RHS) { f |= FL_CONVERGED; M.sc[SC_RNORM2 * M.K + k] = 0.0; M.coliters[k] = M.ctl->iter; }
            M.colflags[k] = f;
        }
    }
}

// s = r - alpha v  (in place on r), fused with (s,s): a column whose ||s|| already meets the tolerance stops at
// the half step (FL_HALF: omega = 0, so k_update_xrp reduces to x += alpha p^ and finds it converged); when every
// column has, the second half of the iteration (the sweeps on s and t = A s^) is skipped (ctl->finish_half).
template <int KC, int VEC>
__global__ void __launch_bounds__(kThreads) k_update_s(DeviceModel M) {
    __shared__ double smem[(kThreads / 32) * kMaxDots * 2 * 32];
    __shared__ double tot[kMaxDots * kMaxK];
    if (M.ctl->all_done) return;
    const int K = M.K, lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kThreads / KC;
    const int nchunk = (K + KC * VEC - 1) / (KC * VEC);
    for (int chunk = 0; chunk < nchunk; ++chunk) {
        const int c = (chunk * KC + lane) * VEC;
        double acc[VEC];
#pragma unroll
        for (int q = 0; q < VEC; ++q) acc[q] = 0.0;
        if (c < K) {
            double alpha[VEC];
            bool any = false;
#pragma unroll
            for (int q = 0; q < VEC; ++q) { alpha[q] = M.sc[SC_ALPHA * K + c + q]; any |= alpha[q] != 0.0; }
            if (any)       // frozen columns (alpha = 0): s = r, nothing to do
                for (int i = M.row_lo + blockIdx.x * GPB + group; i < M.row_hi; i += gridDim.x * GPB) {
                    const size_t idx = (size_t)i * K + c;
                    Vd<VEC> r = ldv<VEC>(M.r + idx);
                    const Vd<VEC> v = ldv<VEC>(M.v + idx);
#pragma unroll
                    for (int q = 0; q < VEC; ++q) { r.a[q] = fma(-alpha[q], v.a[q], r.a[q]); acc[q] = fma(r.a[q], r.a[q], acc[q]); }
                    stv<VEC>(M.r + idx, r);
                }
        }
        block_dots<1, KC, VEC>(acc, smem, M.partials, K, chunk);
    }
    if (!last_block_arrives(&M.ctl->ticket_s)) return;
    grid_totals<1>(M.partials, tot, K);
    dd_allreduce(M, tot, K);
    __shared__ int not_half;
    if (threadIdx.x == 0) not_half = 0;
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        int f = M.colflags[k];
        if (!(f & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN | FL_PENDING))) {
            const double ss = tot[k];
            if (M.sc[SC_ALPHA * K + k] != 0.0 && ss == ss && ss <= M.tol2 * M.sc[SC_BNORM2 * K + k]) {
                f |= FL_HALF;
                M.sc[SC_OMEGA * K + k] = 0.0; M.sc[SC_BETA * K + k] = 0.0;
                M.colflags[k] = f;
            } else atomicOr(&not_half, 1);
        } else if (f & FL_PENDING) atomicOr(&not_half, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) M.ctl->finish_half = not_half ? 0 : 1;
}

// x += alpha ph + omega sh ; r = s - omega t ; p = r + beta (p - omega v) ; dot (r,r); convergence
// (ph, sh: preconditioned p and s in the sweep precision PT; p and s themselves when m = 1)
template <int KC, int VEC, typename PT>
__global__ void __launch_bounds__(kThreads) k_update_xrp(DeviceModel M, const PT* ph, const PT* sh) {
    __shared__ double smem[(kThreads / 32) * kMaxDots * 2 * 32];
    __shared__ double tot[kMaxDots * kMaxK];
    if (M.ctl->all_done) return;
    const int K = M.K, lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kThreads / KC;
    double* __restrict__ x = M.sp->state_t1;
    const int nchunk = (K + KC * VEC - 1) / (KC * VEC);
    for (int chunk = 0; chunk < nchunk; ++chunk) {
        const int c = (chunk * KC + lane) * VEC;
        double acc[VEC];
#pragma unroll
        for (int q = 0; q < VEC; ++q) acc[q] = 0.0;
        if (c < K) {
            int f[VEC]; double alpha[VEC], omega[VEC], beta[VEC];
            bool any_pending = false, any_active = false;
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                f[q] = M.colflags[c + q];
                alpha[q] = M.sc[SC_ALPHA * K + c + q]; omega[q] = M.sc[SC_OMEGA * K + c + q]; beta[q] = M.sc[SC_BETA * K + c + q];
                any_pending |= (f[q] & FL_PENDING) != 0;
                any_active |= !(f[q] & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN | FL_PENDING));
            }
            if (any_pending || any_active)
                for (int i = M.row_lo + blockIdx.x * GPB + group; i < M.row_hi; i += gridDim.x * GPB) {
                    const size_t idx = (size_t)i * K + c;
                    Vd<VEC> xv = ldv<VEC>(x + idx), rv = ldv<VEC>(M.r + idx), pv = ldv<VEC>(M.p + idx);
                    const Vd<VEC> tv = ldv<VEC>(M.tt + idx), vv = ldv<VEC>(M.v + idx);
                    const Vd<VEC> phv = ldz<PT, VEC>(ph + idx), shv = ldz<PT, VEC>(sh + idx);
#pragma unroll
                    for (int q = 0; q < VEC; ++q) {
                        if (f[q] & FL_PENDING) {
                            xv.a[q] = (f[q] & FL_NAN) ? qnan() : 0.0; rv.a[q] = 0.0; pv.a[q] = 0.0;
                        } else if (!(f[q] & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN))) {
                            xv.a[q] = fma(omega[q], shv.a[q], fma(alpha[q], phv.a[q], xv.a[q]));
                            const double rn = fma(-omega[q], tv.a[q], rv.a[q]);
                            rv.a[q] = rn;
                            pv.a[q] = fma(beta[q], fma(-omega[q], vv.a[q], pv.a[q]), rn);
                            acc[q] = fma(rn, rn, acc[q]);
                        }
                    }
                    stv<VEC>(x + idx, xv); stv<VEC>(M.r + idx, rv); stv<VEC>(M.p + idx, pv);
                }
        }
        block_dots<1, KC, VEC>(acc, smem, M.partials, K, chunk);
    }
    if (!last_block_arrives(&M.ctl->ticket[3])) return;
    grid_totals<1>(M.partials, tot, K);
    dd_allreduce(M, tot, K);
    if (threadIdx.x == 0) M.ctl->iter += 1;
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        int f = M.colflags[k];
        if (f & FL_PENDING) {
            f &= ~FL_PENDING;
            if (f & FL_ZERO_RHS) { f |= FL_CONVERGED; M.sc[SC_RNORM2 * K + k] = 0.0; M.coliters[k] = M.ctl->iter; }
        } else if (!(f & (FL_CONVERGED | FL_BREAKDOWN | FL_NAN))) {
            f &= ~FL_HALF;
            const double rr = tot[k];
            M.sc[SC_RNORM2 * K + k] = rr;
            if (!(rr == rr) || isinf(rr)) f |= FL_NAN;
            else if (rr <= M.tol2 * M.sc[SC_BNORM2 * K + k]) { f |= FL_CONVERGED; M.coliters[k] = M.ctl->iter; }
        }
        M.colflags[k] = f;
    }
    __syncthreads();
    if (threadIdx.x == 0) { M.ctl->finish_half = 0; publish_done(M, K); }
}

// ---------------------------------------------------------------------------------------------
// mass flux across every edge  (reference transport.py:406-429) + running boundary sums
// (postproc_util.py:100-143).  c[t+1] of a ghost cell = its BC value, NaN when unset.
// ---------------------------------------------------------------------------------------------
template <int KC, int VEC>
__global__ void __launch_bounds__(kThreads) k_mass_flux(DeviceModel M) {
    pdl_enter();
    const StepParams& sp = *M.sp;
    const int K = M.K, lane = threadIdx.x % KC, group = threadIdx.x / KC, GPB = kThreads / KC;
    const double dt = sp.dt;
    const double* __restrict__ x = sp.state_t1;
    const size_t EK = (size_t)M.E * K, GK = (size_t)M.E_g * K;
    const int n_ie = M.ie_hi - M.ie_lo, n_own = n_ie + (M.ge_hi - M.ge_lo);     // owned internal + ghost edges
    for (int c = lane * VEC; c < K; c += KC * VEC)
        for (int j = blockIdx.x * GPB + group; j < n_own; j += gridDim.x * GPB) {
            const int e = j < n_ie ? M.ie_lo + j : M.E_int + M.ge_lo + (j - n_ie);
            const int P = M.f1p[e], N = M.f2p[e];
            const double a = (double)sp.adv_t[e], d = sp.cdiff_t[e];
            const Vd<VEC> cP = ldv<VEC>(x + (size_t)P * K + c);
            Vd<VEC> cN;
            if (N < M.n) cN = ldv<VEC>(x + (size_t)N * K + c);
            else {
                cN = ldv<VEC>(sp.bc_t1 + (size_t)(N - M.n) * K + c);
#pragma unroll
                for (int q = 0; q < VEC; ++q) if (cN.a[q] == 0.0) cN.a[q] = qnan();
            }
            Vd<VEC> fa, fd, ft;
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                fa.a[q] = __dmul_rn((a < 0.0 ? __dmul_rn(a, cN.a[q]) : __dmul_rn(a, cP.a[q])), dt);
                fd.a[q] = __dmul_rn(__dmul_rn(d, cN.a[q] - cP.a[q]), dt);
                ft.a[q] = fa.a[q] + fd.a[q];
            }
            const size_t o = (size_t)e * K + c;
            stv<VEC>(M.flux + o, fa); stv<VEC>(M.flux + EK + o, fd); stv<VEC>(M.flux + 2 * EK + o, ft);
            if (e >= M.E_int) {
                if (c == 0) {       // boundary volumes (postproc_util.py:93-95, 112-134): face_flow * dt, NaN skipped
                    const double fv = (double)sp.flowg_t[e - M.E_int] * dt;
                    if (fv == fv) {
                        const size_t gv = (size_t)(e - M.E_int), Eg = (size_t)M.E_g;
                        M.vsum[gv] += fv;
                        M.vsum[Eg + gv] += (fv <= 0.0) ? fv : 0.0;
                        M.vsum[2 * Eg + gv] += (fv >= 0.0) ? fv : 0.0;
                    }
                }
                const size_t g = (size_t)(e - M.E_int) * K + c;
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    const double f = ft.a[q];
                    M.bsum[g + q] += f;
                    M.bsum[GK + g + q] += (f <= 0.0) ? f : f * 0.0;
                    M.bsum[2 * GK + g + q] += (f >= 0.0) ? f : f * 0.0;
                }
            }
        }
}

// sum_i vol[i], sum_i vol[i] * c[i,k]   (postproc_util.py:36-59).  Deterministic two-stage reduction:
// kMassBlocks CTAs each reduce a grid-stride slice in a fixed order into partial[b][2]; the last CTA to
// arrive adds the partials in block order.
constexpr int kMassBlocks = 256;
__global__ void __launch_bounds__(kThreads) k_mass_total(const float* __restrict__ vol, const double* __restrict__ state, int lo, int n, int K, int k,
                                                         double* __restrict__ partial /* [kMassBlocks][2] */, unsigned* ticket,
                                                         double* __restrict__ out /* [2]: volume, mass */) {
    __shared__ double sv[kThreads], sm[kThreads];
    double v = 0.0, m = 0.0;
    for (int i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double vi = (double)vol[i];
        v += vi; m = fma(vi, state[(size_t)i * K + k], m);
    }
    sv[threadIdx.x] = v; sm[threadIdx.x] = m;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) { sv[threadIdx.x] += sv[threadIdx.x + s]; sm[threadIdx.x] += sm[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { partial[2 * blockIdx.x] = sv[0]; partial[2 * blockIdx.x + 1] = sm[0]; }
    if (!last_block_arrives(ticket)) return;
    if (threadIdx.x == 0) {
        double tv = 0.0, tm = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) { tv += __ldcg(partial + 2 * b); tm += __ldcg(partial + 2 * b + 1); }
        out[0] = tv; out[1] = tm;
    }
}

}  // namespace cwr
